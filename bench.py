#!/usr/bin/env python
"""bench.py -- ADMM iterations/s of the B200 hot path on BASELINE.json's metric configs.

Default workload (config.workload) = BASELINE configs[2], the configuration the north-star target is quoted on:
8 partitions x 1M rows x 10k features, 1 % nnz (100 stored values per row), lambda in {0.1, 1, 10} in ONE run,
synthetic (SURVEY.md 8d: uniform distinct columns per row, N(0,1) values, seed 1000+p per partition).  The 8
partitions are sharded over the N ranks (p % N): per-GPU work shrinks as N grows, scaling = "strong".
One "step" = one ADMM iteration = the x-update of every (partition, lambda) reducer + the consensus all-reduce +
the z/u update (jobs/RegressionAdmmTrain.java:281-497; reducers = nblocks x #lambda, :355).  The timed region is
a complete job of K iterations FROM THE COLD STATE z = u = 0 (Gram + Cholesky of every partition included), after
W warm-up iterations of a throw-away job; inputs (0.8 GB CSR + 0.6 GB block-major list per partition, 400 MB per
inverse Hessian) are far larger than the 126 MB L2, so nothing is flushed between iterations.

    python bench.py --gpus N --steps K --warmup W            (N > 1: launched by torch.distributed.run)
    python bench.py --impl reference ...                      (CPU arm: the oracle port, rank 0 only)
    python bench.py --workload cfg2|cfg3|cfg4|cfg5            (cfg2 = 8 x 1M x 1k dense; cfg4 = 8 sparse partitions
                                                               PER GPU, weak scaling; cfg5 = NaiveTrain per-key fits)
    python bench.py --dump-outputs DIR ...                    (also write what the timed path returned in its last step)

Prints ONE JSON line (rank 0).  `value` = iterations/s with inputs resident in HBM; `e2e` = the same job through
the public API from pinned HOST buffers (upload + K iterations + model read-back in the timed region);
`also.cfg2` = the same measurements for configs[1] (round 1's headline line), `parity` = the same kernels on a
row-reduced copy of the workload against the CPU oracle in exact mode.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "ml-ease_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402

WORKLOADS = {
    # name: partitions, rows/partition, features, stored values per row (None = dense), lambdas
    "cfg2": dict(P=8, n=1_000_000, D=1000, nnz=None, lambdas=[1.0], scaling="strong",
                 desc="8 partitions x 1M x 1k dense, lambda=1 (BASELINE configs[1]); partitions sharded p%N over ranks"),
    "cfg3": dict(P=8, n=1_000_000, D=10_000, nnz=100, lambdas=[0.1, 1.0, 10.0], scaling="strong",
                 desc="8 partitions x 1M x 10k, 1% nnz (100/row), lambda in {0.1,1,10} in one run (BASELINE configs[2], the "
                      "north-star target config); partitions sharded p%N over ranks"),
    "cfg4": dict(P=None, n=1_000_000, D=10_000, nnz=100, lambdas=[1.0], scaling="weak",
                 desc="8 partitions PER GPU x 1M x 10k, 1% nnz, lambda=1 (BASELINE configs[3] = 64 partitions on 8 GPUs; "
                      "P = 8*N at N GPUs, batched Gram + Cholesky)"),
}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="cfg3", choices=["cfg2", "cfg3", "cfg4", "cfg5"])
    ap.add_argument("--also", default="cfg2", help="comma list of further workloads measured after the main one and nested under `also` ('' = none)")
    ap.add_argument("--partitions", type=int, default=0, help="override the workload's partition count")
    ap.add_argument("--rows", type=int, default=0, help="override rows per partition")
    ap.add_argument("--features", type=int, default=0, help="override the feature count")
    ap.add_argument("--cpu-rows", type=int, default=0, help="rows per partition of the bounded CPU sample (0 = auto)")
    ap.add_argument("--cpu-iters", type=int, default=0, help="iterations of the CPU sample job (0 = auto)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--hessian-policy", type=int, default=0)
    ap.add_argument("--keys", type=int, default=100_000, help="cfg5: number of NaiveTrain keys")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the timed path returned in its last step as DIR/<workload>_<name>.npy (float32 / float64, "
                         "under 64 MB in all; see write_dump)")
    return ap.parse_args()


def workload(args, name, world):
    wl = dict(WORKLOADS[name])
    wl["name"] = name
    if wl["P"] is None:
        wl["P"] = 8 * world
    if name == args.workload:
        if args.partitions:
            wl["P"] = args.partitions
        if args.rows:
            wl["n"] = args.rows
        if args.features:
            wl["D"] = args.features
        if args.partitions or args.rows or args.features:
            wl["desc"] = "%d partitions x %d x %d %s, lambdas %s (overridden shape)" % (
                wl["P"], wl["n"], wl["D"], "dense" if wl["nnz"] is None else "%d nnz/row" % wl["nnz"], wl["lambdas"])
    return wl


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            j = json.load(f)
        return dict(hbm=float(j["hbm_gbs"]), tf_burst=float(j["bf16_tflops"]), tf_sust=float(j["bf16_tflops_sustained"]), src="measured")
    except Exception:
        return dict(hbm=6650.0, tf_burst=1590.0, tf_sust=1400.0, src="fallback")


# ------------------------------------------------------------------------------------------------ synthetic data
def true_beta(wl, seed=999):
    """beta* of SURVEY 8d.  Dense rows: std 1/sqrt(D).  Sparse rows: std 1/sqrt(nnz per row), so that the margins x.beta*
    have unit variance as in the dense config (1/sqrt(D) would leave a 100-entry row with a margin of std 0.1: no signal)."""
    rng = np.random.default_rng(seed)
    scale = np.sqrt(wl["D"] if wl["nnz"] is None else wl["nnz"])
    return (rng.normal(size=wl["D"]) / scale).astype(np.float32)


def gen_dense(p, n, D, beta, device):
    """Partition p: x ~ N(0,1) fp32, y ~ Bernoulli(sigmoid(x.beta* - 1)); seed 1000+p (SURVEY.md 8d)."""
    import torch
    g = torch.Generator(device=device)
    g.manual_seed(1000 + p)
    X = torch.randn(n, D, generator=g, device=device, dtype=torch.float32)
    b = torch.as_tensor(beta, device=device)
    s = X @ b - 1.0
    y = (torch.rand(n, generator=g, device=device) < torch.sigmoid(s)).to(torch.int32)
    return X, y


def gen_sparse(p, n, D, nnz, beta, device, chunk=250_000):
    """Partition p in CSR form: `nnz` DISTINCT column ids per row, uniform over [0, D) (rows with a repeated id are redrawn
    whole, which leaves the uniform distribution over distinct sets), sorted; values N(0,1) fp32;
    y ~ Bernoulli(sigmoid(x.beta* - 1)); seed 1000+p (SURVEY.md 8d)."""
    import torch
    g = torch.Generator(device=device)
    g.manual_seed(1000 + p)
    cols = torch.empty((n, nnz), dtype=torch.int32, device=device)
    for r0 in range(0, n, chunk):
        r1 = min(n, r0 + chunk)
        if nnz * nnz > D:   # rejection would rarely terminate: take the nnz smallest of D uniform keys per row instead
            cols[r0:r1] = torch.sort(torch.rand(r1 - r0, D, generator=g, device=device).topk(nnz, dim=1)[1].to(torch.int32), dim=1)[0]
            continue
        c = torch.sort(torch.randint(0, D, (r1 - r0, nnz), generator=g, device=device, dtype=torch.int32), dim=1)[0]
        while True:
            idx = (c[:, 1:] == c[:, :-1]).any(1).nonzero().squeeze(1)
            if idx.numel() == 0:
                break
            c[idx] = torch.sort(torch.randint(0, D, (idx.numel(), nnz), generator=g, device=device, dtype=torch.int32), dim=1)[0]
        cols[r0:r1] = c
    vals = torch.randn(n, nnz, generator=g, device=device, dtype=torch.float32)
    b = torch.as_tensor(beta, device=device)
    s = torch.empty(n, device=device, dtype=torch.float32)
    for r0 in range(0, n, chunk):
        r1 = min(n, r0 + chunk)
        s[r0:r1] = (vals[r0:r1] * b[cols[r0:r1].long()]).sum(1) - 1.0
    y = (torch.rand(n, generator=g, device=device) < torch.sigmoid(s)).to(torch.int32)
    rowptr = torch.arange(n + 1, dtype=torch.int64, device=device) * nnz
    return rowptr, cols.reshape(-1), vals.reshape(-1), y


# ------------------------------------------------------------------------------------------------ clocks sampler
class Clocks:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx, self.lines, self.proc = gpu_index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-lms", "25"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._rd, daemon=True).start()
        except Exception:
            self.proc = None

    def _rd(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if self.proc is not None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except Exception:
                self.proc.kill()
        sm, mx, reasons = [], 0.0, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx = max(mx, float(f[2]))
            except ValueError:
                continue
            for nm, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        if not sm:   # timed region shorter than one sampling period: take one reading now (GPU still warm)
            try:
                o = subprocess.run(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits"],
                                   capture_output=True, text=True, timeout=10).stdout.strip()
                f = [x.strip() for x in o.split(",")]
                sm.append(float(f[1])); mx = max(mx, float(f[2]))
                for nm, v in zip(names, f[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(nm)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx or None, "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------ CPU arm (oracle port)
def _cpu_data(wl, rows):
    """The first `rows` rows of every partition of the workload, generated with the same procedure on the CPU generator."""
    from oracle import oracle as orc
    P, D, nnz = wl["P"], wl["D"], wl["nnz"]
    beta = true_beta(wl)
    if nnz is None:
        Xs, ys = [], []
        for p in range(P):
            X, y = gen_dense(p, rows, D, beta, "cpu")
            Xs.append(X.numpy()); ys.append(y.numpy())
        data = orc.Csr.from_dense(np.vstack(Xs), np.concatenate(ys))
    else:
        ci, vv, ys = [], [], []
        for p in range(P):
            _, c, v, y = gen_sparse(p, rows, D, nnz, beta, "cpu", chunk=50_000)
            ci.append(c.numpy()); vv.append(v.numpy()); ys.append(y.numpy())
        data = orc.Csr(np.arange(P * rows + 1, dtype=np.int64) * nnz, np.concatenate(ci), np.concatenate(vv), np.concatenate(ys), n_features=D)
    return data, np.arange(P + 1, dtype=np.int64) * rows


def cpu_arm(args, wl, steps):
    """The reference's CPU path for this metric: the faithful oracle (TRON with the reference's tolerance schedule), one
    single-threaded solve per (partition, lambda) like one Hadoop reducer each (reducers = nblocks x #lambda,
    jobs/RegressionAdmmTrain.java:355), min(P*L, cores) of them in parallel.  It times x-update + z/u update only (no Hadoop job
    launch, shuffle or per-iteration avro re-ingest: this flatters the reference).  Bounded sample: `rows` rows of every
    partition; iterations/s are extrapolated linearly in rows to the full partition size (same pass count, per-pass cost linear
    in nnz), and the same job on a quarter of the rows is timed as well so that the per-pass linearity is evidenced in the line."""
    from oracle import oracle as orc
    cores = os.cpu_count() or 1
    P, L = wl["P"], len(wl["lambdas"])
    threads = min(P * L, cores)
    rows = args.cpu_rows or (250_000 if wl["nnz"] is not None else 10_000)
    rows = min(rows, wl["n"])
    iters = args.cpu_iters or (min(steps, 5) if wl["nnz"] is not None else min(steps, 20))
    data, prs = _cpu_data(wl, rows)
    t0 = time.perf_counter()
    r = orc.admm_run(data, prs, wl["lambdas"], niters=iters, epsilon=0.0, mode="faithful", nthreads=threads)
    dt = time.perf_counter() - t0
    its = r["iters_done"]
    # linearity probe: the first quarter of the sample rows of every partition
    q = max(rows // 4, 1)
    sub, sprs = _cpu_data(wl, q)
    t1 = time.perf_counter()
    r4 = orc.admm_run(sub, sprs, wl["lambdas"], niters=iters, epsilon=0.0, mode="faithful", nthreads=threads)
    dt4 = time.perf_counter() - t1
    scale = rows / float(wl["n"])
    val = its / dt * scale
    return dict(value=val, unit="ADMM iterations/s", cores=threads, cores_used=threads, cores_host=cores, kind="port",
                extrapolated=scale < 1.0, value_on_sample=its / dt, sample_rows_per_partition=rows, full_rows_per_partition=wl["n"],
                sample="%d partitions x %d rows (%.1f%% of %d) x %d features%s, %d lambda(s) = %d single-threaded reducers on %d threads; "
                       "%d iterations in %.1f s (%d sparse passes); iterations/s extrapolated linearly in rows; host has %d cores"
                       % (P, rows, 100 * scale, wl["n"], wl["D"], "" if wl["nnz"] is None else " at %d nnz/row" % wl["nnz"], L, P * L, threads,
                          its, dt, r["passes"], cores),
                linearity={"rows": [q, rows], "seconds": [dt4, dt], "passes": [int(r4["passes"]), int(r["passes"])],
                           "time_ratio_measured": dt / dt4, "rows_ratio": rows / float(q),
                           # the cost of ONE sparse pass is what is linear in the rows; how many passes TRON needs depends on the
                           # conditioning (fewer rows per feature -> more CG steps), so the two samples are compared per pass
                           "seconds_per_pass_per_row": [dt4 / max(int(r4["passes"]), 1) / q, dt / max(int(r["passes"]), 1) / rows]},
                seconds=dt, iters=its, passes=int(r["passes"]))


_REAL_STDOUT = None


def isolate_stdout():
    """The contract is ONE JSON line on stdout.  Libraries (NCCL's version banner, etc.) may write to fd 1 from any
    rank, so fd 1 is pointed at stderr for the whole process and the JSON line is written to the saved descriptor."""
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)


def emit(obj):
    line = (json.dumps(obj) + "\n").encode()
    if _REAL_STDOUT is not None:
        os.write(_REAL_STDOUT, line)
    else:
        sys.stdout.write(line.decode()); sys.stdout.flush()


def log(*a):
    print("[bench]", *a, file=sys.stderr, flush=True)


DUMP_BYTES = 60_000_000   # array data; with the .npy headers a dump stays under 64 MB


def write_dump(path, arrays):
    """Writes each array as path/<name>.npy so that two builds run with the same arguments can be compared output for output.
    When the arrays exceed DUMP_BYTES together, each one is cut to its share of that budget: a sample of its elements
    (flattened, at indices drawn with a fixed seed, in index order) that is the same from run to run."""
    total = sum(a.nbytes for a in arrays.values())
    os.makedirs(path, exist_ok=True)
    for i, (name, a) in enumerate(sorted(arrays.items())):
        assert a.dtype in (np.float32, np.float64), (name, a.dtype)
        if total > DUMP_BYTES:
            keep = int(a.size * DUMP_BYTES // total)
            if keep < a.size:
                a = a.reshape(-1)[np.sort(np.random.default_rng(i).choice(a.size, keep, replace=False))]
        np.save(os.path.join(path, name + ".npy"), a)


# ------------------------------------------------------------------------------------------------ GPU legs
class Ctx:
    pass


def run_admm_workload(cx, wl, K, W, want_e2e):
    """Resident-data leg (`value`) and host-buffer leg (`e2e`) of one ADMM workload on this rank's GPU.  Returns a dict on
    rank 0 (None elsewhere)."""
    import torch
    import torch.distributed as dist
    import mlease_b200 as mb
    from mlease_b200.distributed import shard_partitions

    args, world, rank, dev, local_rank = cx.args, cx.world, cx.rank, cx.dev, cx.local_rank
    P, n, D, nnz, lambdas = wl["P"], wl["n"], wl["D"], wl["nnz"], wl["lambdas"]
    L = len(lambdas)
    sparse = nnz is not None
    my_parts = shard_partitions(P, world, rank)
    beta = true_beta(wl)
    stream = torch.cuda.current_stream().cuda_stream

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def make_session():
        # the whole loop runs in C (mlease_admm_run); with N > 1 the per-iteration exchange is the library's own ncclAllReduce
        s = mb.AdmmSession(P, D, lambdas, device=local_rank, stream=stream, epsilon=0.0, hessian_policy=args.hessian_policy)
        if cx.comm is not None:
            s.set_comm(cx.comm)
        return s

    # ---------------- device-resident leg ("value") ----------------
    t_gen = time.perf_counter()
    sess = make_session()
    host_parts = {}
    for p in my_parts:
        if sparse:
            rp, ci, vv, y = gen_sparse(p, n, D, nnz, beta, dev)
            sess.add_partition_csr(p, rp, ci, vv, y)            # device pointers: D2D copy + block-major list build
            if want_e2e:
                host_parts[p] = tuple(torch.empty(t.shape, dtype=t.dtype, pin_memory=True).copy_(t) for t in (rp, ci, vv, y))
            del rp, ci, vv, y
        else:
            X, y = gen_dense(p, n, D, beta, dev)
            sess.add_partition_dense(p, X, y)                   # device pointers: D2D copy into the padded layout
            if want_e2e:
                host_parts[p] = tuple(torch.empty(t.shape, dtype=t.dtype, pin_memory=True).copy_(t) for t in (X, y))
            del X, y
        torch.cuda.empty_cache()
    torch.cuda.synchronize()
    log("rank %d %s: data + upload %.1f s, free HBM %.1f GB" % (rank, wl["name"], time.perf_counter() - t_gen, torch.cuda.mem_get_info()[0] / 1e9))
    if W > 0:
        sess.run(W)                                             # warm-up: a throw-away job of W iterations
    barrier()
    sess.profile(2)
    st0 = sess.stats()
    clk = Clocks(local_rank); clk.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    done = sess.run(K)
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    clocks = clk.stop()
    st1 = sess.stats()
    prof = sess.profile(0)
    tms = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tms, op=dist.ReduceOp.MAX)
    ms = float(tms.item())
    z_final = np.stack([sess.z(l) for l in range(L)])
    if cx.dump is not None:
        # what a caller of the timed job gets back: z per lambda, x and u of every (partition on this rank, lambda)
        cx.dump[wl["name"] + "_z"] = z_final
        cx.dump[wl["name"] + "_x"] = np.stack([np.stack([sess.x(p, l) for l in range(L)]) for p in my_parts])
        cx.dump[wl["name"] + "_u"] = np.stack([np.stack([sess.u(p, l) for l in range(L)]) for p in my_parts])
    # size-independent invariant of the consensus step: with the unpenalised intercept z0 = mean_p(x_p + u_p), the new duals
    # u_p = float(u_p + x_p - z) sum to zero over ALL partitions (up to float rounding)
    usum = torch.tensor([[float(sess.u(p, l)[-1]) for l in range(L)] for p in my_parts], dtype=torch.float64, device=dev).sum(0)
    if world > 1:
        dist.all_reduce(usum, op=dist.ReduceOp.SUM)
    launches = st1["kernel_launches"] - st0["kernel_launches"]
    last_maxdiff = st1["last_maxdiff"]
    sess.close(); del sess
    torch.cuda.empty_cache()

    # ---------------- end-to-end leg (host buffers, public API) ----------------
    e2e = None
    if want_e2e:
        # untimed warm-up of the host-buffer path (the W iterations above warmed the resident path only): one upload of every
        # partition from the pinned buffers, state allocation, one iteration -- first-touch of the pinned pages, the copy stream,
        # the stream-ordered pool of the list builders
        sw = make_session()
        for p in my_parts:
            (sw.add_partition_csr if sparse else sw.add_partition_dense)(p, *host_parts[p])
        sw.run(1)
        sw.close()
        del sw
        torch.cuda.synchronize()
        barrier()
        t0 = time.perf_counter()
        s2 = make_session()
        h2d = 0
        for p in my_parts:
            hp = host_parts[p]
            (s2.add_partition_csr if sparse else s2.add_partition_dense)(p, *hp)   # pinned host -> device inside the timed region
            h2d += sum(t.numel() * t.element_size() for t in hp)
        torch.cuda.synchronize()
        t_up = time.perf_counter()
        s2.begin()                                              # solver-state allocation (D'^2 buffers) happens here
        torch.cuda.synchronize()
        t_alloc = time.perf_counter()
        done2 = s2.run(K)
        models = [s2.final_model(l) for l in range(L)]          # device -> host read of the job's result
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        phases = {"upload_and_layout_s": t_up - t0, "solver_state_alloc_s": t_alloc - t_up, "iterations_and_readback_s": t0 + dt - t_alloc}
        if cx.dump is not None:
            cx.dump[wl["name"] + "_e2e_final_model"] = np.stack(models)
        tdt = torch.tensor([dt], dtype=torch.float64, device=dev)
        th = torch.tensor([float(h2d)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tdt, op=dist.ReduceOp.MAX); dist.all_reduce(th, op=dist.ReduceOp.SUM)
        e2e = {"value": done2 / float(tdt.item()), "unit": "ADMM iterations/s", "h2d_bytes_per_step": float(th.item()) / done2,
               "d2h_bytes_per_step": (sum(m.nbytes for m in models) + 8 * done2) * world / done2, "seconds": float(tdt.item()), "phases_rank0": phases,
               "note": "upload once (the reference re-ingests every iteration), K iterations, model read-back; timed after one untimed pass of the same path (upload + 1 iteration)"}
        s2.close()
        del s2, host_parts
        torch.cuda.empty_cache()

    if rank != 0:
        return None
    pk = peaks()
    val = done / (ms / 1000.0)
    k1_ms, k1_n = prof["ms"]["k1"], prof["launches"]["k1"]
    gr_ms, gr_n = prof["ms"]["gram"], prof["launches"]["gram"]
    k1_total_bytes = prof["k1_bytes"]
    k1_gbs = (k1_total_bytes / 1e9) / (k1_ms / 1e3) if k1_ms > 0 else None
    traffic, traffic_src = None, None   # DRAM bytes of one steady-state K1 launch from the committed ncu --set full capture (N=1)
    try:
        if world == 1 and wl["name"] in ("cfg2", "cfg3") and (P, n, D) == (WORKLOADS[wl["name"]]["P"], WORKLOADS[wl["name"]]["n"], WORKLOADS[wl["name"]]["D"]):
            tj = json.load(open(os.path.join(ROOT, "profiles", "k1_traffic.json")))[wl["name"]]
            # the captured launch served a known number of (partition, lambda) passes: its DRAM bytes per algorithmic byte, applied to
            # this run's average launch (launches differ in how many problems are still running)
            traffic = tj["traffic_over_algorithmic"] * (k1_total_bytes / max(k1_n, 1))
            traffic_src = ("%s: %.3f GB of DRAM traffic for %.3f GB algorithmic in the captured launch, scaled to this run's average launch "
                           "(a committed capture of this command, not measured by this run)"
                           % (tj["source"], tj["traffic_bytes_per_launch"] / 1e9, tj["algorithmic_bytes_of_captured_launch"] / 1e9))
    except Exception:
        traffic = None
    fused = bool(st1.get("k1_fused"))
    shared_bytes = st1["k1_shared_bytes"] - st0["k1_shared_bytes"]
    roof = {"kernel": (("k1_csr_fused_kernel (score + reweight + gradient of ALL lambdas of a partition in one pass over its rows)" if fused
                        else "k1_csr_fx_kernel (fused score+reweight+gradient over the CSR rows)") if sparse else
                       "k1_dense_kernel (fused score+reweight+gradient, one pass over X)"), "bound": "hbm",
            "achieved": k1_gbs, "peak": pk["hbm"], "unit": "GB/s", "frac": (k1_gbs / pk["hbm"]) if k1_gbs else None, "traffic": traffic,
            "traffic_source": traffic_src, "peak_source": pk["src"] + " hbm_gbs (copy)", "launches": k1_n, "avg_launch_ms": k1_ms / max(k1_n, 1),
            "algorithmic_bytes_per_launch": k1_total_bytes / max(k1_n, 1),
            "algorithmic_bytes": ("(8*nnz + 17*n) per (partition, lambda) pass (SURVEY 8d); the lambdas of a partition share the rows through L2"
                                  if sparse else "n*(4*ldx + 9) per partition pass (SURVEY 8d)"),
            "share_of_step": k1_ms / ms}
    if not sparse:
        roof["emit_bytes_not_counted"] = prof["k1_emit_bytes"]
    else:
        # the same launches with the lambdas of a partition counted as ONE read of its rows (what a fused pass has to move at least)
        sg = (shared_bytes / 1e9) / (k1_ms / 1e3) if k1_ms > 0 else None
        roof["shared_read"] = {"achieved": sg, "frac": (sg / pk["hbm"]) if sg else None, "bytes_per_launch": shared_bytes / max(k1_n, 1),
                               "bytes": "8*nnz + 9*n per partition pass + 8*n per lambda served"}
    gram_tf = (prof["gram_flops"] / 1e12) / (gr_ms / 1e3) if gr_ms > 0 else None
    # CSR Gram: e4m3 operands (tcgen05 kind::f8f6f4).  MEASURED_PEAKS.json holds no fp8 number: the peak used is twice the measured
    # sustained bf16 figure (the f8f6f4 MMA has twice the bf16 rate per SM); the bf16 peak is reported beside it.
    g_peak = 2.0 * pk["tf_sust"] if sparse else pk["tf_sust"]
    roof_gram = {"kernel": "gram_csr_tcgen05_kernel (e4m3 operands assembled from CSR, kind::f8f6f4)" if sparse else "gram_tcgen05_kernel (bf16, kind::f16)",
                 "bound": "tensor", "achieved": gram_tf, "peak": g_peak, "unit": "TFLOP/s", "frac": (gram_tf / g_peak) if gram_tf else None,
                 "frac_of_bf16_sustained": (gram_tf / pk["tf_sust"]) if gram_tf else None, "launches": gr_n,
                 "avg_launch_ms": gr_ms / max(gr_n, 1), "flops": "n*D'*(D'+1) per build actually run (lower triangle; cold-start builds shared across lambdas)",
                 "peak_source": (("2 x " if sparse else "") + pk["src"] + " bf16 sustained" + (" (no fp8 peak in MEASURED_PEAKS.json)" if sparse else "")),
                 "share_of_step": gr_ms / ms}
    out = {"value": val, "ms_per_step": ms / done, "samples_per_s": val * P * n, "iters_done": done, "job_ms": ms,
           "gpu_launches": int(launches), "clocks": clocks, "roofline": roof, "roofline_gram": roof_gram,
           "kernel_ms": prof["ms"], "kernel_launch_counts": prof["launches"],
           "solver": {"k1_passes": st1["k1_passes"] - st0["k1_passes"], "gram_builds": st1["gram_builds"] - st0["gram_builds"],
                      "newton_steps": st1["newton_steps"] - st0["newton_steps"], "rejected": st1["rejected_steps"] - st0["rejected_steps"],
                      "not_converged": st1["not_converged"], "last_maxdiff": last_maxdiff},
           "checks": {"sum_over_partitions_of_u_intercept": [float(v) for v in usum.tolist()], "last_maxdiff": last_maxdiff},
           "z_checksum": float(np.abs(z_final).sum())}
    if e2e:
        out["e2e"] = e2e
    return out


def parity_leg(cx, wl, iters=4):
    """The same kernels (CSR K1, CSR Gram on tcgen05, wide Cholesky, shared cold-start factor) on a row-reduced copy of the
    workload -- same feature count, nnz/row and lambdas -- against the CPU oracle in exact mode at the same iteration count."""
    import torch
    import mlease_b200 as mb
    from oracle import oracle as orc
    small = dict(wl)
    small["P"] = min(wl["P"], 4)
    small["n"] = 3000 if wl["nnz"] is not None else 6000
    data, prs = _cpu_data(small, small["n"])
    L = len(wl["lambdas"])
    t0 = time.perf_counter()
    ref = orc.admm_run(data, prs, wl["lambdas"], niters=iters, mode="exact", epsilon=0.0, nthreads=min(os.cpu_count() or 1, small["P"] * L))
    t_cpu = time.perf_counter() - t0
    with mb.AdmmSession(small["P"], wl["D"], wl["lambdas"], device=cx.local_rank, stream=torch.cuda.current_stream().cuda_stream, epsilon=0.0) as s:
        for p in range(small["P"]):
            r0, r1 = prs[p], prs[p + 1]
            j0, j1 = data.rowptr[r0], data.rowptr[r1]
            if wl["nnz"] is None:
                s.add_partition_dense(p, data.val[j0:j1].reshape(r1 - r0, wl["D"]), data.response[r0:r1])
            else:
                s.add_partition_csr(p, data.rowptr[r0:r1 + 1] - j0, data.colidx[j0:j1], data.val[j0:j1], data.response[r0:r1])
        done = s.run(iters)
        z = np.stack([s.z(l) for l in range(L)])
        nc = s.stats()["not_converged"]
    errs = [float(np.abs(z[l] - ref["z_hist"][-1, l]).max() / np.abs(ref["z_hist"][-1, l]).max()) for l in range(L)]
    tol = 1e-5
    return {"against": "oracle exact mode (oracle/mlease_oracle.cpp), same iteration count", "shape": "%d partitions x %d rows x %d features%s, lambdas %s, %d iterations"
            % (small["P"], small["n"], wl["D"], "" if wl["nnz"] is None else " at %d nnz/row" % wl["nnz"], wl["lambdas"], iters),
            "rel_err_z_per_lambda": errs, "tol": tol, "pass": bool(done == iters and max(errs) < tol and nc == 0), "oracle_seconds": t_cpu}


def run_naive_workload(cx, K, W):
    """BASELINE configs[4]: NaiveTrain per-key fits, `--keys` keys x 1000 rows x 256 dense features, lambda = 1.  Keys are
    independent (replicas only): rank r fits keys r::N in batches of 8192 keys generated on the device before the timed
    region.  One "step" = one NaiveTrain job = a fit of every key of the rank."""
    import torch
    import torch.distributed as dist
    import mlease_b200 as mb
    args, world, rank, dev = cx.args, cx.world, cx.rank, cx.dev
    nk, D, B = 1000, 256, 8192
    keys_total = args.keys
    my_keys = (keys_total + world - 1) // world
    stream = torch.cuda.current_stream().cuda_stream
    g = torch.Generator(device=dev); g.manual_seed(1000 + rank)
    beta = torch.as_tensor((np.random.default_rng(999).normal(size=D) / np.sqrt(D)).astype(np.float32), device=dev)

    def batch(nkeys):
        X = torch.randn(nkeys * nk, D, generator=g, device=dev)
        y = (torch.rand(nkeys * nk, generator=g, device=dev) < torch.sigmoid(X @ beta - 1.0)).to(torch.int32)
        return X, y, np.arange(nkeys + 1, dtype=np.int64) * nk
    sizes = [min(B, my_keys - k0) for k0 in range(0, my_keys, B)]
    batches = {kb: batch(kb) for kb in dict.fromkeys(sizes)}   # full batches share one draw, the last one may be shorter
    for X, y, krs in batches.values():
        for _ in range(max(W, 1)):
            mb.naive_train_dense(X, krs, y, 1.0, device=cx.local_rank, stream=stream)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(K):
        fits = [mb.naive_train_dense(batches[kb][0], batches[kb][2], batches[kb][1], 1.0, device=cx.local_rank, stream=stream) for kb in sizes]
    e1.record()
    torch.cuda.synchronize()
    tms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tms, op=dist.ReduceOp.MAX)
    if rank != 0:
        return None
    if cx.dump is not None and K > 0:
        # the models [keys, D+1] and skipped flags [keys] of rank 0's keys, in key order
        cx.dump["cfg5_models"] = np.concatenate([m for m, _ in fits])
        cx.dump["cfg5_skipped"] = np.concatenate([s for _, s in fits]).astype(np.float32)
    sec = float(tms.item()) / 1e3
    return {"value": K * my_keys * world / sec, "unit": "per-key fits/s", "metric": "NaiveTrain per-key fits/sec", "seconds": sec,
            "keys": my_keys * world, "rows_per_key": nk, "features": D, "scaling": "weak (replicas only)"}


def main():
    args = parse()
    isolate_stdout()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    K, W = args.steps, max(args.warmup, 0)
    if args.workload == "cfg5":
        wl = dict(name="cfg5", P=args.keys, n=1000, D=256, nnz=None, lambdas=[1.0], scaling="weak",
                  desc="NaiveTrain per-key: %d keys x 1k rows x 256 dense features, lambda=1 (BASELINE configs[4])" % args.keys)
    else:
        wl = workload(args, args.workload, world)
    cfg = {"workload": wl["desc"], "name": wl["name"], "partitions": wl["P"], "rows_per_partition": wl["n"], "features": wl["D"],
           "nnz_per_row": wl["nnz"], "lambdas": wl["lambdas"], "num_iters": K,
           "timed_region": "cold-start job of K iterations (z=u=0), Gram + Cholesky of every partition included",
           "l2": "inputs_larger_than_L2 (>= 0.8 GB per partition)",
           "parallelism": "partitions p%%N over %d rank(s); the loop runs in C (mlease_admm_run) with one ncclAllReduce of [L][D']+1 fp64 per iteration inside the library" % world}
    base = {"metric": "ADMM iterations/sec", "unit": "ADMM iterations/s", "n_gpus": args.gpus, "steps": K, "warmup": W,
            "higher_is_better": True, "scaling": wl["scaling"], "vs_baseline": None, "dtype": "f32 data / f64 reductions / bf16 (dense) or e4m3 (CSR) Gram operands",
            "data": "synthetic", "config": cfg}

    if args.impl == "reference":
        if rank != 0:
            return
        if wl["name"] == "cfg5":
            emit({"impl": "reference", "unavailable": "cfg5 (NaiveTrain) has no reference arm in bench.py; see tests/test_gpu_parity.py for its oracle parity"})
            return
        cb = cpu_arm(args, wl, K)
        out = dict(base)
        out.update({"impl": "reference", "value": cb["value"], "ms_per_step": 1000.0 / cb["value"], "n_gpus": args.gpus,
                    "samples_per_s": cb["value"] * wl["P"] * wl["n"], "gpu_launches": 0, "cpu_baseline": cb,
                    "e2e": {"value": cb["value"], "unit": "ADMM iterations/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}})
        emit(out)
        return

    import torch
    import torch.distributed as dist

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    cx = Ctx()
    cx.args, cx.world, cx.rank, cx.local_rank, cx.dev = args, world, rank, local_rank, "cuda:%d" % local_rank
    cx.comm = None
    cx.dump = {} if args.dump_outputs else None
    if world > 1:
        # keep stdout to the single JSON line: NCCL's version banner / debug lines go to a file
        os.environ.setdefault("NCCL_DEBUG_FILE", "/tmp/nccl_debug_%h_%p.log")
        dist.init_process_group("nccl", device_id=torch.device(cx.dev))
        from mlease_b200.distributed import make_comm
        cx.comm = make_comm(local_rank)      # the library's own NCCL communicator; torch.distributed ships its id and times the ranks

    out = dict(base)
    if wl["name"] == "cfg5":
        res = run_naive_workload(cx, K, W)
        if rank == 0:
            out.update(res)
            if cx.dump is not None:
                write_dump(args.dump_outputs, cx.dump)
            emit(out)
        if world > 1:
            dist.destroy_process_group()
        return

    res = run_admm_workload(cx, wl, K, W, not args.no_e2e)
    also = {}
    for name in [a for a in args.also.split(",") if a and a != wl["name"] and a in WORKLOADS]:
        wl2 = workload(args, name, world)
        r2 = run_admm_workload(cx, wl2, K, W, not args.no_e2e)
        if rank == 0:
            r2["config"] = {"workload": wl2["desc"], "partitions": wl2["P"], "rows_per_partition": wl2["n"], "features": wl2["D"],
                            "nnz_per_row": wl2["nnz"], "lambdas": wl2["lambdas"]}
            also[name] = (wl2, r2)
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    out.update(res)
    ok = True
    if world == 1 and not args.no_parity:
        out["parity"] = parity_leg(cx, wl)
        ok = out["parity"]["pass"]
    if world == 1 and not args.no_cpu:
        out["cpu_baseline"] = cpu_arm(args, wl, K)
    if also:
        out["also"] = {}
        for name, (wl2, r2) in also.items():
            if world == 1 and not args.no_cpu:
                r2["cpu_baseline"] = cpu_arm(args, wl2, K)
            out["also"][name] = r2
    if cx.dump is not None:
        write_dump(args.dump_outputs, cx.dump)
    emit(out)
    if world > 1:
        dist.destroy_process_group()
    if not ok:
        raise SystemExit(3)


if __name__ == "__main__":
    main()
