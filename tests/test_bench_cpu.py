"""CPU-side checks of bench.py: the config-3 generator (SURVEY.md 8d: uniform DISTINCT columns per row) and the
`--impl reference` line of the CPU arm (the oracle port on a bounded sample, extrapolation declared in the line)."""
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def test_sparse_generator_distinct_sorted_uniform_and_seeded():
    import bench
    wl = dict(bench.WORKLOADS["cfg3"])
    wl.update(D=300, nnz=20)
    beta = bench.true_beta(wl)
    rp, ci, v, y = (t.numpy() for t in bench.gen_sparse(3, 5000, 300, 20, beta, "cpu", chunk=1200))
    assert rp[0] == 0 and np.all(np.diff(rp) == 20) and len(ci) == len(v) == 5000 * 20
    c = ci.reshape(5000, 20)
    assert np.all(np.diff(c, axis=1) > 0) and c.min() >= 0 and c.max() < 300          # strictly increasing = distinct, sorted
    counts = np.bincount(ci, minlength=300)
    assert counts.min() > 0.7 * counts.mean() and counts.max() < 1.3 * counts.mean()   # uniform over the columns
    assert set(np.unique(y)) <= {0, 1} and 0.1 < y.mean() < 0.6
    rp2, ci2, v2, y2 = (t.numpy() for t in bench.gen_sparse(3, 5000, 300, 20, beta, "cpu", chunk=1200))
    assert np.array_equal(ci, ci2) and np.array_equal(v, v2) and np.array_equal(y, y2)
    _, ci3, _, _ = (t.numpy() for t in bench.gen_sparse(4, 5000, 300, 20, beta, "cpu", chunk=1200))
    assert not np.array_equal(ci, ci3)                                                  # seed 1000 + p


def test_dump_outputs_are_whole_within_budget_and_a_fixed_sample_beyond(tmp_path, monkeypatch):
    import bench
    rng = np.random.default_rng(0)
    arrays = {"cfg3_z": rng.normal(size=(3, 101)), "cfg3_u": rng.normal(size=(2, 3, 101)).astype(np.float32)}
    bench.write_dump(str(tmp_path / "a"), arrays)
    for name, a in arrays.items():
        got = np.load(str(tmp_path / "a" / (name + ".npy")))
        assert got.dtype == a.dtype and np.array_equal(got, a)
    monkeypatch.setattr(bench, "DUMP_BYTES", 2000)
    for d in ("b", "c"):
        bench.write_dump(str(tmp_path / d), arrays)
    sizes = 0
    for name, a in arrays.items():
        b, c = (np.load(str(tmp_path / d / (name + ".npy"))) for d in ("b", "c"))
        assert np.array_equal(b, c) and b.dtype == a.dtype and 0 < b.size < a.size and np.isin(b, a).all()
        sizes += b.nbytes
    assert sizes <= 2000


def test_reference_arm_line_declares_its_sample():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2", "--warmup", "0",
                          "--partitions", "2", "--rows", "4000", "--features", "20000", "--cpu-rows", "1000", "--cpu-iters", "2"],
                         capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    j = json.loads(lines[0])
    assert j["impl"] == "reference" and j["unit"] == "ADMM iterations/s" and j["higher_is_better"] is True
    cb = j["cpu_baseline"]
    assert cb["kind"] == "port" and cb["extrapolated"] is True and cb["cores_used"] <= cb["cores_host"]
    assert cb["sample_rows_per_partition"] == 1000 and cb["full_rows_per_partition"] == 4000
    assert abs(cb["value"] - cb["value_on_sample"] * 0.25) < 1e-9 * max(1.0, cb["value"])
    assert cb["linearity"]["rows"] == [250, 1000] and cb["linearity"]["time_ratio_measured"] > 0
    assert j["e2e"]["h2d_bytes_per_step"] == 0 and j["value"] == cb["value"]
