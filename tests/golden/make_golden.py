#!/usr/bin/env python
"""Regenerates the files under tests/golden/ from a checkout of the reference project (linkedin/ml-ease):

    python tests/golden/make_golden.py <ml-ease checkout>

1. sample_data.npz   -- the reference's only fixture, examples/sample-data.avro, decoded with
                        the minimal Avro object-container reader below (null codec, Pig-style
                        ["null", T] unions) into CSR arrays.  Derived data, not reference source.
2. sklearn_fixed_point.npz -- scikit-learn LogisticRegression (newton-cholesky, tol 1e-12) on
                        that fixture for lambda in {1,10,100}: the ADMM fixed point
                        argmin sum_i w_i logloss + (lambda/2)|beta|^2, intercept unpenalised
                        (jobs/RegressionAdmmTrain.java:381,392-403) -- an INDEPENDENT pin.
3. oracle_frozen.npz -- frozen outputs of oracle/mlease_oracle.cpp (exact + faithful ADMM on the
                        fixture with 4 partitions, objective values, scores, loglik) so that any
                        later edit of the oracle that changes numbers is caught.
4. sample_data_head.avro -- the first HEAD_BLOCKS container blocks of examples/sample-data.avro, byte for
                        byte (header, blocks, sync markers): a valid container of the file's first
                        records, small enough to keep (the whole file is 1.26 MB).
"""
import json
import os
import struct
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
HEAD_BLOCKS = 6


# ----------------------------------------------------------------------------- mini avro reader
class _Buf:
    def __init__(self, b):
        self.b, self.i = b, 0

    def long(self):
        shift, acc = 0, 0
        while True:
            c = self.b[self.i]
            self.i += 1
            acc |= (c & 0x7F) << shift
            if not c & 0x80:
                break
            shift += 7
        return (acc >> 1) ^ -(acc & 1)

    def bytes_(self):
        n = self.long()
        out = self.b[self.i:self.i + n]
        self.i += n
        return out

    def raw(self, n):
        out = self.b[self.i:self.i + n]
        self.i += n
        return out


def _decode(buf, schema):
    if isinstance(schema, list):  # union
        return _decode(buf, schema[buf.long()])
    if isinstance(schema, dict):
        t = schema["type"]
        if t == "record":
            return {f["name"]: _decode(buf, f["type"]) for f in schema["fields"]}
        if t == "array":
            out = []
            while True:
                n = buf.long()
                if n == 0:
                    break
                if n < 0:
                    n = -n
                    buf.long()
                for _ in range(n):
                    out.append(_decode(buf, schema["items"]))
            return out
        return _decode(buf, t)
    if schema == "null":
        return None
    if schema == "string":
        return buf.bytes_().decode()
    if schema == "int" or schema == "long":
        return buf.long()
    if schema == "float":
        return struct.unpack("<f", buf.raw(4))[0]
    if schema == "double":
        return struct.unpack("<d", buf.raw(8))[0]
    if schema == "boolean":
        return buf.raw(1) != b"\0"
    raise ValueError(schema)


def read_avro(path):
    b = _Buf(open(path, "rb").read())
    assert b.raw(4) == b"Obj\x01"
    meta = {}
    while True:
        n = b.long()
        if n == 0:
            break
        for _ in range(abs(n)):
            k = b.bytes_().decode()
            meta[k] = b.bytes_()
    assert meta.get("avro.codec", b"null") == b"null"
    schema = json.loads(meta["avro.schema"])
    sync = b.raw(16)
    recs, nblocks = [], 0
    while b.i < len(b.b):
        cnt = b.long()
        b.long()  # block byte size
        for _ in range(cnt):
            recs.append(_decode(b, schema))
        assert b.raw(16) == sync
        nblocks += 1
    return schema, recs, nblocks


def write_sample_head(path):
    """Copies the header and the first HEAD_BLOCKS blocks of the container at `path` to sample_data_head.avro."""
    raw = open(path, "rb").read()
    b = _Buf(raw)
    assert b.raw(4) == b"Obj\x01"
    while True:
        n = b.long()
        if n == 0:
            break
        for _ in range(abs(n)):
            b.bytes_(), b.bytes_()
    sync = b.raw(16)
    for _ in range(HEAD_BLOCKS):
        b.long()
        b.raw(b.long())
        assert b.raw(16) == sync
    with open(os.path.join(HERE, "sample_data_head.avro"), "wb") as f:
        f.write(raw[:b.i])


def main(ref):
    from oracle import oracle as orc

    src = os.path.join(ref, "examples", "sample-data.avro")
    write_sample_head(src)
    schema, recs, nblocks = read_avro(src)
    names = sorted({f["name"] for r in recs for f in r["features"]}, key=lambda s: int(s))
    assert all(f["term"] in ("", None) for r in recs for f in r["features"])
    gid = {n: i for i, n in enumerate(names)}
    rowptr, colidx, val = [0], [], []
    for r in recs:
        fs = sorted(((gid[f["name"]], f["value"]) for f in r["features"]))
        colidx += [a for a, _ in fs]
        val += [np.float32(v) for _, v in fs]
        rowptr.append(len(colidx))
    response = np.array([r["response"] for r in recs], np.int32)
    weight = np.array([1 if r["weight"] is None else r["weight"] for r in recs], np.float32)
    offset = np.array([0 if r["offset"] is None else r["offset"] for r in recs], np.float32)
    np.savez_compressed(os.path.join(HERE, "sample_data.npz"), rowptr=np.array(rowptr, np.int64),
                        colidx=np.array(colidx, np.int32), val=np.array(val, np.float32), response=response,
                        weight=weight, offset=offset, feature_names=np.array(names), avro_blocks=nblocks)
    print("fixture:", len(recs), "records", len(names), "features", int((response == 1).sum()), "positives", nblocks, "blocks")

    data = orc.Csr(np.array(rowptr), np.array(colidx), np.array(val), response, weight, offset, len(names))
    D = data.n_features

    # 2. sklearn fixed points
    from sklearn.linear_model import LogisticRegression
    from scipy.sparse import csr_matrix
    X = csr_matrix((data.val.astype(np.float64), data.colidx, data.rowptr), shape=(data.nrows, D))
    fp = {}
    for lam in (1.0, 10.0, 100.0):
        clf = LogisticRegression(C=1.0 / lam, fit_intercept=True, solver="newton-cholesky", tol=1e-12, max_iter=1000)
        clf.fit(X.toarray(), (response == 1).astype(int), sample_weight=weight.astype(np.float64))
        fp["lam%g" % lam] = np.concatenate([clf.coef_.ravel(), clf.intercept_])
    np.savez_compressed(os.path.join(HERE, "sklearn_fixed_point.npz"), **fp)

    # 3. frozen oracle outputs
    P = 4
    prs = np.linspace(0, data.nrows, P + 1).astype(np.int64)
    frozen = {}
    ex = orc.admm_run(data, prs, [1.0, 10.0, 100.0], niters=20, mode="exact", nthreads=8)
    fa = orc.admm_run(data, prs, [1.0, 10.0, 100.0], niters=20, mode="faithful", nthreads=8)
    frozen.update(part_rowstart=prs, exact_z_hist=ex["z_hist"], exact_diff_hist=ex["diff_hist"], exact_x_last=ex["x_last"],
                  exact_u_last=ex["u_last"], faithful_z_hist=fa["z_hist"], faithful_eps_hist=fa["eps_hist"],
                  faithful_iters=fa["iters_done"], faithful_passes=fa["passes"])
    rng = np.random.default_rng(7)
    w = rng.normal(0, 0.1, D + 1)
    pm = rng.normal(0, 0.1, D + 1)
    pv = np.full(D + 1, 0.5)
    f, g = orc.objective("grad", data, w, pm, pv)
    frozen.update(obj_w=w, obj_pm=pm, obj_f=f, obj_g=g, obj_hdiag=orc.objective("hessian_diag", data, w, pm, pv))
    model = ex["z_hist"][-1, 0]
    pred = orc.score(data, model)
    ll, cnt = orc.test_loglik(response, pred, weight, combiner_block=128)
    frozen.update(score_pred=pred, loglik=ll, loglik_count=cnt, sample_loglik=orc.sample_test_loglik(data, model))
    np.savez_compressed(os.path.join(HERE, "oracle_frozen.npz"), **frozen)
    for lam, li in ((1.0, 0), (10.0, 1), (100.0, 2)):
        z = ex["z_hist"][-1, li]
        ref = fp["lam%g" % lam]
        print("lambda", lam, "exact ADMM(20) vs sklearn: max|dz|/max|z| =", np.abs(z - ref).max() / np.abs(ref).max(),
              " faithful:", np.abs(fa["z_hist"][-1, li] - ref).max() / np.abs(ref).max())


if __name__ == "__main__":
    main(sys.argv[1])
