"""CPU tests of the block-parallel ingest of the host job layer (ml-ease_b200/host/avro_walk.hpp): the plan-walker readers
and RegressionPrepare must give exactly what the generic (Value-tree) decoder gives -- same rows, same first-seen feature
ids, same keys, same error texts -- whatever the number of threads, blocks and files."""
import ctypes as C
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import avro_util as au  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")


@pytest.fixture(scope="module")
def host():
    import mlease_b200
    mlease_b200.lib()
    h = C.CDLL(os.path.join(ROOT, "ml-ease_b200", "lib", "libmlease_host.so"))
    h.mlease_job_last_error.restype = C.c_char_p
    h.mlease_rows_count.restype = C.c_int64
    h.mlease_rows_feature.restype = C.c_char_p
    h.mlease_rows_key.restype = C.c_char_p
    h.mlease_rows_feature.argtypes = [C.c_void_p, C.c_int32]
    h.mlease_rows_key.argtypes = [C.c_void_p, C.c_int64]
    h.mlease_rows_count.argtypes = [C.c_void_p, C.POINTER(C.c_int64), C.POINTER(C.c_int32)]
    h.mlease_rows_get.argtypes = [C.c_void_p] + [C.c_void_p] * 6
    h.mlease_rows_free.argtypes = [C.c_void_p]
    return h


def _rows(host, path, raw, binary=False, generic=False):
    """-> dict of arrays, or the error text."""
    hd = C.c_void_p()
    rc = host.mlease_rows_read(path.encode(), int(raw), int(binary), int(generic), C.byref(hd))
    if rc != 0:
        return host.mlease_job_last_error().decode()
    nnz, nf = C.c_int64(), C.c_int32()
    n = host.mlease_rows_count(hd, C.byref(nnz), C.byref(nf))
    out = {"rowptr": np.zeros(n + 1, np.int64), "colidx": np.zeros(nnz.value, np.int32), "vals": np.zeros(nnz.value, np.float32),
           "response": np.zeros(n, np.int32), "weight": np.zeros(n, np.float32), "offset": np.zeros(n, np.float32)}
    host.mlease_rows_get(hd, *[out[k].ctypes.data_as(C.c_void_p) for k in ("rowptr", "colidx", "vals", "response", "weight", "offset")])
    out["features"] = [host.mlease_rows_feature(hd, k) for k in range(nf.value)]
    out["keys"] = [host.mlease_rows_key(hd, i) for i in range(n)]
    host.mlease_rows_free(hd)
    return out


def _same(a, b):
    assert isinstance(a, dict) and isinstance(b, dict), (a if isinstance(a, str) else "", b if isinstance(b, str) else "")
    assert a["features"] == b["features"] and a["keys"] == b["keys"]
    for k in ("rowptr", "colidx", "response"):
        assert np.array_equal(a[k], b[k]), k
    for k in ("vals", "weight", "offset"):
        assert np.array_equal(a[k].view(np.uint32), b[k].view(np.uint32)), k   # bit for bit


def _write_cfg(path, **kv):
    with open(path, "w") as f:
        for k, v in kv.items():
            f.write("%s=%s\n" % (k.replace("_", "."), v))
    return path


def _run(host, job, cfg):
    rc = host.mlease_job_run(job.encode(), cfg.encode())
    return rc, host.mlease_job_last_error().decode()


PREPARED = {"type": "record", "name": "RegressionPrepareOutput", "fields": [
    {"name": "key", "type": "string"}, {"name": "response", "type": "int"},
    {"name": "features", "type": {"type": "array", "items": {"type": "record", "name": "feature", "fields": [
        {"name": "name", "type": "string"}, {"name": "term", "type": "string"}, {"name": "value", "type": "float"}]}}},
    {"name": "weight", "type": "float"}, {"name": "offset", "type": "float"}]}


def _random_prepared(rng, n, nfeat_names=40):
    recs = []
    for i in range(n):
        k = int(rng.integers(0, 9))                      # empty feature lists occur
        feats = [{"name": "f%d" % rng.integers(0, nfeat_names), "term": ("" if rng.random() < 0.6 else "t%d" % rng.integers(0, 3)),
                  "value": float(np.float32(rng.normal()))} for _ in range(k)]
        recs.append({"key": str(int(rng.integers(0, 5))), "response": int(rng.integers(0, 2)), "features": feats,
                     "weight": float(np.float32(rng.uniform(0.5, 2))), "offset": float(np.float32(rng.normal(0, 0.1)))})
    return recs


@pytest.mark.parametrize("codec", ["null", "deflate"])
def test_prepared_rows_fast_equals_generic_across_blocks_files_threads(host, tmp_path, monkeypatch, codec):
    rng = np.random.default_rng(3)
    d = tmp_path / "prep"
    au.write_avro(str(d / "part-00000.avro"), PREPARED, _random_prepared(rng, 700), codec=codec, block=64)
    au.write_avro(str(d / "part-00001.avro"), PREPARED, _random_prepared(rng, 300, nfeat_names=60), codec=codec, block=7)
    au.write_avro(str(d / "part-00002.avro"), PREPARED, [], codec=codec)            # a file without blocks
    ref = _rows(host, str(d), raw=False, generic=True)
    assert isinstance(ref, dict) and len(ref["response"]) == 1000 and any(b"\x01" in f for f in ref["features"])
    try:
        for threads in (1, 3, 8):
            assert host.mlease_host_set_threads(threads) == threads
            _same(_rows(host, str(d), raw=False), ref)
    finally:
        host.mlease_host_set_threads(0)
    _same(_rows(host, str(d), raw=False, binary=True), _rows(host, str(d), raw=False, binary=True, generic=True))


def test_raw_pig_style_unions_fast_equals_generic_and_fixture(host, tmp_path):
    """The reference's own fixture schema: every field a ["null", T] union, the feature record itself nullable."""
    npz = np.load(os.path.join(GOLDEN, "sample_data.npz"))
    recs = au.fixture_records(npz)
    p = str(tmp_path / "raw.avro")
    au.write_avro(p, au.PIG_SCHEMA, recs, codec="deflate", block=97)
    fast, gen = _rows(host, p, raw=True), _rows(host, p, raw=True, generic=True)
    _same(fast, gen)
    assert len(fast["response"]) == 1000 and int((fast["response"] == 1).sum()) == 299 and len(fast["features"]) == 200
    # the first blocks of the reference's fixture file itself, as Pig wrote them
    head = _rows(host, os.path.join(GOLDEN, "sample_data_head.avro"), raw=True)
    _same(head, _rows(host, os.path.join(GOLDEN, "sample_data_head.avro"), raw=True, generic=True))
    assert len(head["response"]) == 78


def test_error_texts_are_the_generic_readers(host, tmp_path):
    sch = {"type": "record", "name": "r", "fields": [
        {"name": "response", "type": ["null", "int", "long"]},
        {"name": "features", "type": ["null", {"type": "array", "items": {"type": "record", "name": "f", "fields": [
            {"name": "name", "type": ["null", "string"]}, {"name": "term", "type": "string"}, {"name": "value", "type": "double"}]}}]}]}
    ok = {"response": 1, "features": [{"name": "a", "term": "", "value": 0.5}]}
    cases = {"null_features": [ok, dict(ok, features=None)], "null_name": [ok, {"response": 0, "features": [{"name": None, "term": "", "value": 1.0}]}],
             "no_response": [ok, dict(ok, response=None)], "bad_response": [ok, dict(ok, response=7)]}
    for name, recs in cases.items():
        p = str(tmp_path / (name + ".avro"))
        au.write_avro(p, sch, recs * 3, block=2)
        f, g = _rows(host, p, raw=True), _rows(host, p, raw=True, generic=True)
        assert isinstance(f, str) and f == g, (name, f, g)
    # prepared reader: the reserved intercept name
    p = str(tmp_path / "icpt.avro")
    au.write_avro(p, PREPARED, [{"key": "0", "response": 1, "features": [{"name": "(INTERCEPT)", "term": "", "value": 1.0}], "weight": 1.0, "offset": 0.0}])
    f, g = _rows(host, p, raw=False), _rows(host, p, raw=False, generic=True)
    assert isinstance(f, str) and f == g and "(INTERCEPT)" in f
    # truncated data file: an error from both, never an overrun
    good = str(tmp_path / "good.avro")
    au.write_avro(good, PREPARED, _random_prepared(np.random.default_rng(0), 50), block=10)
    blob = open(good, "rb").read()
    bad = str(tmp_path / "bad.avro")
    open(bad, "wb").write(blob[:len(blob) * 2 // 3])
    f, g = _rows(host, bad, raw=False), _rows(host, bad, raw=False, generic=True)
    assert isinstance(f, str) and isinstance(g, str) and "avro" in f and "avro" in g


def test_unusual_schema_falls_back_to_the_generic_reader(host, tmp_path):
    """A weight stored as a string is not something the plan walker takes: the generic reader handles the file."""
    sch = {"type": "record", "name": "r", "fields": [
        {"name": "response", "type": "int"}, {"name": "weight", "type": "string"},
        {"name": "features", "type": {"type": "array", "items": {"type": "record", "name": "f", "fields": [
            {"name": "name", "type": "string"}, {"name": "term", "type": "string"}, {"name": "value", "type": "float"}]}}}]}
    p = str(tmp_path / "odd.avro")
    au.write_avro(p, sch, [{"response": 1, "weight": "x", "features": [{"name": "a", "term": "b", "value": 2.0}]}] * 5)
    _same(_rows(host, p, raw=True), _rows(host, p, raw=True, generic=True))


@pytest.mark.parametrize("mapkey", ["pkey", ""])
def test_prepare_job_fast_equals_generic(host, tmp_path, monkeypatch, mapkey):
    """RegressionPrepare on the plan walker (block-parallel, records encoded directly) writes the records the generic job writes:
    map.key branch and the seeded random-key branch with click replicates (the key stream is a counter: one draw per record)."""
    npz = np.load(os.path.join(GOLDEN, "sample_data.npz"))
    recs = au.fixture_records(npz, with_key=lambda i: i % 4)
    au.write_avro(str(tmp_path / "in" / "part-0.avro"), au.pig_schema_with_key(), recs[:600], block=53, codec="deflate")
    au.write_avro(str(tmp_path / "in" / "part-1.avro"), au.pig_schema_with_key(), recs[600:], block=400)
    outs = {}
    for mode in ("fast", "generic"):
        monkeypatch.setenv("MLEASE_HOST_GENERIC_INGEST", "1" if mode == "generic" else "0")
        kv = dict(input_paths=str(tmp_path / "in"), output_path=str(tmp_path / ("out_" + mode)), num_blocks=5, num_click_replicates=3, random_seed=11)
        if mapkey:
            kv["map_key"] = mapkey
        rc, err = _run(host, "RegressionPrepare", _write_cfg(str(tmp_path / (mode + ".job")), **kv))
        assert rc == 0, err
        outs[mode] = au.read_dir(str(tmp_path / ("out_" + mode)))
    assert len(outs["fast"]) == len(outs["generic"]) >= 1000
    assert outs["fast"] == outs["generic"]
    # and the prepared output reads back the same through both readers
    _same(_rows(host, str(tmp_path / "out_fast"), raw=False), _rows(host, str(tmp_path / "out_generic"), raw=False, generic=True))


def test_model_files_direct_encoder_equals_value_tree_encoder(host, tmp_path):
    """iter-i/{u,init-value,model}, final-model, models: the direct encoder (feature name / term bytes prepared once per file)
    writes the records the Value-tree encoder writes; large models span several container blocks."""
    rng = np.random.default_rng(5)
    D, M = 3000, 9
    names = ["f%d" % k if k % 3 else "f%d\x01t%d" % (k, k % 7) for k in range(D)]
    keys = ["%s#%d" % ("1.0" if m % 2 else "0.1", m) for m in range(M)]
    coefs = rng.normal(size=(M, D + 1)).astype(np.float32)
    ux = rng.normal(size=(M, D + 1)).astype(np.float32)
    nb = ("\0".join(names) + "\0").encode()
    kb = ("\0".join(keys) + "\0").encode()
    for with_ux in (False, True):
        outs = []
        for generic in (0, 1):
            p = str(tmp_path / ("m%d%d.avro" % (with_ux, generic)))
            rc = host.mlease_models_write(p.encode(), D, nb, M, kb, coefs.ctypes.data_as(C.c_void_p), ux.ctypes.data_as(C.c_void_p) if with_ux else None, generic)
            assert rc == 0, host.mlease_job_last_error().decode()
            outs.append(au.read_avro(p)[1])
        assert outs[0] == outs[1] and len(outs[0]) == M
        r0 = outs[0][0]
        assert r0["key"] == keys[0] and r0["model"][0] == {"name": "(INTERCEPT)", "term": "", "value": float(coefs[0, D])}
        assert r0["model"][1 + 3] == {"name": "f3", "term": "t3", "value": float(coefs[0, 3])} and r0["model"][1 + 4]["term"] == "" and ("uplusx" in r0) == with_ux


def test_test_job_output_transcoder_equals_generic(host, tmp_path):
    """RegressionTest's output (input record with unions removed + pred, jobs/RegressionTest.java:198-236) written by copying the
    record bytes without the union indices, block-parallel: same records as decode -> append pred -> encode; a record that does
    not fit the union-free schema (a null response) sends the file through the generic path, which reports it as before."""
    npz = np.load(os.path.join(GOLDEN, "sample_data.npz"))
    recs = au.fixture_records(npz, with_key=lambda i: i % 3)
    src = str(tmp_path / "t.avro")
    au.write_avro(src, au.pig_schema_with_key(), recs, block=111, codec="deflate")
    pred = np.random.default_rng(1).normal(size=len(recs)).astype(np.float32)
    outs = []
    for generic in (0, 1):
        o = str(tmp_path / ("o%d.avro" % generic))
        rc = host.mlease_test_output_write(src.encode(), o.encode(), pred.ctypes.data_as(C.c_void_p), C.c_int64(len(pred)), generic)
        assert rc == 0, host.mlease_job_last_error().decode()
        outs.append(au.read_avro(o))
    assert outs[0][0] == outs[1][0] and outs[0][0]["name"] == "AdmmTestOutput" and outs[0][0]["fields"][-1] == {"name": "pred", "type": "float"}
    assert outs[0][1] == outs[1][1] and len(outs[0][1]) == len(recs)
    assert [np.float32(r["pred"]) for r in outs[0][1][:50]] == list(pred[:50]) and outs[0][1][7]["features"][0]["name"] == recs[7]["features"][0]["name"]
    # a null in a field that the union-free schema makes mandatory: both report the generic encoder's error
    bad = str(tmp_path / "bad.avro")
    au.write_avro(bad, au.pig_schema_with_key(), recs[:20] + [dict(recs[20], response=None)] + recs[21:40], block=7)
    errs = []
    for generic in (0, 1):
        rc = host.mlease_test_output_write(bad.encode(), str(tmp_path / "ob.avro").encode(), pred.ctypes.data_as(C.c_void_p), C.c_int64(len(pred)), generic)
        assert rc != 0
        errs.append(host.mlease_job_last_error().decode())
    assert errs[0] == errs[1] and "null" in errs[0]


def test_scored_records_reader_equals_generic(host, tmp_path):
    """RegressionTestLoglik reads (response, pred, weight) of the Test job's output: the plan walker skips the feature lists."""
    npz = np.load(os.path.join(GOLDEN, "sample_data.npz"))
    recs = au.fixture_records(npz)
    src = str(tmp_path / "t.avro")
    au.write_avro(src, au.PIG_SCHEMA, recs, block=90)
    pred = np.random.default_rng(2).normal(size=len(recs)).astype(np.float32)
    scored = str(tmp_path / "scored.avro")
    assert host.mlease_test_output_write(src.encode(), scored.encode(), pred.ctypes.data_as(C.c_void_p), C.c_int64(len(pred)), 0) == 0
    host.mlease_scored_read.restype = C.c_int64
    got = []
    for generic in (0, 1):
        r, p, w = np.zeros(len(recs), np.int32), np.zeros(len(recs), np.float32), np.zeros(len(recs), np.float32)
        n = host.mlease_scored_read(scored.encode(), C.c_int64(len(recs)), r.ctypes.data_as(C.c_void_p), p.ctypes.data_as(C.c_void_p), w.ctypes.data_as(C.c_void_p), generic)
        assert n == len(recs), host.mlease_job_last_error().decode()
        got.append((r, p, w))
    for a, b in zip(got[0], got[1]):
        assert np.array_equal(a, b)
    assert np.array_equal(got[0][1], pred) and np.array_equal(got[0][0], npz["response"].astype(np.int32)) and (got[0][2] == 1).all()
    # records without pred: the reference's error text from both
    errs = []
    for generic in (0, 1):
        n = host.mlease_scored_read(src.encode(), C.c_int64(0), None, None, None, generic)
        assert n == -1
        errs.append(host.mlease_job_last_error().decode())
    assert errs[0] == errs[1] == "response/pred is null"


def _random_case(rng):
    """A random record schema in the family the jobs read (fields present / absent / nullable, numeric types varied, extra fields,
    shuffled order) with matching records."""
    def nullable(t, p=0.5):
        return ["null", t] if rng.random() < p else t
    item_fields = [{"name": "name", "type": nullable("string", 0.4)}, {"name": "value", "type": nullable(str(rng.choice(["float", "double", "int", "long"])), 0.4)}]
    has_term = rng.random() < 0.7
    if has_term:
        item_fields.append({"name": "term", "type": nullable("string", 0.4)})
    if rng.random() < 0.3:
        item_fields.append({"name": "junk", "type": "long"})
    rng.shuffle(item_fields)
    item = {"type": "record", "name": "feat", "fields": item_fields}
    feats_t = {"type": "array", "items": (["null", item] if rng.random() < 0.5 else item)}
    fields = [{"name": "features", "type": (["null", feats_t] if rng.random() < 0.5 else feats_t)}]
    present = {}
    for nm, types in (("key", ["string", "int", "long"]), ("response", ["int", "boolean", "long"]), ("click", ["int", "boolean"]), ("label", ["int"]),
                      ("weight", ["float", "double", "int", "string"]), ("offset", ["float", "double", "long"])):
        if rng.random() < (0.85 if nm in ("response", "key") else 0.5):
            t = str(rng.choice(types, p=None if nm != "weight" else [0.4, 0.3, 0.25, 0.05]))
            present[nm] = t
            fields.append({"name": nm, "type": nullable(t)})
    if rng.random() < 0.5:
        fields.append({"name": "extra", "type": {"type": "record", "name": "ex", "fields": [
            {"name": "tags", "type": {"type": "array", "items": "string"}}, {"name": "d", "type": ["null", "double"]}, {"name": "b", "type": "boolean"}]}})
    rng.shuffle(fields)
    schema = {"type": "record", "name": "rec", "fields": fields}

    def val(t, fld):
        is_union = isinstance(fld["type"], list)
        if is_union and rng.random() < 0.15:
            return None
        if t == "string":
            return str(rng.integers(0, 4)) if fld["name"] == "key" else "w%d" % rng.integers(0, 3)
        if t == "boolean":
            return bool(rng.integers(0, 2))
        if t in ("int", "long"):
            return int(rng.integers(-1, 2)) if fld["name"] in ("response", "click", "label") else int(rng.integers(0, 5))
        return float(np.float32(rng.normal()))
    recs = []
    for _ in range(int(rng.integers(0, 60))):
        r = {}
        for f in fields:
            if f["name"] == "features":
                if isinstance(f["type"], list) and rng.random() < 0.1:
                    r["features"] = None
                    continue
                fl = []
                for _k in range(int(rng.integers(0, 6))):
                    e = {}
                    for itf in item_fields:
                        t = itf["type"][1] if isinstance(itf["type"], list) else itf["type"]
                        if itf["name"] == "name":
                            e["name"] = None if (isinstance(itf["type"], list) and rng.random() < 0.05) else "n%d" % rng.integers(0, 12)
                        elif itf["name"] == "term":
                            e["term"] = None if (isinstance(itf["type"], list) and rng.random() < 0.3) else ("" if rng.random() < 0.5 else "t%d" % rng.integers(0, 3))
                        elif itf["name"] == "junk":
                            e["junk"] = int(rng.integers(0, 1000))
                        else:
                            e["value"] = None if (isinstance(itf["type"], list) and rng.random() < 0.1) else (int(rng.integers(-3, 4)) if t in ("int", "long") else float(np.float32(rng.normal())))
                    fl.append(e)
                r["features"] = fl
            elif f["name"] == "extra":
                r["extra"] = {"tags": ["a"] * int(rng.integers(0, 3)), "d": None if rng.random() < 0.5 else 1.5, "b": True}
            else:
                r[f["name"]] = val(present[f["name"]], f)
        recs.append(r)
    return schema, recs


def test_random_schemas_fast_reader_equals_generic_reader(host, tmp_path):
    """Seeded fuzz over the schema family the jobs read: whatever the generic reader returns -- rows or an error text -- the
    plan-walker reader returns too (schemas it does not take, e.g. a string weight, fall back to the generic reader)."""
    rng = np.random.default_rng(2024)
    n_rows = n_err = 0
    for case in range(120):
        schema, recs = _random_case(rng)
        p = str(tmp_path / ("c%d.avro" % case))
        au.write_avro(p, schema, recs, block=int(rng.integers(1, 9)), codec=str(rng.choice(["null", "deflate"])))
        raw, binary = bool(rng.integers(0, 2)), bool(rng.integers(0, 2))
        f, g = _rows(host, p, raw=raw, binary=binary), _rows(host, p, raw=raw, binary=binary, generic=True)
        if isinstance(g, str):
            assert f == g, (case, f, g)
            n_err += 1
        else:
            _same(f, g)
            n_rows += 1
    assert n_rows >= 20 and n_err >= 5, (n_rows, n_err)


def test_random_schemas_prepare_job_fast_equals_generic(host, tmp_path, monkeypatch):
    """The same fuzz through RegressionPrepare: identical output records or identical error text, for map.key on fields of every
    scalar type (printed as Java's toString), on a missing field, and for the seeded random-key branch with click replicates."""
    rng = np.random.default_rng(99)
    n_ok = n_err = 0
    for case in range(60):
        schema, recs = _random_case(rng)
        if rng.random() < 0.7:   # most cases: a record stream the job accepts (int response, lists and names present)
            schema["fields"] = [f for f in schema["fields"] if f["name"] not in ("response", "click", "label")] + [{"name": "response", "type": ["null", "int"]}]
            for r in recs:
                r["response"] = int(rng.integers(0, 2))
                r["features"] = r["features"] or []
                for e in r["features"]:
                    e["name"] = e["name"] or "n0"
            if not recs:
                continue
        d = tmp_path / ("in%d" % case)
        au.write_avro(str(d / "part-0.avro"), schema, recs, block=int(rng.integers(1, 9)), codec=str(rng.choice(["null", "deflate"])))
        names = [f["name"] for f in schema["fields"] if f["name"] != "features"]
        mapkey = "" if rng.random() < 0.4 else str(rng.choice(names + ["nosuchfield"]))
        res = []
        for mode in ("fast", "generic"):
            monkeypatch.setenv("MLEASE_HOST_GENERIC_INGEST", "1" if mode == "generic" else "0")
            kv = dict(input_paths=str(d), output_path=str(tmp_path / ("o%d_%s" % (case, mode))), num_blocks=4, num_click_replicates=2, random_seed=case)
            if mapkey:
                kv["map_key"] = mapkey
            rc, err = _run(host, "RegressionPrepare", _write_cfg(str(tmp_path / "c.job"), **kv))
            res.append(err if rc else au.read_dir(kv["output_path"]))
        assert type(res[0]) is type(res[1]) and res[0] == res[1], (case, mapkey, res[0] if isinstance(res[0], str) else "", res[1] if isinstance(res[1], str) else "")
        n_ok += not isinstance(res[0], str)
        n_err += isinstance(res[0], str)
    assert n_ok >= 15 and n_err >= 5, (n_ok, n_err)
