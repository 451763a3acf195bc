"""CPU tests of the host job layer (ml-ease_b200/host): avro codec, job config, RegressionPrepare (pure host),
deterministic partition-id logic bit-exact against the oracle."""
import ctypes as C
import os
import sys

import numpy as np
import pytest

from oracle import oracle as orc

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import avro_util as au  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")


@pytest.fixture(scope="module")
def host():
    import mlease_b200
    mlease_b200.lib()   # loads libmlease_b200.so first
    h = C.CDLL(os.path.join(ROOT, "ml-ease_b200", "lib", "libmlease_host.so"))
    h.mlease_job_last_error.restype = C.c_char_p
    return h


def _run(host, job, cfg_path):
    rc = host.mlease_job_run(job.encode(), cfg_path.encode())
    return rc, host.mlease_job_last_error().decode()


def _write_cfg(path, **kv):
    with open(path, "w") as f:
        f.write("# test job\n")
        for k, v in kv.items():
            f.write("%s=%s\n" % (k.replace("_", "."), v))
    return path


def test_avro_round_trip_python_to_cpp_to_python(host, tmp_path):
    npz = np.load(os.path.join(GOLDEN, "sample_data.npz"))
    recs = au.fixture_records(npz)[:250]
    src = str(tmp_path / "in.avro")
    au.write_avro(src, au.PIG_SCHEMA, recs, codec="deflate", block=37)
    for codec in ("null", "deflate"):
        dst = str(tmp_path / ("out_%s.avro" % codec))
        n, nb = C.c_int64(0), C.c_int64(0)
        assert host.mlease_avro_copy(src.encode(), dst.encode(), codec.encode(), C.byref(n), C.byref(nb)) == 0, host.mlease_job_last_error()
        assert n.value == 250 and nb.value == 7
        _, back, _ = au.read_avro(dst)
        assert back == au.read_avro(src)[1]


def test_cpp_reader_decodes_the_reference_fixture(host, tmp_path):
    """The first 6 blocks of the reference's examples/sample-data.avro as Pig wrote them (tests/golden/make_golden.py)."""
    dst = str(tmp_path / "copy.avro")
    n, nb = C.c_int64(0), C.c_int64(0)
    src = os.path.join(GOLDEN, "sample_data_head.avro")
    assert host.mlease_avro_copy(src.encode(), dst.encode(), b"deflate", C.byref(n), C.byref(nb)) == 0
    assert n.value == 78 and nb.value == 6             # Pig wrote 13 records per block
    _, recs, _ = au.read_avro(dst)
    npz = np.load(os.path.join(GOLDEN, "sample_data.npz"))
    for r in recs:   # the npz keeps each row's features sorted by column id; the file keeps Pig's order
        r["features"].sort(key=lambda f: int(f["name"]))
    assert recs == au.fixture_records(npz)[:78]


def test_prepare_keys_and_partition_ids_bit_exact_vs_oracle(host):
    rng = np.random.default_rng(0)
    n, nblocks, reps = 500, 7, 3
    base = rng.integers(0, nblocks, n).astype(np.int32)
    resp = rng.integers(0, 2, n).astype(np.int32)
    w = rng.uniform(0.1, 3, n)
    vp = C.c_void_p
    for mode in (0, 1):
        keys = np.full((n, reps), -1, np.int32); nk = np.zeros(n, np.int32); ow = np.zeros(n, np.float32)
        assert host.mlease_prepare_keys(C.c_int64(n), base.ctypes.data_as(vp), resp.ctypes.data_as(vp), w.ctypes.data_as(vp), nblocks, reps,
                                        mode, keys.ctypes.data_as(vp), nk.ctypes.data_as(vp), ow.ctypes.data_as(vp)) == 0
        k2, nk2, w2 = orc.prepare(base, resp, w, nblocks, reps, bool(mode))
        np.testing.assert_array_equal(keys, k2); np.testing.assert_array_equal(nk, nk2); np.testing.assert_array_equal(ow, w2)
    names = ["item%d" % i for i in rng.permutation(40)] + ["10", "9", "a#b"]
    lam = np.array([10.0, 0.1, 1.0], np.float32)
    packed = b"".join(s.encode() + b"\0" for s in names)
    ids = np.zeros((3, len(names)), np.int32); part = np.zeros_like(ids); hp = np.zeros_like(ids)
    assert host.mlease_partition_ids(len(names), packed, lam.ctypes.data_as(vp), 3, 5, ids.ctypes.data_as(vp), part.ctypes.data_as(vp),
                                     hp.ctypes.data_as(vp)) == 0
    i2, p2, h2 = orc.partition_ids(names, lam, 5)
    np.testing.assert_array_equal(ids, i2); np.testing.assert_array_equal(part, p2); np.testing.assert_array_equal(hp, h2)
    buf = C.create_string_buffer(64)
    for f in (1.0, 0.1, 100.0, 1e-4, 1e7, 0.001, float(np.float32(0.01) / np.float32(10)), 12345.678):
        host.mlease_java_float_to_string(C.c_float(f), buf, 64)
        assert buf.value.decode() == orc.java_float_to_string(f)


def test_prepare_job_map_key_and_click_replicates(host, tmp_path):
    npz = np.load(os.path.join(GOLDEN, "sample_data.npz"))
    recs = au.fixture_records(npz, with_key=lambda i: i % 4)
    au.write_avro(str(tmp_path / "in" / "part-0.avro"), au.pig_schema_with_key(), recs, block=300)
    # (1) map.key branch: deterministic, bit exact (jobs/RegressionPrepare.java:101-107)
    cfg = _write_cfg(str(tmp_path / "p1.job"), input_paths=str(tmp_path / "in"), output_path=str(tmp_path / "out1"), map_key="pkey", num_blocks=4)
    rc, err = _run(host, "RegressionPrepare", cfg)
    assert rc == 0, err
    out = au.read_dir(str(tmp_path / "out1"))
    assert len(out) == 1000
    for i, (a, b) in enumerate(zip(recs, out)):
        assert b["key"] == str(i % 4) and b["response"] == a["response"] and b["weight"] == 1.0 and b["offset"] == 0.0
        assert [(f["name"], f["term"], np.float32(f["value"])) for f in b["features"]] == [(f["name"], "", np.float32(f["value"])) for f in a["features"]]
    # (2) random-key branch with num.click.replicates: positives appear `reps` times on consecutive partitions, weight / reps
    cfg = _write_cfg(str(tmp_path / "p2.job"), input_paths=str(tmp_path / "in"), output_path=str(tmp_path / "out2"), num_blocks=5,
                     num_click_replicates=3, random_seed=7)
    rc, err = _run(host, "RegressionPrepare", cfg)
    assert rc == 0, err
    out = au.read_dir(str(tmp_path / "out2"))
    npos = int((npz["response"] == 1).sum())
    assert len(out) == 1000 + 2 * npos
    i = 0
    for a in recs:
        if a["response"] == 1:
            ks = [int(out[i + j]["key"]) for j in range(3)]
            assert ks[1] == (ks[0] + 1) % 5 and ks[2] == (ks[1] + 1) % 5
            assert all(out[i + j]["weight"] == np.float32(1 / 3) for j in range(3))
            i += 3
        else:
            assert 0 <= int(out[i]["key"]) < 5 and out[i]["weight"] == 1.0
            i += 1
    # (3) wrong map.key -> the reference's IOException text
    cfg = _write_cfg(str(tmp_path / "p3.job"), input_paths=str(tmp_path / "in"), output_path=str(tmp_path / "out3"), map_key="nope", num_blocks=4)
    rc, err = _run(host, "RegressionPrepare", cfg)
    assert rc != 0 and "map.key is wrongly specified" in err


def test_job_config_errors(host, tmp_path):
    cfg = _write_cfg(str(tmp_path / "a.job"), output_base_path=str(tmp_path / "o"), num_blocks=2, regularizer=3)
    open(cfg, "a").write("lambda : 1,10\n")
    rc, err = _run(host, "RegressionAdmmTrain", cfg)
    assert rc != 0 and "Only L1 and L2 regularization supported!" in err
    rc, err = _run(host, "Nope", cfg)
    assert rc != 0 and "unknown job class" in err
    rc, err = _run(host, "RegressionAdmmTrain", str(tmp_path / "missing.job"))
    assert rc != 0 and "cannot open" in err


def test_corrupt_and_truncated_avro_files_are_errors_not_overruns(host, tmp_path):
    """Every read of file content is bounds-checked (ADVICE r1): a truncated or corrupted container is an error message."""
    npz = np.load(os.path.join(GOLDEN, "sample_data.npz"))
    src = str(tmp_path / "in.avro")
    au.write_avro(src, au.PIG_SCHEMA, au.fixture_records(npz)[:60], block=20)
    raw = open(src, "rb").read()
    n, nb = C.c_int64(0), C.c_int64(0)
    for name, blob in (("trunc_mid", raw[:len(raw) // 2]), ("trunc_tail", raw[:-5]), ("trunc_head", raw[:40]),
                       ("bad_len", raw[:-400] + b"\xff\xff\xff\xff\xff\xff\xff\xff\xff\xff\x7f" + raw[-389:])):
        bad = str(tmp_path / (name + ".avro"))
        open(bad, "wb").write(blob)
        rc = host.mlease_avro_copy(bad.encode(), str(tmp_path / "o.avro").encode(), b"null", C.byref(n), C.byref(nb))
        assert rc != 0, name
        assert "avro" in host.mlease_job_last_error().decode(), name


def test_prepare_key_strings_and_strict_partition_keys_follow_java(host, tmp_path):
    """map.key values print as Java's toString ("1.0" for a float/double 1, not "1.000000"); the `response` field itself must
    exist as an int (Util.getIntAvro, jobs/RegressionPrepare.java:159); AdmmTrain's partition keys go through Integer.parseInt
    (:558): "1.9" or "3abc" are NumberFormatExceptions, not partition 1 / 3."""
    schema = {"type": "record", "name": "r", "fields": [
        {"name": "features", "type": {"type": "array", "items": {"type": "record", "name": "f", "fields": [
            {"name": "name", "type": "string"}, {"name": "term", "type": "string"}, {"name": "value", "type": "float"}]}}},
        {"name": "response", "type": ["null", "int"]}, {"name": "fkey", "type": "double"}, {"name": "gkey", "type": "float"}]}
    recs = [{"features": [{"name": "a", "term": "", "value": 1.0}], "response": i % 2, "fkey": float(i % 3), "gkey": 0.5 + i % 2} for i in range(12)]
    au.write_avro(str(tmp_path / "in" / "p.avro"), schema, recs)
    for mk, expect in (("fkey", ["0.0", "1.0", "2.0"]), ("gkey", ["0.5", "1.5"])):
        cfg = _write_cfg(str(tmp_path / (mk + ".job")), input_paths=str(tmp_path / "in"), output_path=str(tmp_path / ("out_" + mk)), map_key=mk, num_blocks=3)
        rc, err = _run(host, "RegressionPrepare", cfg)
        assert rc == 0, err
        assert sorted({r["key"] for r in au.read_dir(str(tmp_path / ("out_" + mk)))}) == expect
    recs2 = [dict(r, response=None) for r in recs]
    au.write_avro(str(tmp_path / "in2" / "p.avro"), schema, recs2)
    cfg = _write_cfg(str(tmp_path / "nr.job"), input_paths=str(tmp_path / "in2"), output_path=str(tmp_path / "out_nr"), map_key="fkey", num_blocks=3)
    rc, err = _run(host, "RegressionPrepare", cfg)
    assert rc != 0 and ("response" in err)
    # AdmmTrain on prepared data whose keys are "0.0", "1.0", "2.0": rejected before any GPU work
    cfg = _write_cfg(str(tmp_path / "t.job"), input_paths=str(tmp_path / "out_fkey"), output_base_path=str(tmp_path / "o"), num_blocks=3, regularizer=2)
    open(cfg, "a").write("lambda=1\n")
    rc, err = _run(host, "RegressionAdmmTrain", cfg)
    assert rc != 0 and 'For input string: "' in err
