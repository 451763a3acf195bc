"""CPU checks of the C-ABI boundary: the library loads, exports every symbol include/mlease_b200.h declares,
and every compute entry point fails loudly without a CUDA device (no CPU fallback)."""
import ctypes as C
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _has_gpu():
    try:
        import torch
        return torch.cuda.is_available()
    except Exception:
        return False


def test_header_symbols_are_exported():
    import mlease_b200
    from mlease_b200._native import EXPORTED, SO_PATH
    hdr = open(os.path.join(ROOT, "include", "mlease_b200.h")).read()
    declared = sorted(set(re.findall(r"\b(mlease_[a-z_0-9]+)\s*\(", hdr)) - {"mlease_allreduce_fn"})
    lib = C.CDLL(SO_PATH)
    missing = [s for s in declared if not hasattr(lib, s)]
    assert not missing, missing
    assert sorted(EXPORTED) == declared, (sorted(set(declared) ^ set(EXPORTED)))
    assert mlease_b200.lib().mlease_abi_version() == 2


@pytest.mark.skipif(_has_gpu(), reason="checks the no-GPU failure mode")
def test_no_cpu_fallback():
    import mlease_b200 as mb
    with pytest.raises(mb.MleaseError, match="no CPU fallback"):
        mb.AdmmSession(2, 10, [1.0])
    with pytest.raises(mb.MleaseError, match="no CPU fallback"):
        mb.score(np.zeros((2, 3), np.float32), np.zeros(4))
    with pytest.raises(mb.MleaseError, match="no CPU fallback"):
        mb.test_loglik([1, 0], [0.1, 0.2])
    with pytest.raises(mb.MleaseError, match="no CPU fallback"):
        mb.naive_train_dense(np.zeros((4, 3), np.float32), [0, 4], [1, 0, 1, 0], 1.0)


def test_config_validation_happens_before_device_use():
    import mlease_b200 as mb
    with pytest.raises(mb.MleaseError, match="Only L1 and L2"):
        mb.AdmmSession(2, 10, [1.0], regularizer=7)
    if not _has_gpu():   # regularizer = 1 (L1 z-update) is a valid config: it gets as far as the device check
        with pytest.raises(mb.MleaseError, match="no CPU fallback"):
            mb.AdmmSession(2, 10, [1.0], regularizer=1)


def test_product_package_never_imports_the_oracle():
    """Nothing under ml-ease_b200/ may import, link or execute anything under oracle/."""
    pkg = os.path.join(ROOT, "ml-ease_b200")
    bad = re.compile(r"(import\s+oracle|from\s+oracle|mlease_oracle|oracle/|orc_[a-z_]+\()")
    for dp, _, fs in os.walk(pkg):
        for f in fs:
            if f.endswith((".py", ".cu", ".cuh", ".h", ".hpp", ".cpp")):
                txt = open(os.path.join(dp, f), errors="ignore").read()
                assert not bad.search(txt), os.path.join(dp, f)


def test_device_library_reads_only_known_environment_variables():
    """The device library takes no tuning switches from the environment: one test hook (segment lists off, so the per-problem
    CSR K1 kernels run) and two diagnostics that only print.  A code path selected by an environment variable is a path
    that neither the tests nor the benchmark run."""
    csrc = os.path.join(ROOT, "ml-ease_b200", "csrc")
    names = set()
    for f in os.listdir(csrc):
        names |= set(re.findall(r'getenv\(\s*"([^"]+)"', open(os.path.join(csrc, f)).read()))
    assert names == {"MLEASE_NO_FUSED_K1", "MLEASE_DEBUG", "MLEASE_UPLOAD_TRACE"}, sorted(names)


def test_tools_and_bench_scripts_parse():
    """The GPU-side scripts cannot run here, but they must at least be valid Python and bench.py must keep its CLI contract."""
    import ast
    import glob
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    for path in glob.glob(os.path.join(root, "tools", "*.py")) + [os.path.join(root, "bench.py"), os.path.join(root, "__graft_entry__.py")]:
        ast.parse(open(path).read(), filename=path)
    out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--help"], capture_output=True, text=True, timeout=120)
    assert out.returncode == 0
    for flag in ("--gpus", "--steps", "--warmup", "--impl"):
        assert flag in out.stdout


def test_headers_are_plain_c99(tmp_path):
    """The drop-in boundary is a C ABI: both headers compile as C99 (what cgo / JNI shims / ctypes-generators include)."""
    import subprocess
    src = tmp_path / "hc.c"
    src.write_text('#include "mlease_b200.h"\n#include "mlease_host.h"\nint main(void) { return 0; }\n')
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Wextra", "-pedantic", "-Werror", "-I", os.path.join(ROOT, "include"), "-fsyntax-only", str(src)])


def test_jni_shim_type_checks_links_and_matches_the_java_class(tmp_path):
    """integration/jni/: the reference-side binding (INTEGRATION.md section 2).  No JDK here, so the C shim is compiled as pedantic C99
    against a stub jni.h carrying the JNI specification's signatures and linked against libmlease_b200.so / libmlease_host.so with no undefined symbols
    (it cannot drift from the header); its exported natives are exactly the `native` methods NativeAdmm.java declares."""
    import re
    import subprocess
    from mlease_b200 import build as _b
    _b.build()
    so = str(tmp_path / "libjni_check.so")
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Wextra", "-pedantic", "-Werror", "-fPIC", "-shared", "-I", os.path.join(ROOT, "tests", "jni_stub"),
                           "-I", os.path.join(ROOT, "include"), os.path.join(ROOT, "integration", "jni", "mlease_b200_jni.c"),
                           "-L", os.path.join(ROOT, "ml-ease_b200", "lib"), "-lmlease_host", "-lmlease_b200", "-Wl,--no-undefined", "-o", so])
    syms = subprocess.run(["nm", "-D", "--defined-only", so], capture_output=True, text=True, check=True).stdout
    for cls, count in (("NativeAdmm", 13), ("NativeOps", 3), ("NativeIngest", 6)):
        exported = set(re.findall(r"Java_com_linkedin_mlease_regression_gpu_" + cls + r"_(\w+)", syms))
        java = open(os.path.join(ROOT, "integration", "jni", cls + ".java")).read()
        declared = set(re.findall(r"\bnative\s+[\w\[\]]+\s+(\w+)\s*\(", java))
        assert exported == declared and len(declared) == count, (cls, sorted(exported ^ declared))


def test_jni_shim_runs_against_a_fake_jnienv_and_the_device_test_double(tmp_path):
    """The shim is also EXECUTED: tests/jni_stub/run_shim.c implements the JNIEnv entries it uses (arrays handed out as copies, so a
    result reaches the caller only if the shim releases it with mode 0) and drives NativeAdmm / NativeOps against the test double of
    the device library (tests/fake_device/), comparing with direct C ABI calls, and NativeIngest against an avro file."""
    import subprocess
    import sys
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import avro_util as au
    import numpy as np
    from mlease_b200 import build as _b
    _b.build()
    exe = str(tmp_path / "run_shim")
    lib = os.path.join(ROOT, "ml-ease_b200", "lib")
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Wextra", "-Werror", "-O1", "-I", os.path.join(ROOT, "tests", "jni_stub"), "-I", os.path.join(ROOT, "include"), "-o", exe,
                           os.path.join(ROOT, "tests", "jni_stub", "run_shim.c"), os.path.join(ROOT, "integration", "jni", "mlease_b200_jni.c"),
                           os.path.join(ROOT, "tests", "fake_device", "fake_mlease_b200.c"), "-L", lib, "-lmlease_host", "-lmlease_b200", "-Wl,-rpath," + lib, "-lm"])
    schema = {"type": "record", "name": "RegressionPrepareOutput", "fields": [
        {"name": "key", "type": "string"}, {"name": "response", "type": "int"},
        {"name": "features", "type": {"type": "array", "items": {"type": "record", "name": "feature", "fields": [
            {"name": "name", "type": "string"}, {"name": "term", "type": "string"}, {"name": "value", "type": "float"}]}}},
        {"name": "weight", "type": "float"}, {"name": "offset", "type": "float"}]}
    recs = [{"key": str(i % 2), "response": i % 2, "features": [{"name": "f%d" % ((i + j) % 5), "term": "", "value": 1.0} for j in range(3)], "weight": 1.0, "offset": 0.0}
            for i in range(20)]
    p = str(tmp_path / "prep.avro")
    au.write_avro(p, schema, recs, block=6)
    out = subprocess.run([exe, p, "20", "60", "5", "f0"], capture_output=True, text=True)
    assert out.returncode == 0 and "JNI shim OK" in out.stdout, out.stdout + out.stderr
