"""Drop-in check: the reference's OWN, unmodified programs - its C++ and C functional tests, its migration sample and its
Python binding with the Python test - built against this repository's headers and run on this library (host backend).
Their sources are not part of this repository: `build()` compiles them into oracle/_ref/tests (oracle/install_ref.sh)
when it finds a reference checkout (__graft_entry__.REFERENCE_SRC); skipped without them."""
import os
import subprocess
import sys

import pytest

from conftest import ROOT

BUILT = os.path.join(ROOT, "oracle", "_ref", "tests")
pytestmark = pytest.mark.skipif(not os.path.exists(os.path.join(BUILT, "mlsl_test")),
                                reason="the reference's test programs are not built (oracle/install_ref.sh)")
MLSLRUN = os.path.join(ROOT, "bin", "mlslrun")


@pytest.fixture(scope="module")
def built(tmp_path_factory):
    d = tmp_path_factory.mktemp("refsrc")
    # the reference's Python binding looks for $MLSL_ROOT/.../libmlsl.so on LD_LIBRARY_PATH: give it this library
    os.makedirs(d / "root" / "intel64" / "lib")
    os.symlink(os.path.join(ROOT, "mlsl_b200", "lib", "libmlsl_b200.so"), d / "root" / "intel64" / "lib" / "libmlsl.so")
    return d


def _run(cmd, extra_env=None, n=4):
    env = dict(os.environ, MLSL_BACKEND="host", MLSL_HEAP_SIZE_GB="0.25", MLSL_WATCHDOG_SEC="60")
    env.update(extra_env or {})
    r = subprocess.run([MLSLRUN, "-n", str(n), "--timeout", "150"] + cmd, env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT,
                       timeout=200)
    return r.returncode, r.stdout.decode("utf-8", "replace")   # the reference prints a non-ASCII byte in its quantisation report


@pytest.mark.parametrize("args", [["1", "0", "0", "0"], ["2", "1", "1", "0"], ["4", "1", "0", "1"], ["2", "0", "1", "1"], ["1", "1", "1", "1"]])
def test_reference_cpp_functional_test(built, args):
    rc, out = _run([os.path.join(BUILT, "mlsl_test")] + args)
    assert rc == 0 and out.count("PASSED") == 144 and "FAILED" not in out, out[-2000:]   # 144: what the reference itself prints


@pytest.mark.parametrize("args", [["1", "0"], ["2", "1"], ["4", "1"], ["2", "0", "1"]])
def test_reference_c_functional_test(built, args):
    rc, out = _run([os.path.join(BUILT, "cmlsl_test")] + args)
    assert rc == 0 and out.count("PASSED") > 100 and "FAILED" not in out, out[-2000:]


def test_reference_sample_and_example(built):
    rc, out = _run([os.path.join(BUILT, "mlsl_sample")])
    assert rc == 0 and "PASSED" in out and "FAILED" not in out, out[-1000:]
    rc, out = _run([os.path.join(BUILT, "mlsl_example"), "2"])
    assert rc == 0 and out.count("exited normally") == 4, out[-1000:]


def test_reference_cpp_functional_test_with_quantization_plugin(built):
    """its quantisation mode asks for dl_comp_* entry points: the sample plug-in exports them"""
    rc, out = _run([os.path.join(BUILT, "mlsl_test"), "1", "0", "0", "0", os.path.join(ROOT, "bin", "libmlsl_quant_sample.so")])
    assert rc == 0 and out.count("PASSED") == 144 and "FAILED" not in out, out[-2000:]


@pytest.mark.parametrize("args", [["1", "0"], ["2", "1"], ["4", "1"]])
def test_reference_python_binding_and_test(built, args):
    root = str(built / "root")
    env = {"MLSL_ROOT": root, "LD_LIBRARY_PATH": os.path.join(root, "intel64", "lib"), "PYTHONPATH": os.path.join(BUILT, "python")}
    rc, out = _run([sys.executable, os.path.join(BUILT, "python", "mlsl_test.py")] + args, env)
    assert rc == 0 and out.count("PASSED") >= 40 and "FAILED" not in out, out[-2000:]
