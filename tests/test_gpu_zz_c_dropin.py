"""The literal drop-in (INTEGRATION.md §1, lib/kvbm-kernels/cuda/stubs.c:4-7): ONE C binary built against the six reference
symbols runs with this repo's libkvbm_kernels.so and must print the same bytes it printed with the reference's own kernels
compiled unmodified under the same file name (stored in tests/golden/ by tests/golden/make_reference_goldens.py).  No
Python in the data path."""
import os
import shutil
import subprocess

import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CUDA = "/usr/local/cuda"
REF_OUTPUT = os.path.join(ROOT, "tests", "golden", "reference_kernels_dropin.txt")


def build_dropin(exe):
    """Compiles tests/c/kernels_dropin.c to `exe`, linked against this repo's libkvbm_kernels.so by file name."""
    gcc = shutil.which("gcc")
    if not gcc or not os.path.exists(os.path.join(CUDA, "lib64", "libcudart.so")):
        pytest.skip("gcc or libcudart are not installed")
    r = subprocess.run([gcc, "-std=c99", "-Wall", "-I", os.path.join(CUDA, "include"), os.path.join(ROOT, "tests", "c", "kernels_dropin.c"),
                        "-o", str(exe), "-L", os.path.join(ROOT, "dynamo_b200"), "-lkvbm_kernels", "-L", os.path.join(CUDA, "lib64"), "-lcudart"],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr


def run_dropin(exe, libdir):
    """Runs `exe` with the libkvbm_kernels.so found in `libdir`; returns (exit code, output)."""
    env = dict(os.environ, LD_LIBRARY_PATH=f"{libdir}:{os.path.join(CUDA, 'lib64')}:" + os.environ.get("LD_LIBRARY_PATH", ""))
    p = subprocess.run([str(exe)], capture_output=True, text=True, env=env, timeout=120)
    return p.returncode, p.stdout + p.stderr


def test_same_binary_same_output_with_either_library(tmp_path):
    exe = tmp_path / "dropin"
    build_dropin(exe)
    rc, out = run_dropin(exe, os.path.join(ROOT, "dynamo_b200"))
    assert rc == 0 and out.strip().endswith("done") and "k3_roundtrip 1" in out, out
    assert "k1_edges 0 0 1" in out and "k4_edges 0 1" in out and "k2_bad_dtype 1" in out, out
    with open(REF_OUTPUT) as f:
        ref = f.read()
    assert out == ref, f"ours:\n{out}\nreference:\n{ref}"
