"""Records what the reference's own kernels compute for the inputs of the GPU tests that compare against them.

    python tests/golden/make_reference_goldens.py [--out DIR]        (on a B200, with oracle/_ref built)

oracle/_ref/libkvbm_kernels_ref.so is the reference's lib/kvbm-kernels/cuda/tensor_kernels.cu compiled unmodified for
sm_100 (`make -C oracle ref`, which needs the reference source tree).  The tests compare this library's kernels with the
files written here, so they run where the reference is not available:

  reference_vectorized_copy_sha256.npy                 [512, 32] uint8: SHA-256 of every output row of K1 on
                                                       tests/test_gpu_kernels.py:reference_copy_case() (16 MiB of output)
  reference_block_from_universal_position_encoded.npy  [2 layouts (NHD, HND), nl*no, chunk] float32: K3 on the
                                                       position-encoded universal tensor
  reference_kernels_dropin.txt                         what tests/c/kernels_dropin.c prints when it runs on the
                                                       reference library
"""
import argparse
import ctypes as C
import os
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

from tests import kats  # noqa: E402
from tests.test_gpu_kernels import (REF_COPY_SHA256, REF_POSITION_BLOCKS, block_from_universal_position_encoded,  # noqa: E402
                                    launch_reference_copy_case, row_sha256)
from tests.test_gpu_zz_c_dropin import REF_OUTPUT, build_dropin, run_dropin  # noqa: E402

REF_SO = os.path.join(ROOT, "oracle", "_ref", "libkvbm_kernels_ref.so")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=HERE)
    out = ap.parse_args().out
    os.makedirs(out, exist_ok=True)
    if not os.path.exists(REF_SO):
        raise SystemExit(f"{REF_SO} is not built (make -C oracle ref, with the reference source tree present)")
    R = C.CDLL(REF_SO)
    R.kvbm_kernels_launch_vectorized_copy.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_int, C.c_void_p]
    R.kvbm_kernels_launch_block_from_universal.argtypes = [C.c_void_p, C.c_void_p] + [C.c_size_t] * 6 + [C.c_int, C.c_int, C.c_void_p]

    theirs, pool, perm, dperm = launch_reference_copy_case(R.kvbm_kernels_launch_vectorized_copy)
    assert bool((theirs[dperm] == pool[perm]).all()), "the reference kernel did not copy"
    np.save(os.path.join(out, os.path.basename(REF_COPY_SHA256)), row_sha256(theirs.cpu().numpy()))

    blocks = np.stack([np.stack(block_from_universal_position_encoded(R.kvbm_kernels_launch_block_from_universal, layout))
                       for layout in (kats.NHD, kats.HND)])
    np.save(os.path.join(out, os.path.basename(REF_POSITION_BLOCKS)), blocks)

    with tempfile.TemporaryDirectory() as tmp:
        exe = os.path.join(tmp, "dropin")
        build_dropin(exe)
        os.symlink(REF_SO, os.path.join(tmp, "libkvbm_kernels.so"))
        rc, text = run_dropin(exe, tmp)
    assert rc == 0, text
    with open(os.path.join(out, os.path.basename(REF_OUTPUT)), "w") as f:
        f.write(text)
    print("wrote", out, blocks.shape)


if __name__ == "__main__":
    main()
