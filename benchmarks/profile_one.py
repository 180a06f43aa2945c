"""Launches ONE variant of the config-2 same-GPU transfer a few times (for ncu captures).

    ncu --set full -k regex:kvbm -c 2 python benchmarks/profile_one.py --which ours
    which: ours | ours:<warps>,<stages>,<tile>[,<pending>[,<ctas>]] | simt | k1 | ref | torch
"""
import argparse
import ctypes as C
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from dynamo_b200 import kernels as K  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--which", default="ours")
ap.add_argument("--iters", type=int, default=3)
ap.add_argument("--blocks", type=int, default=256)
ap.add_argument("--pool", type=int, default=1024)
a = ap.parse_args()
torch.cuda.set_device(0)
nl, nbp, n, region = 32, a.pool, a.blocks, 32768


def pool():
    bufs = [torch.empty(2 * nbp * region, dtype=torch.uint8, device="cuda") for _ in range(nl)]
    base = torch.tensor([b.data_ptr() for b in bufs], dtype=torch.int64, device="cuda")
    return bufs, base, K.PagedLayout(base.data_ptr(), region, region * nbp, region, nl, 2, nbp)


sb, sbase, src = pool()
db, dbase, dst = pool()
for t in sb:
    t.random_(0, 256)
sid = torch.from_numpy(np.random.default_rng(0).permutation(nbp)[:n].astype(np.int32)).cuda()
did = torch.from_numpy(np.random.default_rng(1).permutation(nbp)[:n].astype(np.int32)).cuda()
d = K.PagedDst(dst, sid.data_ptr(), did.data_ptr(), 0, 0)
sp = int(torch.cuda.current_stream().cuda_stream)
ptr_s = torch.tensor([sb[l].data_ptr() + o * region * nbp + int(b) * region for b in sid.tolist() for l in range(nl) for o in range(2)], dtype=torch.int64, device="cuda")
ptr_d = torch.tensor([db[l].data_ptr() + o * region * nbp + int(b) * region for b in did.tolist() for l in range(nl) for o in range(2)], dtype=torch.int64, device="cuda")
torch.cuda.synchronize()
w = a.which
if w == "torch":
    big_a = torch.empty(n * nl * 2 * region, dtype=torch.uint8, device="cuda")
    big_b = torch.empty_like(big_a)
    torch.cuda.synchronize()
torch.cuda.cudart().cudaProfilerStart()   # use with: ncu --profile-from-start off
for _ in range(a.iters):
    if w.startswith("ours"):
        opts = K.PagedCopyOpts()
        if ":" in w:
            v = [int(x) for x in w.split(":")[1].split(",")]
            opts = K.PagedCopyOpts(warps_per_cta=v[0], stages=v[1], tile_bytes=v[2], stores_in_flight=v[3] if len(v) > 3 else 0, max_ctas=v[4] if len(v) > 4 else 0)
        K.check(K.paged_copy(src, [d], n, 0, nl, 0, opts, sp))
    elif w == "simt":
        K.check(K.paged_copy(src, [d], n, 0, nl, 0, K.PagedCopyOpts(force_simt=1), sp))
    elif w == "k1":
        K.check(K.vectorized_copy(ptr_s.data_ptr(), ptr_d.data_ptr(), region, ptr_s.numel(), sp))
    elif w == "ref":
        R = C.CDLL(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "oracle", "_ref", "libkvbm_kernels_ref.so"))
        R.kvbm_kernels_launch_vectorized_copy.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_int, C.c_void_p]
        assert R.kvbm_kernels_launch_vectorized_copy(ptr_s.data_ptr(), ptr_d.data_ptr(), region, ptr_s.numel(), sp) == 0
    else:
        big_b.copy_(big_a)
    torch.cuda.synchronize()
torch.cuda.cudart().cudaProfilerStop()
print("done", w)
