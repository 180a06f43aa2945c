"""Geometry sweep of the paged-copy kernel on one GPU (same-device gather->scatter, HBM bound).

    python benchmarks/sweep.py [--blocks 256] [--out gpurun_out/sweep.json]

Times config 2's workload (Llama-3-8B bf16, 4k ctx: 256 blocks x 32 layers x K/V x 32 KiB = 512 MiB,
vLLM layer-separate pools of 1024 blocks, random block tables) for several (warps, stages, tile, ctas)
and prints GB/s of algorithmic bytes moved (read + write) next to torch's copy_ on the same volume.
Also times the reference's own K1 kernel (oracle/_ref) driven like executor/cuda.rs:234-327 if present.
"""
import argparse
import ctypes as C
import json
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from dynamo_b200 import kernels as K  # noqa: E402


def timed(fn, iters=20, warm=5, flush=None):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(iters):
        if flush is not None:
            flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        e1.synchronize()
        ts.append(e0.elapsed_time(e1))
    return float(np.median(ts)), float(np.min(ts))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--blocks", type=int, default=256)
    ap.add_argument("--pool", type=int, default=1024)
    ap.add_argument("--layers", type=int, default=32)
    ap.add_argument("--inner", type=int, default=1024)
    ap.add_argument("--out", default="gpurun_out/sweep.json")
    ap.add_argument("--peer", action="store_true", help="destination pool on cuda:1 (NVLink peer stores)")
    ap.add_argument("--pull", action="store_true", help="with --peer: SOURCE pool on cuda:1, kernel on cuda:0 reads over NVLink")
    ap.add_argument("--fine", action="store_true", help="second-round sweep: CTA count x ring shape")
    a = ap.parse_args()
    torch.cuda.set_device(0)
    ddev = "cuda:0"
    if a.peer:
        from dynamo_b200.physical import TransferManager
        _m = TransferManager(device=0)
        _m.enable_peer_access(1)
        ddev = "cuda:1"
    nl, nbp, n = a.layers, a.pool, a.blocks
    region = 16 * a.inner * 2

    def pool(dev="cuda:0"):
        bufs = [torch.empty(2 * nbp * region, dtype=torch.uint8, device=dev) for _ in range(nl)]
        base = torch.tensor([b.data_ptr() for b in bufs], dtype=torch.int64, device="cuda:0")
        return bufs, base, K.PagedLayout(base.data_ptr(), region, region * nbp, region, nl, 2, nbp)

    sb, sbase, src = pool(ddev if a.pull else "cuda:0")
    db, dbase, dst = pool("cuda:0" if a.pull else ddev)
    for t in sb:
        t.random_(0, 256)
    sid = torch.from_numpy(np.random.default_rng(0).permutation(nbp)[:n].astype(np.int32)).cuda()
    did = torch.from_numpy(np.random.default_rng(1).permutation(nbp)[:n].astype(np.int32)).cuda()
    d = K.PagedDst(dst, sid.data_ptr(), did.data_ptr(), 0, 0)
    sp = int(torch.cuda.current_stream().cuda_stream)
    bytes_moved = n * nl * 2 * region
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    results = []

    big_a = torch.empty(bytes_moved, dtype=torch.uint8, device="cuda:0")
    big_b = torch.empty(bytes_moved, dtype=torch.uint8, device=ddev)
    med, best = timed(lambda: big_b.copy_(big_a), flush=flush)
    results.append(dict(name="torch.copy_", ms=med, gbs_rw=2 * bytes_moved / med / 1e6))
    print(results[-1], flush=True)

    cfgs = [  # (warps, stages, pending stores, tile, ctas)
        (4, 3, 1, 16384, 0), (2, 3, 1, 32768, 0), (8, 3, 1, 8192, 0), (4, 6, 3, 8192, 0),
        (6, 2, 1, 16384, 0), (3, 2, 1, 32768, 0), (12, 2, 1, 8192, 0), (16, 3, 1, 4096, 0),
        (4, 3, 1, 16384, 74), (4, 3, 1, 16384, 32), (4, 3, 1, 16384, 16),
    ]
    if a.fine:
        cfgs = []
        for shape in [(4, 3, 1, 16384), (4, 6, 3, 8192), (2, 3, 1, 32768), (8, 3, 1, 8192), (2, 6, 3, 16384), (4, 4, 2, 8192)]:
            for ctas in (64, 74, 96, 111, 128, 148):
                cfgs.append((*shape, ctas))
    if a.peer:   # NVLink-bound: how few SMs saturate the link, and how many stores must be in flight
        cfgs = [(4, 3, 1, 16384, 0), (4, 6, 3, 8192, 0), (4, 6, 5, 8192, 0), (2, 6, 4, 16384, 0),
                (4, 3, 1, 16384, 74), (4, 3, 1, 16384, 32), (4, 3, 1, 16384, 16), (4, 3, 1, 16384, 8),
                (4, 6, 4, 8192, 32), (4, 6, 4, 8192, 16), (4, 6, 4, 8192, 8), (2, 6, 4, 16384, 16),
                (2, 6, 4, 16384, 8), (4, 12, 10, 4096, 16), (4, 3, 2, 16384, 16), (1, 6, 4, 32768, 16), (1, 6, 4, 32768, 32)]
    for warps, stages, pend, tile, ctas in cfgs:
        opts = K.PagedCopyOpts(warps_per_cta=warps, stages=stages, tile_bytes=tile, max_ctas=ctas, stores_in_flight=pend)
        rc = K.paged_copy(src, [d], n, 0, nl, 0, opts, sp)
        if rc != 0:
            print("rc", rc, warps, stages, tile)
            continue
        med, best = timed(lambda: K.paged_copy(src, [d], n, 0, nl, 0, opts, sp), flush=flush)
        results.append(dict(name="paged_tma", warps=warps, stages=stages, pending=pend, tile=tile, ctas=ctas,
                            ms=med, ms_min=best, gbs_rw=2 * bytes_moved / med / 1e6))
        print(results[-1], flush=True)
    opts = K.PagedCopyOpts(force_simt=1)
    med, best = timed(lambda: K.paged_copy(src, [d], n, 0, nl, 0, opts, sp), flush=flush)
    results.append(dict(name="paged_simt", ms=med, gbs_rw=2 * bytes_moved / med / 1e6))
    print(results[-1], flush=True)

    # legacy ABI (pointer tables) ours vs the reference kernel
    ptr_s = torch.tensor([sb[l].data_ptr() + o * region * nbp + int(b) * region for b in sid.tolist() for l in range(nl) for o in range(2)],
                         dtype=torch.int64, device="cuda")
    ptr_d = torch.tensor([db[l].data_ptr() + o * region * nbp + int(b) * region for b in did.tolist() for l in range(nl) for o in range(2)],
                         dtype=torch.int64, device="cuda")
    npairs = ptr_s.numel()
    med, best = timed(lambda: K.vectorized_copy(ptr_s.data_ptr(), ptr_d.data_ptr(), region, npairs, sp), flush=flush)
    results.append(dict(name="ours_K1_abi", ms=med, gbs_rw=2 * bytes_moved / med / 1e6))
    print(results[-1], flush=True)
    ref = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "oracle", "_ref", "libkvbm_kernels_ref.so")
    if os.path.exists(ref):
        R = C.CDLL(ref)
        R.kvbm_kernels_launch_vectorized_copy.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_int, C.c_void_p]
        med, best = timed(lambda: R.kvbm_kernels_launch_vectorized_copy(ptr_s.data_ptr(), ptr_d.data_ptr(), region, npairs, sp), flush=flush)
        results.append(dict(name="reference_K1_sm100", ms=med, gbs_rw=2 * bytes_moved / med / 1e6))
        print(results[-1], flush=True)
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    json.dump(results, open(a.out, "w"), indent=1)


if __name__ == "__main__":
    main()
