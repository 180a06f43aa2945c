#!/usr/bin/env python
"""bench.py -- KV-cache transfer GB/s (+ decode TTFT delta) for the prefill->decode hand-off.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Workload = BASELINE.json configs[1]: Llama-3-8B bf16, 4 k-token context, paged KV block_size=16
  -> 256 blocks x 32 layers x {K,V} x 32 KiB regions = 512 MiB per destination, random (non-contiguous)
  block tables on both sides, vLLM layer-separate pools ([2, num_blocks, 16, 8, 128] per layer).
A "step" is one gather -> NVLink -> scatter of that request's KV.

  N = 1      source and destination pools on the same GPU (HBM-bound: 512 MiB read + 512 MiB written)
  N > 1      rank 0 = prefill GPU, ranks 1..N-1 = decode GPUs, one process per GPU, pools mapped into each other through
             CUDA IPC.  --direction pull (default): every decode GPU launches the transfer kernel itself and READS its
             blocks from the prefill pool over NVLink (the decode-side READ of vLLM's NixlConnector); --direction push:
             rank 0 launches ONE kernel that stores to all decode pools (measured: SM-issued peer stores cap at 706 GB/s
             per destination, peer loads reach 775; profiles/r02_copylab_{push,pull}.jsonl).

  value      GB/s of destination bytes, kernel launched through the C ABI with block tables already in HBM; K launches back
             to back, each bracketed by its own pair of CUDA events: the step time is the MEDIAN of the K per-launch device
             times (max over ranks); total / K of the same K steps is kept too (`ms_per_step_mean`)
  e2e        same metric through the host API (TransferManager.execute_transfer / execute_fanout): block tables arrive as
             HOST lists every step, are uploaded inside the timed region, and the step ends when the host observes the
             completion word the kernel writes back.  (KV pages are device-resident by definition of the path.)
  parity     EVERY moved region on EVERY destination is compared on the device with the bytes the source must have held
             (closed-form pattern; the cast through the golden fp8->bf16 table of tests/golden), and every block that was
             not a destination must still be zero.  A mismatch makes the run exit non-zero.
  gpu_baselines   the reference's GPU paths on the same pools, outside the timed regions (rank 0): its own K1 kernel driven
             like kvbm-physical executor/cuda.rs:234-327, per-chunk cudaMemcpyAsync (v1 D2D), the driver's batched memcpy
             (K4), one contiguous copy (the DMA ceiling), the two-hop GPU->pinned->GPU plan.
  --impl reference   the reference's own CPU path for this hand-off (execute_memcpy_transfer,
             lib/kvbm-physical/src/transfer/executor/memcpy.rs:30-165, restated in oracle/kvbm_oracle.c because no Rust
             toolchain exists here) on the host cores, same workload, same pool size.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True   # the benchmark leaves the tree as it found it (it may be read-only)

import numpy as np  # noqa: E402

# ---- workload geometry; defaults = BASELINE configs[1] (Llama-3-8B, bf16, block_size 16, 4k ctx) ----
NL, OUTER, PAGE, KV_HEADS, HEAD_DIM, DTYPE_BYTES = 32, 2, 16, 8, 128, 2
INNER = KV_HEADS * HEAD_DIM
REGION = PAGE * INNER * DTYPE_BYTES          # 32 KiB (destination side)
SRC_REGION = REGION                          # differs only with --cast fp8 (16 KiB fp8 source regions)
CTX_TOKENS = 4096
N_BLOCKS = CTX_TOKENS // PAGE                # 256
POOL_BLOCKS = 1024                           # pool per GPU: 1024 blocks = 2 GiB (transfer touches 512 MiB of it)
BYTES_PER_DST = N_BLOCKS * NL * OUTER * REGION
MODEL_NAME = "Llama-3-8B bf16"
CAST = 0
REPLICATE = False
NVLS = False
TOPOLOGY = "fanout"
DIRECTION = "pull"


def configure(args):
    """Non-default workloads (other BASELINE configs) for the numbers under profiles/; the driver uses defaults."""
    global NL, KV_HEADS, INNER, REGION, SRC_REGION, CTX_TOKENS, N_BLOCKS, POOL_BLOCKS, BYTES_PER_DST, MODEL_NAME, CAST
    global REPLICATE, NVLS, TOPOLOGY, DIRECTION
    if args.model == "llama70b-tp4":       # configs[3]: 80 layers, 2 of 8 KV heads per rank -> 8 KiB regions
        NL, KV_HEADS, MODEL_NAME = 80, 2, "Llama-3-70B TP=4 shard bf16"
    elif args.model == "mixtral":          # configs[4]: same KV geometry as Llama-3-8B
        MODEL_NAME = "Mixtral-8x7B bf16"
    INNER = KV_HEADS * HEAD_DIM
    REGION = PAGE * INNER * DTYPE_BYTES
    SRC_REGION = REGION
    if args.cast == "fp8":                 # configs[2]: fp8 KV source, bf16 destination, cast fused in the kernel
        CAST, SRC_REGION, MODEL_NAME = 1, REGION // 2, MODEL_NAME.replace("bf16", "fp8->bf16")
    CTX_TOKENS = args.ctx
    N_BLOCKS = CTX_TOKENS // PAGE
    POOL_BLOCKS = args.pool_blocks or max(1024, 2 * N_BLOCKS)
    BYTES_PER_DST = N_BLOCKS * NL * OUTER * REGION
    REPLICATE = args.replicate
    NVLS = bool(args.nvls) and args.replicate and args.gpus > 1
    TOPOLOGY = args.topology
    DIRECTION = args.direction
    if args.gpus == 1 or NVLS or REPLICATE:
        DIRECTION = "push"                 # one payload read once and stored N times is a source-side operation


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, copy read+write)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


NVLINK_PEER_GBS_GUIDE = 770.0   # B200_PROFILING.md: measured peer copy per direction on this pool; nominal 900


class ClockSampler:
    """nvidia-smi clocks/throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def wait_first_sample(self, timeout_s):
        t0 = time.time()
        while self.proc and not self.rows and time.time() - t0 < timeout_s:
            time.sleep(0.005)

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1]))
                mx.append(float(r[2]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# =====================================================================================================
# reference arm / cpu_baseline: the reference's CPU path (oracle port), host cores
# =====================================================================================================
def numa_interleave():
    """MPOL_INTERLEAVE over every NUMA node for the pages allocated from here on (what `numactl --interleave=all` does).
    Without it the whole pool lands on the node of the allocating thread and the all-cores figure swings 2x between boxes."""
    try:
        nodes = sorted(int(d[4:]) for d in os.listdir("/sys/devices/system/node") if d.startswith("node") and d[4:].isdigit())
        if len(nodes) < 2:
            return f"{len(nodes)} NUMA node"
        mask = 0
        for n in nodes:
            mask |= 1 << n
        libc = C.CDLL(None, use_errno=True)
        m = C.c_ulong(mask)
        rc = libc.syscall(238, 3, C.byref(m), C.c_ulong(max(nodes) + 2))   # SYS_set_mempolicy, MPOL_INTERLEAVE
        return f"pages interleaved over {len(nodes)} NUMA nodes" if rc == 0 else f"set_mempolicy failed (errno {C.get_errno()})"
    except Exception as e:   # pragma: no cover
        return f"NUMA policy unavailable ({type(e).__name__})"


def cpu_path(steps, warmup, threads):
    """Times execute_memcpy_transfer on host memory for the same request and the SAME pool size as the GPU arm."""
    from oracle import oracle as O
    mk = lambda: O.Layout(O.LW, POOL_BLOCKS, NL, OUTER, PAGE, INNER, DTYPE_BYTES, block_dim=O.BLOCK_IS_SECOND_DIM)
    src, dst = mk(), mk()
    rng = np.random.default_rng(1234)
    for b in src.buffers:   # touch every page once with non-trivial bytes
        b[:] = rng.integers(0, 256, 4096, dtype=np.uint8).repeat(b.size // 4096)
    for b in dst.buffers:
        b[:] = 1
    sid = np.random.default_rng(10).permutation(POOL_BLOCKS)[:N_BLOCKS]
    did = np.random.default_rng(100).permutation(POOL_BLOCKS)[:N_BLOCKS]
    times = []
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        O.execute_memcpy_transfer(src, dst, sid, did, nthreads=threads)
        dt = time.perf_counter() - t0
        if i >= warmup:
            times.append(dt)
    ok = all(dst.block_checksum(int(d)) == src.block_checksum(int(s)) for s, d in zip(sid[:8], did[:8]))
    return times, ok


def host_threads():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    cores = host_threads()
    numa = numa_interleave()
    t1, ok1 = cpu_path(2, 1, 1)
    times, ok = cpu_path(args.steps, args.warmup, cores)
    med = statistics.median(times)
    gbs = BYTES_PER_DST / med / 1e9
    v1 = BYTES_PER_DST / statistics.median(t1) / 1e9
    line = {
        "impl": "reference", "metric": "kv_transfer_gbs", "value": round(gbs, 3), "unit": "GB/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(1e3 * med, 4),
        "ms_per_step_mean": round(1e3 * sum(times) / len(times), 4),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": workload_config(args.gpus),
        "cpu_baseline": {"value": round(gbs, 3), "unit": "GB/s", "cores": cores, "kind": "port", "single_thread_value": round(v1, 3),
                         "sample": f"{len(times)} x the full {N_BLOCKS}-block/{BYTES_PER_DST >> 20} MiB request (median), execute_memcpy_transfer "
                                   f"restated in C (oracle/kvbm_oracle.c), {cores} pinned threads over the chunk list, {numa}; the "
                                   f"reference's own loop is single-threaded: {v1:.2f} GB/s on 1 core; bit-exact={ok and ok1}"},
        "e2e": {"value": round(gbs, 3), "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)
    return 0


def workload_config(n_gpus):
    if n_gpus == 1:
        topo = "same-GPU gather->scatter"
    elif TOPOLOGY == "pairs":
        topo = f"{n_gpus // 2} x (1 prefill -> 1 decode) rank pairs, {DIRECTION} over CUDA IPC mappings"
    elif NVLS:
        topo = f"1 prefill -> {n_gpus - 1} decode GPUs, ONE write per tile to an NVLink multicast mapping (NVLS; the switch fans out)"
    elif DIRECTION == "pull":
        topo = f"1 prefill -> {n_gpus - 1} decode GPUs; every decode GPU pulls its blocks (NVLink peer loads via CUDA IPC mappings)"
    else:
        topo = f"1 prefill -> {n_gpus - 1} decode GPUs (NVLink peer stores via CUDA IPC mappings)"
    return {"workload": f"{MODEL_NAME} KV hand-off, {CTX_TOKENS // 1024}k ctx, block_size={PAGE}: {N_BLOCKS} blocks x {NL} layers x K/V x "
                        f"{REGION // 1024} KiB = {BYTES_PER_DST / 2**20:.0f} MiB per destination" + (" (identical payload to every destination)" if REPLICATE else ""),
            "topology": topo, "direction": DIRECTION if n_gpus > 1 else "local",
            "layout": "LayerSeparate/BlockIsSecondDim (vLLM [2,num_blocks,16,8,128] per layer)",
            "pool_blocks": POOL_BLOCKS,
            "block_tables": "random permutation (seeded), non-contiguous on both sides",
            "cache": f"inputs larger than L2 ({(BYTES_PER_DST + BYTES_PER_DST * SRC_REGION // REGION) / 2**20:.0f} MiB touched per step vs 126 MB L2), no flush needed",
            "bytes_per_destination": BYTES_PER_DST}


# =====================================================================================================
# closed-form pool contents: every rank can say what ANY source region holds without talking to the source
# =====================================================================================================
def pattern_terms(torch, dev, region):
    i = torch.arange(region, dtype=torch.int64, device=dev)
    a = (i * 131 + (i >> 8) * 17 + (i >> 13) * 5).to(torch.uint8)                    # [region]
    b = (torch.arange(POOL_BLOCKS, dtype=torch.int64, device=dev) * 7919 // 3).to(torch.uint8)   # [pool]
    return a, b


def pattern_const(layer, outer):
    return (layer * 37 + outer * 101 + 11) & 255


def fill_source(torch, bufs, dev, region):
    a, b = pattern_terms(torch, dev, region)
    for l, buf in enumerate(bufs):
        v = buf.view(OUTER, POOL_BLOCKS, region)
        for o in range(OUTER):
            torch.add(a[None, :], b[:, None], out=v[o])          # uint8 arithmetic wraps mod 256
            v[o] += pattern_const(l, o)


def verify_destination(torch, dst_bufs, dev, sid, did, cast, lut=None, src_region=None):
    """Compares every moved region of this destination with what the source held; returns (regions checked, mismatching
    regions, untouched blocks that changed)."""
    a, b = pattern_terms(torch, dev, src_region or SRC_REGION)
    s = torch.as_tensor(np.asarray(sid, dtype=np.int64), device=dev)
    d = torch.as_tensor(np.asarray(did, dtype=np.int64), device=dev)
    untouched = torch.ones(POOL_BLOCKS, dtype=torch.bool, device=dev)
    untouched[d] = False
    keep = untouched.nonzero().flatten()
    bad = changed = checked = 0
    for l, buf in enumerate(dst_bufs):
        v = buf.view(OUTER, POOL_BLOCKS, REGION)
        for o in range(OUTER):
            want = a[None, :] + b[s][:, None] + pattern_const(l, o)               # [n_blocks, src_region] uint8
            got = v[o].index_select(0, d)
            if cast:
                want = lut[want.long()]                                              # int16 bf16 bit patterns
                got = got.view(torch.int16)
            bad += int((want != got).any(dim=1).sum().item())
            checked += int(s.numel())
            changed += int(v[o].index_select(0, keep).any(dim=1).sum().item())
    return checked, bad, changed


def golden_lut(torch, dev):
    t = np.load(os.path.join(ROOT, "tests", "golden", "fp8_e4m3_to_bf16_torch.npy"))
    return torch.as_tensor(t.astype(np.uint16).view(np.int16).copy(), device=dev)


DUMP_SAMPLES = 4 << 20   # bytes sampled over all destinations: 16 MiB of float32 per run


def dump_destination(torch, out_dir, name, dst_bufs, dev, did, n_samples):
    """Writes out_dir/<name>.npy: a fixed, seeded sample of the bytes this destination received, read the way its owner
    reads them (layer, K/V, position in the block table, byte), each byte as a float32 in 0..255."""
    per_layer = OUTER * N_BLOCKS * REGION
    idx = np.sort(np.random.default_rng(7).integers(0, NL * per_layer, n_samples, dtype=np.int64))
    layer, rest = np.divmod(idx, per_layer)
    outer, rest = np.divmod(rest, N_BLOCKS * REGION)
    j, byte = np.divmod(rest, REGION)
    offset = torch.as_tensor(outer * (POOL_BLOCKS * REGION) + np.asarray(did, dtype=np.int64)[j] * REGION + byte, device=dev)
    bounds = np.searchsorted(layer, np.arange(NL + 1))
    got = torch.cat([dst_bufs[l][offset[bounds[l]:bounds[l + 1]]] for l in range(NL)])
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, name + ".npy"), got.float().cpu().numpy())


# =====================================================================================================
# ours
# =====================================================================================================
def run_ours(args):
    import torch
    import torch.distributed as dist
    from dynamo_b200 import kernels as K
    from dynamo_b200.disagg import assign_roles
    from dynamo_b200.kernels import PagedCopyOpts, PagedDst, PagedLayout
    from dynamo_b200.physical import BlockDimension, LayoutConfig, StorageKind, TransferManager, TransferOptions

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world == 1 and args.gpus > 1:
        raise SystemExit("launch with torch.distributed.run for --gpus > 1")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a GPU: the KV transfer path has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dev = f"cuda:{local}"
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device(dev))

    def barrier():
        if world > 1:
            dist.barrier()

    def allmax(x):
        t = torch.tensor([float(x)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def allsum(x):
        t = torch.tensor([int(x)], dtype=torch.int64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return int(t.item())

    cfg = LayoutConfig(POOL_BLOCKS, NL, OUTER, PAGE, INNER, dtype_width_bytes=DTYPE_BYTES)
    src_cfg = cfg if not CAST else LayoutConfig(POOL_BLOCKS, NL, OUTER, PAGE, INNER, dtype_width_bytes=1, allow_fp8=True)
    mgr = TransferManager(device=local, worker_id=rank + 1)
    roles = assign_roles(world, TOPOLOGY)
    is_src = roles.is_source(rank)
    is_dst = roles.is_destination(rank)
    my_dsts = roles.destinations.get(rank, [])          # destination ranks this rank is the source of
    n_dst = len(roles.destinations[roles.sources[0]])   # destinations per source (same for every source)
    n_src = len(roles.sources)
    my_src = roles.source_of(rank) if is_dst else None
    my_dst_index = roles.destinations[my_src].index(rank) if is_dst else -1
    pull = DIRECTION == "pull" and world > 1
    launcher = is_dst if pull else is_src

    def register(bufs, c=None):
        return mgr.register_layer_separate(c or cfg, [b.data_ptr() for b in bufs], [b.numel() for b in bufs],
                                           BlockDimension.BlockIsSecondDim, StorageKind.Device, local)

    def make_pool(region):
        return [torch.empty(OUTER * POOL_BLOCKS * region, dtype=torch.uint8, device=dev) for _ in range(NL)]

    src_bufs = dst_bufs = None
    h_src_local = h_dst_local = None
    if is_src:
        src_bufs = make_pool(SRC_REGION)
        fill_source(torch, src_bufs, dev, SRC_REGION)
        h_src_local = register(src_bufs, src_cfg)
    flag_buf = torch.zeros(64, dtype=torch.int32, device=dev)   # [0]=done flag of this destination
    mc_group, mc_base = None, 0
    if NVLS:
        # every rank (the source included: the root of the reference's ncclBcast keeps a copy too) binds one pool
        # allocation to the multicast object; layers lie back to back in it
        from dynamo_b200.disagg import share_fd
        from dynamo_b200.physical import MulticastGroup
        per_layer = OUTER * POOL_BLOCKS * REGION
        tag = os.environ.get("MASTER_PORT", "0")
        if rank == 0:
            mc_group = MulticastGroup.create(world, NL * per_layer, shareable=True)
            share_fd(0, world, mc_group.export_fd(), "mc-" + tag)
        else:
            mc_group = MulticastGroup.from_fd(share_fd(rank, world, None, "mc-" + tag), world, NL * per_layer)
        mc_group.add_device(local)
        barrier()
        pool_ptr = mc_group.bind_local(local)

        class _Raw:
            def __init__(self, ptr, nbytes):
                self.__cuda_array_interface__ = {"shape": (nbytes,), "typestr": "|u1", "data": (int(ptr), False), "version": 2}
        whole = torch.as_tensor(_Raw(pool_ptr, NL * per_layer), device=dev)
        whole.zero_()
        dst_bufs = [whole[l * per_layer:(l + 1) * per_layer] for l in range(NL)]
        h_dst_local = register(dst_bufs)
        torch.cuda.synchronize()
        barrier()
        if is_src:
            mc_base = mc_group.map(local)
    elif is_dst:
        dst_bufs = make_pool(REGION)
        for b in dst_bufs:
            b.zero_()
        h_dst_local = register(dst_bufs)
    torch.cuda.synchronize()

    # ---- exchange layout metadata (CUDA IPC handles inside): sources map the decode pools, decode ranks the prefill pool
    flag_cfg = LayoutConfig(1, 1, 1, 1, 128, dtype_width_bytes=2)
    h_dsts, peer_flags, h_src_remote, blobs = [], [], None, None
    if world > 1:
        h_flag_local = mgr.register_fully_contiguous(flag_cfg, flag_buf.data_ptr(), 256, StorageKind.Device, local)
        mine = (mgr.export_metadata(h_dst_local) if (is_dst and not NVLS) else b"",
                mgr.export_metadata(h_flag_local),
                mgr.export_metadata(h_src_local) if is_src else b"")
        blobs = [None] * world
        dist.all_gather_object(blobs, mine)
        if is_src:
            if NVLS:
                per_layer = OUTER * POOL_BLOCKS * REGION
                h_mc = mgr.register_layer_separate(cfg, [mc_base + l * per_layer for l in range(NL)], [per_layer] * NL,
                                                   BlockDimension.BlockIsSecondDim, StorageKind.Device, local)
                h_dsts = [h_mc] * len(my_dsts)
            else:
                h_dsts = [mgr.import_metadata(blobs[r][0]) for r in my_dsts]
            peer_flags = [mgr.memory_region(mgr.import_metadata(blobs[r][1]), 0, 0, 0)[0] for r in my_dsts]
        if pull and is_dst:
            h_src_remote = mgr.import_metadata(blobs[my_src][2])
    else:
        h_dsts = [h_dst_local]
        peer_flags = [flag_buf.data_ptr()]

    # ---- block tables (every rank can derive every table: the seeds are the contract) ----
    def tables(sort=False):
        s = [np.random.default_rng(10 + (0 if REPLICATE else d)).permutation(POOL_BLOCKS)[:N_BLOCKS] for d in range(n_dst)]
        t = [np.random.default_rng(100 + (0 if NVLS else d)).permutation(POOL_BLOCKS)[:N_BLOCKS] for d in range(n_dst)]
        if sort:
            s, t = [np.sort(x) for x in s], [np.sort(x) for x in t]
        return s, t
    sids, dids = tables()
    stream = torch.cuda.Stream(device=dev)
    sp = int(stream.cuda_stream)
    K_steps, W = args.steps, args.warmup

    def ev():
        return torch.cuda.Event(enable_timing=True)

    # device descriptors straight from the registered layouts (same numbers the manager uses)
    keep = []

    def desc(h, region):
        bases = [mgr.memory_region(h, 0, l, 0)[0] for l in range(NL)]
        t = torch.tensor(bases, dtype=torch.int64, device=dev)
        keep.append(t)
        return PagedLayout(t.data_ptr(), region, region * POOL_BLOCKS, region, NL, OUTER, POOL_BLOCKS)

    def dev_ids(x):
        t = torch.from_numpy(np.ascontiguousarray(x, dtype=np.int32)).to(dev)
        keep.append(t)
        return t

    ws = torch.zeros(K.sync_workspace_words(NL), dtype=torch.int32, device=dev)

    def make_launch(s_tabs, d_tabs):
        """Returns launch(epoch) for this rank's role (None when this rank launches nothing)."""
        if not launcher:
            return None
        if pull:
            d_src = desc(h_src_remote, SRC_REGION)
            dd = [PagedDst(desc(h_dst_local, REGION), dev_ids(s_tabs[my_dst_index]).data_ptr(), dev_ids(d_tabs[my_dst_index]).data_ptr(),
                           flag_buf.data_ptr(), 0)]
        else:
            d_src = desc(h_src_local, SRC_REGION)
            shared = dev_ids(s_tabs[0])
            dd = []
            for d in range(len(h_dsts)):
                s_ids = shared if REPLICATE else dev_ids(s_tabs[d])
                dd.append(PagedDst(desc(h_dsts[d], REGION), s_ids.data_ptr(), dev_ids(d_tabs[d]).data_ptr(), peer_flags[d], 0))

        def launch(epoch):
            opts = PagedCopyOpts(epoch=epoch, sync_workspace=ws.data_ptr(), multicast=1 if NVLS else 0)
            K.check(K.paged_copy(d_src, dd, N_BLOCKS, 0, NL, CAST, opts, sp), "paged_copy")
        return launch

    def timed_leg(launch, steps, epoch0):
        """K steps back to back, every launch bracketed by its own pair of CUDA events on the launching stream.  Returns
        (median of the K per-launch device times, total / K), both max over ranks.  Ranks that only receive (push mode) wait
        ON THE DEVICE for the last step's done flag, so the total covers the landing of the last byte."""
        barrier()
        starts, ends = [ev() for _ in range(steps)], [ev() for _ in range(steps)]
        first, last = ev(), ev()
        first.record(stream)
        if launch is not None:
            for i in range(steps):          # back to back, no host sync: each launch bracketed by its own pair of events
                starts[i].record(stream)
                launch(epoch0 + i + 1)
                ends[i].record(stream)
        elif world > 1 and is_dst and not pull:
            K.check(K.wait_flag(flag_buf.data_ptr(), epoch0 + steps, sp))   # device-side: all K steps landed here
        last.record(stream)
        stream.synchronize()
        torch.cuda.synchronize()
        barrier()
        total = first.elapsed_time(last)
        med = statistics.median(starts[i].elapsed_time(ends[i]) for i in range(steps)) if launch is not None else 0.0
        return allmax(med), allmax(total / steps)

    # ================= leg 1: `value` -- C ABI, block tables resident in HBM =================
    launch = make_launch(sids, dids)
    barrier()
    if launch is not None:
        with torch.cuda.stream(stream):
            for i in range(W):
                launch(i + 1)
        stream.synchronize()
    if world > 1 and is_dst and not pull:
        K.check(K.wait_flag(flag_buf.data_ptr(), W, sp))
        stream.synchronize()
    torch.cuda.synchronize()
    # the clock sampler (an nvidia-smi child) starts BEFORE the barrier that opens the timed region: spawning it takes
    # ~0.1 s on an 8-GPU box, which ranks that are already timing would otherwise count as transfer time
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
        sampler.wait_first_sample(2.0)
    launches0 = K.launch_count()
    value_ms_med, value_ms_mean = timed_leg(launch, K_steps, W)
    launches_value = K.launch_count() - launches0

    # ================= leg 2: `e2e` -- host API, host block tables every step =================
    e2e_times = []
    sid_l = [np.ascontiguousarray(s, dtype=np.uint64) for s in sids]   # host block tables (numpy, zero-copy into the ABI)
    did_l = [np.ascontiguousarray(d, dtype=np.uint64) for d in dids]

    def step():
        o = TransferOptions(cast_mode=CAST, multicast=1 if NVLS else 0)
        if pull:
            note = mgr.execute_transfer(h_src_remote, sid_l[my_dst_index], h_dst_local, did_l[my_dst_index], o)
        elif len(h_dsts) == 1 or NVLS:
            note = mgr.execute_transfer(h_src_local, sid_l[0], h_dsts[0], did_l[0], o)
        else:
            note = mgr.execute_fanout(h_src_local, h_dsts, sid_l, did_l, REPLICATE, o)
        note.wait(60.0)
    if launcher:
        for _ in range(W):
            step()
    torch.cuda.synchronize()
    barrier()
    h2d0 = mgr.h2d_bytes()
    launches1 = K.launch_count()
    t_all0 = time.perf_counter()
    if launcher:
        for _ in range(K_steps):
            t0 = time.perf_counter()
            step()
            e2e_times.append(time.perf_counter() - t0)
    torch.cuda.synchronize()
    barrier()
    e2e_wall = allmax(time.perf_counter() - t_all0)
    launches_e2e = K.launch_count() - launches1
    h2d_per_step = allsum((mgr.h2d_bytes() - h2d0) // max(1, K_steps))
    launches_all = allsum(launches_value + launches_e2e)
    e2e_p50 = allmax(1e3 * statistics.median(e2e_times) if e2e_times else 0.0)
    clocks = sampler.stop() if rank == 0 else None

    # ================= parity: every moved region on every destination (not timed) =================
    lut = golden_lut(torch, dev) if CAST else None
    checked = bad = changed = 0
    if is_dst:
        checked, bad, changed = verify_destination(torch, dst_bufs, dev, sids[my_dst_index], dids[my_dst_index], CAST, lut)
    checked, bad, changed = allsum(checked), allsum(bad), allsum(changed)
    parity = {"blocks_checked": "all", "regions_checked": checked, "regions_mismatching": bad, "untouched_blocks_changed": changed,
              "destinations": n_dst * n_src, "ok": bad == 0 and changed == 0 and checked == n_dst * n_src * N_BLOCKS * NL * OUTER,
              "how": "device-side comparison of every moved (block, layer, K/V) region with the closed-form source pattern"
                     + (" through the golden fp8->bf16 table (tests/golden)" if CAST else "") + "; every non-destination block must still be zero"}
    ok = parity["ok"]
    if args.dump_outputs and is_dst:
        dump_destination(torch, args.dump_outputs, f"received_kv_rank{rank}", dst_bufs, dev, dids[my_dst_index],
                         DUMP_SAMPLES // (n_dst * n_src))

    # ================= extras (not timed): sorted tables, GPU baselines, the other transfer modes =================
    extras = {}
    if not args.quick:
        s2, d2 = tables(sort=True)
        l2 = make_launch(s2, d2)
        e0 = W + K_steps
        if l2 is not None:
            for i in range(3):
                l2(e0 + 1 + i)
        if world > 1 and is_dst and not pull:
            K.check(K.wait_flag(flag_buf.data_ptr(), e0 + 3, sp))
        stream.synchronize()
        sm, _ = timed_leg(l2, 10, e0 + 3)
        extras["sorted_block_tables"] = {"ms_per_step": round(sm, 5),
                                         "value": round(BYTES_PER_DST * n_dst * n_src / (sm * 1e-3) / 1e9, 2), "unit": "GB/s",
                                         "note": "same request with both block tables sorted ascending (SURVEY 8d asks both)"}
        if world > 1 and not NVLS and not CAST and not REPLICATE and TOPOLOGY == "fanout":
            st = selftest_modes(torch, dist, mgr, dict(world=world, rank=rank, local=local, dev=dev, is_src=is_src, is_dst=is_dst,
                                                       dst_bufs=dst_bufs, h_dst_local=h_dst_local, h_src_local=h_src_local,
                                                       h_src_remote=h_src_remote, my_dst_index=my_dst_index, n_dst=n_dst, blobs=blobs,
                                                       h_dsts=h_dsts, sids=sids, dids=dids, barrier=barrier, allsum=allsum))
            extras["selftest"] = st
            ok = ok and st["all_ok"]
        if rank == 0 and not CAST and not NVLS:
            extras["gpu_baselines"] = gpu_baselines(torch, K, mgr, h_src_local, h_dsts[0], sids[0], dids[0], dev, world)
        barrier()
        if REPLICATE and world > 1:
            # the ncclBcast baseline is a separate single-process program that opens its own communicators on every GPU: the
            # other ranks must leave their GPUs idle meanwhile, so they wait on the (CPU-side) rendezvous store, not in an
            # NCCL barrier whose kernel would spin on the device
            store = dist.distributed_c10d._get_default_store()
            if rank == 0:
                extras.setdefault("gpu_baselines", {})["nccl_bcast_per_region"] = nccl_bcast_baseline()
                store.set("kvbm_bench_nccl_baseline_done", "1")
            else:
                store.wait(["kvbm_bench_nccl_baseline_done"])
        barrier()

    if rank == 0:
        total_dst_bytes = BYTES_PER_DST * n_dst * n_src
        ms_per_step = value_ms_med
        value = total_dst_bytes / (ms_per_step * 1e-3) / 1e9
        e2e_ms = 1e3 * e2e_wall / K_steps
        e2e_val = total_dst_bytes / (e2e_ms * 1e-3) / 1e9
        peak, peak_src = peaks()
        gb = extras.get("gpu_baselines", {})
        if world == 1:
            alg = BYTES_PER_DST * SRC_REGION // REGION + BYTES_PER_DST   # B_src read once + B_dst written, per launch (SURVEY §8d)
            roof = {"bound": "hbm", "achieved": round(alg / (ms_per_step * 1e-3) / 1e9, 2), "peak": peak, "unit": "GB/s",
                    "frac": round(alg / (ms_per_step * 1e-3) / 1e9 / peak, 4), "traffic": ncu_traffic("n1"), "peak_source": peak_src,
                    "kernel": f"kvbm_paged_copy_kernel<{CAST}>", "algorithmic_bytes_per_launch": alg,
                    "frac_of_mean_step": round(alg / (value_ms_mean * 1e-3) / 1e9 / peak, 4)}
        else:
            # NVLink: bytes that cross the source GPU's port per step / step time, against a contiguous peer copy measured
            # on THIS box in this process (gpu_baselines.memcpy_whole) -- else the guide's 770 GB/s
            measured = gb.get("memcpy_whole", {}).get("gbs")
            nv_peak = measured or NVLINK_PEER_GBS_GUIDE
            per_src = value / n_src
            roof = {"bound": "nvlink", "achieved": round(per_src, 2), "peak": round(nv_peak, 1), "unit": "GB/s",
                    "frac": round(per_src / nv_peak, 4), "frac_of_nominal_900": round(per_src / 900.0, 4),
                    "traffic": ncu_traffic("n2") if world == 2 else None, "sources": n_src,
                    "peak_source": ("contiguous cudaMemcpyAsync rank0 -> rank1 measured in this run (gpu_baselines.memcpy_whole)" if measured else
                                    "B200_PROFILING.md measured peer copy 770 GB/s per direction") + "; nominal 900",
                    "kernel": "kvbm_paged_copy_kernel<0>", "algorithmic_bytes_per_launch": (total_dst_bytes // n_src) // (n_dst if pull else 1),
                    "launches_per_step": n_dst if pull else 1,
                    "hbm_read_gbs_source": round((BYTES_PER_DST * SRC_REGION // REGION) * (1 if REPLICATE else n_dst) / (ms_per_step * 1e-3) / 1e9, 2)}
            if NVLS:   # the source sends the payload ONCE; the switch delivers it to every bound GPU
                egress = BYTES_PER_DST / (ms_per_step * 1e-3) / 1e9
                roof.update({"achieved": round(egress, 2), "frac": round(egress / nv_peak, 4), "algorithmic_bytes_per_launch": BYTES_PER_DST,
                             "nvls": True, "delivered_gbs_all_destinations": round(value, 2),
                             "note": "achieved = NVLink egress of the source (1x payload); value = bytes delivered to the N-1 decode GPUs"})
        line = {
            "metric": "kv_transfer_gbs", "value": round(value, 2), "unit": "GB/s", "n_gpus": world, "steps": K_steps,
            "warmup": W, "ms_per_step": round(ms_per_step, 5), "ms_per_step_mean": round(value_ms_mean, 5),
            "value_of_mean_step": round(total_dst_bytes / (value_ms_mean * 1e-3) / 1e9, 2),
            "timing": "K steps back to back; ms_per_step = median of the K per-launch CUDA-event intervals (one event pair per launch on the launching stream), max over ranks; *_mean = first-event-to-last-event of the same K steps / K (includes the gaps between launches)",
            "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u8", "data": "synthetic", "config": workload_config(world),
            "e2e": {"value": round(e2e_val, 2), "unit": "GB/s", "ms_per_step": round(e2e_ms, 5), "p50_ms": round(e2e_p50, 5),
                    "h2d_bytes_per_step": int(h2d_per_step), "d2h_bytes_per_step": 4 * (n_dst * n_src if pull else n_src),
                    "what": "TransferManager.execute_%s with host block-id lists; id upload, launch and completion-word "
                            "read-back inside the timed region%s" % ("transfer" if (pull or n_dst == 1) else "fanout",
                                                                     " (one call per decode rank, max over ranks)" if pull else "")},
            "gpu_launches": int(launches_all),
            "gpu_launches_detail": {"value_leg_rank0": int(launches_value), "e2e_leg_rank0": int(launches_e2e),
                                    "launching_ranks": (n_dst * n_src) if pull else n_src},
            "roofline": roof, "clocks": clocks, "parity": parity, "bit_exact_probe": ok,
        }
        line.update(extras)
        cores = host_threads()
        if not args.no_cpu_baseline:
            numa = numa_interleave()
            ours_ms = e2e_p50
            if world == 1:
                t1, ok1 = cpu_path(2, 1, 1)
                tn, okn = cpu_path(6, 2, cores)
                v1 = BYTES_PER_DST / statistics.median(t1) / 1e9
                vn = BYTES_PER_DST / statistics.median(tn) / 1e9
                line["cpu_baseline"] = {"value": round(vn, 3), "unit": "GB/s", "cores": cores, "kind": "port",
                                        "single_thread_value": round(v1, 3),
                                        "sample": f"6 x the full {N_BLOCKS}-block/{BYTES_PER_DST >> 20} MiB request with {cores} pinned threads (median), "
                                                  f"{numa}, pool of {POOL_BLOCKS} blocks like the GPU arm; the reference's loop is "
                                                  f"single-threaded: {v1:.2f} GB/s on 1 core (2 repeats); bit-exact={ok1 and okn}"}
                cpu_ms = 1e3 * statistics.median(tn)
                # decode-visible TTFT = T_prefill + T_transfer + T_first_decode (lib/mocker/src/common/utils.rs:14-40): only
                # T_transfer differs between the arms
                line["ttft"] = {"model": "T_prefill + T_transfer + T_first_decode; only T_transfer changes",
                                "transfer_ms_p50": round(ours_ms, 4), "reference_cpu_transfer_ms_p50": round(cpu_ms, 3),
                                "mocker_default_64GBs_ms": round(BYTES_PER_DST / 64e9 * 1e3, 3),
                                "decode_ttft_drop_ms_vs_cpu_path": round(cpu_ms - ours_ms, 3)}
            else:
                # fan-out: every decode GPU's KV is complete when the slowest transfer completes; the CPU path copies the
                # N-1 requests one after another on the host cores
                tn, okn = cpu_path(3, 1, cores)
                cpu_ms = 1e3 * statistics.median(tn)
                line["ttft"] = {"model": "T_prefill + T_transfer + T_first_decode; only T_transfer changes",
                                "fan_out": n_dst, "transfer_ms_p50_all_destinations": round(ours_ms, 4),
                                "reference_cpu_transfer_ms_p50_per_destination": round(cpu_ms, 3),
                                "reference_cpu_transfer_ms_all_destinations": round(cpu_ms * n_dst, 3),
                                "mocker_default_64GBs_ms_per_destination": round(BYTES_PER_DST / 64e9 * 1e3, 3),
                                "decode_ttft_drop_ms_vs_cpu_path_last_destination": round(cpu_ms * n_dst - ours_ms, 3),
                                "cpu_cores": cores}
        print(json.dumps(line), flush=True)
    barrier()
    if mc_group is not None:
        mc_group.detach()
    mgr.close()
    if world > 1:
        dist.destroy_process_group()
    return 0 if ok else 1


# -----------------------------------------------------------------------------------------------------
# extras
# -----------------------------------------------------------------------------------------------------
def selftest_modes(torch, dist, mgr, env):
    """The transfer modes the headline run did not use, each over the full request with the full parity check, so a
    multi-GPU box exercises push, pull and the fused cast in both directions in one driver-run command."""
    from dynamo_b200.physical import BlockDimension, LayoutConfig, StorageKind, TransferOptions
    world, local, dev = env["world"], env["local"], env["dev"]
    is_src, is_dst = env["is_src"], env["is_dst"]
    dst_bufs, h_dst_local, h_src_local = env["dst_bufs"], env["h_dst_local"], env["h_src_local"]
    my_dst_index, n_dst = env["my_dst_index"], env["n_dst"]
    blobs, h_dsts = env["blobs"], env["h_dsts"]
    sids, dids = env["sids"], env["dids"]
    barrier, allsum = env["barrier"], env["allsum"]
    lut = golden_lut(torch, dev)
    out = {}
    sid_l = [np.ascontiguousarray(s, dtype=np.uint64) for s in sids]
    did_l = [np.ascontiguousarray(d, dtype=np.uint64) for d in dids]
    # rank 0's pool mapped into every decode rank (for pull) even when the headline run pushed
    h_src_remote = env["h_src_remote"]
    if is_dst and h_src_remote is None:
        h_src_remote = mgr.import_metadata(blobs[0][2])
    # an fp8 copy of the source pool for the cast modes (same closed-form pattern at 16 KiB regions)
    r8 = REGION // 2
    h_src8 = h_src8_remote = None
    cfg8 = LayoutConfig(POOL_BLOCKS, NL, OUTER, PAGE, INNER, dtype_width_bytes=1, allow_fp8=True)
    if is_src:
        src8 = [torch.empty(OUTER * POOL_BLOCKS * r8, dtype=torch.uint8, device=dev) for _ in range(NL)]
        fill_source(torch, src8, dev, r8)
        h_src8 = mgr.register_layer_separate(cfg8, [b.data_ptr() for b in src8], [b.numel() for b in src8],
                                             BlockDimension.BlockIsSecondDim, StorageKind.Device, local)
    torch.cuda.synchronize()
    b8 = [None] * world
    dist.all_gather_object(b8, mgr.export_metadata(h_src8) if is_src else b"")
    if is_dst:
        h_src8_remote = mgr.import_metadata(b8[0])

    def run(name, how, cast):
        if is_dst:
            for b in dst_bufs:
                b.zero_()
        torch.cuda.synchronize()
        barrier()
        t0 = time.perf_counter()
        o = TransferOptions(cast_mode=cast)
        if how == "pull" and is_dst:
            mgr.execute_transfer(h_src8_remote if cast else h_src_remote, sid_l[my_dst_index], h_dst_local, did_l[my_dst_index], o).wait(60.0)
        elif how == "push" and is_src:
            src = h_src8 if cast else h_src_local
            if len(h_dsts) == 1:
                mgr.execute_transfer(src, sid_l[0], h_dsts[0], did_l[0], o).wait(60.0)
            else:
                mgr.execute_fanout(src, h_dsts, sid_l, did_l, False, o).wait(60.0)
        torch.cuda.synchronize()
        barrier()
        wall = time.perf_counter() - t0
        c = b = ch = 0
        if is_dst:
            c, b, ch = verify_destination(torch, dst_bufs, dev, sids[my_dst_index], dids[my_dst_index], cast, lut, src_region=r8 if cast else REGION)
        c, b, ch = allsum(c), allsum(b), allsum(ch)
        out[name] = {"ok": b == 0 and ch == 0 and c == n_dst * N_BLOCKS * NL * OUTER, "regions_checked": c, "regions_mismatching": b,
                     "untouched_blocks_changed": ch, "wall_ms_incl_barriers": round(1e3 * wall, 2)}

    run("push", "push", 0)
    run("pull", "pull", 0)
    run("push_cast_fp8_to_bf16", "push", 1)
    run("pull_cast_fp8_to_bf16", "pull", 1)     # receiver-side up-cast: fp8 bytes on the wire, bf16 written locally
    out["all_ok"] = all(v["ok"] for v in out.values())
    out["what"] = "each mode moves the full request once through TransferManager and is verified region by region like `parity`"
    return out


def gpu_baselines(torch, K, mgr, h_src, h_dst, sid, did, dev, world, iters=5):
    """The reference's GPU paths for the same request on the same pools, wall clock per transfer (host work included,
    stream synchronised), medians of `iters`.  rank 0 -> first destination (a peer mapping when N > 1)."""
    from dynamo_b200.kernels import MemcpyBatchMode
    res = {"note": "rank 0 -> its first destination, host work included, median of %d; NOT part of any timed region of `value`/`e2e`" % iters}
    sbase = np.array([mgr.memory_region(h_src, 0, l, 0)[0] for l in range(NL)], dtype=np.uint64)
    dbase = np.array([mgr.memory_region(h_dst, 0, l, 0)[0] for l in range(NL)], dtype=np.uint64)
    sid = np.asarray(sid, dtype=np.uint64)
    did = np.asarray(did, dtype=np.uint64)
    stream = torch.cuda.Stream(device=dev)
    sp = int(stream.cuda_stream)
    npairs = N_BLOCKS * NL * OUTER
    payload = npairs * REGION

    def host_tables():
        # the reference's host loop (cuda.rs:258-283): (block, layer, outer) order, 2 x nb*nl*no addresses; numpy stands in
        # for 32 768 memory_region() calls -- generous to the reference
        o = np.arange(OUTER, dtype=np.uint64)
        s = (sbase[None, :, None] + sid[:, None, None] * np.uint64(REGION) + o[None, None, :] * np.uint64(REGION * POOL_BLOCKS)).reshape(-1)
        d = (dbase[None, :, None] + did[:, None, None] * np.uint64(REGION) + o[None, None, :] * np.uint64(REGION * POOL_BLOCKS)).reshape(-1)
        return s, d

    def timed(fn, moved=payload):
        fn()
        torch.cuda.synchronize()
        ts = []
        for _ in range(iters):
            t0 = time.perf_counter()
            fn()
            ts.append(time.perf_counter() - t0)
        ms = 1e3 * statistics.median(ts)
        return {"ms": round(ms, 4), "gbs": round(moved / (ms * 1e-3) / 1e9, 2)}

    pin_s = torch.empty(npairs, dtype=torch.int64).pin_memory()
    pin_d = torch.empty(npairs, dtype=torch.int64).pin_memory()
    dev_s = torch.empty(npairs, dtype=torch.int64, device=dev)
    dev_d = torch.empty(npairs, dtype=torch.int64, device=dev)
    done = torch.cuda.Event()

    def k1_flow(launch):
        s, d = host_tables()
        pin_s.numpy()[:] = s.view(np.int64)
        pin_d.numpy()[:] = d.view(np.int64)
        with torch.cuda.stream(stream):
            dev_s.copy_(pin_s, non_blocking=True)
            dev_d.copy_(pin_d, non_blocking=True)
            rc = launch(dev_s.data_ptr(), dev_d.data_ptr(), REGION, npairs, sp)
            assert rc == 0, rc
            done.record(stream)
        done.synchronize()          # pointers_transfered_event.synchronize() + completion, cuda.rs:324

    ref_so = os.path.join(ROOT, "oracle", "_ref", "libkvbm_kernels_ref.so")
    if os.path.exists(ref_so):
        R = C.CDLL(ref_so)
        R.kvbm_kernels_launch_vectorized_copy.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_int, C.c_void_p]
        res["ref_k1_flow"] = dict(timed(lambda: k1_flow(R.kvbm_kernels_launch_vectorized_copy)),
                                  what="the reference's tensor_kernels.cu K1 (compiled unmodified for sm_100) driven like "
                                       "kvbm-physical executor/cuda.rs:234-327: host pointer tables, 2 x H2D, launch, host sync")
    res["ours_k1_flow"] = dict(timed(lambda: k1_flow(K.vectorized_copy)),
                               what="the same flow through this library's drop-in K1 symbol")
    s, d = host_tables()
    sl, dl = [int(x) for x in s], [int(x) for x in d]
    s_arr = (C.c_void_p * npairs)(*sl)
    d_arr = (C.c_void_p * npairs)(*dl)
    raw = K.lib().kvbm_kernels_memcpy_batch

    def per_chunk(mode):
        K.check(raw(s_arr, d_arr, REGION, npairs, int(mode), sp))
        stream.synchronize()
    res["memcpy_per_chunk"] = dict(timed(lambda: per_chunk(MemcpyBatchMode.FallbackOnly)),
                                   what="one cudaMemcpyAsync per (block, layer, K/V) chunk = the v1 D2D path "
                                        "(block/transfer/cuda.rs:299-391) and UCX cuda_ipc behaviour")
    if K.is_memcpy_batch_available():
        try:
            res["memcpy_batch"] = dict(timed(lambda: per_chunk(MemcpyBatchMode.BatchWithoutFallback)),
                                       what="cudaMemcpyBatchAsync over the same chunk list (K4, tensor_kernels.cu:389-473)")
        except Exception as e:   # the driver may refuse peer batches
            res["memcpy_batch"] = {"unavailable": str(e)[:120]}
    try:
        # the contiguous DMA ceiling: ONE cudaMemcpyAsync of the request's byte count, rank 0's GPU -> the next GPU (a buffer this
        # process allocates there itself; peer access enabled so that the copy goes over NVLink), CUDA events on the stream
        big_a = torch.empty(payload, dtype=torch.uint8, device=dev)
        if world == 1 or torch.cuda.device_count() < 2:
            big_b = torch.empty(payload, dtype=torch.uint8, device=dev)
            where = "its own HBM"
        else:
            peer = (torch.cuda.current_device() + 1) % torch.cuda.device_count()
            mgr.enable_peer_access(peer)
            big_b = torch.empty(payload, dtype=torch.uint8, device=f"cuda:{peer}")
            torch.cuda.synchronize(peer)
            where = f"GPU {peer} over NVLink"
        srcs = (C.c_void_p * 1)(big_a.data_ptr())
        dsts = (C.c_void_p * 1)(big_b.data_ptr())

        def whole():
            K.check(raw(srcs, dsts, payload, 1, int(MemcpyBatchMode.FallbackOnly), sp))
            stream.synchronize()
        whole()
        evs = []
        for _ in range(iters + 3):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            K.check(raw(srcs, dsts, payload, 1, int(MemcpyBatchMode.FallbackOnly), sp))
            e1.record(stream)
            e1.synchronize()
            evs.append(e0.elapsed_time(e1))
        dev_ms = statistics.median(evs)
        r = timed(whole)
        res["memcpy_whole"] = {"ms": r["ms"], "device_ms": round(dev_ms, 4), "gbs": round(payload / (dev_ms * 1e-3) / 1e9, 2), "wall_gbs": r["gbs"],
                               "what": f"one contiguous {payload >> 20} MiB cudaMemcpyAsync, rank 0 -> {where} (DMA engines): the measured copy "
                                       "ceiling of this box; gbs = CUDA events on the stream, wall_gbs includes the host's launch + sync"}
        del big_a, big_b
    except Exception as e:
        res["memcpy_whole"] = {"unavailable": str(e)[:160]}
    # two-hop plan GPU -> pinned -> GPU (strategy.rs:222-233, executor/mod.rs:357-416): what the reference does when direct
    # GPU RDMA is not allowed
    try:
        from dynamo_b200.physical import LayoutConfig, StorageKind
        bcfg = LayoutConfig(N_BLOCKS, NL, OUTER, PAGE, INNER, dtype_width_bytes=DTYPE_BYTES)
        bounce = torch.empty(bcfg.required_bytes(), dtype=torch.uint8).pin_memory()
        h_b = mgr.register_fully_contiguous(bcfg, bounce.data_ptr(), bounce.numel(), StorageKind.Pinned)
        ident = np.arange(N_BLOCKS, dtype=np.uint64)

        def two_hop():
            mgr.execute_transfer(h_src, sid, h_b, ident).wait(60.0)
            mgr.execute_transfer(h_b, ident, h_dst, did).wait(60.0)
        res["two_hop_pinned"] = dict(timed(two_hop), what="Device -> Pinned bounce -> Device (our kernels on both hops; PCIe-bound)")
        mgr.unregister(h_b)
    except Exception as e:
        res["two_hop_pinned"] = {"unavailable": str(e)[:160]}
    return res


def nccl_bcast_baseline():
    """The reference's replicate path: one grouped ncclBcast per region (kvbm-engine collectives/nccl.rs:321-356), as the
    stand-alone binary benchmarks/nccl_bcast_baseline (single process, one communicator per GPU).  Run on 64 blocks
    (4096 regions, 128 MiB): with the full 256-block request (16 384 broadcasts per rank in ONE group) NCCL 2.27 does not
    finish within minutes on this box (profiles/r02_nccl_bcast_n2_*.json), and the rate is flat in the size anyway."""
    exe = os.path.join(ROOT, "benchmarks", "nccl_bcast_baseline")
    if not os.path.exists(exe):
        return {"unavailable": "benchmarks/nccl_bcast_baseline not built (needs nccl.h at build time)"}
    try:
        r = subprocess.run([exe, "--blocks", str(min(N_BLOCKS, 64)), "--pool", str(POOL_BLOCKS), "--layers", str(NL), "--iters", "3", "--warmup", "1"],
                           capture_output=True, text=True, timeout=60)
        for ln in r.stdout.splitlines():
            if ln.startswith("{"):
                d = json.loads(ln)
                d["note"] = "64 of the request's 256 blocks per broadcast group (the full request does not complete in one NCCL group)"
                return d
        return {"unavailable": (r.stderr or r.stdout)[-200:]}
    except Exception as e:
        return {"unavailable": str(e)[:160]}


def ncu_traffic(which):
    """dram (N=1) / NVLink (N=2) bytes per launch of the dominant kernel from the committed ncu summary (profiles/), or None."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    try:
        d = json.load(open(p))
        return d["paged_copy_n1_dram_bytes_per_launch"] if which == "n1" else d.get("paged_copy_n2_nvlink_bytes_per_launch")
    except Exception:
        return None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--quick", action="store_true", help="skip the untimed extras (sorted tables, GPU baselines, mode self-test)")
    # non-default workloads (other BASELINE configs); results of these runs live in profiles/
    ap.add_argument("--model", default="llama8b", choices=["llama8b", "llama70b-tp4", "mixtral"])
    ap.add_argument("--ctx", type=int, default=4096, help="context tokens (blocks = ctx/16)")
    ap.add_argument("--cast", default="none", choices=["none", "fp8"])
    ap.add_argument("--replicate", action="store_true", help="same blocks to every destination (CollectiveOps::broadcast)")
    ap.add_argument("--nvls", action="store_true", help="with --replicate: write once to an NVLink multicast mapping (the switch fans out)")
    ap.add_argument("--pool-blocks", type=int, default=0)
    ap.add_argument("--direction", default="pull", choices=["pull", "push"],
                    help="N > 1: pull = every decode GPU launches and reads the prefill pool (default); push = the prefill GPU stores to all")
    ap.add_argument("--topology", default="fanout", choices=["fanout", "pairs"],
                    help="fanout: rank 0 -> ranks 1..N-1 (default); pairs: rank r -> rank r+N/2 (TP-sharded prefill -> decode)")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="after the timed steps, write a seeded sample of the KV bytes every destination received to "
                         "DIR/received_kv_rank<r>.npy (float32, 16 MiB in all; identical inputs on every run)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs samples the GPU transfer (--impl ours)")
    configure(args)
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else max(args.warmup, 1)
    if args.impl == "reference":
        return run_reference(args)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
