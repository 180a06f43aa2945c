"""CPU tests of the host library (libkvbm_physical.so): the reference's pure-arithmetic unit tests, the
strategy table, block validation, the Memcpy strategy against the oracle, ABI symbol presence.

Reference tests mirrored (relative to /root/reference/lib/kvbm-physical/src):
  layout/fully_contiguous.rs:356-424, layout/layer_separate.rs:345-430       layout KATs
  transfer/strategy.rs:288-503                                               strategy tables
  transfer/validation.rs:227-465                                             validation
  transfer/tests/local_transfers.rs (System/Pinned rows)                     Memcpy strategy
"""
import ctypes as C
import itertools
import os
import subprocess

import numpy as np
import pytest

from dynamo_b200 import _lib, kernels as K, physical as P
from dynamo_b200.physical import (BlockDimension, ErrorCode, KvbmError, LayoutConfig, StorageKind, TransferManager,
                                  TransferOptions, TransferStrategy)
from oracle import oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def std_cfg(nb, **kw):
    base = dict(num_blocks=nb, num_layers=2, outer_dim=2, page_size=16, inner_dim=128, dtype_width_bytes=2)
    base.update(kw)
    return LayoutConfig(**base)


@pytest.fixture()
def mgr():
    m = TransferManager(device=-1, worker_id=7)   # host-only manager: works without a GPU
    yield m
    m.close()


# ------------------------------------------------------------------ ABI surface
def _exported(path):
    out = subprocess.run(["nm", "-D", "--defined-only", path], capture_output=True, text=True, check=True).stdout
    return {line.split()[-1] for line in out.splitlines() if line.strip()}


def _declared(header):
    import re
    txt = open(os.path.join(ROOT, "include", header)).read()
    return set(re.findall(r"\b(kvbm_[a-z0-9_]+)\s*\(", txt))


def test_kernels_library_exports_every_declared_symbol():
    syms = _exported(_lib.KERNELS_SO)
    declared = _declared("kvbm_kernels.h")
    assert declared, "header parse failed"
    assert declared <= syms, declared - syms
    assert set(K.EXPORTED_SYMBOLS) == declared
    # the six reference symbols, by name (tensor_kernels.cu:306,332,360,389,477,551)
    for s in ["kvbm_kernels_launch_universal_from_block", "kvbm_kernels_launch_block_from_universal",
              "kvbm_kernels_has_memcpy_batch_async", "kvbm_kernels_memcpy_batch", "kvbm_kernels_is_stub_build",
              "kvbm_kernels_launch_vectorized_copy"]:
        assert s in syms


def test_physical_library_exports_every_declared_symbol():
    syms = _exported(_lib.PHYSICAL_SO)
    declared = _declared("kvbm_physical.h")
    assert declared <= syms, declared - syms
    assert set(P.EXPORTED_SYMBOLS) == declared


def test_library_loads_without_gpu_and_reports_real_build():
    assert K.is_using_stubs() is False
    assert K.is_memcpy_batch_available() is True
    # reference no-op / NULL semantics hold before any CUDA call is made (tensor_kernels.cu:396-402,555-561)
    assert K.vectorized_copy(0, 0, 0, 3, 0) == 0 and K.vectorized_copy(0, 0, 64, 0, 0) == 0
    assert K.vectorized_copy(0, 0, 64, 3, 0) == K.CUDA_ERROR_INVALID_VALUE
    assert K.memcpy_batch(None, None, 64, 3, K.MemcpyBatchMode.FallbackOnly, 0) == K.CUDA_ERROR_INVALID_VALUE


def test_paged_copy_rejects_nonzero_reserved_option_fields():
    """kvbm_paged_copy_opts.reserved0 / reserved1 must be 0.  The slots once selected L2 cache hints and diagnostic ring
    variants that did not copy; a caller that still sets them gets cudaErrorInvalidValue, before any CUDA call, instead of
    a transfer.  The arguments are otherwise well-formed; their addresses are never dereferenced."""
    region, nl, no, nb = 4096, 2, 2, 8
    layout = lambda base: K.PagedLayout(base, no * region, region, region, nl, no, nb)
    dst = K.PagedDst(layout(0x200000), 0x300000, 0x400000, 0, 0)
    for field, value in (("reserved0", 1), ("reserved1", 2)):
        opts = K.PagedCopyOpts(**{field: value})
        assert K.paged_copy(layout(0x100000), [dst], 4, 0, nl, K.CastMode.NONE, opts) == K.CUDA_ERROR_INVALID_VALUE, field


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "dynamo_b200")
    for base, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".cpp", ".hpp", ".h")):
                txt = open(os.path.join(base, f), errors="replace").read()
                assert "kvbm_oracle" not in txt and "from oracle" not in txt and "import oracle" not in txt, f


def test_cuda_strategy_without_device_fails_loudly(mgr):
    cfg = std_cfg(4)
    buf = np.zeros(cfg.required_bytes(), dtype=np.uint8)
    dev_like = mgr.register_fully_contiguous(cfg, buf.ctypes.data, buf.size, StorageKind.Device)
    pin = mgr.register_fully_contiguous(cfg, buf.ctypes.data, buf.size, StorageKind.Pinned)
    with pytest.raises(KvbmError) as e:
        mgr.execute_transfer(pin, [0], dev_like, [1])
    assert e.value.code == ErrorCode.CUDA and "no CPU fallback" in e.value.msg


# ------------------------------------------------------------------ layouts
def test_config_helpers_and_validation():
    cfg = std_cfg(10, num_layers=4)
    assert cfg.required_bytes() == 10 * 4 * 2 * 16 * 128 * 2      # fully_contiguous.rs:372-373
    assert cfg.bytes_per_block() == 4 * 2 * 16 * 128 * 2
    cfg.validate()
    for bad in [dict(num_blocks=0), dict(outer_dim=3), dict(outer_dim=0), dict(dtype_width_bytes=1),
                dict(dtype_width_bytes=3), dict(dtype_width_bytes=16), dict(alignment=3), dict(page_size=0)]:
        with pytest.raises(KvbmError) as e:
            std_cfg(4, **bad).validate()
        assert e.value.code == ErrorCode.CONFIG
    std_cfg(4, dtype_width_bytes=1, allow_fp8=True).validate()


def test_fc_memory_region_kat(mgr):
    cfg = std_cfg(2)
    R = 16 * 128 * 2
    h = mgr.register_fully_contiguous(cfg, 0x1000, cfg.required_bytes(), StorageKind.System)
    assert mgr.is_fully_contiguous(h)
    assert mgr.memory_region(h, 0, 0, 0) == (0x1000, R)
    assert mgr.memory_region(h, 0, 0, 1) == (0x1000 + R, R)
    assert mgr.memory_region(h, 0, 1, 0) == (0x1000 + 2 * R, R)
    assert mgr.memory_region(h, 1, 0, 0) == (0x1000 + 2 * 2 * R, R)
    for bad in [(2, 0, 0), (0, 2, 0), (0, 0, 2)]:
        with pytest.raises(KvbmError) as e:
            mgr.memory_region(h, *bad)
        assert e.value.code == ErrorCode.RANGE
    with pytest.raises(KvbmError) as e:   # "Memory region too small for layout" fully_contiguous.rs:166-172
        mgr.register_fully_contiguous(cfg, 0x1000, cfg.required_bytes() - 1, StorageKind.System)
    assert e.value.code == ErrorCode.CONFIG and "too small" in e.value.msg


def test_lw_memory_region_kat(mgr):
    cfg = std_cfg(2)
    per_layer = 2 * 2 * 16 * 128 * 2
    R = 16 * 128 * 2
    h = mgr.register_layer_separate(cfg, [0x1000, 0x1000 + per_layer], [per_layer] * 2, BlockDimension.BlockIsFirstDim,
                                    StorageKind.System)
    assert not mgr.is_fully_contiguous(h)
    assert mgr.memory_region(h, 0, 0, 0) == (0x1000, R)
    assert mgr.memory_region(h, 0, 1, 0) == (0x1000 + per_layer, R)
    assert mgr.memory_region(h, 0, 0, 1) == (0x1000 + R, R)
    h2 = mgr.register_layer_separate(cfg, [0x1000, 0x9000], [per_layer] * 2, BlockDimension.BlockIsSecondDim,
                                     StorageKind.System)
    assert mgr.memory_region(h2, 1, 0, 0) == (0x1000 + R, R)          # block_stride = region
    assert mgr.memory_region(h2, 0, 1, 1) == (0x9000 + 2 * R, R)      # outer_stride = region * num_blocks
    with pytest.raises(KvbmError):   # layer_separate.rs:163-169
        mgr.register_layer_separate(cfg, [0x1000], [per_layer], BlockDimension.BlockIsFirstDim, StorageKind.System)


def test_layouts_agree_with_oracle_on_random_geometry(mgr):
    rng = np.random.default_rng(0)
    for _ in range(20):
        nb, nl, no = int(rng.integers(1, 9)), int(rng.integers(1, 6)), int(rng.integers(1, 3))
        page, inner, dt = int(rng.integers(1, 33)), int(rng.integers(1, 300)), int(rng.choice([2, 4, 8]))
        cfg = LayoutConfig(nb, nl, no, page, inner, dtype_width_bytes=dt)
        bd = int(rng.integers(0, 2))
        per_layer = nb * no * page * inner * dt
        bases = [0x10000 + i * (per_layer + 4096) for i in range(nl)]
        h_fc = mgr.register_fully_contiguous(cfg, 0x5000, cfg.required_bytes(), StorageKind.System)
        h_lw = mgr.register_layer_separate(cfg, bases, [per_layer] * nl, BlockDimension(bd), StorageKind.System)
        o_fc = O.Layout(O.FC, nb, nl, no, page, inner, dt, bases=[0x5000])
        o_lw = O.Layout(O.LW, nb, nl, no, page, inner, dt, block_dim=bd, bases=bases)
        for b, l, o in itertools.product(range(nb), range(nl), range(no)):
            assert mgr.memory_region(h_fc, b, l, o) == o_fc.memory_region(b, l, o)
            assert mgr.memory_region(h_lw, b, l, o) == o_lw.memory_region(b, l, o)


# ------------------------------------------------------------------ strategy table (strategy.rs:288-503)
S, Pn, D, Dk = StorageKind.System, StorageKind.Pinned, StorageKind.Device, StorageKind.Disk


@pytest.mark.parametrize("src,dst,want", [
    (S, S, TransferStrategy.Memcpy), (S, Pn, TransferStrategy.Memcpy), (Pn, S, TransferStrategy.Memcpy),
    (Pn, Pn, TransferStrategy.Memcpy), (Pn, D, TransferStrategy.CudaAsyncH2D), (D, Pn, TransferStrategy.CudaAsyncD2H),
    (D, D, TransferStrategy.CudaAsyncD2D), (S, Dk, TransferStrategy.NixlWrite), (Pn, Dk, TransferStrategy.NixlWrite),
    (Dk, S, TransferStrategy.NixlReadFlipped), (Dk, Pn, TransferStrategy.NixlReadFlipped),
])
def test_direct_strategies(src, dst, want):
    plan = P.select_direct_strategy(src, dst)
    assert not plan.two_hop and plan.first == want


def test_two_hop_and_gds_strategies():
    p = P.select_direct_strategy(D, Dk)
    assert p.two_hop and (p.first, p.bounce_location, p.second) == (TransferStrategy.CudaAsyncD2H, Pn, TransferStrategy.NixlWrite)
    p = P.select_direct_strategy(Dk, D)
    assert p.two_hop and (p.first, p.bounce_location, p.second) == (TransferStrategy.NixlReadFlipped, Pn, TransferStrategy.CudaAsyncH2D)
    p = P.select_direct_strategy(Dk, Dk)
    assert p.two_hop and (p.first, p.second) == (TransferStrategy.NixlReadFlipped, TransferStrategy.NixlWrite)
    assert P.select_direct_strategy(D, Dk, allow_gds=True).first == TransferStrategy.NixlWrite
    assert P.select_direct_strategy(Dk, D, allow_gds=True).first == TransferStrategy.NixlRead
    for a, b in [(S, D), (D, S)]:      # the reference panics (strategy.rs:161,165); we return an error
        with pytest.raises(KvbmError) as e:
            P.select_direct_strategy(a, b)
        assert e.value.code == ErrorCode.UNSUPPORTED and "not supported" in e.value.msg


def test_remote_strategies():
    """strategy.rs:443-503 (select_direct_strategy with dst_is_remote) and select_strategy / select_remote_strategy_v2 (:78-108, 245-281)."""
    W, RF = TransferStrategy.NixlWrite, TransferStrategy.NixlReadFlipped
    # test_host_to_remote
    for k in (S, Pn):
        p = P.select_direct_strategy(k, k, dst_is_remote=True)
        assert not p.two_hop and p.first == W
    # test_device_to_remote_without_rdma / with_rdma
    p = P.select_direct_strategy(D, S, dst_is_remote=True)
    assert p.two_hop and (p.first, p.bounce_location, p.second) == (TransferStrategy.CudaAsyncD2H, Pn, W)
    p = P.select_direct_strategy(D, D, allow_gpu_rdma=True, dst_is_remote=True)
    assert not p.two_hop and p.first == W
    # test_disk_to_remote
    p = P.select_direct_strategy(Dk, S, dst_is_remote=True)
    assert p.two_hop and (p.first, p.bounce_location, p.second) == (W, Pn, W)
    # select_strategy: both local = the direct table
    assert P.select_strategy(D, True, D, True).first == TransferStrategy.CudaAsyncD2D
    assert P.select_strategy(Pn, True, S, True).first == TransferStrategy.Memcpy
    # exactly one side local: push = NixlWrite, pull = NixlReadFlipped
    assert P.select_strategy(Pn, True, Pn, False).first == W
    assert P.select_strategy(S, False, Pn, True).first == RF
    assert P.select_strategy(D, True, D, False, allow_gpu_rdma=True).first == W
    assert P.select_strategy(D, False, D, True, allow_gpu_rdma=True).first == RF
    for args, text in [((D, False, D, False), "Both src and dst are remote"),
                       ((Dk, True, S, False), "Neither local nor remote disk transfers are supported over NIXL"),
                       ((S, False, Dk, True), "Neither local nor remote disk transfers are supported over NIXL"),
                       ((D, True, S, False), "GPU RDMA is disabled"), ((Pn, False, D, True), "GPU RDMA is disabled")]:
        with pytest.raises(KvbmError) as e:
            P.select_strategy(*args)
        assert e.value.code == ErrorCode.UNSUPPORTED and text in e.value.msg


# ------------------------------------------------------------------ validation.rs
def test_validate_block_transfer_codes():
    P.validate_block_transfer([0, 1], [2, 3], 4, 4)
    P.validate_block_transfer([], [], 4, 4)
    cases = [(([0, 1], [2], 4, 4, False), ErrorCode.LENGTH_MISMATCH),
             (([0, 1], [2, 2], 4, 4, False), ErrorCode.DUPLICATE_DST),
             (([0, 1], [1, 2], 4, 4, True), ErrorCode.OVERLAP),
             (([0, 4], [1, 2], 4, 4, False), ErrorCode.RANGE),
             (([0, 1], [1, 9], 4, 4, False), ErrorCode.RANGE)]
    for args, code in cases:
        with pytest.raises(KvbmError) as e:
            P.validate_block_transfer(*args)
        assert e.value.code == code
    P.validate_block_transfer([0, 1], [1, 2], 4, 4, False)   # overlap only matters for the same layout
    # agrees with the oracle on random id lists
    rng = np.random.default_rng(1)
    a = O.Layout(O.FC, 8, 2, 2, 16, 128, 2, bases=[0x1000])
    b = O.Layout(O.FC, 8, 2, 2, 16, 128, 2, bases=[0x1000])
    omap = {O.OK: None, O.ERR_LENGTH_MISMATCH: ErrorCode.LENGTH_MISMATCH, O.ERR_DUP_DST: ErrorCode.DUPLICATE_DST,
            O.ERR_OVERLAP: ErrorCode.OVERLAP, O.ERR_RANGE: ErrorCode.RANGE}
    for _ in range(200):
        n = int(rng.integers(0, 5))
        s, d = rng.integers(0, 10, n), rng.integers(0, 10, n + int(rng.integers(0, 2) == 0 and n > 3))
        same = bool(rng.integers(0, 2))
        want = omap[O.validate_block_transfer(s, d, a, a if same else b)]
        try:
            P.validate_block_transfer(list(s), list(d), 8, 8, same)
            got = None
        except KvbmError as e:
            got = ErrorCode(e.code)
        assert got == want, (s, d, same)


# ------------------------------------------------------------------ Memcpy strategy == config 1 plumbing
KINDS = ["FC", "LWf", "LWs"]


def host_layout(mgr, kind, nb, storage=StorageKind.System, fill=0, **kw):
    """Returns (handle, oracle twin sharing the SAME numpy memory)."""
    okw = dict(nl=2, no=2, page=16, inner=128, dt=2)
    okw.update(kw)
    cfg = LayoutConfig(nb, okw["nl"], okw["no"], okw["page"], okw["inner"], dtype_width_bytes=okw["dt"])
    if kind == "FC":
        twin = O.Layout(O.FC, nb, okw["nl"], okw["no"], okw["page"], okw["inner"], okw["dt"], fill=fill)
        h = mgr.register_fully_contiguous(cfg, twin.buffers[0].ctypes.data, twin.buffers[0].size, storage)
    else:
        bd = O.BLOCK_IS_FIRST_DIM if kind == "LWf" else O.BLOCK_IS_SECOND_DIM
        twin = O.Layout(O.LW, nb, okw["nl"], okw["no"], okw["page"], okw["inner"], okw["dt"], block_dim=bd, fill=fill)
        h = mgr.register_layer_separate(cfg, [b.ctypes.data for b in twin.buffers], [b.size for b in twin.buffers],
                                        BlockDimension(bd), storage)
    return h, twin


@pytest.mark.parametrize("sk,dk", list(itertools.product(KINDS, repeat=2)))
@pytest.mark.parametrize("mode", [None, range(0, 1), range(1, 2)], ids=["full", "layer0", "layer1"])
def test_memcpy_strategy_matches_oracle_with_guards(mgr, sk, dk, mode):
    hs, src = host_layout(mgr, sk, 6)
    hd, dst = host_layout(mgr, dk, 6, storage=StorageKind.Pinned)
    _, ref = host_layout(mgr, dk, 6)
    src.fill_blocks([0, 1], -1)
    for t in (dst, ref):
        t.fill_blocks([2, 5], 0xFF)
    note = mgr.execute_transfer(hs, [0, 1], hd, [3, 4], TransferOptions(layer_range=mode))
    assert note.is_complete()                      # memcpy is synchronous: completed() (memcpy.rs:91-92)
    O.execute_memcpy_transfer(src, ref, [0, 1], [3, 4], mode)
    for a, b in zip(dst.buffers, ref.buffers):
        assert np.array_equal(a, b)
    want = src.block_checksums([0, 1], mode)
    got = dst.block_checksums([3, 4], mode)
    assert [got[3], got[4]] == [want[0], want[1]]


def test_execute_transfer_error_paths(mgr):
    hs, _ = host_layout(mgr, "FC", 4)
    hd, _ = host_layout(mgr, "FC", 4)
    h3, _ = host_layout(mgr, "FC", 4, nl=3)
    h64, _ = host_layout(mgr, "LWf", 4, inner=64)
    def code(fn):
        with pytest.raises(KvbmError) as e:
            fn()
        return e.value.code
    assert code(lambda: mgr.execute_transfer(hs, [0, 1], hd, [2])) == ErrorCode.LENGTH_MISMATCH
    assert code(lambda: mgr.execute_transfer(hs, [0, 1], hd, [2, 2])) == ErrorCode.DUPLICATE_DST
    assert code(lambda: mgr.execute_transfer(hs, [0, 1], hs, [1, 2])) == ErrorCode.OVERLAP
    assert code(lambda: mgr.execute_transfer(hs, [0, 9], hd, [1, 2])) == ErrorCode.RANGE
    assert code(lambda: mgr.execute_transfer(hs, [0], h3, [1])) == ErrorCode.INCOMPATIBLE
    assert code(lambda: mgr.execute_transfer(hs, [0], h64, [1])) == ErrorCode.INCOMPATIBLE
    assert code(lambda: mgr.execute_transfer(hs, [0], hd, [1], TransferOptions(layer_range=range(0, 3)))) == ErrorCode.RANGE
    assert code(lambda: mgr.execute_transfer(hs, [0], 0xdead, [1])) == ErrorCode.HANDLE
    assert code(lambda: mgr.execute_transfer(hs, [0], hd, [1], TransferOptions(cast_mode=1))) == ErrorCode.INCOMPATIBLE
    mgr.execute_transfer(hs, [], hd, [])           # empty transfer is fine


def test_config1_cpu_handoff_plumbing(mgr):
    # BASELINE configs[0]: Llama-3-8B geometry (32 KiB regions), LW/BlockIsSecondDim, random tables, fewer layers
    nb, n = 64, 32
    hs, src = host_layout(mgr, "LWs", nb, nl=4, inner=1024)
    hd, dst = host_layout(mgr, "LWs", nb, nl=4, inner=1024)
    rng = np.random.default_rng(1234)
    for b in src.buffers:
        b[:] = rng.integers(0, 256, b.size, dtype=np.uint8)
    sid = np.random.default_rng(0).permutation(nb)[:n]
    did = np.random.default_rng(1).permutation(nb)[:n]
    before = mgr.bytes_moved()
    mgr.execute_transfer(hs, list(sid), hd, list(did)).wait()
    assert mgr.bytes_moved() - before == n * 4 * 2 * 32768
    want = src.block_checksums(sid)
    for s, d in zip(sid, did):
        assert dst.block_checksum(int(d)) == want[int(s)]
    untouched = sorted(set(range(nb)) - set(int(x) for x in did))
    assert not dst.region_bytes(untouched[0], 0, 0).any()


def test_metadata_roundtrip_same_process_and_version_check(mgr):
    hs, src = host_layout(mgr, "LWs", 4)
    blob = mgr.export_metadata(hs)
    h2 = mgr.import_metadata(blob)
    assert h2 != hs
    for b, l, o in itertools.product(range(4), range(2), range(2)):
        assert mgr.memory_region(h2, b, l, o) == mgr.memory_region(hs, b, l, o)
    bad = bytearray(blob)
    bad[8] = 99           # version field (layout/serialize.rs: version checked on deserialize)
    with pytest.raises(KvbmError) as e:
        mgr.import_metadata(bytes(bad))
    assert e.value.code == ErrorCode.VERSION
    with pytest.raises(KvbmError):
        mgr.import_metadata(blob[:20])
    with pytest.raises(KvbmError):
        mgr.import_metadata(b"x" * len(blob))


def test_multicast_group_fails_loudly_without_a_driver():
    """No GPU / no libcuda here: the NVLS entry points must say so instead of pretending (no CPU fallback)."""
    from dynamo_b200.physical import KvbmError, MulticastGroup, multicast_supported
    import torch
    if torch.cuda.is_available():
        pytest.skip("CPU-only check")
    assert multicast_supported(0) is False
    with pytest.raises(KvbmError) as ei:
        MulticastGroup.create(2, 1 << 21)
    assert "driver" in str(ei.value).lower() or "cuda" in str(ei.value).lower()


def test_public_headers_are_plain_c(tmp_path):
    """The drop-in boundary is a C ABI: include/*.h must compile as C99 (no C++-isms, no torch types), and a C caller can
    name every struct a binding needs."""
    import shutil
    gcc = shutil.which("gcc")
    cuda_inc = "/usr/local/cuda/include"
    if not gcc or not os.path.exists(os.path.join(cuda_inc, "cuda_runtime_api.h")):
        pytest.skip("gcc or the CUDA headers are not installed")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    src = tmp_path / "abi.c"
    src.write_text('#include "kvbm_kernels.h"\n#include "kvbm_physical.h"\n#include "kvbm_router.h"\n'
                   "int main(void) {\n"
                   "  static kvbm_paged_layout l; static kvbm_paged_dst d; static kvbm_paged_copy_opts o;\n"
                   "  static kvbm_layout_config c; static kvbm_transfer_options t; static kvbm_transfer_plan p;\n"
                   "  (void)l; (void)d; (void)o; (void)c; (void)t; (void)p;\n"
                   "  return kvbm_kernels_is_stub_build() ? 1 : 0;\n}\n")
    r = subprocess.run([gcc, "-std=c99", "-Wall", "-Wextra", "-pedantic", "-Werror", "-fsyntax-only", "-I", os.path.join(root, "include"),
                        "-I", cuda_inc, str(src)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr


@pytest.mark.parametrize("kinds", [("LWs", "LWs"), ("FC", "FC"), ("LWs", "FC")])
def test_config1_sized_host_transfer_is_bit_exact_when_split_over_threads(mgr, kinds):
    """BASELINE configs[0] geometry (Llama-3-8B: 32 layers x K/V x 32 KiB regions), 96 of 192 blocks = 192 MiB: large enough
    that the Memcpy strategy splits the chunk list over host threads; BLAKE3 per block must equal the oracle's copy."""
    nb, n = 192, 96
    kw = dict(nl=32, no=2, page=16, inner=1024, dt=2)
    hs, src = host_layout(mgr, kinds[0], nb, **kw)
    hd, dst = host_layout(mgr, kinds[1], nb, **kw)
    _, ref = host_layout(mgr, kinds[1], nb, **kw)
    rng = np.random.default_rng(1234)
    for b in src.buffers:
        b[:] = rng.integers(0, 256, b.size, dtype=np.uint8)
    sid = np.random.default_rng(0).permutation(nb)[:n]
    did = np.random.default_rng(1).permutation(nb)[:n]
    note = mgr.execute_transfer(hs, sid.astype(np.uint64), hd, did.astype(np.uint64))
    assert note.is_complete()          # memcpy.rs:91-92: synchronous, already complete
    O.execute_memcpy_transfer(src, ref, sid, did)
    for got, want in zip(dst.buffers, ref.buffers):
        assert np.array_equal(got, want)
    # BLAKE3 by position (local_transfers.rs:108-171): destination block i carries the checksum of source block i
    want, got = src.block_checksums(sid.tolist()), dst.block_checksums(did.tolist())
    assert [got[int(d)] for d in did] == [want[int(s)] for s in sid]


@pytest.mark.parametrize("as_numpy", [True, False])
@pytest.mark.parametrize("replicate", [True, False])
def test_fanout_over_host_layouts_matches_oracle(mgr, as_numpy, replicate):
    """execute_fanout / CollectiveOps::broadcast semantics on the Memcpy strategy (host pools): every destination gets its own
    (src, dst) table -- or the same source blocks when replicating -- and equals the oracle's copy."""
    nb, n, nd = 24, 9, 3
    hs, src = host_layout(mgr, "LWs", nb)
    rng = np.random.default_rng(77)
    for b in src.buffers:
        b[:] = rng.integers(0, 256, b.size, dtype=np.uint8)
    dsts = [host_layout(mgr, "LWs", nb) for _ in range(nd)]
    refs = [host_layout(mgr, "LWs", nb)[1] for _ in range(nd)]
    sids = [rng.permutation(nb)[:n] for _ in range(nd)]
    if replicate:
        sids = [sids[0]] * nd
    dids = [rng.permutation(nb)[:n] for _ in range(nd)]
    conv = (lambda a: a.astype(np.uint64)) if as_numpy else (lambda a: [int(x) for x in a])
    note = mgr.execute_fanout(hs, [h for h, _ in dsts], [conv(s) for s in sids], [conv(d) for d in dids], replicate)
    assert note.is_complete()
    for (h, twin), ref, s, d in zip(dsts, refs, sids, dids):
        O.execute_memcpy_transfer(src, ref, s, d)
        for got, want in zip(twin.buffers, ref.buffers):
            assert np.array_equal(got, want)


def test_c_program_drives_the_host_abi(tmp_path):
    """tests/c/host_abi_smoke.c: a C99 program (no Python, no torch) registers pools, transfers, exchanges the
    SerializedLayout handshake and sees errors as codes -- the drop-in boundary used the way a cgo/JNI/Rust binding would."""
    import shutil
    gcc = shutil.which("gcc")
    cuda_inc = "/usr/local/cuda/include"
    if not gcc or not os.path.exists(os.path.join(cuda_inc, "cuda_runtime_api.h")):
        pytest.skip("gcc or the CUDA headers are not installed")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    libdir = os.path.join(root, "dynamo_b200")
    exe = tmp_path / "host_abi_smoke"
    r = subprocess.run([gcc, "-std=c99", "-Wall", "-Wextra", "-pedantic", "-Werror", "-I", os.path.join(root, "include"), "-I", cuda_inc,
                        os.path.join(root, "tests", "c", "host_abi_smoke.c"), "-o", str(exe), "-L", libdir, "-lkvbm_physical",
                        "-lkvbm_kernels", f"-Wl,-rpath,{libdir}"], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    r = subprocess.run([str(exe)], capture_output=True, text=True, timeout=60)
    assert r.returncode == 0 and "host ABI ok" in r.stdout, r.stdout + r.stderr


# ------------------------------------------------------------------ round-2 additions
def test_router_library_exports_every_declared_symbol():
    import re
    from dynamo_b200 import router as R
    syms = _exported(R.ROUTER_SO)
    txt = open(os.path.join(ROOT, "include", "kvbm_router.h")).read()
    declared = set(re.findall(r"\b((?:kvr|dynamo)_[a-z0-9_]+)\s*\(", txt)) - {"dynamo_kv_event_callback"}
    assert {"dynamo_llm_init", "dynamo_kv_event_publish_stored", "dynamo_kv_event_publish_removed", "kvr_tree_find_matches"} <= declared
    assert declared <= syms, declared - syms


def _blob_with_identity(blob: bytes, identity: int) -> bytes:
    """BlobHeader (transfer_manager.cpp): magic[8] version fully_contiguous block_dim storage device_id n_allocs (6 x u32)
    worker_id pid (2 x u64) -> the process identity sits at byte offset 40."""
    import struct
    return blob[:40] + struct.pack("<Q", identity) + blob[48:]


def test_remote_host_layout_without_mapping_is_descriptor_only(mgr):
    """ADVICE r1: a System/Pinned layout exported by ANOTHER process has no IPC handle; its addresses mean nothing here.
    It is importable as a descriptor (geometry + memory_region arithmetic) but every transfer touching it is refused."""
    cfg = std_cfg(4)
    buf = np.zeros(cfg.required_bytes(), dtype=np.uint8)
    local = mgr.register_fully_contiguous(cfg, buf.ctypes.data, buf.size, StorageKind.System)
    other = np.zeros(cfg.required_bytes(), dtype=np.uint8)
    h_other = mgr.register_fully_contiguous(cfg, other.ctypes.data, other.size, StorageKind.System)
    blob = mgr.export_metadata(h_other)
    same = mgr.import_metadata(blob)                                   # same process: usable as before
    mgr.execute_transfer(local, [0], same, [1])
    import struct
    me = struct.unpack("<Q", blob[40:48])[0]
    assert me >> 32, "the process identity must carry a nonce above the pid (pid alone collides across PID namespaces)"
    foreign = mgr.import_metadata(_blob_with_identity(blob, me ^ (0x5a5a << 32)))   # same pid, different process nonce
    assert mgr.memory_region(foreign, 1, 0, 0)[1] == cfg.region_size()
    for a, b in ((local, foreign), (foreign, local)):
        with pytest.raises(KvbmError) as e:
            mgr.execute_transfer(a, [0], b, [1])
        assert e.value.code == ErrorCode.UNSUPPORTED and "not addressable" in e.value.msg
    # ... unless the importer names its OWN mapping of that memory (shared memory between worker processes): then the layout
    # is a usable remote -- a push into it is select_strategy's NixlWrite, executed as the memcpy it is on one host
    view = np.zeros(cfg.required_bytes(), dtype=np.uint8)               # stands for this process's mapping of the peer's pool
    mapped = mgr.import_metadata(_blob_with_identity(blob, me ^ (0x5a5a << 32)), local_bases=[view.ctypes.data])
    buf[:] = np.arange(buf.size, dtype=np.uint64).astype(np.uint8)
    mgr.execute_transfer(local, [2], mapped, [3])
    bpb = cfg.required_bytes() // cfg.num_blocks
    assert np.array_equal(view[3 * bpb:4 * bpb], buf[2 * bpb:3 * bpb]) and not view[:3 * bpb].any()
    plan = mgr.select_strategy(local, mapped)
    assert not plan.two_hop and plan.first == TransferStrategy.NixlWrite
    assert mgr.select_strategy(mapped, local).first == TransferStrategy.NixlReadFlipped
    assert mgr.select_strategy(local, same).first == TransferStrategy.Memcpy
    with pytest.raises(KvbmError) as e:                                 # both sides another process's: the reference's error
        mgr.execute_transfer(mapped, [0], mapped, [1])
    assert "Both src and dst are remote" in e.value.msg
    with pytest.raises(KvbmError) as e:                                 # one address per allocation
        mgr.import_metadata(_blob_with_identity(blob, me ^ (0x5a5a << 32)), local_bases=[view.ctypes.data, view.ctypes.data])
    assert "allocations" in e.value.msg


def test_two_hop_plan_needs_a_bounce_buffer_and_kv_layout_overrides_are_rejected(mgr):
    """executor/mod.rs:514-527 error texts; transfer/mod.rs:128-147 rejects pairs that would need a transformation."""
    from dynamo_b200.physical import TransferOptions
    cfg = std_cfg(4)
    a = np.zeros(cfg.required_bytes(), dtype=np.uint8)
    b = np.zeros(cfg.required_bytes(), dtype=np.uint8)
    ha = mgr.register_fully_contiguous(cfg, a.ctypes.data, a.size, StorageKind.System)
    hb = mgr.register_fully_contiguous(cfg, b.ctypes.data, b.size, StorageKind.System)
    # Unknown <-> known is "Unsupported" (executor/mod.rs:56-60) and rejected with the reference's text
    with pytest.raises(KvbmError) as e:
        mgr.execute_transfer(ha, [0], hb, [1], TransferOptions(dst_kv_layout=2))
    assert e.value.code == ErrorCode.UNSUPPORTED and "Layout transformation not supported: src=Unknown, dst=UniversalPP" in e.value.msg
    # a supported pair needs num_heads (config.rs:118-126) ...
    with pytest.raises(KvbmError) as e:
        mgr.execute_transfer(ha, [0], hb, [1], TransferOptions(src_kv_layout=4, dst_kv_layout=1))
    assert e.value.code == ErrorCode.CONFIG and "num_heads_required_for_kv_block_layout" in e.value.msg
    mgr.execute_transfer(ha, [0], hb, [1], TransferOptions(src_kv_layout=2, dst_kv_layout=2))   # same layout: plain copy
    # ... and a CUDA strategy: the permuting launch has no CPU twin in the product (the oracle is test infrastructure)
    cfg_h = std_cfg(4, num_heads=2)
    hc = mgr.register_fully_contiguous(cfg_h, a.ctypes.data, a.size, StorageKind.System)
    hd = mgr.register_fully_contiguous(cfg_h, b.ctypes.data, b.size, StorageKind.System)
    with pytest.raises(KvbmError) as e:
        mgr.execute_transfer(hc, [0], hd, [1], TransferOptions(src_kv_layout=4, dst_kv_layout=1))
    assert e.value.code == ErrorCode.UNSUPPORTED and "only on the CUDA strategies" in e.value.msg
    # Device<->System stay "not supported", exactly like strategy.rs:150-160 (there is no implicit staging)
    dev_like = mgr.register_fully_contiguous(cfg, a.ctypes.data, a.size, StorageKind.Device)
    with pytest.raises(KvbmError) as e:
        mgr.execute_transfer(dev_like, [0], hb, [1])
    assert e.value.code == ErrorCode.UNSUPPORTED and "Device to System" in e.value.msg
    with pytest.raises(KvbmError) as e:
        mgr.execute_transfer(hb, [0], dev_like, [1])
    assert e.value.code == ErrorCode.UNSUPPORTED and "System to Device" in e.value.msg
    # capabilities: with GPU RDMA disallowed a cross-GPU D2D becomes TwoHop{D2H, Pinned, H2D}; it needs a CUDA manager and a
    # bounce buffer -- on this host-only manager the plan is selected and then fails loudly for the right reason
    mgr.set_capabilities(allow_gpu_rdma=False)
    try:
        d0 = mgr.register_fully_contiguous(cfg, a.ctypes.data, a.size, StorageKind.Device, 0)
        d1 = mgr.register_fully_contiguous(cfg, b.ctypes.data, b.size, StorageKind.Device, 1)
        with pytest.raises(KvbmError) as e:
            mgr.execute_transfer(d0, [0], d1, [1])
        assert e.value.code == ErrorCode.CUDA and "no CPU fallback" in e.value.msg
    finally:
        mgr.set_capabilities(allow_gpu_rdma=True)


def test_select_transform_kernel_and_requires_transform_kats():
    """transfer/executor/mod.rs:578-655 and layout/kv_block_layout.rs:376-391, case by case."""
    from dynamo_b200.kernels import KvBlockLayout as KV
    from dynamo_b200.physical import TransformKernel as T, requires_transform, select_transform_kernel as sel
    assert sel(KV.OperationalNHD, KV.OperationalNHD) == T.NONE and sel(KV.UniversalTP, KV.UniversalTP) == T.NONE
    assert sel(KV.OperationalNHD, KV.UniversalTP) == T.BlockToUniversal and sel(KV.OperationalHND, KV.UniversalTP) == T.BlockToUniversal
    assert sel(KV.OperationalNHD, KV.UniversalPP) == T.BlockToUniversal and sel(KV.OperationalHND, KV.UniversalPP) == T.BlockToUniversal
    assert sel(KV.UniversalTP, KV.OperationalNHD) == T.UniversalToBlock and sel(KV.UniversalTP, KV.OperationalHND) == T.UniversalToBlock
    assert sel(KV.UniversalPP, KV.OperationalNHD) == T.UniversalToBlock and sel(KV.UniversalPP, KV.OperationalHND) == T.UniversalToBlock
    assert sel(KV.OperationalNHD, KV.OperationalHND) == T.OperationalTranspose
    assert sel(KV.OperationalHND, KV.OperationalNHD) == T.OperationalTranspose
    assert sel(KV.Unknown, KV.OperationalNHD) == T.Unsupported and sel(KV.OperationalNHD, KV.Unknown) == T.Unsupported
    assert sel(KV.Custom, KV.OperationalNHD) == T.Unsupported
    assert sel(KV.Custom, KV.Custom) == T.Unsupported     # the C enum does not carry Custom's dimension order: never assumed equal
    assert sel(KV.UniversalTP, KV.UniversalPP) == T.Unsupported and sel(KV.UniversalPP, KV.UniversalTP) == T.Unsupported  # :87-91 TODO
    assert sel(KV.Unknown, KV.Unknown) == T.NONE
    assert not requires_transform(KV.OperationalNHD, KV.OperationalNHD)
    assert requires_transform(KV.OperationalNHD, KV.UniversalTP) and requires_transform(KV.OperationalHND, KV.OperationalNHD)
    assert requires_transform(KV.Unknown, KV.OperationalNHD) and requires_transform(KV.OperationalNHD, KV.Unknown)
    assert not requires_transform(KV.Unknown, KV.Unknown)


def test_kv_block_layout_of_a_layout_validates_and_travels_with_the_metadata(mgr):
    """fully_contiguous.rs:83-88 / layer_separate.rs:91-101 / config.rs:114-140; serialize.rs carries kv_block_layout."""
    import json
    from dynamo_b200.kernels import KvBlockLayout as KV
    cfg = std_cfg(4, num_heads=2)
    a = np.zeros(cfg.required_bytes(), dtype=np.uint8)
    fc = mgr.register_fully_contiguous(cfg, a.ctypes.data, a.size, StorageKind.System)
    assert mgr.kv_block_layout(fc) == KV.Unknown        # builder default
    mgr.set_kv_block_layout(fc, KV.UniversalTP)
    assert mgr.kv_block_layout(fc) == KV.UniversalTP
    # same-process metadata round trip keeps it
    again = mgr.import_metadata(mgr.export_metadata(fc))
    assert mgr.kv_block_layout(again) == KV.UniversalTP
    # the reference's JSON descriptor names it ("kv_block_layout": "UniversalTP")
    text = mgr.layout_descriptor_json(fc)
    desc = json.loads(text)
    assert mgr.kv_block_layout(mgr.import_descriptor_json(text)) == KV.UniversalTP
    assert "UniversalTP" in json.dumps(desc)
    # layer-separate layouts only carry operational formats
    lay = [np.zeros(cfg.required_bytes() // cfg.num_layers, dtype=np.uint8) for _ in range(cfg.num_layers)]
    lw = mgr.register_layer_separate(cfg, [x.ctypes.data for x in lay], [x.size for x in lay], BlockDimension.BlockIsFirstDim, StorageKind.System)
    mgr.set_kv_block_layout(lw, KV.OperationalNHD)
    with pytest.raises(KvbmError) as e:
        mgr.set_kv_block_layout(lw, KV.UniversalTP)
    assert e.value.code == ErrorCode.CONFIG and "fully contiguous" in e.value.msg
    # num_heads is required, and must divide inner_dim
    plain = mgr.register_fully_contiguous(std_cfg(4), a.ctypes.data, a.size, StorageKind.System)
    with pytest.raises(KvbmError) as e:
        mgr.set_kv_block_layout(plain, KV.OperationalNHD)
    assert "num_heads_required_for_kv_block_layout" in e.value.msg
    odd = mgr.register_fully_contiguous(std_cfg(4, num_heads=3), a.ctypes.data, a.size, StorageKind.System)
    with pytest.raises(KvbmError) as e:
        mgr.set_kv_block_layout(odd, KV.OperationalNHD)
    assert "inner_dim_must_be_divisible" in e.value.msg
    with pytest.raises(KvbmError):
        mgr.set_kv_block_layout(0xdead, KV.OperationalNHD)
    # layouts whose own formats differ: the transfer is a transformation, not a copy -> needs CUDA here
    b = np.zeros(cfg.required_bytes(), dtype=np.uint8)
    nhd = mgr.register_fully_contiguous(cfg, b.ctypes.data, b.size, StorageKind.System)
    mgr.set_kv_block_layout(nhd, KV.OperationalNHD)
    with pytest.raises(KvbmError) as e:
        mgr.execute_transfer(nhd, [0], fc, [1])
    assert e.value.code == ErrorCode.UNSUPPORTED and "only on the CUDA strategies" in e.value.msg


def test_layout_ids_are_reused_and_never_overwrite_a_live_layout(mgr):
    """ADVICE r1: next_layout_id is a u16; registering past 65535 must not clobber a live layout."""
    cfg = std_cfg(2)
    buf = np.zeros(cfg.required_bytes(), dtype=np.uint8)
    keep = mgr.register_fully_contiguous(cfg, buf.ctypes.data, buf.size, StorageKind.System)
    seen = set()
    for _ in range(66000):                                              # wraps the 16-bit id space once
        h = mgr.register_fully_contiguous(cfg, buf.ctypes.data, buf.size, StorageKind.System)
        assert h != keep and h & 0xFFFF != 0
        seen.add(h & 0xFFFF)
        mgr.unregister(h)
    assert len(seen) > 60000
    assert mgr.memory_region(keep, 1, 0, 0)[1] == cfg.region_size()    # the early layout is still the same layout


def test_ctypes_mirrors_have_the_c_struct_layouts(tmp_path):
    """A Python mirror that silently drops (or mis-orders) trailing fields still "works" with zeros -- round 2 lost the
    per-destination flag arrays that way.  Compile a C program that prints sizeof / offsetof of the option structs and
    compare with the ctypes mirrors field by field."""
    import shutil
    from dynamo_b200 import physical as PH
    gcc = shutil.which("gcc")
    cuda_inc = "/usr/local/cuda/include"
    if not gcc or not os.path.exists(os.path.join(cuda_inc, "cuda_runtime_api.h")):
        pytest.skip("gcc or the CUDA headers are not installed")
    structs = {"kvbm_paged_copy_opts": K.PagedCopyOpts, "kvbm_paged_layout": K.PagedLayout, "kvbm_paged_dst": K.PagedDst,
               "kvbm_transfer_options": PH._COptions, "kvbm_layout_config": PH._CConfig, "kvbm_transfer_plan": PH._CPlan,
               "kvbm_transfer_capabilities": PH._CCaps}
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "kvbm_kernels.h"', '#include "kvbm_physical.h"', "int main(void) {"]
    for cname, mirror in structs.items():
        lines.append(f'  printf("{cname} sizeof %zu\\n", sizeof({cname}));')
        for fname, _ in mirror._fields_:
            lines.append(f'  printf("{cname} {fname} %zu\\n", offsetof({cname}, {fname}));')
    lines += ["  return 0;", "}"]
    src, exe = tmp_path / "layout.c", tmp_path / "layout"
    src.write_text("\n".join(lines))
    r = subprocess.run([gcc, "-std=c99", "-I", os.path.join(ROOT, "include"), "-I", cuda_inc, "-o", str(exe), str(src)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr        # a field the mirror names but the header lacks fails right here
    out = subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout
    c = {(a, b): int(v) for a, b, v in (ln.split() for ln in out.splitlines())}
    for cname, mirror in structs.items():
        assert C.sizeof(mirror) == c[(cname, "sizeof")], f"{cname}: ctypes {C.sizeof(mirror)} vs C {c[(cname, 'sizeof')]} bytes"
        for fname, _ in mirror._fields_:
            assert getattr(mirror, fname).offset == c[(cname, fname)], f"{cname}.{fname}"


@pytest.mark.parametrize("dims", [(3, 2, 4, 5, 16), (2, 1, 16, 8, 256), (80, 2, 16, 8, 256), (1, 2, 7, 3, 48), (61, 1, 64, 1, 1152)],
                         ids=lambda d: "nl%d-no%d-nt%d-nh%d-row%d" % d)
def test_permute_stride_table_spells_every_kv_block_layout(dims):
    """The whole address arithmetic of kvbm_paged_permute_kernel is one stride table per side (kvbm_kernels.cu,
    fill_permute_side).  Checked here without a GPU: moving each row with the table's offsets must equal the oracle's
    dim_order permutation (kv_block_layout.rs:85-95) for every ordered pair of formats."""
    from dynamo_b200.kernels import KvBlockLayout as KV
    nl, no, nt, nh, row = dims
    region = nt * nh * row
    block = nl * no * region

    def row_offsets(kv):
        uni, lstep, ostep, hs, ts = K.permute_strides(kv, nl, no, nh, nt, row, block, region)
        l, o, h, t = np.meshgrid(np.arange(nl), np.arange(no), np.arange(nh), np.arange(nt), indexing="ij")
        base = (l * lstep + o * ostep) if uni else (l * no + o) * region      # operational blocks: regions in (layer, outer) order
        return (base + h * hs + t * ts).reshape(-1)

    rng = np.random.default_rng(nl * 7 + nh)
    src = rng.integers(0, 256, block, dtype=np.uint8)
    offs = {kv: row_offsets(kv) for kv in (KV.UniversalTP, KV.UniversalPP, KV.OperationalHND, KV.OperationalNHD)}
    for kv, off in offs.items():                      # a bijection onto the block's rows
        assert np.array_equal(np.sort(off), np.arange(nl * no * nh * nt) * row), kv
    col = np.arange(row)
    for a, oa in offs.items():
        for b, ob in offs.items():
            dst = np.zeros_like(src)
            dst[(ob[:, None] + col).reshape(-1)] = src[(oa[:, None] + col).reshape(-1)]
            assert np.array_equal(dst, O.kv_layout_permute(src, int(a), int(b), nl, no, nt, nh, row)), (a, b)
    assert K.permute_strides(KV.Unknown, nl, no, nh, nt, row, block, region) is None
    assert K.permute_strides(KV.Custom, nl, no, nh, nt, row, block, region) is None
    assert K.permute_strides(KV.OperationalNHD, nl, no, nh, nt, row, block + 8, region) is None      # strides must be multiples of 16


def test_manager_is_reentrant_from_many_threads(mgr):
    """SURVEY 8(b) threading: the reference is called from arbitrary tokio worker threads.  Concurrent execute_transfer,
    register / unregister and notification polling on ONE manager must give the bytes a sequential run gives."""
    import threading
    nb, threads, rounds = 64, 8, 40
    cfg = std_cfg(nb)
    src_t, dst_t, ref_t = (O.Layout(O.FC, nb, 2, 2, 16, 128, 2) for _ in range(3))
    rng = np.random.default_rng(3)
    src_t.buffers[0][:] = rng.integers(0, 256, src_t.buffers[0].size, dtype=np.uint8)
    hs = mgr.register_fully_contiguous(cfg, src_t.buffers[0].ctypes.data, src_t.buffers[0].size, StorageKind.System)
    hd = mgr.register_fully_contiguous(cfg, dst_t.buffers[0].ctypes.data, dst_t.buffers[0].size, StorageKind.Pinned)
    per = nb // threads                                      # thread t owns destination blocks [t*per, (t+1)*per)
    plans = [[(list(map(int, np.random.default_rng(100 * t + r).integers(0, nb, per))),
               list(map(int, t * per + np.random.default_rng(7 * t + r).permutation(per)))) for r in range(rounds)] for t in range(threads)]
    errors = []

    def run(t):
        try:
            scratch = np.zeros(cfg.required_bytes(), dtype=np.uint8)
            for sid, did in plans[t]:
                note = mgr.execute_transfer(hs, sid, hd, did)
                assert note.is_complete()
                h = mgr.register_fully_contiguous(cfg, scratch.ctypes.data, scratch.size, StorageKind.System)   # churn the layout table
                assert mgr.memory_region(h, 1, 1, 1)[1] == cfg.region_size()
                mgr.unregister(h)
        except Exception as e:  # pragma: no cover
            errors.append(repr(e))

    ts = [threading.Thread(target=run, args=(t,)) for t in range(threads)]
    for th in ts:
        th.start()
    for th in ts:
        th.join()
    assert errors == []
    for t in range(threads):                                 # destinations are disjoint per thread: order across threads is irrelevant
        for sid, did in plans[t]:
            O.execute_memcpy_transfer(src_t, ref_t, sid, did)
    assert np.array_equal(dst_t.buffers[0], ref_t.buffers[0])


def test_host_libraries_are_race_free_under_thread_sanitizer(tmp_path):
    """SURVEY 5 (race detection): tests/c/race_check.cpp, built from the library SOURCES with -fsanitize=thread, hammers the
    host-only TransferManager (execute / register / unregister / notifications) and the KV event publisher (RadixTree +
    JSON sinks) from 8 threads.  A data race makes ThreadSanitizer print a report and the run exit non-zero."""
    import pyarrow
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    probe = tmp_path / "p.cpp"
    probe.write_text("int main(){return 0;}\n")
    if subprocess.run(["g++", "-fsanitize=thread", str(probe), "-o", str(tmp_path / "p")], capture_output=True).returncode != 0:
        pytest.skip("g++ has no ThreadSanitizer runtime here")
    xxh = os.path.join(pyarrow.get_include(), "arrow", "vendored", "xxhash")
    cuda = os.environ.get("CUDA_HOME", "/usr/local/cuda")
    exe = tmp_path / "race_check"
    src = [os.path.join(root, p) for p in ("tests/c/race_check.cpp", "dynamo_b200/csrc/host/transfer_manager.cpp",
                                           "dynamo_b200/csrc/host/multicast.cpp", "dynamo_b200/csrc/router/radix_tree.cpp",
                                           "dynamo_b200/csrc/router/kv_events.cpp")]
    cmd = ["g++", "-std=c++17", "-O1", "-g", "-fsanitize=thread", "-fno-omit-frame-pointer", "-pthread", "-I", os.path.join(root, "include"),
           "-I", os.path.join(cuda, "include"), "-I", xxh, *src, "-L", os.path.join(root, "dynamo_b200"), "-lkvbm_kernels",
           "-L", os.path.join(cuda, "lib64"), "-lcudart", "-ldl", f"-Wl,-rpath,{os.path.join(root, 'dynamo_b200')}",
           f"-Wl,-rpath,{os.path.join(cuda, 'lib64')}", "-o", str(exe)]
    b = subprocess.run(cmd, capture_output=True, text=True)
    assert b.returncode == 0, b.stderr[-2000:]
    r = subprocess.run([str(exe)], capture_output=True, text=True, timeout=300, env=dict(os.environ, TSAN_OPTIONS="halt_on_error=1"))
    assert r.returncode == 0 and "race check ok" in r.stdout and "ThreadSanitizer" not in r.stderr, (r.stdout[-500:], r.stderr[-3000:])


def test_metadata_importers_survive_corrupted_input_under_asan_ubsan(tmp_path):
    """The three importers parse bytes that come from other processes.  tests/c/fuzz_import.cpp mutates valid exports (bit
    flips, truncation, 0xff runs, inflated JSON numbers ...) 20 000 times per format and imports them into fresh managers,
    built from the library sources with -fsanitize=address,undefined: an import may only succeed or return an error code.
    (This harness found a length_error escaping the C ABI through an unchecked num_layers; layout sizes are now
    overflow-checked like the reference's saturating_mul, config.rs:64-82.)"""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    probe = tmp_path / "p.cpp"
    probe.write_text("int main(){return 0;}\n")
    if subprocess.run(["g++", "-fsanitize=address,undefined", str(probe), "-o", str(tmp_path / "p")], capture_output=True).returncode != 0:
        pytest.skip("g++ has no AddressSanitizer runtime here")
    cuda = os.environ.get("CUDA_HOME", "/usr/local/cuda")
    exe = tmp_path / "fuzz_import"
    src = [os.path.join(root, p) for p in ("tests/c/fuzz_import.cpp", "dynamo_b200/csrc/host/transfer_manager.cpp", "dynamo_b200/csrc/host/multicast.cpp")]
    cmd = ["g++", "-std=c++17", "-O1", "-g", "-fsanitize=address,undefined", "-fno-sanitize-recover=undefined", "-fno-omit-frame-pointer", "-pthread",
           "-I", os.path.join(root, "include"), "-I", os.path.join(cuda, "include"), *src, "-L", os.path.join(root, "dynamo_b200"), "-lkvbm_kernels",
           "-L", os.path.join(cuda, "lib64"), "-lcudart", "-ldl", f"-Wl,-rpath,{os.path.join(root, 'dynamo_b200')}",
           f"-Wl,-rpath,{os.path.join(cuda, 'lib64')}", "-o", str(exe)]
    b = subprocess.run(cmd, capture_output=True, text=True)
    assert b.returncode == 0, b.stderr[-2000:]
    r = subprocess.run([str(exe), "20000"], capture_output=True, text=True, timeout=600, env=dict(os.environ, ASAN_OPTIONS="detect_leaks=1"))
    assert r.returncode == 0 and "fuzz ok" in r.stdout, (r.stdout[-500:], r.stderr[-3000:])


def test_layout_sizes_are_overflow_checked(mgr):
    """config.rs:64-82 multiplies with saturating_mul; a config whose byte size does not fit can never be registered."""
    huge = LayoutConfig(num_blocks=2**40, num_layers=2**20, outer_dim=2, page_size=2**10, inner_dim=2**10, dtype_width_bytes=2)
    assert huge.required_bytes() == 2**64 - 1
    buf = np.zeros(64, dtype=np.uint8)
    with pytest.raises(KvbmError) as e:
        mgr.register_fully_contiguous(huge, buf.ctypes.data, 2**63, StorageKind.System)
    assert e.value.code == ErrorCode.CONFIG and "overflow" in e.value.msg
    many_layers = std_cfg(1, num_layers=2**30)
    with pytest.raises(KvbmError) as e:
        mgr.register_fully_contiguous(many_layers, buf.ctypes.data, 2**62, StorageKind.System)
    assert e.value.code == ErrorCode.CONFIG
