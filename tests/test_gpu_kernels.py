"""GPU parity tests for the six reference symbols, driven through the C ABI (ctypes).

Mirrors the reference's kernel tests:
  lib/kvbm-kernels/tests/memcpy_batch.rs       (no-ops, H2D+D2H roundtrips over all 3 modes, KAT patterns)
  lib/kvbm-kernels/tests/kernel_roundtrip.rs   (permute roundtrip x dtype x layout, poison fill, empty batch)
  lib/kvbm-kernels/src/tensor_kernels.rs:286-  (universal_roundtrip with +0.25 encoded values)
and compares every result bit-for-bit with the CPU oracle, and with what the reference's own kernels
(tensor_kernels.cu compiled unmodified for sm_100) produced on a B200 for the same inputs, stored under
tests/golden/ by tests/golden/make_reference_goldens.py.
"""
import hashlib
import os

import numpy as np
import pytest
import torch

from dynamo_b200 import kernels as K
from oracle import oracle as O
from tests import kats
from tests.gpu_util import dev_ptr_table, dev_u8, pinned_u8, stream_ptr

pytestmark = pytest.mark.gpu

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
REF_COPY_SHA256 = os.path.join(GOLDEN, "reference_vectorized_copy_sha256.npy")
REF_POSITION_BLOCKS = os.path.join(GOLDEN, "reference_block_from_universal_position_encoded.npy")


def reference_copy_case():
    """512 pairs of one 32 KiB (block, layer, outer) region of Llama-3-8B bf16, gathered from a 1024-region pool and
    scattered in a shuffled order.  Seeded: the reference kernel's output for exactly these inputs is stored."""
    size, pairs = 32768, 512
    rng = np.random.default_rng(139)
    pool = rng.integers(0, 256, (pairs * 2, size), dtype=np.uint8)
    return size, pairs, pool, rng.permutation(pairs * 2)[:pairs], rng.permutation(pairs)


def launch_reference_copy_case(launch):
    """Runs `launch` (a kvbm_kernels_launch_vectorized_copy) on reference_copy_case(); returns (output, pool, perm, dperm)
    on the device, output[dperm[i]] being the copy of pool[perm[i]]."""
    size, pairs, pool, perm, dperm = reference_copy_case()
    pool = torch.from_numpy(pool).cuda()
    out = dev_u8(pairs * size).view(pairs, size)
    st = dev_ptr_table([pool[int(i)].data_ptr() for i in perm])
    dt = dev_ptr_table([out[int(i)].data_ptr() for i in dperm])
    assert launch(st.data_ptr(), dt.data_ptr(), size, pairs, stream_ptr()) == 0
    torch.cuda.synchronize()
    return out, pool, torch.from_numpy(perm).cuda(), torch.from_numpy(dperm).cuda()


def row_sha256(rows: np.ndarray) -> np.ndarray:
    return np.stack([np.frombuffer(hashlib.sha256(r.tobytes()).digest(), dtype=np.uint8) for r in rows])


def block_from_universal_position_encoded(launch_block_from_universal, layout):
    """The position-encoded universal tensor of kernel_roundtrip.rs:418-493 scattered into its nl*no chunks by the given
    kvbm_kernels_launch_block_from_universal; returns the chunks as float32 arrays."""
    d = kats.PERMUTE_DIMS
    uni = kats.position_encoded_universal(**d)
    du = torch.from_numpy(uni.reshape(-1).view(np.uint8).copy()).cuda()
    ut = dev_ptr_table([du.data_ptr()])
    chunks = [dev_u8(w.nbytes, fill=0xDE) for w in kats.make_blocks(uni, layout)]
    bt = dev_ptr_table([t.data_ptr() for t in chunks])
    rc = launch_block_from_universal(ut.data_ptr(), bt.data_ptr(), 1, d["nh"], d["nl"], d["no"], d["nt"], d["hd"], 2, layout,
                                     stream_ptr())
    assert rc == 0
    torch.cuda.synchronize()
    return [c.cpu().numpy().view(np.float32) for c in chunks]


def test_not_a_stub_and_batch_query():
    assert K.is_using_stubs() is False
    assert K.is_memcpy_batch_available() is True   # built with CUDA 12.9


# ---------------------------------------------------------------- K4 memcpy_batch
@pytest.mark.parametrize("mode", list(K.MemcpyBatchMode))
def test_memcpy_batch_noops(mode):
    s = torch.cuda.Stream()
    assert K.memcpy_batch(None, None, 128, 0, mode, stream_ptr(s)) == 0   # memcpy_batch.rs:238-266
    assert K.memcpy_batch(None, None, 0, 5, mode, stream_ptr(s)) == 0     # memcpy_batch.rs:268-299
    assert K.memcpy_batch(None, None, 128, 3, mode, stream_ptr(s)) == K.CUDA_ERROR_INVALID_VALUE


@pytest.mark.parametrize("name,size,pairs,gen", kats.COPY_KATS, ids=[k[0] for k in kats.COPY_KATS])
@pytest.mark.parametrize("mode", list(K.MemcpyBatchMode))
def test_memcpy_batch_h2d_d2h_roundtrip(name, size, pairs, gen, mode):
    # memcpy_batch.rs:120-225: pinned -> device -> pinned (non-default stream is required by the batch API)
    s = torch.cuda.Stream()
    data = kats.copy_kat_data(size, pairs, gen)
    src = [pinned_u8(d) for d in data]
    dev = [dev_u8(size) for _ in range(pairs)]
    dst = [pinned_u8(np.zeros(size, dtype=np.uint8)) for _ in range(pairs)]
    torch.cuda.synchronize()
    rc = K.memcpy_batch([t.data_ptr() for t in src], [t.data_ptr() for t in dev], size, pairs, mode, stream_ptr(s))
    assert rc == 0
    rc = K.memcpy_batch([t.data_ptr() for t in dev], [t.data_ptr() for t in dst], size, pairs, mode, stream_ptr(s))
    assert rc == 0
    s.synchronize()
    for d, out in zip(data, dst):
        assert np.array_equal(out.numpy(), d)


# ---------------------------------------------------------------- K1 vectorized_copy
def test_vectorized_copy_noops_and_null():
    sp = stream_ptr()
    assert K.vectorized_copy(0, 0, 128, 0, sp) == 0
    assert K.vectorized_copy(0, 0, 0, 4, sp) == 0
    assert K.vectorized_copy(0, 0, 128, 4, sp) == K.CUDA_ERROR_INVALID_VALUE


@pytest.mark.parametrize("name,size,pairs,gen", kats.COPY_KATS, ids=[k[0] for k in kats.COPY_KATS])
@pytest.mark.parametrize("table_kind", ["device", "pinned"])
def test_vectorized_copy_d2d_kats(name, size, pairs, gen, table_kind):
    data = kats.copy_kat_data(size, pairs, gen)
    src = [torch.from_numpy(d).cuda() for d in data]
    dst = [dev_u8(size, fill=0xDE) for _ in range(pairs)]
    if table_kind == "device":
        st, dt = dev_ptr_table([t.data_ptr() for t in src]), dev_ptr_table([t.data_ptr() for t in dst])
    else:  # pointer tables may be pinned host memory (tensor_kernels.cu:51-53)
        st = torch.tensor([t.data_ptr() for t in src], dtype=torch.int64).pin_memory()
        dt = torch.tensor([t.data_ptr() for t in dst], dtype=torch.int64).pin_memory()
    assert K.vectorized_copy(st.data_ptr(), dt.data_ptr(), size, pairs, stream_ptr()) == 0
    torch.cuda.synchronize()
    want = [np.zeros(size, dtype=np.uint8) for _ in range(pairs)]
    O.vectorized_copy(data, want, size)
    for w, out in zip(want, dst):
        assert np.array_equal(out.cpu().numpy(), w)


def test_vectorized_copy_h2d_and_d2h_pinned():
    size, pairs = 32768, 40
    rng = np.random.default_rng(5)
    data = [rng.integers(0, 256, size, dtype=np.uint8) for _ in range(pairs)]
    src = [pinned_u8(d) for d in data]
    dev = [dev_u8(size) for _ in range(pairs)]
    back = [pinned_u8(np.zeros(size, dtype=np.uint8)) for _ in range(pairs)]
    a, b, c = (dev_ptr_table([t.data_ptr() for t in x]) for x in (src, dev, back))
    assert K.vectorized_copy(a.data_ptr(), b.data_ptr(), size, pairs, stream_ptr()) == 0
    assert K.vectorized_copy(b.data_ptr(), c.data_ptr(), size, pairs, stream_ptr()) == 0
    torch.cuda.synchronize()
    for d, out in zip(data, back):
        assert np.array_equal(out.numpy(), d)


@pytest.mark.parametrize("size", [1, 7, 15, 16, 17, 999, 4096 + 3, 16384, 16384 + 16, 100_000])
def test_vectorized_copy_every_alignment_phase(size):
    # any alignment / any size must work (tensor_kernels.cu:511-540; 999 B regression in memcpy_batch.rs:401)
    base = torch.from_numpy((np.arange(2 * size + 64, dtype=np.int64) * 7 % 251).astype(np.uint8)).cuda()
    host = base.cpu().numpy()
    for so in (0, 1, 4, 8, 13):
        for do in (0, 2, 4, 8, 15):
            dst = dev_u8(size + 64, fill=0xAA)
            st = dev_ptr_table([base.data_ptr() + so])
            dt = dev_ptr_table([dst.data_ptr() + do])
            assert K.vectorized_copy(st.data_ptr(), dt.data_ptr(), size, 1, stream_ptr()) == 0
            out = dst.cpu().numpy()
            assert np.array_equal(out[do:do + size], host[so:so + size]), (so, do)
            assert (out[:do] == 0xAA).all() and (out[do + size:] == 0xAA).all(), (so, do)


def test_vectorized_copy_one_huge_pair_is_split_over_the_chip():
    # the reference runs a whole pair on one CTA (README.md:123: 5 MiB block -> 2.81 GB/s); we tile it
    size = 5 * 1024 * 1024 + 48
    src = torch.randint(0, 256, (size,), dtype=torch.uint8, device="cuda")
    dst = dev_u8(size)
    st, dt = dev_ptr_table([src.data_ptr()]), dev_ptr_table([dst.data_ptr()])
    assert K.vectorized_copy(st.data_ptr(), dt.data_ptr(), size, 1, stream_ptr()) == 0
    assert torch.equal(src, dst)


def test_vectorized_copy_matches_reference_kernel_bit_for_bit():
    ours, pool, perm, dperm = launch_reference_copy_case(K.vectorized_copy)
    theirs = np.load(REF_COPY_SHA256)          # SHA-256 of every output row the reference kernel wrote
    assert np.array_equal(row_sha256(ours.cpu().numpy()), theirs)
    assert torch.equal(ours[dperm], pool[perm])


# ---------------------------------------------------------------- K2/K3 permute
def test_permute_empty_batch_noop_and_bad_dtype():
    sp = stream_ptr()
    # kernel_roundtrip.rs:362-410
    assert K.universal_from_block(0, 0, 0, 1, 1, 1, 1, 1, K.TensorDataType.F32, K.BlockLayout.NHD, sp) == 0
    assert K.block_from_universal(0, 0, 0, 1, 1, 1, 1, 1, K.TensorDataType.F32, K.BlockLayout.NHD, sp) == 0
    assert K.universal_from_block(0, 0, 2, 1, 1, 1, 1, 1, K.TensorDataType.F32, K.BlockLayout.NHD, sp) == K.CUDA_ERROR_INVALID_VALUE
    assert K.universal_from_block(0, 0, 2, 1, 1, 1, 1, 1, 9, K.BlockLayout.NHD, sp) == K.CUDA_ERROR_INVALID_VALUE  # tensor_kernels.cu:327


def _permute_case(dtype, layout, dims, nb, seed=11):
    nh, nl, no, nt, hd = dims
    npd, elem = kats.DTYPES[dtype], kats.ELEM[dtype]
    rng = np.random.default_rng(seed)
    unis = [(rng.random(dims) * 2 - 1).astype(npd) if dtype != 1 else rng.integers(0, 65536, dims).astype(np.uint16)
            for _ in range(nb)]
    ref_chunks = [c for u in unis for c in kats.make_blocks(u, layout)]
    sp = stream_ptr()
    d_chunks = [torch.from_numpy(c.view(np.uint8).copy()).cuda() for c in ref_chunks]
    d_unis = [dev_u8(u.nbytes, fill=0xDE) for u in unis]
    bt, ut = dev_ptr_table([t.data_ptr() for t in d_chunks]), dev_ptr_table([t.data_ptr() for t in d_unis])
    assert K.universal_from_block(ut.data_ptr(), bt.data_ptr(), nb, nh, nl, no, nt, hd, dtype, layout, sp) == 0
    torch.cuda.synchronize()
    for got, want in zip(d_unis, unis):
        assert np.array_equal(got.cpu().numpy(), want.reshape(-1).view(np.uint8))
    for t in d_chunks:
        t.fill_(0xDE)                                   # poison before the reverse pass
    assert K.block_from_universal(ut.data_ptr(), bt.data_ptr(), nb, nh, nl, no, nt, hd, dtype, layout, sp) == 0
    torch.cuda.synchronize()
    for got, want in zip(d_chunks, ref_chunks):
        assert np.array_equal(got.cpu().numpy(), want.view(np.uint8))
    return unis, ref_chunks


@pytest.mark.parametrize("dtype", [0, 1, 2, 3])
@pytest.mark.parametrize("layout", [kats.NHD, kats.HND])
def test_permute_roundtrip_reference_dims(dtype, layout):
    d = kats.PERMUTE_DIMS   # kernel_roundtrip.rs:241-252
    _permute_case(dtype, layout, (d["nh"], d["nl"], d["no"], d["nt"], d["hd"]), kats.PERMUTE_NB)


@pytest.mark.parametrize("layout", [kats.NHD, kats.HND])
def test_permute_llama70b_tp_reshard_shape(layout):
    # SURVEY §8 a15: per block [8, nl, 2, 16, 128] bf16 (fewer layers to keep the test small) -> 16 B vector path
    _permute_case(1, layout, (8, 4, 2, 16, 128), 3)


@pytest.mark.parametrize("layout", [kats.NHD, kats.HND])
def test_permute_position_encoded_kat_and_reference_kernel(layout):
    ours = block_from_universal_position_encoded(K.lib().kvbm_kernels_launch_block_from_universal, layout)
    want = kats.make_blocks(kats.position_encoded_universal(**kats.PERMUTE_DIMS), layout)
    for got, w in zip(ours, want):
        assert np.array_equal(got, w)
    theirs = np.load(REF_POSITION_BLOCKS)[layout]   # [nl*no, chunk] float32 the reference kernel wrote, per layout
    assert np.array_equal(np.stack(ours), theirs)


def test_universal_roundtrip_quarter_offsets():
    # tensor_kernels.rs:298-470: values (global_idx*inner + offset) + 0.25, nh=2 nl=2 no=2 nt=3 hd=4, nb=2, F32 NHD
    nh, nl, no, nt, hd, nb = 2, 2, 2, 3, 4, 2
    inner, chunk_count = nt * nh * hd, nl * no
    chunks = [np.arange(inner, dtype=np.float32) + (g * inner) + 0.25 for g in range(nb * chunk_count)]
    d_chunks = [torch.from_numpy(c.copy()).cuda() for c in chunks]
    d_unis = [dev_u8(nh * nl * no * nt * hd * 4, fill=0xDE) for _ in range(nb)]
    bt, ut = dev_ptr_table([t.data_ptr() for t in d_chunks]), dev_ptr_table([t.data_ptr() for t in d_unis])
    assert K.universal_from_block(ut.data_ptr(), bt.data_ptr(), nb, nh, nl, no, nt, hd, 2, 0, stream_ptr()) == 0
    torch.cuda.synchronize()
    for b in range(nb):
        u = d_unis[b].cpu().numpy().view(np.float32).reshape(nh, nl, no, nt, hd)
        for h in range(nh):
            for l in range(nl):
                for o in range(no):
                    for t in range(nt):
                        for x in range(hd):
                            off = (t * nh + h) * hd + x
                            assert u[h, l, o, t, x] == ((b * chunk_count + l * no + o) * inner + off) + 0.25


# ---------------------------------------------------------------- v1 fatbin drop-in (DYN_FATBIN_PATH)
def test_v1_fatbin_vectorised_copy_symbol_and_launch_contract():
    """Loads dynamo_b200/vectorized_copy.fatbin the way the v1 block manager does
    (lib/llm/src/block_manager/block/transfer/cuda.rs:85-153,521-548): cuModuleLoadData, symbol
    `vectorised_copy`, grid=min(1024,pairs) x block=256, 0 dynamic smem, pointer tables in pinned memory."""
    from cuda.bindings import driver as drv
    path = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "dynamo_b200", "vectorized_copy.fatbin")
    assert os.path.exists(path), "build() must produce the fatbin"
    torch.cuda.init()
    torch.zeros(1, device="cuda")
    data = open(path, "rb").read()
    err, mod = drv.cuModuleLoadData(data)
    assert err == drv.CUresult.CUDA_SUCCESS, err
    err, fn = drv.cuModuleGetFunction(mod, b"vectorised_copy")
    assert err == drv.CUresult.CUDA_SUCCESS, err
    for size, pairs in [(32768, 160), (999, 7), (5 * 1024 * 1024, 2), (64, 3000)]:
        src = torch.randint(0, 256, (pairs, size), dtype=torch.uint8, device="cuda")
        dst = torch.zeros(pairs, size, dtype=torch.uint8, device="cuda")
        perm = torch.randperm(pairs)
        st = torch.tensor([src[int(i)].data_ptr() for i in perm], dtype=torch.int64).pin_memory()
        dt = torch.tensor([dst[i].data_ptr() for i in range(pairs)], dtype=torch.int64).pin_memory()
        args = np.array([st.data_ptr(), dt.data_ptr(), size, pairs], dtype=np.uint64)
        a0, a1, a2 = (np.array([v], dtype=np.uint64) for v in (st.data_ptr(), dt.data_ptr(), size))
        a3 = np.array([pairs], dtype=np.int32)
        params = np.array([a.ctypes.data for a in (a0, a1, a2, a3)], dtype=np.uint64)
        torch.cuda.synchronize()
        (err,) = drv.cuLaunchKernel(fn, min(1024, pairs), 1, 1, 256, 1, 1, 0, 0, params.ctypes.data, 0)
        assert err == drv.CUresult.CUDA_SUCCESS, err
        torch.cuda.synchronize()
        assert torch.equal(dst, src[perm]), (size, pairs)
    drv.cuModuleUnload(mod)
