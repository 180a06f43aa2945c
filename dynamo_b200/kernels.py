"""ctypes mirror of the reference's safe-ish Rust wrappers (lib/kvbm-kernels/src/tensor_kernels.rs).

Same function names, argument meaning and error behaviour as the Rust crate:
  vectorized_copy      tensor_kernels.rs:232-250   -> kvbm_kernels_launch_vectorized_copy
  memcpy_batch         tensor_kernels.rs:139-175   -> kvbm_kernels_memcpy_batch
  universal_from_block tensor_kernels.rs:177-215   -> kvbm_kernels_launch_universal_from_block
  block_from_universal tensor_kernels.rs:217-...   -> kvbm_kernels_launch_block_from_universal
  is_memcpy_batch_available / is_using_stubs       tensor_kernels.rs:111-137
plus the v2 paged entry point (include/kvbm_kernels.h part 2).  Every function returns the raw
cudaError_t (0 == cudaSuccess) like the FFI does; `check()` turns it into an exception.
"""
from __future__ import annotations

import ctypes as C
import enum
from typing import Optional, Sequence

from . import _lib

MAX_DESTINATIONS = 8


class TensorDataType(enum.IntEnum):
    F16 = 0
    BF16 = 1
    F32 = 2
    F64 = 3


class BlockLayout(enum.IntEnum):
    NHD = 0
    HND = 1


class MemcpyBatchMode(enum.IntEnum):
    BatchedWithFallback = 0
    FallbackOnly = 1
    BatchWithoutFallback = 2


class KvBlockLayout(enum.IntEnum):
    """KVBM_KV_* -- lib/kvbm-physical/src/layout/kv_block_layout.rs:40-76 (dimension order of one block, head_dim innermost)"""
    Unknown = 0
    UniversalTP = 1      # [nh, nl, no, nt, hd]
    UniversalPP = 2      # [nl, nh, no, nt, hd]
    OperationalHND = 3   # [nl, no, nh, nt, hd]
    OperationalNHD = 4   # [nl, no, nt, nh, hd]
    Custom = 5


class CastMode(enum.IntEnum):
    NONE = 0
    FP8E4M3_TO_BF16 = 1
    BF16_TO_FP8E4M3 = 2


CUDA_SUCCESS = 0
CUDA_ERROR_INVALID_VALUE = 1


class CudaError(RuntimeError):
    def __init__(self, code: int, what: str):
        super().__init__(f"{what} failed: cudaError_t={code}")
        self.code = code


def check(code: int, what: str = "kvbm_kernels") -> None:
    if code != CUDA_SUCCESS:
        raise CudaError(code, what)


class PagedLayout(C.Structure):
    """struct kvbm_paged_layout"""
    _fields_ = [
        ("layer_base", C.c_void_p),
        ("block_stride", C.c_uint64),
        ("outer_stride", C.c_uint64),
        ("region_bytes", C.c_uint32),
        ("num_layers", C.c_uint32),
        ("outer_dim", C.c_uint32),
        ("num_blocks", C.c_uint32),
    ]


class PagedDst(C.Structure):
    """struct kvbm_paged_dst"""
    _fields_ = [
        ("layout", PagedLayout),
        ("src_block_ids", C.c_void_p),
        ("dst_block_ids", C.c_void_p),
        ("done_flag", C.c_void_p),
        ("layer_done_flags", C.c_void_p),
    ]


class PermuteSide(C.Structure):
    """struct kvbm_permute_side"""
    _fields_ = [("layout", PagedLayout), ("block_ids", C.c_void_p), ("kv_layout", C.c_int)]


class PagedCopyOpts(C.Structure):
    """struct kvbm_paged_copy_opts"""
    _fields_ = [
        ("epoch", C.c_uint32),
        ("layer_ready_flags", C.c_void_p),
        ("sync_workspace", C.c_void_p),
        ("max_ctas", C.c_int),
        ("warps_per_cta", C.c_int),
        ("stages", C.c_int),
        ("tile_bytes", C.c_int),
        ("force_simt", C.c_int),
        ("completion_flag", C.c_void_p),
        ("completion_value", C.c_uint32),
        ("stores_in_flight", C.c_int),
        ("reserved0", C.c_int),
        ("reserved1", C.c_int),
        ("gate_timeout_ms", C.c_int),
        ("multicast", C.c_int),
        ("gate_mode", C.c_int),
        ("static_schedule", C.c_int),
    ]


def sync_workspace_words(num_layers: int) -> int:
    """KVBM_SYNC_WORKSPACE_WORDS: u32 words of PagedCopyOpts.sync_workspace (per-layer counters + control words)."""
    return int(num_layers) + 4


_configured = False


def lib() -> C.CDLL:
    global _configured
    L = _lib.load(_lib.KERNELS_SO)
    if not _configured:
        vp, sz, i = C.c_void_p, C.c_size_t, C.c_int
        L.kvbm_kernels_launch_vectorized_copy.argtypes = [vp, vp, sz, i, vp]
        L.kvbm_kernels_launch_vectorized_copy.restype = i
        L.kvbm_kernels_memcpy_batch.argtypes = [vp, vp, sz, sz, i, vp]
        L.kvbm_kernels_memcpy_batch.restype = i
        for f in (L.kvbm_kernels_launch_universal_from_block, L.kvbm_kernels_launch_block_from_universal):
            f.argtypes = [vp, vp, sz, sz, sz, sz, sz, sz, i, i, vp]
            f.restype = i
        L.kvbm_kernels_has_memcpy_batch_async.restype = C.c_bool
        L.kvbm_kernels_is_stub_build.restype = C.c_bool
        L.kvbm_kernels_paged_copy_v2.argtypes = [C.POINTER(PagedLayout), C.POINTER(PagedDst), i, i, i, i, i,
                                                 C.POINTER(PagedCopyOpts), vp]
        L.kvbm_kernels_paged_copy_v2.restype = i
        L.kvbm_kernels_paged_permute.argtypes = [C.POINTER(PermuteSide), C.POINTER(PermuteSide), i, i, i, C.c_uint32, C.c_uint32,
                                                 C.c_uint32, vp, C.c_uint32, vp, C.c_uint32, vp]
        L.kvbm_kernels_paged_permute.restype = i
        L.kvbm_kernels_permute_strides.argtypes = [i, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint64, C.c_uint64,
                                                   C.POINTER(C.c_uint64)]
        L.kvbm_kernels_permute_strides.restype = i
        L.kvbm_kernels_set_flags.argtypes = [vp, i, i, C.c_uint32, vp]
        L.kvbm_kernels_set_flags.restype = i
        L.kvbm_kernels_wait_flag.argtypes = [vp, C.c_uint32, vp]
        L.kvbm_kernels_wait_flag.restype = i
        L.kvbm_kernels_stream_wait_event.argtypes = [vp, vp]
        L.kvbm_kernels_stream_wait_event.restype = i
        L.kvbm_kernels_launch_count.restype = C.c_uint64
        L.kvbm_kernels_build_info.restype = C.c_char_p
        _configured = True
    return L


EXPORTED_SYMBOLS = [
    "kvbm_kernels_launch_vectorized_copy", "kvbm_kernels_memcpy_batch",
    "kvbm_kernels_launch_universal_from_block", "kvbm_kernels_launch_block_from_universal",
    "kvbm_kernels_has_memcpy_batch_async", "kvbm_kernels_is_stub_build",
    "kvbm_kernels_paged_copy_v2", "kvbm_kernels_set_flags", "kvbm_kernels_wait_flag", "kvbm_kernels_stream_wait_event",
    "kvbm_kernels_launch_count", "kvbm_kernels_build_info", "kvbm_kernels_gate_would_spin", "kvbm_kernels_paged_permute",
    "kvbm_kernels_permute_strides",
]

GATE_AUTO, GATE_SPIN, GATE_STREAM_WAIT = 0, 1, 2


def gate_would_spin() -> bool:
    """True when gated transfers spin in ONE launch (eager CUDA module loading); False when they gate on the stream."""
    return bool(lib().kvbm_kernels_gate_would_spin())


def is_memcpy_batch_available() -> bool:
    return bool(lib().kvbm_kernels_has_memcpy_batch_async())


def is_using_stubs() -> bool:
    return bool(lib().kvbm_kernels_is_stub_build())


def launch_count() -> int:
    return int(lib().kvbm_kernels_launch_count())


def vectorized_copy(src_ptrs: int, dst_ptrs: int, copy_size_bytes: int, num_pairs: int, stream: int) -> int:
    """src_ptrs/dst_ptrs: address of a DEVICE-ACCESSIBLE table of `num_pairs` pointers."""
    return lib().kvbm_kernels_launch_vectorized_copy(src_ptrs, dst_ptrs, copy_size_bytes, num_pairs, stream)


def memcpy_batch(src_ptrs: Optional[Sequence[int]], dst_ptrs: Optional[Sequence[int]], size_per_copy: int,
                 num_copies: int, mode: MemcpyBatchMode, stream: int) -> int:
    """src_ptrs/dst_ptrs: HOST sequences of addresses (None -> NULL table)."""
    s = (C.c_void_p * len(src_ptrs))(*src_ptrs) if src_ptrs is not None else None
    d = (C.c_void_p * len(dst_ptrs))(*dst_ptrs) if dst_ptrs is not None else None
    return lib().kvbm_kernels_memcpy_batch(s, d, size_per_copy, num_copies, int(mode), stream)


def universal_from_block(universal_ptrs: int, block_ptrs: int, num_blocks: int, nh: int, nl: int, no: int,
                         nt: int, hd: int, dtype: int, layout: int, stream: int) -> int:
    return lib().kvbm_kernels_launch_universal_from_block(universal_ptrs, block_ptrs, num_blocks, nh, nl, no, nt,
                                                          hd, int(dtype), int(layout), stream)


def block_from_universal(universal_ptrs: int, block_ptrs: int, num_blocks: int, nh: int, nl: int, no: int,
                         nt: int, hd: int, dtype: int, layout: int, stream: int) -> int:
    return lib().kvbm_kernels_launch_block_from_universal(universal_ptrs, block_ptrs, num_blocks, nh, nl, no, nt,
                                                          hd, int(dtype), int(layout), stream)


def paged_copy(src: PagedLayout, dsts: Sequence[PagedDst], num_blocks: int, layer_begin: int, layer_end: int,
               cast_mode: int = 0, opts: Optional[PagedCopyOpts] = None, stream: int = 0) -> int:
    arr = (PagedDst * max(1, len(dsts)))(*dsts)
    return lib().kvbm_kernels_paged_copy_v2(C.byref(src), arr, len(dsts), num_blocks, layer_begin, layer_end,
                                            int(cast_mode), C.byref(opts) if opts is not None else None, stream)


def paged_permute(src: PermuteSide, dst: PermuteSide, num_blocks: int, layer_begin: int, layer_end: int, num_heads: int,
                  page_size: int, row_bytes: int, done_flag: int = 0, epoch: int = 0, completion_flag: int = 0,
                  completion_value: int = 0, stream: int = 0) -> int:
    """Blocks src.block_ids[i] -> dst.block_ids[i], every element moved from its place under src.kv_layout to its place under
    dst.kv_layout; row_bytes = head_dim * element size.  include/kvbm_kernels.h (kvbm_kernels_paged_permute)."""
    return lib().kvbm_kernels_paged_permute(C.byref(src), C.byref(dst), num_blocks, layer_begin, layer_end, num_heads, page_size,
                                            row_bytes, done_flag or None, epoch, completion_flag or None, completion_value, stream)


def permute_strides(kv_layout: int, num_layers: int, outer_dim: int, num_heads: int, page_size: int, row_bytes: int,
                    block_stride: int, outer_stride: int):
    """Host-only: (universal, layer_step, outer_step, head_stride, tok_stride) of one side of `paged_permute`, or None."""
    out = (C.c_uint64 * 5)()
    if lib().kvbm_kernels_permute_strides(int(kv_layout), num_layers, outer_dim, num_heads, page_size, row_bytes, block_stride,
                                          outer_stride, out):
        return None
    return bool(out[0]), int(out[1]), int(out[2]), int(out[3]), int(out[4])


def set_flags(flags_ptr: int, first: int, count: int, value: int, stream: int) -> int:
    return lib().kvbm_kernels_set_flags(flags_ptr, first, count, value, stream)


def stream_wait_event(stream: int, event: int) -> int:
    return lib().kvbm_kernels_stream_wait_event(stream, event)


def wait_flag(flag_ptr: int, value: int, stream: int) -> int:
    return lib().kvbm_kernels_wait_flag(flag_ptr, value, stream)
