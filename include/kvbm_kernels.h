/*
 * kvbm_kernels.h -- C ABI of libkvbm_kernels.so, the B200-native (sm_100a) replacement for
 * Dynamo's lib/kvbm-kernels.
 *
 * Part 1 are the six symbols the reference exports and its Rust FFI binds
 *   (/root/reference/lib/kvbm-kernels/cuda/tensor_kernels.cu:306,332,360,389,477,551;
 *    Rust declarations lib/kvbm-kernels/src/tensor_kernels.rs:46-74,89-109).
 * Signatures, enum values, return codes and edge-case behaviour are identical, so this library is a
 * drop-in via LD_LIBRARY_PATH exactly as lib/kvbm-kernels/cuda/stubs.c:4-7 documents.
 *
 * Part 2 are the v2 extensions: the block-table ("paged") gather -> push -> scatter kernel with
 * address arithmetic on the device, multi-destination fan-out over NVLink peer mappings, the fused
 * fp8<->bf16 cast and in-kernel completion / layer-streaming flags.  They replace the host loop +
 * pointer-table upload + host sync of lib/kvbm-physical/src/transfer/executor/cuda.rs:234-327 and
 * the grouped ncclBcast of lib/kvbm-engine/src/collectives/nccl.rs:321-356.
 *
 * No torch types; plain pointers and sizes.  All functions are thread-safe and hold no global state
 * (device attribute queries are cached per device).  Nothing here ever falls back to a CPU copy.
 */
#ifndef KVBM_KERNELS_H
#define KVBM_KERNELS_H

#include <stdbool.h>
#include <stddef.h>
#include <stdint.h>

#if defined(__CUDA_RUNTIME_API_H__) || defined(__DRIVER_TYPES_H__)
/* cudaError_t / cudaStream_t come from the CUDA headers */
#else
typedef int cudaError_t;    /* cudaSuccess == 0, as lib/kvbm-kernels/cuda/stubs.c:14-18 */
typedef void* cudaStream_t; /* opaque */
#endif

#ifdef __cplusplus
extern "C" {
#endif

/* ============================ Part 1: reference ABI (exact) ============================ */

/* tensor_kernels.cu:59-69 */
enum { KVBM_DTYPE_F16 = 0, KVBM_DTYPE_BF16 = 1, KVBM_DTYPE_F32 = 2, KVBM_DTYPE_F64 = 3 };
enum { KVBM_BLOCK_LAYOUT_NHD = 0, KVBM_BLOCK_LAYOUT_HND = 1 };
/* tensor_kernels.cu:371-375 */
enum {
  KVBM_MEMCPY_BATCHED_WITH_FALLBACK = 0,
  KVBM_MEMCPY_FALLBACK_ONLY = 1,
  KVBM_MEMCPY_BATCH_WITHOUT_FALLBACK = 2,
};

/* Replaces tensor_kernels.cu:551-571 (K1).  src_ptrs/dst_ptrs are DEVICE-ACCESSIBLE tables (device
 * or pinned host) of num_pairs pointers; every pair copies copy_size_bytes; any alignment; src/dst
 * may be device, peer-device or pinned-host memory.  num_pairs==0 || copy_size_bytes==0 ->
 * cudaSuccess before the NULL checks; NULL table -> cudaErrorInvalidValue. */
cudaError_t kvbm_kernels_launch_vectorized_copy(void** src_ptrs, void** dst_ptrs,
                                                size_t copy_size_bytes, int num_pairs,
                                                cudaStream_t stream);

/* Replaces tensor_kernels.cu:389-473 (K4).  HOST pointer tables, consumed before return. */
cudaError_t kvbm_kernels_memcpy_batch(const void* const* src_ptrs, void* const* dst_ptrs,
                                      size_t size_per_copy, size_t num_copies, int mode,
                                      cudaStream_t stream);

/* Replaces tensor_kernels.cu:306-330 (K2): block stacks [nl*no chunks of NHD|HND] -> universal
 * [nh,nl,no,nt,hd].  Tables are device-accessible. Unknown dtype -> cudaErrorInvalidValue. */
cudaError_t kvbm_kernels_launch_universal_from_block(void* const* universal_ptrs,
                                                     const void* const* block_ptrs,
                                                     size_t num_blocks, size_t nh, size_t nl,
                                                     size_t no, size_t nt, size_t hd, int dtype,
                                                     int layout, cudaStream_t stream);

/* Replaces tensor_kernels.cu:332-356 (K3): the inverse. */
cudaError_t kvbm_kernels_launch_block_from_universal(const void* const* universal_ptrs,
                                                     void* const* block_ptrs, size_t num_blocks,
                                                     size_t nh, size_t nl, size_t no, size_t nt,
                                                     size_t hd, int dtype, int layout,
                                                     cudaStream_t stream);

/* tensor_kernels.cu:360-368 */
bool kvbm_kernels_has_memcpy_batch_async(void);
/* tensor_kernels.cu:477-481: always false -- this is a real CUDA build. */
bool kvbm_kernels_is_stub_build(void);

/* ============================ Part 2: v2 extensions ============================ */

#define KVBM_MAX_DESTINATIONS 8
/* u32 words of kvbm_paged_copy_opts.sync_workspace for a source pool of `num_layers` layers */
#define KVBM_SYNC_WORKSPACE_WORDS(num_layers) ((num_layers) + 4)

/* Geometry of one KV pool as the kernel sees it.  It is the device form of
 * Layout::memory_region (lib/kvbm-physical/src/layout/mod.rs:73-78):
 *   addr(block, layer, outer) = layer_base[layer] + block*block_stride + outer*outer_stride
 * FullyContiguous pools (fully_contiguous.rs:158-162) set layer_base[l] = base + l*layer_stride;
 * LayerSeparate pools (layer_separate.rs:171-184) pass their per-layer allocations directly.
 * layer_base is a DEVICE-ACCESSIBLE array of num_layers addresses (uploaded once per pool). */
typedef struct kvbm_paged_layout {
  const uint64_t* layer_base;
  uint64_t block_stride;
  uint64_t outer_stride;
  uint32_t region_bytes; /* page_size * inner_dim * dtype_width_bytes */
  uint32_t num_layers;
  uint32_t outer_dim;
  uint32_t num_blocks;
} kvbm_paged_layout;

/* One destination of a transfer: its pool, the block table pair and optional in-band signals.
 * block id arrays are DEVICE-ACCESSIBLE int32[num_blocks]. */
typedef struct kvbm_paged_dst {
  kvbm_paged_layout layout;      /* layer_base may hold PEER addresses (NVLink-mapped) */
  const int32_t* src_block_ids;  /* blocks to gather from the source pool */
  const int32_t* dst_block_ids;  /* where they are scattered in this destination */
  uint32_t* done_flag;           /* nullable; set to `epoch` (st.release.sys) once every byte landed */
  uint32_t* layer_done_flags;    /* nullable; [num_layers]; entry l set to `epoch` when layer l landed */
} kvbm_paged_dst;

enum { KVBM_GATE_AUTO = 0, KVBM_GATE_SPIN = 1, KVBM_GATE_STREAM_WAIT = 2 };

enum {
  KVBM_CAST_NONE = 0,
  KVBM_CAST_FP8E4M3_TO_BF16 = 1, /* exact; NaN codes -> 0x7fc0 */
  KVBM_CAST_BF16_TO_FP8E4M3 = 2, /* round-to-nearest-even, saturate-to-finite */
};

typedef struct kvbm_paged_copy_opts {
  uint32_t epoch;                 /* value written to done flags / compared with ready flags (>=) */
  const uint32_t* layer_ready_flags; /* nullable; [num_layers]; layer l is read only after flag >= epoch */
  uint32_t* sync_workspace;       /* device u32[KVBM_SYNC_WORKSPACE_WORDS(num_layers)], zeroed (left zeroed by every launch):
                                     per-layer landed-item counters, then the launch's control words (rings finished, abort,
                                     tile-scheduler tickets).  Required iff any flag or gating is used; without it the
                                     library lends the launch a slot of a small per-device pool for the tile scheduler. */
  int max_ctas;                   /* 0 = default (one CTA per SM: an SM moves at most ~50 GB/s per direction, the HBM-bound copy wants
                                     them all); smaller values leave SMs to the engine -- 16 CTAs saturate an NVLink peer */
  int warps_per_cta;              /* 0 = default (4).  Two warps -- a producer and a consumer -- form one ring. */
  int stages;                     /* 0 = default */
  int tile_bytes;                 /* 0 = default */
  int force_simt;                 /* 1 = never use the TMA path (diagnostics) */
  uint32_t* completion_flag;      /* nullable; device-visible (e.g. mapped pinned host) word set to
                                     completion_value once EVERY destination has landed: lets the host
                                     observe completion without cudaEventQuery polling */
  uint32_t completion_value;
  int stores_in_flight;           /* 0 = default (max(1, stages/3)): slots that may still be draining to the destination;
                                     stages - stores_in_flight loads are kept in flight ahead */
  int reserved0;                  /* must be 0 (keeps the offsets of the fields below); non-zero -> cudaErrorInvalidValue */
  int reserved1;                  /* must be 0 (keeps the offsets of the fields below); non-zero -> cudaErrorInvalidValue */
  int gate_timeout_ms;            /* gated transfers: a layer_ready wait longer than this aborts the launch (completion word
                                     becomes 0xFFFFFFFF, done flags are not written) instead of hanging the GPU; 0 = 10 s */
  int multicast;                  /* NVLS: non-zero = dsts[0].layout.layer_base[] hold NVLink MULTICAST addresses (a mapping of a
                                     CUmulticastObject, see kvbm_mc_group_* in kvbm_physical.h).  The payload is written ONCE
                                     (1 = multimem.st from shared memory, 2 = TMA bulk store) and the NVSwitch delivers it to every
                                     device bound to the object; dsts[1..] contribute only their done / layer_done flags.  This is
                                     the replacement of the grouped ncclBcast (kvbm-engine collectives/nccl.rs:421-462): egress of
                                     the source GPU is 1x the payload instead of Nx.  Requires cast_mode NONE, 16-byte strides. */
  int gate_mode;                  /* how layer_ready_flags are waited for: KVBM_GATE_AUTO (0) = warps of the ONE launch spin on
                                     the flags when the process loads CUDA modules eagerly (CUDA_MODULE_LOADING=EAGER), else
                                     the wait moves to the stream (cuStreamWaitValue32 + a single-layer launch per layer) so
                                     that nothing resident spins while some other kernel of the process is still being loaded
                                     lazily -- see kvbm_kernels_gate_would_spin(); KVBM_GATE_SPIN (1) / KVBM_GATE_STREAM_WAIT
                                     (2) force either behaviour.  gate_timeout_ms applies to the spinning form only. */
  int static_schedule;            /* diagnostics: 1 = split the tiles round-robin over the rings instead of the dynamic
                                     (ticket) tile scheduler */
} kvbm_paged_copy_opts;

/* Gather `num_blocks` non-contiguous blocks x layers [layer_begin, layer_end) x outer from `src`,
 * push them to `num_dsts` destinations and scatter them into their block tables, optionally casting.
 * One launch, one-sided (no receiver kernel), stream-ordered, never blocks the host.
 * When all destinations share one src_block_ids pointer the payload is read from HBM once and stored
 * num_dsts times (replicate); otherwise each destination's blocks are gathered separately. */
cudaError_t kvbm_kernels_paged_copy_v2(const kvbm_paged_layout* src, const kvbm_paged_dst* dsts,
                                       int num_dsts, int num_blocks, int layer_begin,
                                       int layer_end, int cast_mode,
                                       const kvbm_paged_copy_opts* opts, cudaStream_t stream);

/* ---- layout-transforming hand-off (TP / PP re-shard while the blocks move) ------------------------------------------------
 * KvBlockLayout (lib/kvbm-physical/src/layout/kv_block_layout.rs:40-95): the order of the four permutable dimensions of one
 * block, head_dim (one "row" of row_bytes) always innermost.  The reference selects a transform kernel for a pair of these
 * (transfer/executor/mod.rs:46-100) but never runs one inside a transfer -- validate_layout_compatibility rejects the pair
 * (executor/cuda.rs:69) and K2 / K3 are only reachable through host-built pointer tables.  Here the transform is part of the
 * paged gather -> scatter: no pointer tables, block ids resolved on the device, either pool may be a peer's (NVLink). */
enum {
  KVBM_KV_UNKNOWN = 0,
  KVBM_KV_UNIVERSAL_TP = 1,    /* [nh, nl, no, nt, hd] */
  KVBM_KV_UNIVERSAL_PP = 2,    /* [nl, nh, no, nt, hd] */
  KVBM_KV_OPERATIONAL_HND = 3, /* [nl, no, nh, nt, hd] */
  KVBM_KV_OPERATIONAL_NHD = 4, /* [nl, no, nt, nh, hd] */
  KVBM_KV_CUSTOM = 5,          /* named by the wire format only; no kernel */
};

typedef struct kvbm_permute_side {
  kvbm_paged_layout layout;  /* operational formats: any paged pool, the (block, layer, outer) region holds [nt, nh, hd] or
                                [nh, nt, hd].  Universal formats: the pool must be fully contiguous -- layer_base[0] +
                                id * block_stride is the start of num_layers * outer_dim * region_bytes contiguous bytes */
  const int32_t* block_ids;  /* device-accessible int32[num_blocks] */
  int kv_layout;             /* KVBM_KV_* (1..4) */
} kvbm_permute_side;

/* Block src.block_ids[i] of `src` -> block dst.block_ids[i] of `dst`, layers [layer_begin, layer_end), every element moved
 * from its position under src.kv_layout to its position under dst.kv_layout (equal layouts = plain copy).  Both sides must
 * agree on num_layers, outer_dim and region_bytes = page_size * num_heads * row_bytes; row_bytes (head_dim * element size)
 * must be a multiple of 16 in 16..65536 (powers of two take the shift-and-mask walk) and every stride a multiple of 16
 * (cudaErrorInvalidValue otherwise).  `done_flag`
 * (nullable, device-visible) receives `epoch` with system scope after the last byte landed, `completion_flag` likewise
 * `completion_value` (a one-thread signal launch behind the permuting launch; none when both are NULL).  Stream-ordered. */
cudaError_t kvbm_kernels_paged_permute(const kvbm_permute_side* src, const kvbm_permute_side* dst, int num_blocks,
                                       int layer_begin, int layer_end, uint32_t num_heads, uint32_t page_size,
                                       uint32_t row_bytes, uint32_t* done_flag, uint32_t epoch, uint32_t* completion_flag,
                                       uint32_t completion_value, cudaStream_t stream);

/* Host-only (no GPU): the stride table kvbm_kernels_paged_permute walks with for one side.  out[0] = 1 when offsets count
 * from the block's first byte (universal formats) or 0 when they count from the (layer, outer) region's first byte; the
 * element (layer l, outer o, head h, token t) then sits at  [out[0] ? l * out[1] + o * out[2] : 0] + h * out[3] + t * out[4].
 * Returns non-zero for formats without a kernel or strides that are not multiples of 16. */
int kvbm_kernels_permute_strides(int kv_layout, uint32_t num_layers, uint32_t outer_dim, uint32_t num_heads, uint32_t page_size,
                                 uint32_t row_bytes, uint64_t block_stride, uint64_t outer_stride, uint64_t out[5]);

/* 1 when KVBM_GATE_AUTO would let the transfer's warps spin on the ready flags (eager module loading detected through
 * cuModuleGetLoadingMode), 0 when it would gate on the stream instead. */
int kvbm_kernels_gate_would_spin(void);

/* Small helpers so hosts without a CUDA binding (ctypes, cgo, JNI) can drive the flags. */
cudaError_t kvbm_kernels_set_flags(uint32_t* flags, int first, int count, uint32_t value,
                                   cudaStream_t stream);
cudaError_t kvbm_kernels_wait_flag(const uint32_t* flag, uint32_t value, cudaStream_t stream);
/* cudaStreamWaitEvent for hosts without a CUDA binding: `event` is a raw cudaEvent_t / CUevent handle.  With
 * set_flags this turns an engine's existing per-layer event into a device-side ready flag on a helper stream. */
cudaError_t kvbm_kernels_stream_wait_event(cudaStream_t stream, void* event);

/* Number of kernel launches issued by this library since load (bench accounting). */
uint64_t kvbm_kernels_launch_count(void);
/* "sm_100a" build tag + whether the TMA path is compiled in. */
const char* kvbm_kernels_build_info(void);

#ifdef __cplusplus
}
#endif
#endif /* KVBM_KERNELS_H */
