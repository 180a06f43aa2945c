// libkvbm_kernels.so -- sm_100a KV-block transfer kernels behind the reference C ABI
// (see include/kvbm_kernels.h for the contract and the reference lines each entry replaces).
#include <cuda_runtime_api.h>

#include "../../../include/kvbm_kernels.h"
#include "copy_engine.cuh"

#include <algorithm>
#include <atomic>
#include <mutex>
#include <cstdio>
#include <vector>

namespace kvbm {

// ------------------------------------------------------------------------------------------------
// launch bookkeeping
// ------------------------------------------------------------------------------------------------
static std::atomic<uint64_t> g_launches{0};

struct DeviceInfo {
  int sm_count = 0;
  int max_smem_optin = 0;
};

static cudaError_t preload_kernels();

static cudaError_t device_info(DeviceInfo* out)
{
  constexpr int kMaxDev = 64;
  static std::atomic<int> sm[kMaxDev];
  static std::atomic<int> smem[kMaxDev];
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return e;
  if (dev < 0 || dev >= kMaxDev) return cudaErrorInvalidDevice;
  int s = sm[dev].load(std::memory_order_acquire);
  if (s == 0) {
    int a = 0, b = 0;
    if ((e = cudaDeviceGetAttribute(&a, cudaDevAttrMultiProcessorCount, dev)) != cudaSuccess) return e;
    if ((e = cudaDeviceGetAttribute(&b, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev)) != cudaSuccess) return e;
    // CUDA loads kernels lazily and a first-time load can wait for the device to go idle.  A transfer kernel
    // that is spinning on layer-ready flags would then deadlock against the very first launch of the tiny
    // flag kernel that is supposed to release it -- so every kernel of this library is loaded up front.
    if ((e = preload_kernels()) != cudaSuccess) return e;
    smem[dev].store(b, std::memory_order_release);
    sm[dev].store(a, std::memory_order_release);
    s = a;
  }
  out->sm_count = s;
  out->max_smem_optin = smem[dev].load(std::memory_order_acquire);
  return cudaSuccess;
}

static int default_ctas(const DeviceInfo& di) { return di.sm_count; }

// Ring geometry of one launch.
struct RingCfg {
  int rings;        // R rings per CTA (2 warps each)
  int stages;       // S (input slots per ring)
  int pending;      // P (TMA stores allowed to keep draining their slot); loads ahead = S - P
  int batch;        // largest scheduler ticket, items
  uint32_t tile;    // source bytes per slot
  uint32_t smem;    // dynamic shared memory bytes
  uint32_t out_tile;  // cast only
};

// Defaults measured on B200 (benchmarks/copylab.cu -> profiles/r02_copylab_*.jsonl).  One SM moves at most ~50 GB/s per
// direction through the TMA however many rings it runs, so the HBM-bound copy wants (nearly) every SM: 132-148 CTAs copy
// 512 MiB HBM->HBM in 0.170 ms (cudaMemcpy 0.173, reference K1 0.177-0.178); 74 CTAs sit at the per-SM limit and are
// sensitive to every instruction of the per-item chain.  A whole 32 KiB region per bulk op halves that chain's share;
// smaller regions get more rings per CTA instead (~192 KiB of slots per CTA either way).  16 CTAs saturate an NVLink
// peer: callers that overlap the transfer with compute pass max_ctas.
constexpr int kDefaultStages = 6;
constexpr uint32_t kDefaultTile = 32768;
constexpr int kDefaultBatch = 8;

static uint32_t round_up(uint32_t x, uint32_t m) { return (x + m - 1) / m * m; }

// cast: 0 none, 1 up (out = 2x), 2 down (out = x/2).  `warps` is the legacy knob: 2 warps make one ring.
static RingCfg make_ring(const DeviceInfo& di, uint32_t unit_bytes, int warps, int stages, int tile, int cast, int pending = 0)
{
  RingCfg c{};
  c.batch = kDefaultBatch;
  // default tile: the whole unit when it is small, else kDefaultTile pieces
  uint32_t t = tile > 0 ? static_cast<uint32_t>(tile) : std::min<uint32_t>(std::max<uint32_t>(unit_bytes, 16), kDefaultTile);
  t = round_up(t, 32);
  // rings per CTA: as many as keep ~32 KiB x S of slots busy (1 for 32 KiB tiles, 2 for 16 KiB, 4 for <= 8 KiB)
  c.rings = warps > 0 ? std::max(1, std::min(warps, 16) / 2) : static_cast<int>(std::max<uint32_t>(1, std::min<uint32_t>(4, kDefaultTile / t)));
  const uint32_t budget = static_cast<uint32_t>(di.max_smem_optin) - 1024;
  for (;;) {
    const uint32_t out = cast == 1 ? 2 * t : (cast == 2 ? t / 2 : 0);
    // default depth: ~96 KiB of slots per ring (small tiles get more slots), at least 3, at most 12
    int s = stages > 0 ? stages : kDefaultStages;
    s = std::max(2, std::min(s, kMaxStages));  // one slot cannot overlap a load with a store
    while (s > 2 && cta_smem_bytes(c.rings, s, t, out) > budget) --s;
    if (cta_smem_bytes(c.rings, s, t, out) <= budget) {
      c.stages = s;
      c.pending = pending > 0 ? std::min(pending, s - 1) : std::max(1, s / 3);  // 2 of 6
      c.tile = t;
      c.out_tile = out;
      c.smem = cta_smem_bytes(c.rings, s, t, out);
      return c;
    }
    if (t > 1024)
      t = round_up(t / 2, 32);
    else if (c.rings > 1)
      c.rings /= 2;
    else {
      c.stages = 2;
      c.pending = 1;
      c.tile = t;
      c.out_tile = out;
      c.smem = cta_smem_bytes(1, 2, t, out);
      return c;
    }
  }
}

// ------------------------------------------------------------------------------------------------
// Scheduler words for launches that bring no workspace (legacy callers, opts == NULL): a small per-device pool of
// zeroed 4-word slots.  A slot is handed to one launch at a time: an event recorded behind the launch tells when it
// may be reused (the kernel leaves the words zeroed).  No free slot, or a stream that is being captured into a
// graph, simply means a static tile schedule for that launch -- never a wait.
// ------------------------------------------------------------------------------------------------
struct SchedPool {
  static constexpr int kSlots = 64;
  std::mutex mu;
  uint32_t* words = nullptr;  // kSlots * 4
  cudaEvent_t ev[kSlots] = {};
  bool used[kSlots] = {};
  int next = 0;
  bool failed = false;
};
static SchedPool g_pools[64];

static uint32_t* sched_acquire(int dev, cudaStream_t stream, int* slot_out)
{
  *slot_out = -1;
  cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
  if (cudaStreamIsCapturing(stream, &cap) != cudaSuccess || cap != cudaStreamCaptureStatusNone) {
    (void)cudaGetLastError();
    return nullptr;
  }
  SchedPool& p = g_pools[dev];
  std::lock_guard<std::mutex> lk(p.mu);
  if (p.failed) return nullptr;
  if (!p.words) {
    if (cudaMalloc(&p.words, SchedPool::kSlots * 16) != cudaSuccess || cudaMemset(p.words, 0, SchedPool::kSlots * 16) != cudaSuccess) {
      (void)cudaGetLastError();
      p.failed = true;
      p.words = nullptr;
      return nullptr;
    }
    for (int i = 0; i < SchedPool::kSlots; ++i)
      if (cudaEventCreateWithFlags(&p.ev[i], cudaEventDisableTiming) != cudaSuccess) {
        (void)cudaGetLastError();
        p.failed = true;
        return nullptr;
      }
  }
  for (int n = 0; n < SchedPool::kSlots; ++n) {
    const int i = (p.next + n) % SchedPool::kSlots;
    if (p.used[i]) {
      if (cudaEventQuery(p.ev[i]) != cudaSuccess) {
        (void)cudaGetLastError();
        continue;
      }
      p.used[i] = false;
    }
    p.used[i] = true;  // busy until sched_release records its event (and that event completes)
    p.next = (i + 1) % SchedPool::kSlots;
    *slot_out = i;
    return p.words + 4 * i;
  }
  return nullptr;
}

static void sched_release(int dev, int slot, cudaStream_t stream)
{
  if (slot < 0) return;
  SchedPool& p = g_pools[dev];
  std::lock_guard<std::mutex> lk(p.mu);
  if (cudaEventRecord(p.ev[slot], stream) != cudaSuccess) {
    (void)cudaGetLastError();
    // cannot tell when the launch ends: retire the slot for good rather than risk sharing it
  }
}

// ------------------------------------------------------------------------------------------------
// K1: pointer-pair copy (legacy ABI).  Hardware-scheduled SIMT: one CTA per (pair, 32 KiB chunk) -- or one warp per
// pair when pairs are small -- 4 independent 16 B loads in flight per thread (8 and 4 are equal on HBM, 4 is a little
// better when the source is pinned host memory: profiles/r02_k1_unroll_sweep.txt), the alignment ladder of the reference.
// The CTA scheduler is the dynamic load balancer here, so the ABI needs no workspace and the library no state.
// ------------------------------------------------------------------------------------------------
constexpr uint32_t kPairChunk = 32768;
constexpr uint32_t kPairSmall = 4096;
constexpr int kPairUnroll = 4;
constexpr int kPairThreads = 256;

__global__ void __launch_bounds__(kPairThreads)
kvbm_pair_copy_kernel(void* const* __restrict__ src_ptrs, void* const* __restrict__ dst_ptrs, size_t copy_size,
                      uint32_t chunks_per_pair, uint64_t num_pairs)
{
  const uint64_t bid = blockIdx.x + static_cast<uint64_t>(gridDim.x) * blockIdx.y;
  if (copy_size <= kPairSmall) {  // warp per pair
    const uint64_t pair = bid * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (pair >= num_pairs) return;
    group_copy_simt<kPairUnroll>(static_cast<uint8_t*>(dst_ptrs[pair]), static_cast<const uint8_t*>(src_ptrs[pair]), copy_size,
                                 threadIdx.x & 31, 32);
    return;
  }
  const uint64_t pair = bid / chunks_per_pair;
  if (pair >= num_pairs) return;
  const uint32_t chunk = static_cast<uint32_t>(bid - pair * chunks_per_pair);
  const size_t off = static_cast<size_t>(chunk) * kPairChunk;
  const size_t left = copy_size - off;
  // chunk boundaries are multiples of 32 KiB, so the alignment class of (src, dst) is the same for every chunk
  group_copy_simt<kPairUnroll>(static_cast<uint8_t*>(dst_ptrs[pair]) + off, static_cast<const uint8_t*>(src_ptrs[pair]) + off,
                               left < kPairChunk ? left : kPairChunk, threadIdx.x, blockDim.x);
}

// ------------------------------------------------------------------------------------------------
// v2: block-table (paged) gather -> push -> scatter, addresses computed on the device
// ------------------------------------------------------------------------------------------------
struct PagedArgs {
  kvbm_paged_layout src;
  kvbm_paged_layout dst[kMaxDst];
  const int32_t* src_ids[kMaxDst];
  const int32_t* dst_ids[kMaxDst];
  int ndst;        // destinations
  int replicate;   // 1: all destinations share src_ids[0] -> read once, store ndst times
  uint32_t n_blocks;
  uint32_t layer_begin, n_layers;  // layers [layer_begin, layer_begin + n_layers)
  uint32_t outer;
  uint32_t tiles_per_region;
  uint32_t tile;      // source bytes per piece
  uint32_t dst_num, dst_den;  // destination bytes = source bytes * dst_num / dst_den (cast)
};

struct PagedGen {
  PagedArgs a;
  // item order (layer-major so a layer completes early for streaming):
  //   item = (((layer * n_blocks + block) * outer + o) * fan + d) * tiles_per_region + t
  // where fan = ndst for distinct payloads (destinations interleaved -> all NVLink ports busy) and 1
  // when replicating.
  __device__ __forceinline__ void get(uint32_t item, Piece& p) const
  {
    uint32_t r = item / a.tiles_per_region;
    const uint32_t t = item - r * a.tiles_per_region;
    uint32_t d = 0;
    if (!a.replicate) {
      const uint32_t r2 = r / a.ndst;
      d = r - r2 * a.ndst;
      r = r2;
    }
    uint32_t r2 = r / a.outer;
    const uint32_t o = r - r2 * a.outer;
    r = r2;
    r2 = r / a.n_blocks;
    const uint32_t blk = r - r2 * a.n_blocks;
    const uint32_t layer = a.layer_begin + r2;

    const uint64_t soff = static_cast<uint64_t>(t) * a.tile;
    const uint32_t left = a.src.region_bytes - static_cast<uint32_t>(soff);
    p.bytes = left < a.tile ? left : a.tile;
    p.layer = static_cast<int>(layer);
    const uint64_t doff = soff * a.dst_num / a.dst_den;
    const int32_t sb = __ldg(a.src_ids[d] + blk);
    p.src = reinterpret_cast<const uint8_t*>(__ldg(a.src.layer_base + layer) + static_cast<uint64_t>(sb) * a.src.block_stride +
                                             static_cast<uint64_t>(o) * a.src.outer_stride + soff);
    if (a.replicate) {
      p.ndst = a.ndst;
#pragma unroll
      for (int k = 0; k < kMaxDst; ++k) {
        if (k < a.ndst) {
          const int32_t db = __ldg(a.dst_ids[k] + blk);
          p.dst[k] = reinterpret_cast<uint8_t*>(__ldg(a.dst[k].layer_base + layer) +
                                                static_cast<uint64_t>(db) * a.dst[k].block_stride +
                                                static_cast<uint64_t>(o) * a.dst[k].outer_stride + doff);
        }
      }
    } else {
      p.ndst = 1;
      const int32_t db = __ldg(a.dst_ids[d] + blk);
      // select destination d without dynamic indexing of a kernel-parameter array of structs
      const uint64_t* lb = a.dst[0].layer_base;
      uint64_t bs = a.dst[0].block_stride, os = a.dst[0].outer_stride;
#pragma unroll
      for (int k = 1; k < kMaxDst; ++k)
        if (k == static_cast<int>(d)) {
          lb = a.dst[k].layer_base;
          bs = a.dst[k].block_stride;
          os = a.dst[k].outer_stride;
        }
      p.dst[0] = reinterpret_cast<uint8_t*>(__ldg(lb + layer) + static_cast<uint64_t>(db) * bs +
                                            static_cast<uint64_t>(o) * os + doff);
    }
  }
};

struct PagedSyncArgs {
  const uint32_t* layer_ready;
  uint32_t* layer_counters;  // [num_layers] (user workspace) or null
  uint32_t* ctl;             // 3 control words: rings finished, abort, scheduler tickets; null = static schedule
  uint32_t* done_flag[kMaxDst];
  uint32_t* layer_done[kMaxDst];
  uint32_t* completion_flag;
  uint32_t completion_value;
  uint32_t epoch;
  uint64_t gate_timeout_ns;
  int num_flag_dsts;  // destinations that get flags (== data destinations unless multicast)
};

__device__ __forceinline__ StreamSync make_sync(const PagedSyncArgs& s, const PagedArgs& a, uint32_t total, int R)
{
  StreamSync ss{};
  ss.gate = s.layer_ready != nullptr;
  ss.want_layers = false;
  ss.want_done = s.completion_flag != nullptr;
  ss.layer_ready = s.layer_ready;
  ss.layer_counters = s.layer_counters;
  ss.ctl = s.ctl;
  ss.epoch = s.epoch;
  ss.gate_timeout_ns = s.gate_timeout_ns;
  ss.completion_flag = s.completion_flag;
  ss.completion_value = s.completion_value;
  ss.total_rings = gridDim.x * R;
  ss.items_per_layer = total / a.n_layers;
  ss.ndst = s.num_flag_dsts;
  ss.layer_begin = static_cast<int>(a.layer_begin);
  ss.layer_end = static_cast<int>(a.layer_begin + a.n_layers);
#pragma unroll
  for (int d = 0; d < kMaxDst; ++d) {
    ss.done_flag[d] = s.done_flag[d];
    ss.layer_done[d] = s.layer_done[d];
    if (d < s.num_flag_dsts && s.layer_done[d] != nullptr) ss.want_layers = true;
    if (d < s.num_flag_dsts && s.done_flag[d] != nullptr) ss.want_done = true;
  }
  if (ss.layer_counters == nullptr) ss.want_layers = false;
  return ss;
}

template <int CAST, bool FAST>
__global__ void __launch_bounds__(512, 1)
kvbm_paged_copy_kernel(const __grid_constant__ PagedGen gen, const __grid_constant__ PagedSyncArgs sync,
                       uint32_t total, int S, int P, int batch, int static_schedule, uint32_t out_tile, int allow_tma, int multimem)
{
  extern __shared__ __align__(128) uint8_t smem[];
  const int R = blockDim.x >> 6;
  const int ring_ndst = gen.a.replicate ? gen.a.ndst : 1;
  const StreamSync ss = make_sync(sync, gen.a, total, R);
  RingParams rp{S, P, batch, gen.a.tile, out_tile, allow_tma != 0, static_schedule != 0, CAST == KVBM_CAST_NONE && multimem != 0};
  run_rings<CAST, FAST>(smem, gen, total, ring_ndst, rp, ss);
}

// ------------------------------------------------------------------------------------------------
// K2 / K3: block stacks <-> universal.  Index peel identical in meaning to the reference
// (tensor_kernels.cu:150-228) but done per 16-byte vector when a head row allows it, and with
// 32-bit arithmetic; one thread moves VEC bytes.
// ------------------------------------------------------------------------------------------------
template <int VEC, bool TO_UNIVERSAL>
__global__ void __launch_bounds__(256)
kvbm_permute_kernel(void* const* universal_ptrs, void* const* block_ptrs, uint64_t total_units,
                    uint32_t units_per_block, uint32_t nh, uint32_t nl, uint32_t no, uint32_t nt,
                    uint32_t hdv /* row length in VEC units */, int layout)
{
  const uint64_t stride = static_cast<uint64_t>(blockDim.x) * gridDim.x;
  for (uint64_t u = static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x; u < total_units; u += stride) {
    const uint32_t b = static_cast<uint32_t>(u / units_per_block);
    const uint32_t residual = static_cast<uint32_t>(u - static_cast<uint64_t>(b) * units_per_block);
    uint32_t tmp = residual;
    const uint32_t hd_i = tmp % hdv;
    tmp /= hdv;
    const uint32_t nt_i = tmp % nt;
    tmp /= nt;
    const uint32_t no_i = tmp % no;
    tmp /= no;
    const uint32_t nl_i = tmp % nl;
    const uint32_t nh_i = tmp / nl;
    const uint32_t chunk_off = layout == KVBM_BLOCK_LAYOUT_NHD ? ((nt_i * nh) + nh_i) * hdv + hd_i
                                                               : ((nh_i * nt) + nt_i) * hdv + hd_i;
    uint8_t* chunk = static_cast<uint8_t*>(block_ptrs[static_cast<size_t>(b) * nl * no + nl_i * no + no_i]) +
                     static_cast<size_t>(chunk_off) * VEC;
    uint8_t* uni = static_cast<uint8_t*>(universal_ptrs[b]) + static_cast<size_t>(residual) * VEC;
    uint8_t* d = TO_UNIVERSAL ? uni : chunk;
    const uint8_t* s = TO_UNIVERSAL ? chunk : uni;
    const bool aligned = ((reinterpret_cast<uintptr_t>(d) | reinterpret_cast<uintptr_t>(s)) & (VEC - 1)) == 0;
    if (!aligned) {
      // buffers only promise element alignment (>= 2 B): move the unit as 16-bit pieces
#pragma unroll
      for (int k = 0; k < VEC / 2; ++k)
        reinterpret_cast<uint16_t*>(d)[k] = reinterpret_cast<const uint16_t*>(s)[k];
    } else if (VEC == 16)
      *reinterpret_cast<uint4*>(d) = *reinterpret_cast<const uint4*>(s);
    else if (VEC == 8)
      *reinterpret_cast<uint2*>(d) = *reinterpret_cast<const uint2*>(s);
    else if (VEC == 4)
      *reinterpret_cast<uint32_t*>(d) = *reinterpret_cast<const uint32_t*>(s);
    else
      *reinterpret_cast<uint16_t*>(d) = *reinterpret_cast<const uint16_t*>(s);
  }
}

// Fast path of K2 / K3 for head rows that are a power-of-two number of 16-byte vectors (hd*elem = 64 B ... 4 KiB: every
// real KV geometry).  One CTA per (block, layer, outer) chunk -- the hardware CTA scheduler balances the SMs -- and one
// warp per head: for a fixed head the universal side is ONE contiguous run of nt rows and the chunk side is nt rows at a
// constant stride (NHD) or contiguous as well (HND), so a lane's addresses advance by shifts and adds: no division per
// vector (the reference peels 5 div/mod per ELEMENT, tensor_kernels.cu:150-187) and 8 independent 16 B loads per lane
// are in flight before the first store.
template <bool TO_UNIVERSAL>
__global__ void __launch_bounds__(256)
kvbm_permute_rows_kernel(void* const* __restrict__ universal_ptrs, void* const* __restrict__ block_ptrs, uint32_t nh, uint32_t nl,
                         uint32_t no, uint32_t nt, uint32_t log2_v /* 16 B vectors per head row */, uint32_t elem, int layout)
{
  const uint32_t chunk_id = blockIdx.x;  // (b * nl + nl_i) * no + no_i
  const uint32_t b = chunk_id / (nl * no);
  const uint32_t rem = chunk_id - b * (nl * no);
  const uint32_t nl_i = rem / no, no_i = rem - nl_i * no;
  uint8_t* chunk = static_cast<uint8_t*>(block_ptrs[chunk_id]);
  uint8_t* uni = static_cast<uint8_t*>(universal_ptrs[b]);
  const uint32_t V = 1u << log2_v;
  const uint32_t row = V << 4;            // bytes per head row
  const uint32_t run = nt << log2_v;      // 16 B vectors of one head on the universal side
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarps = blockDim.x >> 5;
  const bool aligned = ((reinterpret_cast<uintptr_t>(chunk) | reinterpret_cast<uintptr_t>(uni)) & 15) == 0;
  for (uint32_t nh_i = warp; nh_i < nh; nh_i += nwarps) {
    uint8_t* u = uni + (static_cast<size_t>((nh_i * nl + nl_i) * no + no_i) * nt << log2_v << 4);
    // chunk-side offset of vector v = (nt_i, c): NHD (nt_i*nh + nh_i)*row + 16c ; HND (nh_i*nt + nt_i)*row + 16c
    const size_t c_base = layout == KVBM_BLOCK_LAYOUT_NHD ? static_cast<size_t>(nh_i) * row : static_cast<size_t>(nh_i) * nt * row;
    const size_t c_stride = layout == KVBM_BLOCK_LAYOUT_NHD ? static_cast<size_t>(nh) * row : row;
    auto chunk_off = [&](uint32_t v) { return c_base + static_cast<size_t>(v >> log2_v) * c_stride + ((v & (V - 1)) << 4); };
    if (aligned) {
      constexpr int U = 8;
      uint32_t v = lane;
      for (; v + (U - 1) * 32 < run; v += U * 32) {
        uint4 x[U];
#pragma unroll
        for (int k = 0; k < U; ++k)
          x[k] = ptx::ld_stream_v4(TO_UNIVERSAL ? chunk + chunk_off(v + k * 32) : u + (static_cast<size_t>(v + k * 32) << 4));
#pragma unroll
        for (int k = 0; k < U; ++k)
          ptx::st_stream_v4(TO_UNIVERSAL ? u + (static_cast<size_t>(v + k * 32) << 4) : chunk + chunk_off(v + k * 32), x[k]);
      }
      for (; v < run; v += 32) {
        const uint4 x = ptx::ld_stream_v4(TO_UNIVERSAL ? chunk + chunk_off(v) : u + (static_cast<size_t>(v) << 4));
        ptx::st_stream_v4(TO_UNIVERSAL ? u + (static_cast<size_t>(v) << 4) : chunk + chunk_off(v), x);
      }
    } else {
      // buffers only promise element alignment: same walk, one element at a time
      const uint32_t per_vec = 16 / elem;
      for (uint32_t e = lane; e < run * per_vec; e += 32) {
        const uint32_t v = e / per_vec, within = (e - v * per_vec) * elem;
        uint8_t* cp = chunk + chunk_off(v) + within;
        uint8_t* up = u + (static_cast<size_t>(v) << 4) + within;
        uint8_t* d = TO_UNIVERSAL ? up : cp;
        const uint8_t* sp = TO_UNIVERSAL ? cp : up;
        if (elem == 2) *reinterpret_cast<uint16_t*>(d) = *reinterpret_cast<const uint16_t*>(sp);
        else if (elem == 4) *reinterpret_cast<uint32_t*>(d) = *reinterpret_cast<const uint32_t*>(sp);
        else *reinterpret_cast<uint2*>(d) = *reinterpret_cast<const uint2*>(sp);
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------
// Paged permute: the K2 / K3 walk with the addresses computed from the pools' layouts and block tables instead of
// host-built pointer tables, and for any pair of KvBlockLayouts (kv_block_layout.rs:85-95).  For a fixed
// (block, layer, outer, head) the nt rows of one head sit at  base + head * head_stride + t * tok_stride  on either side:
//   UniversalTP [nh,nl,no,nt,hd]  base = block + (l*no + o)*nt*row     head_stride = nl*no*nt*row  tok_stride = row
//   UniversalPP [nl,nh,no,nt,hd]  base = block + l*nh*no*nt*row + o*nt*row   head_stride = no*nt*row   tok_stride = row
//   OperationalHND [nl,no,nh,nt,hd]  base = region(l, o)               head_stride = nt*row        tok_stride = row
//   OperationalNHD [nl,no,nt,nh,hd]  base = region(l, o)               head_stride = row           tok_stride = nh*row
// One CTA per (block pair, layer, outer), one warp per head, 8 independent 16 B loads per lane before the first store.
// ------------------------------------------------------------------------------------------------
struct PermuteSide {
  const uint64_t* layer_base;
  const int32_t* ids;
  uint64_t block_stride;
  uint64_t layer_step;   // added per layer on top of layer_base[universal ? 0 : l]
  uint64_t outer_step;
  uint64_t head_stride;
  uint64_t tok_stride;
  int universal;
};

template <bool POW2>
__global__ void __launch_bounds__(256)
kvbm_paged_permute_kernel(const __grid_constant__ PermuteSide S, const __grid_constant__ PermuteSide D, uint32_t layer_begin,
                          uint32_t nlayers, uint32_t no, uint32_t nh, uint32_t nt, uint32_t vpr /* POW2: log2 of, else: 16 B vectors per row */,
                          uint32_t magic /* !POW2: ceil(2^32 / vpr) */)
{
  const uint32_t unit = blockIdx.x;  // (pair * nlayers + l) * no + o
  const uint32_t pair = unit / (nlayers * no);
  const uint32_t rem = unit - pair * (nlayers * no);
  const uint32_t l = layer_begin + rem / no, o = rem % no;
  auto base_of = [&](const PermuteSide& X) {
    return reinterpret_cast<uint8_t*>(static_cast<uintptr_t>(__ldg(X.layer_base + (X.universal ? 0 : l)))) +
           static_cast<uint64_t>(__ldg(X.ids + pair)) * X.block_stride + l * X.layer_step + o * X.outer_step;
  };
  const uint8_t* sb = base_of(S);
  uint8_t* db = base_of(D);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarps = blockDim.x >> 5;
  constexpr int U = 8;
  if (POW2) {
    const uint32_t log2_v = vpr;
    const uint32_t V = 1u << log2_v;
    const uint32_t run = nt << log2_v;  // 16 B vectors of one head
    for (uint32_t h = warp; h < nh; h += nwarps) {
      const uint8_t* sh = sb + h * S.head_stride;
      uint8_t* dh = db + h * D.head_stride;
      auto off = [&](const PermuteSide& X, uint32_t v) { return static_cast<uint64_t>(v >> log2_v) * X.tok_stride + ((v & (V - 1)) << 4); };
      uint32_t v = lane;
      for (; v + (U - 1) * 32 < run; v += U * 32) {
        uint4 x[U];
#pragma unroll
        for (int k = 0; k < U; ++k) x[k] = ptx::ld_stream_v4(sh + off(S, v + k * 32));
#pragma unroll
        for (int k = 0; k < U; ++k) ptx::st_stream_v4(dh + off(D, v + k * 32), x[k]);
      }
      for (; v < run; v += 32) ptx::st_stream_v4(dh + off(D, v), ptx::ld_stream_v4(sh + off(S, v)));
    }
  } else {
    // rows of any whole number of 16 B vectors (head_dim 80, 96, 192, MLA's 576 ...): token = v / V by a multiply-high with
    // ceil(2^32 / V) (exact for v < 2^32 / V; the host checks nt * V against it), so the 8 loads stay independent
    const uint32_t V = vpr;
    const uint32_t run = nt * V;
    for (uint32_t h = warp; h < nh; h += nwarps) {
      const uint8_t* sh = sb + h * S.head_stride;
      uint8_t* dh = db + h * D.head_stride;
      uint32_t v = lane;
      for (; v + (U - 1) * 32 < run; v += U * 32) {
        uint4 x[U];
        uint64_t od[U];
#pragma unroll
        for (int k = 0; k < U; ++k) {
          const uint32_t vk = v + k * 32, t = __umulhi(vk, magic), c = vk - t * V;
          x[k] = ptx::ld_stream_v4(sh + static_cast<uint64_t>(t) * S.tok_stride + (c << 4));
          od[k] = static_cast<uint64_t>(t) * D.tok_stride + (c << 4);
        }
#pragma unroll
        for (int k = 0; k < U; ++k) ptx::st_stream_v4(dh + od[k], x[k]);
      }
      for (; v < run; v += 32) {
        const uint32_t t = __umulhi(v, magic), c = v - t * V;
        ptx::st_stream_v4(dh + static_cast<uint64_t>(t) * D.tok_stride + (c << 4), ptx::ld_stream_v4(sh + static_cast<uint64_t>(t) * S.tok_stride + (c << 4)));
      }
    }
  }
}

__global__ void kvbm_signal_kernel(uint32_t* a, uint32_t va, uint32_t* b, uint32_t vb)
{
  __threadfence_system();
  if (a) ptx::st_release_sys(a, va);
  if (b) ptx::st_release_sys(b, vb);
}

static size_t dtype_size(int dtype)
{
  switch (dtype) {
    case KVBM_DTYPE_F16:
    case KVBM_DTYPE_BF16:
      return 2;
    case KVBM_DTYPE_F32:
      return 4;
    case KVBM_DTYPE_F64:
      return 8;
    default:
      return 0;
  }
}

template <bool TO_UNIVERSAL>
static cudaError_t launch_permute(void* const* universal_ptrs, void* const* block_ptrs, size_t num_blocks,
                                  size_t nh, size_t nl, size_t no, size_t nt, size_t hd, int dtype,
                                  int layout, cudaStream_t stream)
{
  const size_t elem = dtype_size(dtype);
  if (elem == 0) return cudaErrorInvalidValue;  // tensor_kernels.cu:327
  const size_t total_per_block = nh * nl * no * nt * hd;
  if (total_per_block * num_blocks == 0) return cudaSuccess;  // tensor_kernels.cu:238-240
  if (!block_ptrs || !universal_ptrs) return cudaErrorInvalidValue;
  if (layout != KVBM_BLOCK_LAYOUT_NHD && layout != KVBM_BLOCK_LAYOUT_HND) return cudaErrorInvalidValue;
  if (total_per_block * elem >= (1ull << 32)) return cudaErrorInvalidValue;

  // The vector must divide a head row AND every buffer must be aligned to it.  Chunk/universal
  // buffers come from cudaMalloc / torch (>= 256 B aligned) in practice, but the ABI takes raw
  // pointers, so only widen past the element size when the row allows it and keep 2/4/8-byte
  // vectors naturally aligned with the element type.
  const size_t row = hd * elem;
  DeviceInfo di;
  cudaError_t e = device_info(&di);
  if (e != cudaSuccess) return e;
  if (row >= 16 && row <= 4096 && (row & (row - 1)) == 0 && num_blocks * nl * no < (1ull << 31) && nh * nl * no * nt * row < (1ull << 40)) {
    uint32_t log2_v = 0;
    while ((16u << log2_v) < row) ++log2_v;
    const unsigned grid = static_cast<unsigned>(num_blocks * nl * no);
    const int threads = static_cast<int>(std::min<size_t>(8, std::max<size_t>(1, nh))) * 32;
    kvbm_permute_rows_kernel<TO_UNIVERSAL><<<grid, threads, 0, stream>>>(universal_ptrs, block_ptrs, static_cast<uint32_t>(nh),
                                                                          static_cast<uint32_t>(nl), static_cast<uint32_t>(no),
                                                                          static_cast<uint32_t>(nt), log2_v, static_cast<uint32_t>(elem), layout);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    return cudaGetLastError();
  }
  int vec = static_cast<int>(elem);
  if (row % 16 == 0)
    vec = 16;
  else if (row % 8 == 0 && elem <= 8)
    vec = std::max<int>(vec, 8);
  else if (row % 4 == 0 && elem <= 4)
    vec = std::max<int>(vec, 4);
  const uint32_t hdv = static_cast<uint32_t>(row / vec);
  const uint32_t units_per_block = static_cast<uint32_t>(total_per_block * elem / vec);
  const uint64_t total_units = static_cast<uint64_t>(units_per_block) * num_blocks;
  const uint64_t want = (total_units + 255) / 256;
  const int grid = static_cast<int>(std::min<uint64_t>(want, static_cast<uint64_t>(di.sm_count) * 16));
  auto go = [&](auto kern) {
    kern<<<grid, 256, 0, stream>>>(universal_ptrs, block_ptrs, total_units, units_per_block,
                                   static_cast<uint32_t>(nh), static_cast<uint32_t>(nl),
                                   static_cast<uint32_t>(no), static_cast<uint32_t>(nt), hdv, layout);
  };
  switch (vec) {
    case 16: go(kvbm_permute_kernel<16, TO_UNIVERSAL>); break;
    case 8: go(kvbm_permute_kernel<8, TO_UNIVERSAL>); break;
    case 4: go(kvbm_permute_kernel<4, TO_UNIVERSAL>); break;
    default: go(kvbm_permute_kernel<2, TO_UNIVERSAL>); break;
  }
  g_launches.fetch_add(1, std::memory_order_relaxed);
  return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------
// tiny flag kernels
// ------------------------------------------------------------------------------------------------
__global__ void kvbm_set_flags_kernel(uint32_t* flags, int first, int count, uint32_t value)
{
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < count) {
    __threadfence_system();
    ptx::st_release_sys(flags + first + i, value);
  }
}
__global__ void kvbm_wait_flag_kernel(const uint32_t* flag, uint32_t value)
{
  while (ptx::ld_acquire_sys(flag) < value) __nanosleep(100);
}

static cudaError_t preload_kernels()
{
  cudaFuncAttributes attr;
  cudaError_t e;
#define KVBM_PRELOAD(k) \
  if ((e = cudaFuncGetAttributes(&attr, k)) != cudaSuccess) return e;
  KVBM_PRELOAD(kvbm_pair_copy_kernel)
  KVBM_PRELOAD((kvbm_paged_copy_kernel<KVBM_CAST_NONE, false>))
  KVBM_PRELOAD((kvbm_paged_copy_kernel<KVBM_CAST_FP8E4M3_TO_BF16, false>))
  KVBM_PRELOAD((kvbm_paged_copy_kernel<KVBM_CAST_BF16_TO_FP8E4M3, false>))
  KVBM_PRELOAD((kvbm_paged_copy_kernel<KVBM_CAST_NONE, true>))
  KVBM_PRELOAD((kvbm_paged_copy_kernel<KVBM_CAST_FP8E4M3_TO_BF16, true>))
  KVBM_PRELOAD((kvbm_paged_copy_kernel<KVBM_CAST_BF16_TO_FP8E4M3, true>))
  KVBM_PRELOAD(kvbm_set_flags_kernel)
  KVBM_PRELOAD(kvbm_wait_flag_kernel)
  KVBM_PRELOAD(kvbm_paged_permute_kernel<true>)
  KVBM_PRELOAD(kvbm_paged_permute_kernel<false>)
  KVBM_PRELOAD(kvbm_signal_kernel)
  KVBM_PRELOAD((kvbm_permute_rows_kernel<true>))
  KVBM_PRELOAD((kvbm_permute_rows_kernel<false>))
  KVBM_PRELOAD((kvbm_permute_kernel<16, true>))
  KVBM_PRELOAD((kvbm_permute_kernel<8, true>))
  KVBM_PRELOAD((kvbm_permute_kernel<4, true>))
  KVBM_PRELOAD((kvbm_permute_kernel<2, true>))
  KVBM_PRELOAD((kvbm_permute_kernel<16, false>))
  KVBM_PRELOAD((kvbm_permute_kernel<8, false>))
  KVBM_PRELOAD((kvbm_permute_kernel<4, false>))
  KVBM_PRELOAD((kvbm_permute_kernel<2, false>))
#undef KVBM_PRELOAD
  return cudaSuccess;
}

// Stream memory operations (cuStreamWriteValue32 / cuStreamWaitValue32) through the driver entry point:
// the stream's front-end writes / polls the word itself -- no kernel launch, no SM occupied by a spinner.
typedef int (*stream_memop_fn)(cudaStream_t, unsigned long long, uint32_t, unsigned int);
static stream_memop_fn g_write32 = nullptr, g_wait32 = nullptr;
static std::atomic<int> g_memops_state{0};  // 0 unknown, 1 available, -1 unavailable

static bool stream_memops()
{
  int st = g_memops_state.load(std::memory_order_acquire);
  if (st == 0) {
    void *w = nullptr, *q = nullptr;
    cudaDriverEntryPointQueryResult r1, r2;
    bool ok = cudaGetDriverEntryPoint("cuStreamWriteValue32", &w, cudaEnableDefault, &r1) == cudaSuccess && w &&
              cudaGetDriverEntryPoint("cuStreamWaitValue32", &q, cudaEnableDefault, &r2) == cudaSuccess && q;
    (void)cudaGetLastError();
    g_write32 = reinterpret_cast<stream_memop_fn>(w);
    g_wait32 = reinterpret_cast<stream_memop_fn>(q);
    st = ok ? 1 : -1;
    g_memops_state.store(st, std::memory_order_release);
  }
  return st == 1;
}

template <class K>
static cudaError_t set_smem(K kernel, uint32_t bytes)
{
  return cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(bytes));
}

}  // namespace kvbm

using namespace kvbm;

// =================================================================================================
// C ABI -- Part 1 (reference symbols)
// =================================================================================================
extern "C" cudaError_t
kvbm_kernels_launch_vectorized_copy(void** src_ptrs, void** dst_ptrs, size_t copy_size_bytes, int num_pairs,
                                    cudaStream_t stream)
{
  if (num_pairs == 0 || copy_size_bytes == 0) return cudaSuccess;  // tensor_kernels.cu:555-557
  if (!src_ptrs || !dst_ptrs) return cudaErrorInvalidValue;        // :559-561
  if (num_pairs < 0) return cudaErrorInvalidValue;
  DeviceInfo di;
  cudaError_t e = device_info(&di);
  if (e != cudaSuccess) return e;

  const uint64_t pairs = static_cast<uint64_t>(num_pairs);
  uint64_t ctas;
  uint32_t chunks_per_pair = 1;
  if (copy_size_bytes <= kPairSmall) {
    constexpr uint64_t warps = kPairThreads / 32;  // one pair per warp
    ctas = (pairs + warps - 1) / warps;
  } else {
    const uint64_t cpp = (copy_size_bytes + kPairChunk - 1) / kPairChunk;
    if (cpp >= (1ull << 32)) return cudaErrorInvalidValue;
    chunks_per_pair = static_cast<uint32_t>(cpp);
    ctas = pairs * cpp;
  }
  const uint64_t gx = std::min<uint64_t>(ctas, 1ull << 30);
  const uint64_t gy = (ctas + gx - 1) / gx;
  if (gy > 65535) return cudaErrorInvalidValue;
  const dim3 grid(static_cast<unsigned>(gx), static_cast<unsigned>(gy));
  kvbm_pair_copy_kernel<<<grid, kPairThreads, 0, stream>>>(src_ptrs, dst_ptrs, copy_size_bytes, chunks_per_pair, pairs);
  g_launches.fetch_add(1, std::memory_order_relaxed);
  return cudaGetLastError();  // :570
}

extern "C" cudaError_t
kvbm_kernels_memcpy_batch(const void* const* src_ptrs, void* const* dst_ptrs, size_t size_per_copy,
                          size_t num_copies, int mode, cudaStream_t stream)
{
  if (num_copies == 0 || size_per_copy == 0) return cudaSuccess;  // tensor_kernels.cu:396-398
  if (!src_ptrs || !dst_ptrs) return cudaErrorInvalidValue;       // :400-402

  auto one_by_one = [&]() -> cudaError_t {
    for (size_t i = 0; i < num_copies; ++i) {
      cudaError_t e = cudaMemcpyAsync(dst_ptrs[i], src_ptrs[i], size_per_copy, cudaMemcpyDefault, stream);
      if (e != cudaSuccess) return e;
    }
    return cudaSuccess;
  };
  if (mode == KVBM_MEMCPY_FALLBACK_ONLY) return one_by_one();

#if CUDART_VERSION >= 12090
  // Host tables are consumed before returning (the caller may free them immediately: cuda.rs:185-204).
  std::vector<void*> srcs(num_copies), dsts(num_copies);
  std::vector<size_t> sizes(num_copies, size_per_copy), attr_idx(num_copies, 0);
  for (size_t i = 0; i < num_copies; ++i) {
    srcs[i] = const_cast<void*>(src_ptrs[i]);
    dsts[i] = dst_ptrs[i];
  }
  cudaMemcpyAttributes attr = {};
  attr.srcAccessOrder = cudaMemcpySrcAccessOrderStream;
#if CUDART_VERSION >= 13000
  cudaError_t e = cudaMemcpyBatchAsync(dsts.data(), srcs.data(), sizes.data(), num_copies, &attr, attr_idx.data(), 1, stream);
#else
  size_t fail_idx = 0;
  cudaError_t e = cudaMemcpyBatchAsync(dsts.data(), srcs.data(), sizes.data(), num_copies, &attr, attr_idx.data(), 1,
                                       &fail_idx, stream);
#endif
  if (e == cudaErrorNotSupported || e == cudaErrorInvalidValue) {
    if (mode == KVBM_MEMCPY_BATCH_WITHOUT_FALLBACK) return e;
    (void)cudaGetLastError();
    return one_by_one();
  }
  return e;
#else
  if (mode == KVBM_MEMCPY_BATCH_WITHOUT_FALLBACK) return cudaErrorNotSupported;
  return one_by_one();
#endif
}

extern "C" cudaError_t
kvbm_kernels_launch_universal_from_block(void* const* universal_ptrs, const void* const* block_ptrs,
                                         size_t num_blocks, size_t nh, size_t nl, size_t no, size_t nt, size_t hd,
                                         int dtype, int layout, cudaStream_t stream)
{
  return launch_permute<true>(universal_ptrs, const_cast<void* const*>(reinterpret_cast<const void* const*>(block_ptrs)),
                              num_blocks, nh, nl, no, nt, hd, dtype, layout, stream);
}

extern "C" cudaError_t
kvbm_kernels_launch_block_from_universal(const void* const* universal_ptrs, void* const* block_ptrs,
                                         size_t num_blocks, size_t nh, size_t nl, size_t no, size_t nt, size_t hd,
                                         int dtype, int layout, cudaStream_t stream)
{
  return launch_permute<false>(const_cast<void* const*>(reinterpret_cast<const void* const*>(universal_ptrs)), block_ptrs,
                               num_blocks, nh, nl, no, nt, hd, dtype, layout, stream);
}

static bool fill_permute_side(const kvbm_permute_side& in, uint32_t nl, uint32_t no, uint32_t nh, uint32_t nt, uint32_t row, PermuteSide* out)
{
  const uint64_t head_run = static_cast<uint64_t>(nt) * row;
  PermuteSide p{};
  p.layer_base = in.layout.layer_base;
  p.ids = in.block_ids;
  p.block_stride = in.layout.block_stride;
  switch (in.kv_layout) {
    case KVBM_KV_UNIVERSAL_TP:
      p.universal = 1;
      p.layer_step = no * head_run;
      p.outer_step = head_run;
      p.head_stride = static_cast<uint64_t>(nl) * no * head_run;
      p.tok_stride = row;
      break;
    case KVBM_KV_UNIVERSAL_PP:
      p.universal = 1;
      p.layer_step = static_cast<uint64_t>(nh) * no * head_run;
      p.outer_step = head_run;
      p.head_stride = no * head_run;
      p.tok_stride = row;
      break;
    case KVBM_KV_OPERATIONAL_HND:
      p.outer_step = in.layout.outer_stride;
      p.head_stride = head_run;
      p.tok_stride = row;
      break;
    case KVBM_KV_OPERATIONAL_NHD:
      p.outer_step = in.layout.outer_stride;
      p.head_stride = row;
      p.tok_stride = static_cast<uint64_t>(nh) * row;
      break;
    default:
      return false;
  }
  if ((p.block_stride | p.outer_step) & 15) return false;
  *out = p;
  return true;
}

// Host-only view of the stride table the permuting kernel walks with (no GPU needed): lets the CPU suite check the
// address arithmetic of every KvBlockLayout against the oracle's dim_order definition, at sizes no GPU test allocates.
extern "C" int
kvbm_kernels_permute_strides(int kv_layout, uint32_t num_layers, uint32_t outer_dim, uint32_t num_heads, uint32_t page_size,
                             uint32_t row_bytes, uint64_t block_stride, uint64_t outer_stride, uint64_t out[5])
{
  if (!out) return 1;
  kvbm_permute_side side{};
  side.layout.block_stride = block_stride;
  side.layout.outer_stride = outer_stride;
  side.kv_layout = kv_layout;
  PermuteSide p;
  if (!fill_permute_side(side, num_layers, outer_dim, num_heads, page_size, row_bytes, &p)) return 1;
  out[0] = p.universal ? 1 : 0;  // 1: offsets are relative to the block's start; 0: relative to the (layer, outer) region
  out[1] = p.layer_step;
  out[2] = p.outer_step;
  out[3] = p.head_stride;
  out[4] = p.tok_stride;
  return 0;
}

extern "C" cudaError_t
kvbm_kernels_paged_permute(const kvbm_permute_side* src, const kvbm_permute_side* dst, int num_blocks, int layer_begin,
                           int layer_end, uint32_t num_heads, uint32_t page_size, uint32_t row_bytes, uint32_t* done_flag,
                           uint32_t epoch, uint32_t* completion_flag, uint32_t completion_value, cudaStream_t stream)
{
  if (num_blocks < 0 || layer_begin < 0 || layer_end < layer_begin) return cudaErrorInvalidValue;
  const bool signal = done_flag || completion_flag;
  auto finish = [&]() -> cudaError_t {
    if (!signal) return cudaSuccess;
    kvbm_signal_kernel<<<1, 1, 0, stream>>>(done_flag, epoch, completion_flag, completion_value);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    return cudaGetLastError();
  };
  if (num_blocks == 0 || layer_end == layer_begin) return finish();
  if (!src || !dst || !src->block_ids || !dst->block_ids || !src->layout.layer_base || !dst->layout.layer_base) return cudaErrorInvalidValue;
  const uint32_t nl = src->layout.num_layers, no = src->layout.outer_dim;
  if (nl == 0 || no == 0 || nl != dst->layout.num_layers || no != dst->layout.outer_dim || static_cast<uint32_t>(layer_end) > nl) return cudaErrorInvalidValue;
  if (row_bytes < 16 || row_bytes > 65536 || (row_bytes & 15) || num_heads == 0 || page_size == 0) return cudaErrorInvalidValue;
  const uint64_t region = static_cast<uint64_t>(page_size) * num_heads * row_bytes;
  if (region != src->layout.region_bytes || region != dst->layout.region_bytes) return cudaErrorInvalidValue;
  PermuteSide S, D;
  if (!fill_permute_side(*src, nl, no, num_heads, page_size, row_bytes, &S) ||
      !fill_permute_side(*dst, nl, no, num_heads, page_size, row_bytes, &D))
    return cudaErrorInvalidValue;
  const uint64_t units = static_cast<uint64_t>(num_blocks) * (layer_end - layer_begin) * no;
  if (units >= (1ull << 31)) return cudaErrorInvalidValue;
  const int threads = static_cast<int>(std::min<uint32_t>(8, num_heads)) * 32;
  const unsigned grid = static_cast<unsigned>(units);
  const uint32_t lb = static_cast<uint32_t>(layer_begin), nlay = static_cast<uint32_t>(layer_end - layer_begin);
  if ((row_bytes & (row_bytes - 1)) == 0) {
    uint32_t log2_v = 0;
    while ((16u << log2_v) < row_bytes) ++log2_v;
    kvbm_paged_permute_kernel<true><<<grid, threads, 0, stream>>>(S, D, lb, nlay, no, num_heads, page_size, log2_v, 0u);
  } else {
    const uint32_t V = row_bytes >> 4;
    const uint64_t magic = ((1ull << 32) + V - 1) / V;
    if (static_cast<uint64_t>(page_size) * V >= (1ull << 32) / V) return cudaErrorInvalidValue;  // exactness bound of the multiply-high division
    kvbm_paged_permute_kernel<false><<<grid, threads, 0, stream>>>(S, D, lb, nlay, no, num_heads, page_size, V, static_cast<uint32_t>(magic));
  }
  g_launches.fetch_add(1, std::memory_order_relaxed);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return e;
  return finish();
}

extern "C" bool
kvbm_kernels_has_memcpy_batch_async(void)
{
#if CUDART_VERSION >= 12090
  return true;
#else
  return false;
#endif
}

extern "C" bool
kvbm_kernels_is_stub_build(void)
{
  return false;
}

// =================================================================================================
// C ABI -- Part 2 (v2 extensions)
// =================================================================================================
static cudaError_t
paged_copy_impl(const kvbm_paged_layout* src, const kvbm_paged_dst* dsts, int num_dsts, int num_blocks,
                int layer_begin, int layer_end, int cast_mode, const kvbm_paged_copy_opts* opts,
                cudaStream_t stream)
{
  if (num_blocks == 0 || num_dsts == 0 || layer_end == layer_begin) return cudaSuccess;
  if (!src || !dsts) return cudaErrorInvalidValue;
  if (num_blocks < 0 || num_dsts < 0 || num_dsts > KVBM_MAX_DESTINATIONS) return cudaErrorInvalidValue;
  if (layer_begin < 0 || layer_end < layer_begin || static_cast<uint32_t>(layer_end) > src->num_layers)
    return cudaErrorInvalidValue;
  if (cast_mode < KVBM_CAST_NONE || cast_mode > KVBM_CAST_BF16_TO_FP8E4M3) return cudaErrorInvalidValue;
  if (!src->layer_base || src->region_bytes == 0) return cudaErrorInvalidValue;
  const uint32_t num = cast_mode == KVBM_CAST_FP8E4M3_TO_BF16 ? 2 : 1;
  const uint32_t den = cast_mode == KVBM_CAST_BF16_TO_FP8E4M3 ? 2 : 1;
  if (cast_mode == KVBM_CAST_BF16_TO_FP8E4M3 && (src->region_bytes & 1)) return cudaErrorInvalidValue;

  kvbm_paged_copy_opts o{};
  if (opts) o = *opts;
  if (o.reserved0 != 0 || o.reserved1 != 0) return cudaErrorInvalidValue;

  // NVLS: dsts[0] is addressed through a multicast mapping and carries the payload for every bound device; the
  // other entries only name the flags of the remaining receivers.
  const bool mc = o.multicast != 0;
  if (mc && (cast_mode != KVBM_CAST_NONE || (src->region_bytes & 3) || (src->block_stride & 3) || (src->outer_stride & 3) ||
             (dsts[0].layout.block_stride & 15) || (dsts[0].layout.outer_stride & 15)))
    return cudaErrorInvalidValue;
  const int data_dsts = mc ? 1 : num_dsts;

  PagedGen gen{};
  PagedSyncArgs sync{};
  gen.a.src = *src;
  gen.a.ndst = data_dsts;
  gen.a.replicate = 1;
  sync.num_flag_dsts = num_dsts;
  for (int d = 0; d < num_dsts; ++d) {
    const kvbm_paged_dst& D = dsts[d];
    sync.done_flag[d] = D.done_flag;
    sync.layer_done[d] = D.layer_done_flags;
    if (d >= data_dsts) continue;
    // same compatibility rules as execute_cuda_transfer (executor/cuda.rs:52-67) + region size match
    // (executor/memcpy.rs:143-153), adjusted for the element-width change of a cast
    if (!D.layout.layer_base || !D.src_block_ids || !D.dst_block_ids) return cudaErrorInvalidValue;
    if (D.layout.num_layers != src->num_layers || D.layout.outer_dim != src->outer_dim) return cudaErrorInvalidValue;
    if (static_cast<uint64_t>(D.layout.region_bytes) * den != static_cast<uint64_t>(src->region_bytes) * num)
      return cudaErrorInvalidValue;
    gen.a.dst[d] = D.layout;
    gen.a.src_ids[d] = D.src_block_ids;
    gen.a.dst_ids[d] = D.dst_block_ids;
    if (D.src_block_ids != dsts[0].src_block_ids) gen.a.replicate = 0;
  }
  if (data_dsts == 1) gen.a.replicate = 1;
  sync.completion_flag = o.completion_flag;
  sync.completion_value = o.completion_value;
  sync.layer_ready = o.layer_ready_flags;
  sync.epoch = o.epoch;
  sync.gate_timeout_ns = static_cast<uint64_t>(o.gate_timeout_ms > 0 ? o.gate_timeout_ms : 10000) * 1000000ull;
  if (o.layer_ready_flags && !o.sync_workspace) return cudaErrorInvalidValue;  // the abort word lives in the workspace
  bool needs_ws = o.completion_flag != nullptr;
  for (int d = 0; d < num_dsts; ++d)
    if (dsts[d].done_flag || dsts[d].layer_done_flags) needs_ws = true;
  if (needs_ws && !o.sync_workspace) return cudaErrorInvalidValue;

  DeviceInfo di;
  cudaError_t e = device_info(&di);
  if (e != cudaSuccess) return e;
  RingCfg rc = make_ring(di, src->region_bytes, o.warps_per_cta, o.stages, o.tile_bytes, cast_mode, o.stores_in_flight);

  gen.a.n_blocks = static_cast<uint32_t>(num_blocks);
  gen.a.layer_begin = static_cast<uint32_t>(layer_begin);
  gen.a.n_layers = static_cast<uint32_t>(layer_end - layer_begin);
  gen.a.outer = src->outer_dim;
  gen.a.tile = rc.tile;
  gen.a.tiles_per_region = (src->region_bytes + rc.tile - 1) / rc.tile;
  gen.a.dst_num = num;
  gen.a.dst_den = den;
  const uint64_t fan = gen.a.replicate ? 1 : static_cast<uint64_t>(data_dsts);
  const uint64_t total = static_cast<uint64_t>(gen.a.n_layers) * gen.a.n_blocks * gen.a.outer * fan * gen.a.tiles_per_region;
  if (total >= (1ull << 31)) return cudaErrorInvalidValue;

  const uint64_t rings_needed = (total + rc.batch - 1) / rc.batch;
  const uint64_t ctas_needed = (rings_needed + rc.rings - 1) / rc.rings;
  // Default: one CTA per SM (see the note at kDefaultTile); max_ctas leaves SMs to whatever the engine is running.
  int cap = o.max_ctas > 0 ? o.max_ctas : default_ctas(di);
  const int grid = static_cast<int>(std::min<uint64_t>(ctas_needed, static_cast<uint64_t>(cap)));
  const int allow_tma = o.force_simt ? 0 : 1;
  const uint32_t total32 = static_cast<uint32_t>(total);

  // control words: the caller's workspace ([num_layers] layer counters, then 3 control words) or a pool slot
  int dev = 0, pool_slot = -1;
  if (o.sync_workspace) {
    sync.layer_counters = o.sync_workspace;
    sync.ctl = o.sync_workspace + src->num_layers;
  } else if (!o.static_schedule && cudaGetDevice(&dev) == cudaSuccess && dev >= 0 && dev < 64) {
    sync.ctl = sched_acquire(dev, stream, &pool_slot);
  }

  auto launch = [&](auto kern) -> cudaError_t {
    cudaError_t err = set_smem(kern, rc.smem);
    if (err == cudaSuccess) {
      kern<<<grid, rc.rings * 64, rc.smem, stream>>>(gen, sync, total32, rc.stages, rc.pending, rc.batch, o.static_schedule,
                                                     rc.out_tile, allow_tma, mc && o.multicast != 2);
      g_launches.fetch_add(1, std::memory_order_relaxed);
      err = cudaGetLastError();
    }
    sched_release(dev, pool_slot, stream);
    return err;
  };
  // the plain hot path gets the kernel with the generality folded away at compile time (copy_engine.cuh, FAST)
  bool any_layer_flags = false;
  for (int d = 0; d < num_dsts; ++d) any_layer_flags = any_layer_flags || dsts[d].layer_done_flags != nullptr;
  const bool fast = !mc && allow_tma && !o.layer_ready_flags && !any_layer_flags &&
                    (gen.a.replicate ? data_dsts : 1) == 1;
  switch (cast_mode) {
    case KVBM_CAST_NONE:
      return fast ? launch(kvbm_paged_copy_kernel<KVBM_CAST_NONE, true>) : launch(kvbm_paged_copy_kernel<KVBM_CAST_NONE, false>);
    case KVBM_CAST_FP8E4M3_TO_BF16:
      return fast ? launch(kvbm_paged_copy_kernel<KVBM_CAST_FP8E4M3_TO_BF16, true>) : launch(kvbm_paged_copy_kernel<KVBM_CAST_FP8E4M3_TO_BF16, false>);
    default:
      return fast ? launch(kvbm_paged_copy_kernel<KVBM_CAST_BF16_TO_FP8E4M3, true>) : launch(kvbm_paged_copy_kernel<KVBM_CAST_BF16_TO_FP8E4M3, false>);
  }
}

// CUDA loads modules lazily by default, and the first launch of a not-yet-loaded kernel (of ANY module in the process)
// can wait for the device to drain -- which never happens while a gated transfer spins on ready flags that the stalled
// launch was supposed to release.  This library preloads its own kernels, but it cannot load the engine's.  So a
// spinning gate is only used when the process runs with eager loading (or the caller insists); otherwise the gate
// moves to the stream front-end: one cuStreamWaitValue32 + one single-layer launch per layer -- nothing resident spins.
static bool eager_module_loading()
{
  static const int mode = [] {
    typedef int (*fn_t)(int*);
    void* f = nullptr;
    cudaDriverEntryPointQueryResult r;
    int m = 0;
    if (cudaGetDriverEntryPoint("cuModuleGetLoadingMode", &f, cudaEnableDefault, &r) == cudaSuccess && f &&
        reinterpret_cast<fn_t>(f)(&m) == 0)
      return m;
    (void)cudaGetLastError();
    return 0;
  }();
  return mode == 1;  // CU_MODULE_EAGER_LOADING
}

extern "C" int
kvbm_kernels_gate_would_spin(void)
{
  return eager_module_loading() ? 1 : 0;
}

extern "C" cudaError_t
kvbm_kernels_paged_copy_v2(const kvbm_paged_layout* src, const kvbm_paged_dst* dsts, int num_dsts, int num_blocks,
                           int layer_begin, int layer_end, int cast_mode, const kvbm_paged_copy_opts* opts,
                           cudaStream_t stream)
{
  const bool gated = opts && opts->layer_ready_flags != nullptr;
  if (!gated || num_blocks == 0 || num_dsts == 0 || layer_end <= layer_begin || !dsts || num_dsts < 0 || num_dsts > KVBM_MAX_DESTINATIONS)
    return paged_copy_impl(src, dsts, num_dsts, num_blocks, layer_begin, layer_end, cast_mode, opts, stream);
  const int mode = opts->gate_mode;
  if (mode < KVBM_GATE_AUTO || mode > KVBM_GATE_STREAM_WAIT) return cudaErrorInvalidValue;
  if (mode == KVBM_GATE_SPIN || (mode == KVBM_GATE_AUTO && eager_module_loading()))
    return paged_copy_impl(src, dsts, num_dsts, num_blocks, layer_begin, layer_end, cast_mode, opts, stream);
  DeviceInfo di;
  cudaError_t e = device_info(&di);
  if (e != cudaSuccess) return e;
  if (!stream_memops()) return mode == KVBM_GATE_AUTO ? paged_copy_impl(src, dsts, num_dsts, num_blocks, layer_begin, layer_end, cast_mode, opts, stream)
                                                       : cudaErrorNotSupported;
  kvbm_paged_copy_opts o = *opts;
  o.layer_ready_flags = nullptr;
  kvbm_paged_dst dd[KVBM_MAX_DESTINATIONS];
  for (int l = layer_begin; l < layer_end; ++l) {
    const bool last = l + 1 == layer_end;
    // CU_STREAM_WAIT_VALUE_GEQ: the stream front-end polls the word, no SM is occupied
    if (g_wait32(stream, reinterpret_cast<unsigned long long>(opts->layer_ready_flags + l), opts->epoch, 0) != 0) return cudaErrorUnknown;
    for (int d = 0; d < num_dsts; ++d) {
      dd[d] = dsts[d];
      if (!last) dd[d].done_flag = nullptr;
    }
    o.completion_flag = last ? opts->completion_flag : nullptr;
    if ((e = paged_copy_impl(src, dd, num_dsts, num_blocks, l, l + 1, cast_mode, &o, stream)) != cudaSuccess) return e;
  }
  return cudaSuccess;
}

extern "C" cudaError_t
kvbm_kernels_set_flags(uint32_t* flags, int first, int count, uint32_t value, cudaStream_t stream)
{
  if (count == 0) return cudaSuccess;
  if (!flags || count < 0 || first < 0) return cudaErrorInvalidValue;
  DeviceInfo di;
  cudaError_t e = device_info(&di);
  if (e != cudaSuccess) return e;
  if (count == 1 && stream_memops()) {
    // CU_STREAM_WRITE_VALUE_DEFAULT (0): memory fence before the write => release semantics for prior work
    if (g_write32(stream, reinterpret_cast<unsigned long long>(flags + first), value, 0) == 0) return cudaSuccess;
  }
  kvbm_set_flags_kernel<<<(count + 127) / 128, 128, 0, stream>>>(flags, first, count, value);
  g_launches.fetch_add(1, std::memory_order_relaxed);
  return cudaGetLastError();
}

extern "C" cudaError_t
kvbm_kernels_wait_flag(const uint32_t* flag, uint32_t value, cudaStream_t stream)
{
  if (!flag) return cudaErrorInvalidValue;
  DeviceInfo di;
  cudaError_t e = device_info(&di);
  if (e != cudaSuccess) return e;
  if (stream_memops()) {
    // CU_STREAM_WAIT_VALUE_GEQ (0): wait until (int32)(*flag - value) >= 0
    if (g_wait32(stream, reinterpret_cast<unsigned long long>(flag), value, 0) == 0) return cudaSuccess;
  }
  kvbm_wait_flag_kernel<<<1, 1, 0, stream>>>(flag, value);
  g_launches.fetch_add(1, std::memory_order_relaxed);
  return cudaGetLastError();
}

extern "C" cudaError_t
kvbm_kernels_stream_wait_event(cudaStream_t stream, void* event)
{
  if (!event) return cudaErrorInvalidValue;
  return cudaStreamWaitEvent(stream, static_cast<cudaEvent_t>(event), 0);
}

extern "C" uint64_t
kvbm_kernels_launch_count(void)
{
  return g_launches.load(std::memory_order_relaxed);
}

extern "C" const char*
kvbm_kernels_build_info(void)
{
  return "libkvbm_kernels sm_100a tma=cp.async.bulk cast=e4m3<->bf16";
}
