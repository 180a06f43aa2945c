// The warp-specialised TMA ring that every paged KV transfer kernel in this library is built from.
//
//     HBM (paged source) --cp.async.bulk--> smem slot --cp.async.bulk--> HBM / NVLink peer (1..N) / multicast
//
// A ring is TWO warps sharing S shared-memory slots of `tile` bytes:
//   * the PRODUCER warp claims work from a grid-wide dynamic tile scheduler (atomic tickets, guided batch size),
//     turns the claimed items into addresses with all 32 lanes at once (block-table lookups are SIMD), waits for the
//     layer's ready flag when the transfer is gated, and issues the bulk loads (completion counted in bytes on the
//     slot's `full` mbarrier).  It never waits for data.
//   * the CONSUMER warp waits for `full`, issues the bulk stores (or converts fp8<->bf16 / stores SIMT / multimem),
//     hands the slot back through the `empty` mbarrier once the store has read it, and publishes per-layer and
//     whole-transfer completion.  It never computes an address.
// A CTA holds R such rings.  Why dynamic scheduling: SMs of a B200 do not move bytes at the same rate (two dies, L2
// slice distance) -- with a static split the slowest ring finished 80-100 us after the fastest on a 170 us copy
// (benchmarks/copylab.cu, profiles/r02_copylab_n1.jsonl); with tickets all rings finish within ~5 us.
#pragma once
#include "ptx.cuh"

namespace kvbm {

constexpr int kMaxDst = 8;
constexpr int kMaxStages = 16;
constexpr int kMaxBatch = 32;  // items claimed per ticket (one per producer lane)

// One unit of work: `bytes` (of source) from `src` to each of dst[0..ndst).
struct Piece {
  const uint8_t* src;
  uint8_t* dst[kMaxDst];
  uint32_t bytes;  // source bytes
  int ndst;
  int layer;  // for layer-streaming flags (0 when unused)
};

// ------------------------------------------------------------------------------------------
// SIMT ladder for pieces TMA cannot take.  Same alignment contract as the reference K1 kernel
// (/root/reference/lib/kvbm-kernels/cuda/tensor_kernels.cu:511-540): the widest vector both
// pointers allow, byte tail.  `tid`/`nthr` = the cooperating group (a warp or a whole CTA);
// 8 independent 16 B loads in flight per thread on the aligned path.
// ------------------------------------------------------------------------------------------
template <int U = 8>
__device__ __forceinline__ void group_copy_simt(uint8_t* dst, const uint8_t* src, size_t bytes, uint32_t tid, uint32_t nthr)
{
  const uintptr_t both = reinterpret_cast<uintptr_t>(dst) | reinterpret_cast<uintptr_t>(src);
  size_t done = 0;
  if ((both & 15) == 0) {
    const size_t n = bytes >> 4;
    const uint4* s = reinterpret_cast<const uint4*>(src);
    uint4* d = reinterpret_cast<uint4*>(dst);
    size_t i = tid;
    for (; i + static_cast<size_t>(U - 1) * nthr < n; i += static_cast<size_t>(U) * nthr) {
      uint4 v[U];
#pragma unroll
      for (int u = 0; u < U; ++u) v[u] = ptx::ld_stream_v4(s + i + static_cast<size_t>(u) * nthr);
#pragma unroll
      for (int u = 0; u < U; ++u) ptx::st_stream_v4(d + i + static_cast<size_t>(u) * nthr, v[u]);
    }
    for (; i < n; i += nthr) ptx::st_stream_v4(d + i, ptx::ld_stream_v4(s + i));
    done = n << 4;
  } else if ((both & 7) == 0) {
    const size_t n = bytes >> 3;
    const uint2* s = reinterpret_cast<const uint2*>(src);
    uint2* d = reinterpret_cast<uint2*>(dst);
#pragma unroll 4
    for (size_t i = tid; i < n; i += nthr) d[i] = s[i];
    done = n << 3;
  } else if ((both & 3) == 0) {
    const size_t n = bytes >> 2;
    const uint32_t* s = reinterpret_cast<const uint32_t*>(src);
    uint32_t* d = reinterpret_cast<uint32_t*>(dst);
#pragma unroll 4
    for (size_t i = tid; i < n; i += nthr) d[i] = s[i];
    done = n << 2;
  }
#pragma unroll 4
  for (size_t i = done + tid; i < bytes; i += nthr) dst[i] = src[i];
}

__device__ __forceinline__ void warp_copy_simt(uint8_t* dst, const uint8_t* src, uint32_t bytes, int lane)
{
  group_copy_simt(dst, src, bytes, static_cast<uint32_t>(lane), 32u);
}

__device__ __forceinline__ bool piece_tma_ok(const Piece& p)
{
  uintptr_t m = reinterpret_cast<uintptr_t>(p.src) | p.bytes;
#pragma unroll
  for (int d = 0; d < kMaxDst; ++d)
    if (d < p.ndst) m |= reinterpret_cast<uintptr_t>(p.dst[d]);
  return (m & 15) == 0 && p.bytes != 0;
}

// Layer-streaming / completion hooks shared by the rings.  All pointers may be null.
// `ctl` is three zeroed words the launch owns: [0] rings finished, [1] abort, [2] scheduler tickets.  They are left
// zeroed by the last ring to finish, so the same words serve the next launch.
struct StreamSync {
  const uint32_t* layer_ready;  // wait until layer_ready[l] >= epoch before reading layer l
  uint32_t* layer_counters;     // [num_layers] zeroed: items of layer l that have landed
  uint32_t* ctl;                // see above; null = static tile schedule, no completion signals
  uint32_t* done_flag[kMaxDst];
  uint32_t* layer_done[kMaxDst];
  uint32_t* completion_flag;    // extra whole-transfer flag (host-mapped memory allowed)
  uint32_t completion_value;
  uint32_t epoch;
  uint32_t total_rings;
  uint32_t items_per_layer;
  int ndst;
  int layer_begin, layer_end;
  uint64_t gate_timeout_ns;  // a gated wait longer than this aborts the transfer instead of spinning forever
  bool gate;         // layer_ready present: reads of a layer wait for its flag
  bool want_layers;  // some destination wants per-layer done flags
  bool want_done;    // some whole-transfer flag is wanted
};

// Ring geometry / behaviour of one launch (uniform across the grid).
struct RingParams {
  int S;              // slots per ring
  int P;              // TMA stores allowed to keep draining their slot (loads ahead = S - P)
  int batch;          // largest ticket (items), <= kMaxBatch
  uint32_t tile_in;   // source bytes per slot
  uint32_t tile_out;  // cast rings: bytes per output buffer (2 of them)
  bool allow_tma;
  bool static_schedule;  // diagnostics: round-robin batches even when control words exist
  bool multimem;      // TMA load + multimem.st from smem to an NVLS multicast address (byte copies only);
                      // otherwise TMA load + TMA store
};

// Per-slot control block the producer fills before it arms the slot's `full` barrier.
struct SlotCtl {
  uint64_t src;
  uint64_t dst[kMaxDst];
  uint32_t bytes;  // bit31: the payload arrives in the slot by TMA; otherwise the consumer moves it SIMT from `src`
  uint32_t layer;  // bit31: end of this ring's stream
};
constexpr uint32_t kSlotTma = 0x80000000u;
constexpr uint32_t kSlotEnd = 0x80000000u;

// shared memory of one ring: [full[S] | empty[S]] mbarriers (16 * kMaxStages bytes), SlotCtl[kMaxStages]
__host__ __device__ constexpr uint32_t ring_ctl_bytes() { return 16u * kMaxStages + static_cast<uint32_t>(sizeof(SlotCtl)) * kMaxStages; }

struct RingSmem {
  uint32_t full0, empty0;  // shared-space addresses of the barrier arrays
  SlotCtl* ctl;
  uint32_t in0;   // S * tile_in
  uint32_t out0;  // 2 * tile_out (cast only)
};

// Flag polls are relaxed loads; one acquire fence follows a successful probe (an ld.acquire.sys per poll would
// invalidate L1 every time and, measured, slowed the co-resident compute kernel).
// Returns false when the flag was not released within gate_timeout_ns or another ring already gave up: a spinning
// kernel that waits for work which can never be submitted (e.g. because a lazy module load is itself waiting for this
// kernel) must not hang the GPU; the ring then records the abort and stops claiming work.
__device__ __forceinline__ bool wait_layer_ready(const StreamSync& ss, int layer, int lane)
{
  uint32_t ok = 1;
  if (lane == 0) {
    const uint64_t t0 = ptx::globaltimer_ns();
    uint32_t polls = 0;
    while (ptx::ld_relaxed_sys(ss.layer_ready + layer) < ss.epoch) {
      __nanosleep(128);
      if ((++polls & 255u) == 0) {
        if (ptx::ld_relaxed_sys(ss.ctl + 1) != 0) {
          ok = 0;
          break;
        }
        if (ptx::globaltimer_ns() - t0 > ss.gate_timeout_ns) {
          ok = 0;
          atomicExch(ss.ctl + 1, 1u);
          break;
        }
      }
    }
    ptx::fence_acq_rel_sys();
  }
  ok = __shfl_sync(0xffffffffu, ok, 0);
  return ok != 0;
}

// `count` more items of `layer` have landed (stores complete, ordered before this call by the caller).
__device__ __forceinline__ void arrive_layer(const StreamSync& ss, int layer, uint32_t count)
{
  const uint32_t old = ptx::atom_add_acq_rel_gpu(ss.layer_counters + layer, count);
  if (old + count == ss.items_per_layer) {
    ss.layer_counters[layer] = 0;  // leave the workspace zeroed for the next launch
    ptx::fence_acq_rel_sys();      // once per layer for the whole grid: everything acquired above is released below
#pragma unroll
    for (int d = 0; d < kMaxDst; ++d)
      if (d < ss.ndst && ss.layer_done[d] != nullptr) ptx::st_relaxed_sys(ss.layer_done[d] + layer, ss.epoch);
  }
}

// This ring is finished (its stores have landed).  The last ring to get here re-zeroes the control words and
// publishes the whole-transfer signals.
__device__ __forceinline__ void arrive_transfer(const StreamSync& ss)
{
  if (ss.ctl == nullptr) return;
  const uint32_t old = ptx::atom_add_acq_rel_gpu(ss.ctl, 1u);
  if (old != ss.total_rings - 1) return;
  ss.ctl[0] = 0;
  ss.ctl[2] = 0;
  const bool aborted = atomicExch(ss.ctl + 1, 0u) != 0;
  if (aborted && ss.layer_counters != nullptr)  // partial layer counts must not leak into the next launch
    for (int l = ss.layer_begin; l < ss.layer_end; ++l) ss.layer_counters[l] = 0;
  if (!ss.want_done) return;
  ptx::fence_acq_rel_sys();
  if (!aborted) {
#pragma unroll
    for (int d = 0; d < kMaxDst; ++d)
      if (d < ss.ndst && ss.done_flag[d] != nullptr) ptx::st_relaxed_sys(ss.done_flag[d], ss.epoch);
  }
  // 0xFFFFFFFF = "this transfer gave up waiting for a layer": destinations are NOT told it completed
  if (ss.completion_flag != nullptr) ptx::st_relaxed_sys(ss.completion_flag, aborted ? 0xFFFFFFFFu : ss.completion_value);
}

// smem -> NVLink multicast address (multimem rings): one store, the switch delivers it to every bound device
__device__ __forceinline__ void warp_store_from_smem_mc(uint8_t* dst, uint32_t src_smem, uint32_t bytes, int lane)
{
  uint4* d = reinterpret_cast<uint4*>(dst);
  const uint32_t n = bytes >> 4;
  for (uint32_t i = lane; i < n; i += 32) {
    uint4 v;
    asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(src_smem + i * 16));
    ptx::multimem_st_v4(d + i, v);
  }
}
// global -> multicast for pieces the TMA load cannot take (the launcher guarantees 4-byte granularity)
__device__ __forceinline__ void warp_copy_simt_mc(uint8_t* dst, const uint8_t* src, uint32_t bytes, int lane)
{
  const uintptr_t both = reinterpret_cast<uintptr_t>(src) | reinterpret_cast<uintptr_t>(dst) | bytes;
  if ((both & 15) == 0) {
    const uint4* s = reinterpret_cast<const uint4*>(src);
    uint4* d = reinterpret_cast<uint4*>(dst);
    for (uint32_t i = lane; i < (bytes >> 4); i += 32) ptx::multimem_st_v4(d + i, ptx::ld_stream_v4(s + i));
  } else {
    const uint32_t* s = reinterpret_cast<const uint32_t*>(src);
    uint32_t* d = reinterpret_cast<uint32_t*>(dst);
    for (uint32_t i = lane; i < (bytes >> 2); i += 32) ptx::multimem_st_b32(d + i, s[i]);
  }
}

template <bool UP>
__device__ __forceinline__ void convert_smem(uint32_t in_smem, uint32_t out_smem, uint32_t src_bytes, int lane);
template <bool UP>
__device__ __forceinline__ void warp_cast_simt(uint8_t* dst, const uint8_t* src, uint32_t src_bytes, int lane);

// ------------------------------------------------------------------------------------------
// Producer warp.  Gen::get(item, Piece&) is called by up to `batch` lanes at once (one item each).
// Work is claimed in ITEMS: the first ticket of every ring is static (ring r takes items [r*B, (r+1)*B) -- no atomic
// on the ramp), later tickets come from ss.ctl[2] and shrink towards the end of the transfer (guided self-scheduling)
// so that all rings run dry together.  Without control words the schedule is a static round-robin of batches.
// ------------------------------------------------------------------------------------------
// FAST = the plain hot path, known at compile time: one destination, TMA load + TMA store, no gating and no per-layer
// flags.  A ring is ONE instruction stream per direction, so every instruction of the per-item chain costs
// its full latency (~10 ns); folding the run-time generality away is worth 10 % on the HBM-bound copy
// (profiles/r02_copylab_libsweep.jsonl vs r02_copylab_engine.jsonl).
template <int CAST, bool FAST, class Gen>
__device__ __forceinline__ void ring_producer(const Gen& gen, uint32_t total, uint32_t my_ring, uint32_t nrings,
                                              const RingSmem& sm, int ndst_rt, const RingParams& rp, const StreamSync& ss)
{
  const int lane = threadIdx.x & 31;
  const int ndst = FAST ? 1 : ndst_rt;
  const bool allow_tma = FAST ? true : rp.allow_tma;
  const bool gate = FAST ? false : ss.gate;
  const int S = rp.S;
  const uint32_t B = static_cast<uint32_t>(rp.batch);
  const bool dynamic = ss.ctl != nullptr && !rp.static_schedule;
  int ready_layer = gate ? ss.layer_begin - 1 : 0x7fffffff;
  uint32_t k = 0;          // tickets taken
  uint32_t last_start = 0;
  int slot = 0;            // slot of the next item; `wait_parity` = parity the producer waits for on empty[slot]
  uint32_t wait_parity = 1;
  bool aborted = false;

  while (!aborted) {
    uint32_t item0, cnt;
    if (k == 0) {
      item0 = my_ring * B;
      cnt = B;
    } else if (dynamic) {
      const uint32_t remaining = total > last_start ? total - last_start : 0;
      uint32_t want = remaining / (4u * nrings);
      want = want < 1u ? 1u : (want > B ? B : want);
      uint32_t t = 0;
      if (lane == 0) t = atomicAdd(ss.ctl + 2, want);
      item0 = nrings * B + __shfl_sync(0xffffffffu, t, 0);
      cnt = want;
    } else {
      item0 = (my_ring + k * nrings) * B;
      cnt = B;
    }
    ++k;
    last_start = item0;
    if (item0 >= total) break;
    cnt = min(cnt, total - item0);

    Piece p;
    p.src = nullptr;
    p.bytes = 0;
    p.ndst = ndst;
    p.layer = 0;
    uint32_t meta = 0;  // bytes | kSlotTma
    if (static_cast<uint32_t>(lane) < cnt) {
      gen.get(item0 + lane, p);
      bool ok = allow_tma && piece_tma_ok(p);
      if (CAST != 0) ok = ok && (p.bytes & 31) == 0;  // both sides whole 16 B vectors
      meta = p.bytes | (ok ? kSlotTma : 0u);
    }
    for (uint32_t i = 0; i < cnt; ++i) {
      const uint64_t src_i = __shfl_sync(0xffffffffu, reinterpret_cast<uint64_t>(p.src), i);
      const uint32_t meta_i = __shfl_sync(0xffffffffu, meta, i);
      const int layer_i = FAST ? 0 : __shfl_sync(0xffffffffu, p.layer, i);
      uint64_t dst_i[kMaxDst];
#pragma unroll
      for (int d = 0; d < kMaxDst; ++d)
        if (d < ndst) dst_i[d] = __shfl_sync(0xffffffffu, reinterpret_cast<uint64_t>(p.dst[d]), i);
      if (!FAST && layer_i > ready_layer) {
        if (!wait_layer_ready(ss, layer_i, lane)) {  // gate timeout: abandon the rest (the abort is recorded)
          aborted = true;
          break;
        }
        ready_layer = layer_i;
      }
      if (lane == 0) {
        ptx::mbar_wait(sm.empty0 + 8 * slot, wait_parity);
        SlotCtl& c = sm.ctl[slot];
        c.src = src_i;
#pragma unroll
        for (int d = 0; d < kMaxDst; ++d)
          if (d < ndst) c.dst[d] = dst_i[d];
        c.layer = static_cast<uint32_t>(layer_i);
        c.bytes = meta_i;
        const uint32_t bytes_i = meta_i & ~kSlotTma;
        if (meta_i & kSlotTma) {
          ptx::mbar_arrive_expect_tx(sm.full0 + 8 * slot, bytes_i);
          ptx::bulk_g2s(sm.in0 + slot * rp.tile_in, reinterpret_cast<const void*>(src_i), bytes_i, sm.full0 + 8 * slot);
        } else {
          ptx::mbar_arrive(sm.full0 + 8 * slot);
        }
      }
      if (++slot == S) {
        slot = 0;
        wait_parity ^= 1u;
      }
    }
    __syncwarp();
  }
  // end of this ring's stream
  if (lane == 0) {
    ptx::mbar_wait(sm.empty0 + 8 * slot, wait_parity);
    sm.ctl[slot].layer = kSlotEnd;
    sm.ctl[slot].bytes = 0;
    ptx::mbar_arrive(sm.full0 + 8 * slot);
  }
}

// ------------------------------------------------------------------------------------------
// Consumer warp.  CAST: 0 byte-exact, 1 fp8->bf16, 2 bf16->fp8.
// Layer completion is published eagerly: whenever the consumer would stall on an empty ring, or moves to another
// layer, it drains its stores and adds what it finished to the layer's counter -- so a receiver that releases
// layer l+1 only after seeing layer l done can never dead-lock against a producer blocked on l+1's gate.
// ------------------------------------------------------------------------------------------
template <int CAST, bool FAST>
__device__ __forceinline__ void ring_consumer(const RingSmem& sm, int ndst_rt, const RingParams& rp, const StreamSync& ss)
{
  const int lane = threadIdx.x & 31;
  const int ndst = FAST ? 1 : ndst_rt;
  const bool multimem = FAST ? false : rp.multimem;
  const bool want_layers = FAST ? false : ss.want_layers;
  const int S = rp.S;
  const int P = rp.P;
  const bool deferred_release = CAST == 0 && !multimem;  // TMA stores read the input slot asynchronously
  uint32_t deferred = 0;  // bit (q & 31): item q's slot is handed back once its bulk store has read it
  int cur_layer = -1;
  uint32_t unpublished = 0;

  // every store issued so far has landed and is ordered before the atomics that follow
  auto drain = [&]() {
    if (lane == 0) {
      ptx::bulk_wait<0>();
      ptx::fence_proxy_async_global();
    }
    __syncwarp();
  };
  auto release_upto = [&](uint32_t q_end) {  // lane 0: hand back every deferred slot of items < q_end (all within 32 items)
    while (deferred != 0) {
      const int b = __ffs(static_cast<int>(deferred)) - 1;
      // bit b belongs to the youngest item j < q_end with (j & 31) == b
      const uint32_t j = ((q_end - 1 - static_cast<uint32_t>(b)) & ~31u) + static_cast<uint32_t>(b);
      ptx::mbar_arrive(sm.empty0 + 8 * (j % S));
      deferred &= deferred - 1;
    }
  };
  auto publish = [&](uint32_t q_now) {
    drain();
    if (lane == 0) {
      if (deferred_release) release_upto(q_now);
      arrive_layer(ss, cur_layer, unpublished);
    }
    unpublished = 0;
  };

  uint32_t q = 0;
  int slot = 0;          // slot of item q
  uint32_t parity = 0;   // parity the consumer waits for on full[slot]
  int rel_slot = 0;      // slot of item q - P (the next deferred release)
  for (;; ++q) {
    if (want_layers && unpublished != 0) {
      uint32_t ready = 0;
      if (lane == 0) ready = ptx::mbar_try_wait(sm.full0 + 8 * slot, parity) ? 1u : 0u;
      ready = __shfl_sync(0xffffffffu, ready, 0);
      if (!ready) publish(q);
    }
    ptx::mbar_wait(sm.full0 + 8 * slot, parity);  // every lane observes the slot (control block + landed bytes)
    const SlotCtl& c = sm.ctl[slot];
    const uint32_t meta_layer = c.layer;
    if (meta_layer & kSlotEnd) break;
    const uint32_t meta_bytes = c.bytes;
    const uint32_t bytes = meta_bytes & ~kSlotTma;
    const bool tma = (meta_bytes & kSlotTma) != 0;
    const int layer = static_cast<int>(meta_layer);
    const uint32_t in = sm.in0 + slot * rp.tile_in;
    if (want_layers && unpublished != 0 && layer != cur_layer) publish(q);
    cur_layer = layer;

    if (!tma) {
      // SIMT from global to global; the slot carries only the addresses
      const uint8_t* src = reinterpret_cast<const uint8_t*>(c.src);
      for (int d = 0; d < ndst; ++d) {
        uint8_t* dst = reinterpret_cast<uint8_t*>(c.dst[d]);
        if (CAST == 0 && multimem)
          warp_copy_simt_mc(dst, src, bytes, lane);
        else if (CAST == 0)
          warp_copy_simt(dst, src, bytes, lane);
        else
          warp_cast_simt<CAST == 1>(dst, src, bytes, lane);
      }
      __syncwarp();
      if (lane == 0) {
        ptx::mbar_arrive(sm.empty0 + 8 * slot);
        ptx::bulk_commit();  // always one group per item (possibly empty) so the wait_group counts hold
      }
    } else if (CAST == 0 && !multimem) {
      if (lane == 0) {
#pragma unroll
        for (int d = 0; d < kMaxDst; ++d)
          if (d < ndst) ptx::bulk_s2g(reinterpret_cast<void*>(c.dst[d]), in, bytes);
        ptx::bulk_commit();
        deferred |= 1u << (q & 31);
      }
    } else if (CAST == 0) {  // multimem: the warp's stores have read the slot, so it is released right away
      warp_store_from_smem_mc(reinterpret_cast<uint8_t*>(c.dst[0]), in, bytes, lane);
      __syncwarp();
      if (lane == 0) {
        ptx::mbar_arrive(sm.empty0 + 8 * slot);
        ptx::bulk_commit();
      }
    } else {
      const uint32_t dst_bytes = CAST == 1 ? bytes * 2 : bytes / 2;
      const uint32_t ob = sm.out0 + (q & 1) * rp.tile_out;
      if (lane == 0) ptx::bulk_wait_read<1>();  // store q-2 (same out buffer) has been read out
      __syncwarp();
      convert_smem<CAST == 1>(in, ob, bytes, lane);
      ptx::fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) {
        ptx::mbar_arrive(sm.empty0 + 8 * slot);  // the input slot is free as soon as it has been converted
#pragma unroll
        for (int d = 0; d < kMaxDst; ++d)
          if (d < ndst) ptx::bulk_s2g(reinterpret_cast<void*>(c.dst[d]), ob, dst_bytes);
        ptx::bulk_commit();
      }
    }
    if (deferred_release) {
      if (lane == 0) {
        // stores q-P+1..q may still be reading their slots; everything older has left shared memory
        if (P == 1)
          ptx::bulk_wait_read<1>();
        else if (P == 2)
          ptx::bulk_wait_read<2>();
        else
          ptx::bulk_wait_read_n(P);
        if (q >= static_cast<uint32_t>(P)) {
          const uint32_t bit = 1u << ((q - P) & 31);
          if (deferred & bit) {
            ptx::mbar_arrive(sm.empty0 + 8 * rel_slot);
            deferred &= ~bit;
          }
        }
      }
      if (q >= static_cast<uint32_t>(P) && ++rel_slot == S) rel_slot = 0;
    }
    ++unpublished;
    if (++slot == S) {
      slot = 0;
      parity ^= 1u;
    }
  }

  drain();
  if (lane == 0) {
    if (want_layers && unpublished != 0) arrive_layer(ss, cur_layer, unpublished);
    arrive_transfer(ss);
  }
}

// ------------------------------------------------------------------------------------------
// Conversion helpers of the cast rings.
// ------------------------------------------------------------------------------------------
template <bool UP>
__device__ __forceinline__ void convert_smem(uint32_t in_smem, uint32_t out_smem, uint32_t src_bytes,
                                             int lane)
{
  if (UP) {
    // 16 fp8 in (16 B) -> 16 bf16 out (32 B) per lane-iteration
    for (uint32_t off = lane * 16; off < src_bytes; off += 32 * 16) {
      uint4 v;
      asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(in_smem + off));
      uint32_t w[4] = {v.x, v.y, v.z, v.w};
      uint32_t o[8];
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        o[2 * k] = ptx::e4m3x2_to_bf16x2(static_cast<uint16_t>(w[k] & 0xffff));
        o[2 * k + 1] = ptx::e4m3x2_to_bf16x2(static_cast<uint16_t>(w[k] >> 16));
      }
      asm volatile("st.shared.v4.u32 [%0], {%1,%2,%3,%4};" ::"r"(out_smem + 2 * off), "r"(o[0]), "r"(o[1]), "r"(o[2]), "r"(o[3]) : "memory");
      asm volatile("st.shared.v4.u32 [%0], {%1,%2,%3,%4};" ::"r"(out_smem + 2 * off + 16), "r"(o[4]), "r"(o[5]), "r"(o[6]), "r"(o[7]) : "memory");
    }
  } else {
    // 16 bf16 in (32 B) -> 16 fp8 out (16 B)
    for (uint32_t off = lane * 32; off < src_bytes; off += 32 * 32) {
      uint4 a, b;
      asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(a.x), "=r"(a.y), "=r"(a.z), "=r"(a.w) : "r"(in_smem + off));
      asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(b.x), "=r"(b.y), "=r"(b.z), "=r"(b.w) : "r"(in_smem + off + 16));
      uint32_t w[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
      uint32_t o[4];
#pragma unroll
      for (int k = 0; k < 4; ++k)
        o[k] = static_cast<uint32_t>(ptx::bf16x2_to_e4m3x2(w[2 * k])) |
               (static_cast<uint32_t>(ptx::bf16x2_to_e4m3x2(w[2 * k + 1])) << 16);
      asm volatile("st.shared.v4.u32 [%0], {%1,%2,%3,%4};" ::"r"(out_smem + off / 2), "r"(o[0]), "r"(o[1]), "r"(o[2]), "r"(o[3]) : "memory");
    }
  }
}

// SIMT conversion straight from global to global for pieces TMA cannot take (any alignment).
template <bool UP>
__device__ __forceinline__ void warp_cast_simt(uint8_t* dst, const uint8_t* src, uint32_t src_bytes,
                                               int lane)
{
  if (UP) {
    uint16_t* d = reinterpret_cast<uint16_t*>(dst);
    const uint32_t pairs = src_bytes >> 1;
    for (uint32_t i = lane; i < pairs; i += 32) {
      uint16_t two = static_cast<uint16_t>(src[2 * i]) | (static_cast<uint16_t>(src[2 * i + 1]) << 8);
      uint32_t r = ptx::e4m3x2_to_bf16x2(two);
      d[2 * i] = static_cast<uint16_t>(r & 0xffff);
      d[2 * i + 1] = static_cast<uint16_t>(r >> 16);
    }
    if ((src_bytes & 1) && lane == 0)
      d[src_bytes - 1] = static_cast<uint16_t>(ptx::e4m3x2_to_bf16x2(src[src_bytes - 1]) & 0xffff);
  } else {
    const uint16_t* s = reinterpret_cast<const uint16_t*>(src);
    const uint32_t elems = src_bytes >> 1;
    for (uint32_t i = lane; i < elems; i += 32)
      dst[i] = static_cast<uint8_t>(ptx::bf16x2_to_e4m3x2(s[i]) & 0xff);
  }
}

// ------------------------------------------------------------------------------------------
// One CTA = R rings.  Shared memory: [R x ring_ctl_bytes()] [R x S x tile_in] [R x 2 x tile_out]
// ------------------------------------------------------------------------------------------
__host__ __device__ constexpr uint32_t cta_smem_bytes(int R, int S, uint32_t tile_in, uint32_t tile_out)
{
  return static_cast<uint32_t>(R) * (ring_ctl_bytes() + static_cast<uint32_t>(S) * tile_in + 2u * tile_out);
}

template <int CAST, bool FAST, class Gen>
__device__ __forceinline__ void run_rings(uint8_t* smem, const Gen& gen, uint32_t total, int ndst, const RingParams& rp,
                                          const StreamSync& ss)
{
  const int warp = threadIdx.x >> 5;
  const int R = blockDim.x >> 6;
  const int ring = warp >> 1;
  const bool producer = (warp & 1) == 0;
  uint8_t* ctl = smem + ring * ring_ctl_bytes();
  RingSmem sm;
  sm.full0 = ptx::smem_addr(ctl);
  sm.empty0 = sm.full0 + 8 * kMaxStages;
  sm.ctl = reinterpret_cast<SlotCtl*>(ctl + 16 * kMaxStages);
  uint8_t* in_base = smem + R * ring_ctl_bytes();
  sm.in0 = ptx::smem_addr(in_base + static_cast<size_t>(ring) * rp.S * rp.tile_in);
  sm.out0 = ptx::smem_addr(in_base + static_cast<size_t>(R) * rp.S * rp.tile_in + static_cast<size_t>(ring) * 2 * rp.tile_out);
  if (producer && (threadIdx.x & 31) == 0) {
    for (int s = 0; s < rp.S; ++s) {
      ptx::mbar_init(sm.full0 + 8 * s, 1);
      ptx::mbar_init(sm.empty0 + 8 * s, 1);
    }
    ptx::mbar_fence_init();
  }
  __syncthreads();
  const uint32_t nrings = gridDim.x * R;
  const uint32_t my_ring = blockIdx.x * R + ring;
  if (producer)
    ring_producer<CAST, FAST>(gen, total, my_ring, nrings, sm, ndst, rp, ss);
  else
    ring_consumer<CAST, FAST>(sm, ndst, rp, ss);
}

}  // namespace kvbm
