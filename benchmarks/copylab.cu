// copylab -- design-space study of the paged KV copy on one B200 (and, with --peer, over NVLink to GPU 1).
// Bench-only: nothing here ships.  Stand-alone (cudart only) so a GPU call does not pay a torch import.
//
//   benchmarks/copylab [--peer push|pull] [--blocks 256] [--pool 1024] [--iters 30] [--only NAME]
//
// Workload = BASELINE configs[1]: 256 blocks x 32 layers x K/V x 32 KiB regions from a 1024-block layer-separate pool
// (random block tables both sides).  Prints one JSON object per variant:
//   ws_*      warp-specialised TMA ring: producer warp (descriptors + cp.async.bulk g2s), consumer warp (s2g), dynamic
//             or static tile scheduler
//   simt_*    SIMT gather/scatter, one CTA per region, U independent 16 B (or 32 B) loads in flight per thread
//   lib       the product library's kvbm_kernels_paged_copy_v2 (dlopen dynamo_b200/libkvbm_kernels.so)
//   ref_k1    the reference K1 recompiled (oracle/_ref), device pointer tables
//   memcpy    cudaMemcpyAsync of the same byte count, contiguous
#include <cuda_runtime.h>
#include <dlfcn.h>

#include <algorithm>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <numeric>
#include <random>
#include <string>
#include <vector>

#include "../dynamo_b200/csrc/kernels/copy_engine.cuh"
#include "../include/kvbm_kernels.h"

using namespace kvbm;

#define CK(x)                                                                                     \
  do {                                                                                            \
    cudaError_t e_ = (x);                                                                         \
    if (e_ != cudaSuccess) {                                                                      \
      fprintf(stderr, "CUDA error %s at %s:%d: %s\n", cudaGetErrorName(e_), __FILE__, __LINE__, #x); \
      exit(2);                                                                                    \
    }                                                                                             \
  } while (0)

struct Layout {
  const uint64_t* layer_base;
  uint64_t block_stride, outer_stride;
  uint32_t region;
};
struct Job {
  Layout src, dst;
  const int32_t* sid;
  const int32_t* did;
  uint32_t n_blocks, n_layers, outer;
  uint32_t tile, tiles_per_region;
  uint32_t total;  // items
};

__device__ __forceinline__ void item_addr(const Job& j, uint32_t item, uint64_t& s, uint64_t& d, uint32_t& bytes)
{
  uint32_t r = item / j.tiles_per_region;
  const uint32_t t = item - r * j.tiles_per_region;
  uint32_t r2 = r / j.outer;
  const uint32_t o = r - r2 * j.outer;
  r = r2;
  r2 = r / j.n_blocks;
  const uint32_t blk = r - r2 * j.n_blocks;
  const uint32_t layer = r2;
  const uint64_t off = static_cast<uint64_t>(t) * j.tile;
  const uint32_t left = j.src.region - static_cast<uint32_t>(off);
  bytes = left < j.tile ? left : j.tile;
  s = __ldg(j.src.layer_base + layer) + static_cast<uint64_t>(__ldg(j.sid + blk)) * j.src.block_stride + o * j.src.outer_stride + off;
  d = __ldg(j.dst.layer_base + layer) + static_cast<uint64_t>(__ldg(j.did + blk)) * j.dst.block_stride + o * j.dst.outer_stride + off;
}

using kvbm::ptx::mbar_arrive;

// ------------------------------------------------------------------------------------------------------------
// ws: R rings per CTA, each = 1 producer warp + 1 consumer warp, S slots of `tile` bytes.
// sched: 0 static (item = first + k*stride in batches of B), 1 dynamic (atomic tickets of B items)
// ------------------------------------------------------------------------------------------------------------
struct WsParams {
  int S, P, B, sched, store_mode, guide;  // store_mode 0 = TMA bulk store, 1 = SIMT st.v4 from smem by the consumer warp, 2 = st.v8 (256-bit)
  uint32_t* counter;               // [0] tickets, [1] finished rings
  unsigned long long* times;       // optional [grid*R][3]: start, first data, end
};

__global__ void __launch_bounds__(256, 1) ws_copy_kernel(const __grid_constant__ Job job, const __grid_constant__ WsParams wp)
{
  extern __shared__ __align__(128) uint8_t smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int R = blockDim.x >> 6;
  const int ring = warp >> 1;
  const bool producer = (warp & 1) == 0;
  const int S = wp.S;
  // per ring: full[S] empty[S] dst[S] bytes[S] (8 B each, 32*S bytes, padded to 1 KiB), then the slots
  uint8_t* ctl = smem + ring * 1024;
  uint64_t* full = reinterpret_cast<uint64_t*>(ctl);
  uint64_t* empty = full + S;
  volatile uint64_t* sdst = reinterpret_cast<volatile uint64_t*>(empty + S);
  volatile uint32_t* sbytes = reinterpret_cast<volatile uint32_t*>(const_cast<uint64_t*>(sdst) + S);
  uint8_t* slots = smem + R * 1024 + static_cast<size_t>(ring) * S * job.tile;
  const uint32_t full0 = ptx::smem_addr(full), empty0 = ptx::smem_addr(empty), slot0 = ptx::smem_addr(slots);
  const unsigned long long t_start = wp.times ? ptx::globaltimer_ns() : 0;

  if (producer && lane == 0) {
    for (int s = 0; s < S; ++s) {
      ptx::mbar_init(full0 + 8 * s, 1);
      ptx::mbar_init(empty0 + 8 * s, 1);
    }
    ptx::mbar_fence_init();
  }
  __syncthreads();

  const uint32_t nrings = gridDim.x * R;
  const uint32_t my = blockIdx.x * R + ring;  // global ring index
  const uint32_t B = wp.B;
  const uint32_t nbatches = (job.total + B - 1) / B;

  if (producer) {
    uint32_t q = 0;  // items issued by this ring
    uint32_t k = 0;
    uint32_t last_start = 0;
    for (;;) {
      uint32_t item0, cnt;
      if (wp.sched == 2) {
        // guided self-scheduling in ITEMS: the first batch is static (no atomic on the ramp), later ones are tickets whose
        // size shrinks towards the end so that all rings finish together
        if (k == 0) {
          item0 = my * B;
        } else {
          const uint32_t remaining = job.total > last_start ? job.total - last_start : 0;
          uint32_t want = remaining / (wp.guide * nrings);
          want = want < 1 ? 1 : (want > B ? B : want);
          uint32_t t = 0;
          if (lane == 0) t = atomicAdd(wp.counter, want);
          item0 = nrings * B + __shfl_sync(0xffffffffu, t, 0);
          cnt = want;
        }
        if (k == 0) cnt = B;
        ++k;
        last_start = item0;
        if (item0 >= job.total) break;
        cnt = min(cnt, job.total - item0);
      } else {
        uint32_t batch;
        if (wp.sched == 1) {
          uint32_t t = 0;
          if (lane == 0) t = atomicAdd(wp.counter, 1u);
          batch = __shfl_sync(0xffffffffu, t, 0);
        } else {
          batch = my + k * nrings;
          ++k;
        }
        if (batch >= nbatches) break;
        item0 = batch * B;
        cnt = min(B, job.total - item0);
      }
      uint64_t s = 0, d = 0;
      uint32_t bytes = 0;
      if (lane < cnt) item_addr(job, item0 + lane, s, d, bytes);
      for (uint32_t i = 0; i < cnt; ++i, ++q) {
        const uint64_t si = __shfl_sync(0xffffffffu, s, i), di = __shfl_sync(0xffffffffu, d, i);
        const uint32_t bi = __shfl_sync(0xffffffffu, bytes, i);
        const int slot = q % S;
        if (lane == 0) {
          ptx::mbar_wait(empty0 + 8 * slot, ((q / S) & 1) ^ 1);
          sdst[slot] = di;
          sbytes[slot] = bi;
          ptx::mbar_arrive_expect_tx(full0 + 8 * slot, bi);
          ptx::bulk_g2s(slot0 + slot * job.tile, reinterpret_cast<const void*>(si), bi, full0 + 8 * slot);
        }
      }
      __syncwarp();
    }
    // tell the consumer how many items this ring produced: a zero-byte "end" marker in the next slot
    if (lane == 0) {
      const int slot = q % S;
      ptx::mbar_wait(empty0 + 8 * slot, ((q / S) & 1) ^ 1);
      sbytes[slot] = 0;
      ptx::mbar_arrive_expect_tx(full0 + 8 * slot, 0);
      if (wp.sched >= 1) {
        const uint32_t old = atomicAdd(wp.counter + 1, 1u);
        if (old == nrings - 1) {  // last ring to run dry: leave the scheduler words zeroed for the next launch
          wp.counter[0] = 0;
          wp.counter[1] = 0;
        }
      }
    }
  } else {
    unsigned long long t_first = 0;
    uint32_t q = 0;
    for (;; ++q) {
      const int slot = q % S;
      ptx::mbar_wait(full0 + 8 * slot, (q / S) & 1);
      const uint32_t bytes = sbytes[slot];
      if (bytes == 0) break;
      if (q == 0 && wp.times) t_first = ptx::globaltimer_ns();
      uint8_t* dst = reinterpret_cast<uint8_t*>(sdst[slot]);
      const uint32_t sa = slot0 + slot * job.tile;
      if (wp.store_mode == 0) {
        if (lane == 0) {
          ptx::bulk_s2g(dst, sa, bytes);
          ptx::bulk_commit();
          // store q-P has finished reading its slot -> hand it back to the producer
          ptx::bulk_wait_read_n(wp.P);
          if (q >= static_cast<uint32_t>(wp.P)) mbar_arrive(empty0 + 8 * ((q - wp.P) % S));
        }
      } else if (wp.store_mode == 1) {
        uint4* d4 = reinterpret_cast<uint4*>(dst);
        for (uint32_t i = lane; i < (bytes >> 4); i += 32) {
          uint4 v;
          asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(sa + i * 16));
          ptx::st_stream_v4(d4 + i, v);
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(empty0 + 8 * slot);
      } else {
        for (uint32_t i = lane; i < (bytes >> 5); i += 32) {
          uint4 a, b;
          asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(a.x), "=r"(a.y), "=r"(a.z), "=r"(a.w) : "r"(sa + i * 32));
          asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(b.x), "=r"(b.y), "=r"(b.z), "=r"(b.w) : "r"(sa + i * 32 + 16));
          asm volatile("st.global.L1::no_allocate.v8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(dst + i * 32), "r"(a.x), "r"(a.y), "r"(a.z),
                       "r"(a.w), "r"(b.x), "r"(b.y), "r"(b.z), "r"(b.w)
                       : "memory");
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(empty0 + 8 * slot);
      }
    }
    if (lane == 0 && wp.store_mode == 0) {
      // the P slots still owned by draining stores are never reused: just wait for the writes themselves
      ptx::bulk_wait<0>();
    }
    if (wp.times && lane == 0) {
      unsigned long long* t = wp.times + 3ull * my;
      t[0] = t_start;
      t[1] = t_first;
      t[2] = ptx::globaltimer_ns();
    }
  }
}

// ------------------------------------------------------------------------------------------------------------
// ws_engine: the PRODUCT engine (copy_engine.cuh run_rings) on the lab's job, to compare with the lab ring above
// ------------------------------------------------------------------------------------------------------------
struct JobGen {
  Job j;
  __device__ __forceinline__ void get(uint32_t item, Piece& p) const
  {
    uint64_t s, d;
    uint32_t bytes;
    item_addr(j, item, s, d, bytes);
    p.src = reinterpret_cast<const uint8_t*>(s);
    p.dst[0] = reinterpret_cast<uint8_t*>(d);
    p.bytes = bytes;
    p.ndst = 1;
    p.layer = 0;
  }
};

__global__ void __launch_bounds__(512, 1) ws_engine_kernel(const __grid_constant__ JobGen gen, uint32_t* ctl, int S, int P, int B)
{
  extern __shared__ __align__(128) uint8_t smem[];
  StreamSync ss{};
  ss.ctl = ctl;
  ss.total_rings = gridDim.x * (blockDim.x >> 6);
  ss.layer_end = 1;
  RingParams rp{S, P, B, gen.j.tile, 0, true, false, false};
  run_rings<0, true>(smem, gen, gen.j.total, 1, rp, ss);
}

// ------------------------------------------------------------------------------------------------------------
// simt: one CTA per `rpc` regions; T threads; each thread keeps U x 16 B loads in flight
// ------------------------------------------------------------------------------------------------------------
template <int U, bool V8>
__global__ void __launch_bounds__(256) simt_copy_kernel(const __grid_constant__ Job job, uint32_t regions, uint32_t rpc)
{
  for (uint32_t rr = 0; rr < rpc; ++rr) {
    const uint32_t r = blockIdx.x * rpc + rr;
    if (r >= regions) return;
    uint64_t s, d;
    uint32_t bytes;
    item_addr(job, r * job.tiles_per_region, s, d, bytes);  // tiles_per_region == 1 for this kernel
    constexpr int W = V8 ? 32 : 16;
    const uint32_t n = job.src.region / W;
    const uint8_t* sp = reinterpret_cast<const uint8_t*>(s);
    uint8_t* dp = reinterpret_cast<uint8_t*>(d);
    for (uint32_t base = 0; base < n; base += U * blockDim.x) {
      if (V8) {
        uint32_t v[U][8];
#pragma unroll
        for (int u = 0; u < U; ++u) {
          const uint32_t i = base + u * blockDim.x + threadIdx.x;
          if (i < n)
            asm volatile("ld.global.L1::no_allocate.v8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                         : "=r"(v[u][0]), "=r"(v[u][1]), "=r"(v[u][2]), "=r"(v[u][3]), "=r"(v[u][4]), "=r"(v[u][5]), "=r"(v[u][6]), "=r"(v[u][7])
                         : "l"(sp + static_cast<size_t>(i) * 32));
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
          const uint32_t i = base + u * blockDim.x + threadIdx.x;
          if (i < n)
            asm volatile("st.global.L1::no_allocate.v8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(dp + static_cast<size_t>(i) * 32), "r"(v[u][0]),
                         "r"(v[u][1]), "r"(v[u][2]), "r"(v[u][3]), "r"(v[u][4]), "r"(v[u][5]), "r"(v[u][6]), "r"(v[u][7])
                         : "memory");
        }
      } else {
        uint4 v[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
          const uint32_t i = base + u * blockDim.x + threadIdx.x;
          if (i < n) v[u] = ptx::ld_stream_v4(sp + static_cast<size_t>(i) * 16);
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
          const uint32_t i = base + u * blockDim.x + threadIdx.x;
          if (i < n) ptx::st_stream_v4(dp + static_cast<size_t>(i) * 16, v[u]);
        }
      }
    }
  }
}

__global__ void verify_kernel(const __grid_constant__ Job job, uint32_t regions, unsigned long long* bad)
{
  const uint32_t r = blockIdx.x;
  if (r >= regions) return;
  Job j = job;
  j.tile = j.src.region;
  j.tiles_per_region = 1;
  uint64_t s, d;
  uint32_t bytes;
  item_addr(j, r, s, d, bytes);
  const uint4* a = reinterpret_cast<const uint4*>(s);
  const uint4* b = reinterpret_cast<const uint4*>(d);
  unsigned long long n = 0;
  for (uint32_t i = threadIdx.x; i < bytes / 16; i += blockDim.x) {
    uint4 x = a[i], y = b[i];
    if (x.x != y.x || x.y != y.y || x.z != y.z || x.w != y.w) ++n;
  }
  if (n) atomicAdd(bad, n);
}

__global__ void fill_kernel(uint4* p, size_t n, uint32_t seed)
{
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < n; i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    uint32_t x = static_cast<uint32_t>(i) * 2654435761u ^ seed;
    x ^= x >> 15;
    x *= 2246822519u;
    p[i] = make_uint4(x, x ^ 0x9e3779b9u, x * 3u + 1u, x >> 3);
  }
}

// ------------------------------------------------------------------------------------------------------------
struct Timing {
  double med_ms, min_ms, b2b_ms;
};

template <class F>
static Timing time_it(F&& launch, cudaStream_t st, int iters, int warm = 5)
{
  for (int i = 0; i < warm; ++i) launch();
  CK(cudaStreamSynchronize(st));
  std::vector<float> ts;
  cudaEvent_t e0, e1;
  CK(cudaEventCreate(&e0));
  CK(cudaEventCreate(&e1));
  for (int i = 0; i < iters; ++i) {
    CK(cudaEventRecord(e0, st));
    launch();
    CK(cudaEventRecord(e1, st));
    CK(cudaEventSynchronize(e1));
    float ms;
    CK(cudaEventElapsedTime(&ms, e0, e1));
    ts.push_back(ms);
  }
  std::sort(ts.begin(), ts.end());
  Timing t;
  t.med_ms = ts[ts.size() / 2];
  t.min_ms = ts[0];
  CK(cudaEventRecord(e0, st));
  for (int i = 0; i < iters; ++i) launch();
  CK(cudaEventRecord(e1, st));
  CK(cudaEventSynchronize(e1));
  float ms;
  CK(cudaEventElapsedTime(&ms, e0, e1));
  t.b2b_ms = ms / iters;
  CK(cudaEventDestroy(e0));
  CK(cudaEventDestroy(e1));
  return t;
}

int main(int argc, char** argv)
{
  int blocks = 256, pool = 1024, layers = 32, iters = 30;
  std::string peer, only;
  bool quick = false;
  for (int i = 1; i < argc; ++i) {
    std::string a = argv[i];
    auto next = [&]() { return std::string(i + 1 < argc ? argv[++i] : ""); };
    if (a == "--blocks") blocks = atoi(next().c_str());
    else if (a == "--pool") pool = atoi(next().c_str());
    else if (a == "--layers") layers = atoi(next().c_str());
    else if (a == "--iters") iters = atoi(next().c_str());
    else if (a == "--peer") peer = next();
    else if (a == "--only") only = next();
    else if (a == "--quick") quick = true;
  }
  const uint32_t region = 32768, outer = 2;
  int ndev = 0;
  CK(cudaGetDeviceCount(&ndev));
  int sdev = 0, ddev = 0;  // where the pools live; the kernel always runs on device 0
  if (!peer.empty()) {
    if (ndev < 2) {
      fprintf(stderr, "--peer needs 2 GPUs\n");
      return 1;
    }
    CK(cudaSetDevice(0));
    CK(cudaDeviceEnablePeerAccess(1, 0));
    if (peer == "pull") sdev = 1;
    else ddev = 1;
  }
  const size_t per_layer = static_cast<size_t>(outer) * pool * region;
  std::vector<uint64_t> sb(layers), db(layers);
  for (int l = 0; l < layers; ++l) {
    void* p;
    CK(cudaSetDevice(sdev));
    CK(cudaMalloc(&p, per_layer));
    fill_kernel<<<1024, 256>>>(static_cast<uint4*>(p), per_layer / 16, 1234u + l);
    sb[l] = reinterpret_cast<uint64_t>(p);
    CK(cudaSetDevice(ddev));
    CK(cudaMalloc(&p, per_layer));
    CK(cudaMemset(p, 0, per_layer));
    db[l] = reinterpret_cast<uint64_t>(p);
  }
  CK(cudaSetDevice(sdev));
  CK(cudaDeviceSynchronize());
  CK(cudaSetDevice(ddev));
  CK(cudaDeviceSynchronize());
  CK(cudaSetDevice(0));
  std::vector<int32_t> perm(pool);
  std::iota(perm.begin(), perm.end(), 0);
  std::mt19937 r0(0), r1(1);
  std::shuffle(perm.begin(), perm.end(), r0);
  std::vector<int32_t> sid(perm.begin(), perm.begin() + blocks);
  std::shuffle(perm.begin(), perm.end(), r1);
  std::vector<int32_t> did(perm.begin(), perm.begin() + blocks);
  uint64_t *d_sb, *d_db;
  int32_t *d_sid, *d_did;
  CK(cudaMalloc(&d_sb, layers * 8));
  CK(cudaMalloc(&d_db, layers * 8));
  CK(cudaMalloc(&d_sid, blocks * 4));
  CK(cudaMalloc(&d_did, blocks * 4));
  CK(cudaMemcpy(d_sb, sb.data(), layers * 8, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(d_db, db.data(), layers * 8, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(d_sid, sid.data(), blocks * 4, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(d_did, did.data(), blocks * 4, cudaMemcpyHostToDevice));
  uint32_t* d_counter;
  unsigned long long *d_times, *d_bad;
  CK(cudaMalloc(&d_counter, 64));
  CK(cudaMemset(d_counter, 0, 64));
  CK(cudaMalloc(&d_times, 3 * 8 * 4096));
  CK(cudaMalloc(&d_bad, 8));

  Job job{};
  job.src = Layout{d_sb, region, static_cast<uint64_t>(region) * pool, region};
  job.dst = Layout{d_db, region, static_cast<uint64_t>(region) * pool, region};
  job.sid = d_sid;
  job.did = d_did;
  job.n_blocks = blocks;
  job.n_layers = layers;
  job.outer = outer;
  const uint32_t regions = blocks * layers * outer;
  const double bytes = static_cast<double>(regions) * region;

  cudaStream_t st;
  CK(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
  int sms = 0;
  CK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, 0));

  auto clear_dst = [&]() {
    CK(cudaSetDevice(ddev));
    for (int l = 0; l < layers; ++l) CK(cudaMemset(reinterpret_cast<void*>(db[l]), 0, per_layer));
    CK(cudaDeviceSynchronize());
    CK(cudaSetDevice(0));
  };
  auto verify = [&]() -> unsigned long long {
    // runs on the device that owns the destination when pushing (peer reads of the source are fine)
    CK(cudaMemset(d_bad, 0, 8));
    verify_kernel<<<regions, 256>>>(job, regions, d_bad);
    CK(cudaDeviceSynchronize());
    unsigned long long bad = 0;
    CK(cudaMemcpy(&bad, d_bad, 8, cudaMemcpyDeviceToHost));
    return bad;
  };
  auto report = [&](const char* name, const std::string& cfg, const Timing& t, unsigned long long bad, const std::string& extra = "") {
    printf("{\"name\":\"%s\",%s\"med_ms\":%.5f,\"min_ms\":%.5f,\"b2b_ms\":%.5f,\"gbs_med\":%.1f,\"gbs_b2b\":%.1f,\"mismatch16\":%llu%s}\n", name,
           cfg.c_str(), t.med_ms, t.min_ms, t.b2b_ms, bytes / t.med_ms / 1e6, bytes / t.b2b_ms / 1e6, bad, extra.c_str());
    fflush(stdout);
  };
  auto want = [&](const char* n) { return only.empty() || only == n; };

  // ---------------- contiguous memcpy of the same volume ----------------
  if (want("memcpy")) {
    void *a, *b;
    CK(cudaSetDevice(sdev));
    CK(cudaMalloc(&a, static_cast<size_t>(bytes)));
    CK(cudaSetDevice(ddev));
    CK(cudaMalloc(&b, static_cast<size_t>(bytes)));
    CK(cudaSetDevice(0));
    Timing t = time_it([&]() { CK(cudaMemcpyAsync(b, a, static_cast<size_t>(bytes), cudaMemcpyDefault, st)); }, st, iters);
    report("memcpy", "", t, 0);
    CK(cudaFree(a));
    CK(cudaFree(b));
  }

  // ---------------- warp-specialised TMA ring ----------------
  if (want("ws")) {
    CK(cudaFuncSetAttribute(ws_copy_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    struct C {
      int grid, R, S, P, B, sched, tile, store, guide = 0;
    };
    std::vector<C> cfgs;
    const bool remote = !peer.empty();
    if (!remote && quick) {
      for (int guide : {1, 2, 4})
        for (int B : {8, 4}) {
          cfgs.push_back({148, 1, 6, 2, B, 2, 32768, 0, guide});
          cfgs.push_back({132, 1, 6, 1, B, 2, 16384, 0, guide});
          cfgs.push_back({74, 2, 6, 2, B, 2, 16384, 0, guide});
          cfgs.push_back({148, 1, 12, 4, B, 2, 16384, 0, guide});
        }
      cfgs.push_back({148, 1, 6, 2, 2, 1, 32768, 0});
      cfgs.push_back({132, 1, 6, 1, 8, 1, 16384, 0});
      cfgs.push_back({74, 2, 6, 2, 8, 1, 16384, 0});
      cfgs.push_back({37, 4, 3, 1, 4, 2, 16384, 0, 2});
      cfgs.push_back({32, 4, 3, 1, 4, 2, 16384, 0, 2});
      cfgs.push_back({16, 4, 3, 1, 4, 2, 16384, 0, 2});
      cfgs.push_back({16, 2, 6, 2, 4, 2, 16384, 0, 2});
      cfgs.push_back({8, 4, 3, 1, 4, 2, 16384, 0, 2});
    } else if (!remote) {
      for (int sched : {1, 0})
        for (int grid : {148, 74}) {
          cfgs.push_back({grid, 1, 6, 2, 8, sched, 32768, 0});
          cfgs.push_back({grid, 2, 3, 1, 8, sched, 32768, 0});
          cfgs.push_back({grid, 2, 6, 2, 8, sched, 16384, 0});
          cfgs.push_back({grid, 1, 12, 4, 8, sched, 16384, 0});
          cfgs.push_back({grid, 4, 3, 1, 8, sched, 16384, 0});
        }
      for (int grid : {111, 132, 296})
        for (int tile : {32768, 16384}) cfgs.push_back({grid, 1, tile == 32768 ? 3 : 6, 1, 8, 1, tile, 0});
      cfgs.push_back({148, 1, 6, 2, 4, 1, 32768, 0});
      cfgs.push_back({148, 1, 6, 2, 2, 1, 32768, 0});
      cfgs.push_back({148, 1, 6, 2, 16, 1, 32768, 0});
      cfgs.push_back({148, 1, 6, 2, 32, 1, 32768, 0});
      cfgs.push_back({148, 1, 6, 1, 8, 1, 32768, 0});
      cfgs.push_back({148, 1, 6, 3, 8, 1, 32768, 0});
      cfgs.push_back({148, 1, 4, 1, 8, 1, 32768, 0});
      cfgs.push_back({148, 1, 3, 1, 8, 1, 32768, 0});
      cfgs.push_back({148, 1, 2, 1, 8, 1, 32768, 0});
      cfgs.push_back({148, 1, 4, 1, 8, 1, 16384, 0});
      cfgs.push_back({148, 1, 8, 2, 8, 1, 8192, 0});
      cfgs.push_back({148, 2, 8, 2, 8, 1, 8192, 0});
      cfgs.push_back({148, 1, 6, 2, 8, 1, 32768, 1});
      cfgs.push_back({148, 2, 3, 1, 8, 1, 32768, 1});
      cfgs.push_back({148, 4, 3, 1, 8, 1, 16384, 1});
      cfgs.push_back({148, 4, 3, 1, 8, 1, 16384, 2});
    } else {
      for (int store : {0, 1, 2})
        for (int grid : {148, 74, 32, 16}) {
          cfgs.push_back({grid, 1, 6, 2, 4, 2, 32768, store, 2});
          cfgs.push_back({grid, 2, 6, 3, 4, 2, 16384, store, 2});
          cfgs.push_back({grid, 4, 6, 3, 4, 2, 8192, store, 2});
        }
      cfgs.push_back({32, 4, 3, 1, 8, 1, 16384, 0});
      cfgs.push_back({32, 2, 6, 5, 8, 1, 16384, 0});
      cfgs.push_back({64, 1, 6, 5, 8, 1, 32768, 0});
      cfgs.push_back({64, 1, 6, 1, 8, 1, 32768, 0});
    }
    for (const C& c : cfgs) {
      Job j = job;
      j.tile = c.tile;
      j.tiles_per_region = (region + c.tile - 1) / c.tile;
      j.total = regions * j.tiles_per_region;
      const size_t smem = c.R * 1024 + static_cast<size_t>(c.R) * c.S * c.tile;
      if (smem > 227 * 1024) continue;
      WsParams wp{c.S, c.P, c.B, c.sched, c.store, c.guide > 0 ? c.guide : 2, d_counter, nullptr};
      clear_dst();
      auto launch = [&]() { ws_copy_kernel<<<c.grid, 64 * c.R, smem, st>>>(j, wp); };
      launch();
      CK(cudaStreamSynchronize(st));
      CK(cudaGetLastError());
      const unsigned long long bad = verify();
      Timing t = time_it(launch, st, iters);
      // one extra launch with the timeline
      WsParams wt = wp;
      wt.times = d_times;
      ws_copy_kernel<<<c.grid, 64 * c.R, smem, st>>>(j, wt);
      CK(cudaStreamSynchronize(st));
      const int nr = c.grid * c.R;
      std::vector<unsigned long long> tm(3 * nr);
      CK(cudaMemcpy(tm.data(), d_times, tm.size() * 8, cudaMemcpyDeviceToHost));
      unsigned long long t0 = ~0ull, tend = 0, first_end = ~0ull;
      std::vector<double> ramp, ends;
      for (int i = 0; i < nr; ++i) t0 = std::min(t0, tm[3 * i]);
      for (int i = 0; i < nr; ++i) {
        ramp.push_back((tm[3 * i + 1] - t0) / 1e3);
        ends.push_back((tm[3 * i + 2] - t0) / 1e3);
        tend = std::max(tend, tm[3 * i + 2]);
        first_end = std::min(first_end, tm[3 * i + 2]);
      }
      std::sort(ramp.begin(), ramp.end());
      char cfg[256], extra[256];
      snprintf(cfg, sizeof cfg, "\"grid\":%d,\"R\":%d,\"S\":%d,\"P\":%d,\"B\":%d,\"sched\":%d,\"tile\":%d,\"store\":%d,\"guide\":%d,", c.grid, c.R, c.S, c.P, c.B,
               c.sched, c.tile, c.store, c.guide);
      snprintf(extra, sizeof extra, ",\"tl_total_us\":%.1f,\"tl_first_data_med_us\":%.1f,\"tl_first_data_max_us\":%.1f,\"tl_end_spread_us\":%.1f",
               (tend - t0) / 1e3, ramp[ramp.size() / 2], ramp.back(), (tend - first_end) / 1e3);
      report("ws", cfg, t, bad, extra);
    }
  }

  // ---------------- SIMT ----------------
  if (want("simt")) {
    Job j = job;
    j.tile = region;
    j.tiles_per_region = 1;
    j.total = regions;
    auto run = [&](const char* name, auto kern, int threads, int rpc) {
      clear_dst();
      const uint32_t grid = (regions + rpc - 1) / rpc;
      auto launch = [&]() { kern<<<grid, threads, 0, st>>>(j, regions, rpc); };
      launch();
      CK(cudaStreamSynchronize(st));
      CK(cudaGetLastError());
      const unsigned long long bad = verify();
      Timing t = time_it(launch, st, iters);
      char cfg[128];
      snprintf(cfg, sizeof cfg, "\"threads\":%d,\"rpc\":%d,", threads, rpc);
      report(name, cfg, t, bad);
    };
    run("simt_u1", simt_copy_kernel<1, false>, 128, 1);
    run("simt_u4", simt_copy_kernel<4, false>, 128, 1);
    run("simt_u8", simt_copy_kernel<8, false>, 128, 1);
    run("simt_u8", simt_copy_kernel<8, false>, 256, 1);
    run("simt_u16", simt_copy_kernel<16, false>, 128, 1);
    run("simt_u4", simt_copy_kernel<4, false>, 256, 1);
    run("simt_u4", simt_copy_kernel<4, false>, 256, 2);
    run("simt_v8_u4", simt_copy_kernel<4, true>, 128, 1);
    run("simt_v8_u8", simt_copy_kernel<8, true>, 128, 1);
    run("simt_v8_u4", simt_copy_kernel<4, true>, 256, 1);
  }

  // ---------------- the product library and the reference K1 ----------------
  typedef cudaError_t (*k1_fn)(void**, void**, size_t, int, cudaStream_t);
  std::string root = argv[0];
  root = root.substr(0, root.find_last_of('/') == std::string::npos ? 0 : root.find_last_of('/'));
  if (root.empty()) root = ".";
  std::vector<uint64_t> ps, pd;
  for (int b = 0; b < blocks; ++b)
    for (int l = 0; l < layers; ++l)
      for (uint32_t o = 0; o < outer; ++o) {
        ps.push_back(sb[l] + static_cast<uint64_t>(sid[b]) * region + o * static_cast<uint64_t>(region) * pool);
        pd.push_back(db[l] + static_cast<uint64_t>(did[b]) * region + o * static_cast<uint64_t>(region) * pool);
      }
  void **d_ps, **d_pd;
  CK(cudaMalloc(&d_ps, ps.size() * 8));
  CK(cudaMalloc(&d_pd, pd.size() * 8));
  CK(cudaMemcpy(d_ps, ps.data(), ps.size() * 8, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(d_pd, pd.data(), pd.size() * 8, cudaMemcpyHostToDevice));
  if (want("lib")) {
    void* h = dlopen((root + "/../dynamo_b200/libkvbm_kernels.so").c_str(), RTLD_NOW | RTLD_LOCAL);
    if (!h) fprintf(stderr, "lib: %s\n", dlerror());
    if (h) {
      typedef cudaError_t (*paged_fn)(const kvbm_paged_layout*, const kvbm_paged_dst*, int, int, int, int, int, const kvbm_paged_copy_opts*, cudaStream_t);
      paged_fn paged = reinterpret_cast<paged_fn>(dlsym(h, "kvbm_kernels_paged_copy_v2"));
      k1_fn k1 = reinterpret_cast<k1_fn>(dlsym(h, "kvbm_kernels_launch_vectorized_copy"));
      kvbm_paged_layout L{d_sb, region, static_cast<uint64_t>(region) * pool, region, static_cast<uint32_t>(layers), outer, static_cast<uint32_t>(pool)};
      kvbm_paged_dst D{};
      D.layout = L;
      D.layout.layer_base = d_db;
      D.src_block_ids = d_sid;
      D.dst_block_ids = d_did;
      clear_dst();
      auto launch = [&]() { CK(paged(&L, &D, 1, blocks, 0, layers, 0, nullptr, st)); };
      launch();
      CK(cudaStreamSynchronize(st));
      const unsigned long long bad = verify();
      report("lib_paged", "", time_it(launch, st, iters), bad);
      clear_dst();
      auto launch2 = [&]() { CK(k1(d_ps, d_pd, region, static_cast<int>(ps.size()), st)); };
      launch2();
      CK(cudaStreamSynchronize(st));
      const unsigned long long bad2 = verify();
      report("lib_k1", "", time_it(launch2, st, iters), bad2);
    }
  }
  if (want("ref")) {
    void* h = dlopen((root + "/../oracle/_ref/libkvbm_kernels_ref.so").c_str(), RTLD_NOW | RTLD_LOCAL);
    if (!h) fprintf(stderr, "ref: %s\n", dlerror());
    if (h) {
      k1_fn k1 = reinterpret_cast<k1_fn>(dlsym(h, "kvbm_kernels_launch_vectorized_copy"));
      clear_dst();
      auto launch = [&]() { CK(k1(d_ps, d_pd, region, static_cast<int>(ps.size()), st)); };
      launch();
      CK(cudaStreamSynchronize(st));
      const unsigned long long bad = verify();
      report("ref_k1", "", time_it(launch, st, iters), bad);
    }
  }

  if (only == "engine") {
    CK(cudaFuncSetAttribute(ws_engine_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    CK(cudaFuncSetAttribute(ws_copy_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    struct C {
      int grid, R, S, P, B, tile;
    };
    const C cs[] = {{132, 1, 6, 1, 8, 16384}, {74, 2, 6, 2, 8, 16384}, {148, 1, 6, 2, 8, 32768}, {148, 2, 3, 1, 8, 16384}, {16, 2, 6, 2, 4, 16384}, {16, 4, 3, 1, 4, 16384}};
    for (const C& c : cs) {
      Job j = job;
      j.tile = c.tile;
      j.tiles_per_region = (region + c.tile - 1) / c.tile;
      j.total = regions * j.tiles_per_region;
      JobGen g{j};
      char cfg[200];
      snprintf(cfg, sizeof cfg, "\"grid\":%d,\"R\":%d,\"S\":%d,\"P\":%d,\"B\":%d,\"tile\":%d,", c.grid, c.R, c.S, c.P, c.B, c.tile);
      {
        const size_t smem = cta_smem_bytes(c.R, c.S, c.tile, 0);
        clear_dst();
        auto launch = [&]() { ws_engine_kernel<<<c.grid, 64 * c.R, smem, st>>>(g, d_counter, c.S, c.P, c.B); };
        launch();
        CK(cudaStreamSynchronize(st));
        CK(cudaGetLastError());
        const unsigned long long bad = verify();
        report("ws_engine", cfg, time_it(launch, st, iters), bad);
      }
      {
        const size_t smem = c.R * 1024 + static_cast<size_t>(c.R) * c.S * c.tile;
        WsParams wp{c.S, c.P, c.B, 2, 0, 4, d_counter + 8, nullptr};
        clear_dst();
        auto launch = [&]() { ws_copy_kernel<<<c.grid, 64 * c.R, smem, st>>>(j, wp); };
        launch();
        CK(cudaStreamSynchronize(st));
        const unsigned long long bad = verify();
        report("ws_lab", cfg, time_it(launch, st, iters), bad);
      }
    }
  }

  // ---------------- the product library under different options (what does the launcher add?) ----------------
  if (only == "libsweep") {
    void* h = dlopen((root + "/../dynamo_b200/libkvbm_kernels.so").c_str(), RTLD_NOW | RTLD_LOCAL);
    if (!h) fprintf(stderr, "lib: %s\n", dlerror());
    if (h) {
      typedef cudaError_t (*paged_fn)(const kvbm_paged_layout*, const kvbm_paged_dst*, int, int, int, int, int, const kvbm_paged_copy_opts*, cudaStream_t);
      paged_fn paged = reinterpret_cast<paged_fn>(dlsym(h, "kvbm_kernels_paged_copy_v2"));
      kvbm_paged_layout L{d_sb, region, static_cast<uint64_t>(region) * pool, region, static_cast<uint32_t>(layers), outer, static_cast<uint32_t>(pool)};
      kvbm_paged_dst D{};
      D.layout = L;
      D.layout.layer_base = d_db;
      D.src_block_ids = d_sid;
      D.dst_block_ids = d_did;
      uint32_t* ws;
      CK(cudaMalloc(&ws, 4 * (layers + 4)));
      CK(cudaMemset(ws, 0, 4 * (layers + 4)));
      struct V {
        const char* name;
        int ws, stat, warps, ctas, stages, tile, pend, flags = 0;
      };
      uint32_t* d_flags;
      CK(cudaMalloc(&d_flags, 256));
      CK(cudaMemset(d_flags, 0, 256));
      uint32_t* h_word;
      CK(cudaHostAlloc(reinterpret_cast<void**>(&h_word), 64, cudaHostAllocMapped));
      const V vs[] = {{"default_pool", 0, 0, 0, 0, 0, 0, 0},      {"default_ws", 1, 0, 0, 0, 0, 0, 0},       {"static", 0, 1, 0, 0, 0, 0, 0},
                      {"ws_done_flag", 1, 0, 0, 0, 0, 0, 0, 1},    {"ws_done_flag_host_word", 1, 0, 0, 0, 0, 0, 0, 3},
                      {"r1_148", 1, 0, 2, 148, 0, 0, 0},           {"r1_132_p1", 1, 0, 2, 132, 6, 16384, 1},  {"r2_74_p1", 1, 0, 4, 74, 6, 16384, 1},
                      {"r1_148_t32", 1, 0, 2, 148, 6, 32768, 2},   {"r2_148", 1, 0, 4, 148, 3, 16384, 1},     {"r4_74", 1, 0, 8, 74, 3, 16384, 1}};
      for (const V& v : vs) {
        kvbm_paged_copy_opts o{};
        o.sync_workspace = v.ws ? ws : nullptr;
        o.static_schedule = v.stat;
        o.warps_per_cta = v.warps;
        o.max_ctas = v.ctas;
        o.stages = v.stages;
        o.tile_bytes = v.tile;
        o.stores_in_flight = v.pend;
        o.epoch = 1;
        D.done_flag = (v.flags & 1) ? d_flags : nullptr;
        o.completion_flag = (v.flags & 2) ? h_word : nullptr;
        o.completion_value = 7;
        clear_dst();
        auto launch = [&]() { CK(paged(&L, &D, 1, blocks, 0, layers, 0, &o, st)); };
        launch();
        CK(cudaStreamSynchronize(st));
        const unsigned long long bad = verify();
        Timing t = time_it(launch, st, iters);
        char cfg[160];
        snprintf(cfg, sizeof cfg, "\"variant\":\"%s\",", v.name);
        report("libsweep", cfg, t, bad);
      }
    }
  }

  // ---------------- K2 / K3 (block stacks <-> universal), ours vs the reference kernels ----------------
  if (only == "perm" || only.empty()) {
    typedef cudaError_t (*perm_fn)(void* const*, const void* const*, size_t, size_t, size_t, size_t, size_t, size_t, int, int, cudaStream_t);
    typedef cudaError_t (*perm_fn2)(const void* const*, void* const*, size_t, size_t, size_t, size_t, size_t, size_t, int, int, cudaStream_t);
    const size_t nb = 64, nh = 8, nl_ = 80, no_ = 2, nt = 16, hd = 128, el = 2;
    const size_t chunk_bytes = nh * nt * hd * el, block_bytes = chunk_bytes * nl_ * no_;
    uint8_t *uni, *chunks, *back;
    CK(cudaMalloc(&uni, nb * block_bytes));
    CK(cudaMalloc(&chunks, nb * block_bytes));
    CK(cudaMalloc(&back, nb * block_bytes));
    fill_kernel<<<1024, 256>>>(reinterpret_cast<uint4*>(chunks), nb * block_bytes / 16, 99u);
    std::vector<void*> up(nb), cp(nb * nl_ * no_), bp(nb * nl_ * no_);
    // chunk order shuffled so that chunks are NOT laid out like the universal tensor
    std::vector<size_t> order(nb * nl_ * no_);
    std::iota(order.begin(), order.end(), 0);
    std::mt19937 rr(7);
    std::shuffle(order.begin(), order.end(), rr);
    for (size_t b = 0; b < nb; ++b) up[b] = uni + b * block_bytes;
    for (size_t i = 0; i < cp.size(); ++i) {
      cp[i] = chunks + order[i] * chunk_bytes;
      bp[i] = back + order[i] * chunk_bytes;
    }
    void **d_up, **d_cp, **d_bp;
    CK(cudaMalloc(&d_up, up.size() * 8));
    CK(cudaMalloc(&d_cp, cp.size() * 8));
    CK(cudaMalloc(&d_bp, bp.size() * 8));
    CK(cudaMemcpy(d_up, up.data(), up.size() * 8, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(d_cp, cp.data(), cp.size() * 8, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(d_bp, bp.data(), bp.size() * 8, cudaMemcpyHostToDevice));
    const double pbytes = static_cast<double>(nb * block_bytes);
    for (const char* which : {"ours", "ref"}) {
      const std::string path = std::string(which) == "ours" ? root + "/../dynamo_b200/libkvbm_kernels.so" : root + "/../oracle/_ref/libkvbm_kernels_ref.so";
      void* h = dlopen(path.c_str(), RTLD_NOW | RTLD_LOCAL);
      if (!h) {
        fprintf(stderr, "perm %s: %s\n", which, dlerror());
        continue;
      }
      perm_fn k2 = reinterpret_cast<perm_fn>(dlsym(h, "kvbm_kernels_launch_universal_from_block"));
      perm_fn2 k3 = reinterpret_cast<perm_fn2>(dlsym(h, "kvbm_kernels_launch_block_from_universal"));
      for (int layout = 0; layout < 2; ++layout) {
        CK(cudaMemset(uni, 0, nb * block_bytes));
        CK(cudaMemset(back, 0, nb * block_bytes));
        auto l2 = [&]() { CK(k2(d_up, reinterpret_cast<const void* const*>(d_cp), nb, nh, nl_, no_, nt, hd, 1, layout, st)); };
        auto l3 = [&]() { CK(k3(reinterpret_cast<const void* const*>(d_up), d_bp, nb, nh, nl_, no_, nt, hd, 1, layout, st)); };
        Timing t2 = time_it(l2, st, iters);
        Timing t3 = time_it(l3, st, iters);
        CK(cudaStreamSynchronize(st));
        // round trip must reproduce the chunks
        std::vector<uint8_t> a(1 << 20), c(1 << 20);
        CK(cudaMemcpy(a.data(), chunks + (nb * block_bytes / 2), a.size(), cudaMemcpyDeviceToHost));
        CK(cudaMemcpy(c.data(), back + (nb * block_bytes / 2), c.size(), cudaMemcpyDeviceToHost));
        const int same = memcmp(a.data(), c.data(), a.size()) == 0;
        printf("{\"name\":\"perm_%s\",\"layout\":\"%s\",\"k2_ms\":%.5f,\"k3_ms\":%.5f,\"k2_gbs_rw\":%.1f,\"k3_gbs_rw\":%.1f,\"roundtrip_ok\":%d}\n", which,
               layout == 0 ? "NHD" : "HND", t2.med_ms, t3.med_ms, 2 * pbytes / t2.med_ms / 1e6, 2 * pbytes / t3.med_ms / 1e6, same);
        fflush(stdout);
      }
    }
  }
  return 0;
}
