// Inline-PTX wrappers for the sm_100a data-movement primitives used by the KV transfer kernels:
// mbarrier, TMA bulk copies (cp.async.bulk, SASS: UBLKCP), proxy fences, system-scope flags,
// vectorised global ld/st with cache hints and the fp8<->bf16 converts.
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime_api.h>

#include <cstdint>

namespace kvbm {
namespace ptx {

__device__ __forceinline__ uint32_t smem_addr(const void* p)
{
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

// ---------------------------------------------------------------- mbarrier
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count)
{
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init()
{
  // make the initialised barriers visible to the async proxy (TMA unit)
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes)
{
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar)
{
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity)
{
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(bar), "r"(parity)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity)
{
  while (!mbar_try_wait(bar, parity)) {
  }
}

// ---------------------------------------------------------------- TMA bulk copies (1-D)
// global -> shared, completion counted in bytes on an mbarrier.  16 B aligned, size % 16 == 0.
__device__ __forceinline__ void bulk_g2s(uint32_t dst_smem, const void* src_gmem, uint32_t bytes,
                                         uint32_t bar)
{
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
          dst_smem),
      "l"(src_gmem), "r"(bytes), "r"(bar)
      : "memory");
}
// shared -> global (local HBM or an NVLink peer mapping), tracked by bulk async-groups.
__device__ __forceinline__ void bulk_s2g(void* dst_gmem, uint32_t src_smem, uint32_t bytes)
{
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst_gmem),
               "r"(src_smem), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void bulk_commit()
{
  asm volatile("cp.async.bulk.commit_group;" ::: "memory");
}
template <int N>
__device__ __forceinline__ void bulk_wait_read()
{
  asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}
// runtime-selected "at most n groups still reading their smem source" (immediate operand in PTX)
__device__ __forceinline__ void bulk_wait_read_n(int n)
{
  switch (n) {
    case 0: bulk_wait_read<0>(); break;
    case 1: bulk_wait_read<1>(); break;
    case 2: bulk_wait_read<2>(); break;
    case 3: bulk_wait_read<3>(); break;
    case 4: bulk_wait_read<4>(); break;
    case 5: bulk_wait_read<5>(); break;
    case 6: bulk_wait_read<6>(); break;
    case 7: bulk_wait_read<7>(); break;
    case 8: bulk_wait_read<8>(); break;
    case 9: bulk_wait_read<9>(); break;
    case 10: bulk_wait_read<10>(); break;
    case 11: bulk_wait_read<11>(); break;
    case 12: bulk_wait_read<12>(); break;
    case 13: bulk_wait_read<13>(); break;
    case 14: bulk_wait_read<14>(); break;
    default: bulk_wait_read<15>(); break;
  }
}
template <int N>
__device__ __forceinline__ void bulk_wait()
{
  asm volatile("cp.async.bulk.wait_group %0;" ::"n"(N) : "memory");
}
// generic-proxy writes to smem -> visible to the async proxy (before a bulk store reads them)
__device__ __forceinline__ void fence_proxy_async_smem()
{
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
// async-proxy global writes <-> generic proxy ordering (before publishing a flag)
__device__ __forceinline__ void fence_proxy_async_global()
{
  asm volatile("fence.proxy.async.global;" ::: "memory");
}

// ---------------------------------------------------------------- flags (system scope: peers + host)
__device__ __forceinline__ void st_release_sys(uint32_t* p, uint32_t v)
{
  asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
// relaxed system-scope store: pair with ONE preceding fence_acq_rel_sys() when several flags are published together
// (a st.release.sys per flag would repeat the fence)
__device__ __forceinline__ void st_relaxed_sys(uint32_t* p, uint32_t v)
{
  asm volatile("st.relaxed.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t ld_acquire_sys(const uint32_t* p)
{
  uint32_t v;
  asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
// polling load: no L1 invalidation / fence per probe (ld.acquire.sys costs a CCTL.IVALL each time); pair a
// successful probe with fence_acq_rel_sys() once
__device__ __forceinline__ uint32_t ld_relaxed_sys(const uint32_t* p)
{
  uint32_t v;
  asm volatile("ld.relaxed.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ uint64_t globaltimer_ns()
{
  uint64_t t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
__device__ __forceinline__ void fence_acq_rel_sys()
{
  asm volatile("fence.acq_rel.sys;" ::: "memory");
}
__device__ __forceinline__ uint32_t atom_add_acq_rel_gpu(uint32_t* p, uint32_t v)
{
  uint32_t old;
  asm volatile("atom.acq_rel.gpu.global.add.u32 %0, [%1], %2;" : "=r"(old) : "l"(p), "r"(v) : "memory");
  return old;
}

// ---------------------------------------------------------------- 128-bit global access, streaming
__device__ __forceinline__ uint4 ld_stream_v4(const void* p)
{
  uint4 r;
  asm volatile("ld.global.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
               : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
               : "l"(p));
  return r;
}
__device__ __forceinline__ void st_stream_v4(void* p, const uint4& v)
{
  asm volatile("st.global.L1::no_allocate.v4.u32 [%0], {%1,%2,%3,%4};" ::"l"(p), "r"(v.x), "r"(v.y),
               "r"(v.z), "r"(v.w)
               : "memory");
}

// Store to an NVLink multicast (multimem) address: the NVSwitch replicates the write to every device bound to the
// multicast object.  PTX only defines multimem.* instructions on such addresses (it assembles to a plain STG).
__device__ __forceinline__ void multimem_st_v4(void* p, const uint4& v)
{
  asm volatile("multimem.st.weak.global.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(p), "f"(__uint_as_float(v.x)),
               "f"(__uint_as_float(v.y)), "f"(__uint_as_float(v.z)), "f"(__uint_as_float(v.w))
               : "memory");
}
__device__ __forceinline__ void multimem_st_b32(void* p, uint32_t v)
{
  asm volatile("multimem.st.weak.global.b32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}

// ---------------------------------------------------------------- fp8 e4m3fn <-> bf16
// two e4m3 codes (low 16 bits) -> two bf16 (exact).  NaN codes (0x7f/0xff) -> 0x7fc0.
__device__ __forceinline__ uint32_t e4m3x2_to_bf16x2(uint16_t two)
{
  uint32_t h2;
  asm("cvt.rn.f16x2.e4m3x2 %0, %1;" : "=r"(h2) : "h"(two));
  __half2 h = *reinterpret_cast<__half2*>(&h2);
  float2 f = __half22float2(h);
  __nv_bfloat162 b = __floats2bfloat162_rn(f.x, f.y);  // exact: every e4m3 value fits bf16
  uint32_t out = *reinterpret_cast<uint32_t*>(&b);
  if ((two & 0x007f) == 0x007f) out = (out & 0xffff0000u) | 0x7fc0u;
  if ((two & 0x7f00) == 0x7f00) out = (out & 0x0000ffffu) | 0x7fc00000u;
  return out;
}
// two bf16 -> two e4m3 codes, RNE, saturate to +-448; NaN -> 0x7f | sign.
__device__ __forceinline__ uint16_t bf16x2_to_e4m3x2(uint32_t two)
{
  float lo = __uint_as_float(two << 16);
  float hi = __uint_as_float(two & 0xffff0000u);
  uint16_t out;
  asm("cvt.rn.satfinite.e4m3x2.f32 %0, %1, %2;" : "=h"(out) : "f"(hi), "f"(lo));
  // hardware maps NaN to 0x7f; carry the sign bit like the oracle does
  if (lo != lo) out = (out & 0xff00) | 0x7f | ((two >> 8) & 0x80);
  if (hi != hi) out = (out & 0x00ff) | 0x7f00 | ((two >> 16) & 0x8000);
  return out;
}

}  // namespace ptx
}  // namespace kvbm
