/* A C program built against the SIX reference symbols only (lib/kvbm-kernels/src/tensor_kernels.rs:46-109).  The test
 * runs it with LD_LIBRARY_PATH pointing at this repo's libkvbm_kernels.so and requires byte-identical output to what the
 * same binary printed on the reference's own kernels compiled unmodified (oracle/_ref) under the same file name
 * (tests/golden/reference_kernels_dropin.txt): the "swap the .so" drop-in of INTEGRATION.md section 1, literally.
 * Prints a checksum line per case. */
#include <cuda_runtime_api.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

cudaError_t kvbm_kernels_launch_vectorized_copy(void** src_ptrs, void** dst_ptrs, size_t copy_size_bytes, int num_pairs, cudaStream_t stream);
cudaError_t kvbm_kernels_memcpy_batch(const void* const* src, void* const* dst, size_t size_per_copy, size_t num_copies, int mode, cudaStream_t stream);
cudaError_t kvbm_kernels_launch_universal_from_block(void* const* universal_ptrs, const void* const* block_ptrs, size_t num_blocks,
                                                     size_t nh, size_t nl, size_t no, size_t nt, size_t hd, int dtype, int layout,
                                                     cudaStream_t stream);
cudaError_t kvbm_kernels_launch_block_from_universal(const void* const* universal_ptrs, void* const* block_ptrs, size_t num_blocks,
                                                     size_t nh, size_t nl, size_t no, size_t nt, size_t hd, int dtype, int layout,
                                                     cudaStream_t stream);
_Bool kvbm_kernels_has_memcpy_batch_async(void);
_Bool kvbm_kernels_is_stub_build(void);

#define CK(x)                                                                          \
  do {                                                                                 \
    cudaError_t e__ = (x);                                                             \
    if (e__ != cudaSuccess) {                                                          \
      printf("CUDA error %d at %s:%d (%s)\n", (int)e__, __FILE__, __LINE__, #x);      \
      return 2;                                                                        \
    }                                                                                  \
  } while (0)

static uint64_t fnv(const unsigned char* p, size_t n)
{
  uint64_t h = 1469598103934665603ull;
  for (size_t i = 0; i < n; ++i) h = (h ^ p[i]) * 1099511628211ull;
  return h;
}

int main(void)
{
  if (kvbm_kernels_is_stub_build()) {
    puts("stub build");
    return 3;
  }
  CK(cudaSetDevice(0));
  cudaStream_t st;
  CK(cudaStreamCreate(&st));

  /* K1: 37 pairs of 999 bytes (the reference's odd-size case, tests/memcpy_batch.rs:350-431), pointer tables in pinned memory */
  enum { NP = 37, SZ = 999 };
  unsigned char *dsrc, *ddst, *h = malloc(NP * 1024), *back = malloc(NP * 1024);
  CK(cudaMalloc((void**)&dsrc, NP * 1024));
  CK(cudaMalloc((void**)&ddst, NP * 1024));
  for (int i = 0; i < NP * 1024; ++i) h[i] = (unsigned char)((i * 13 + i / 1024) % 256);
  CK(cudaMemcpy(dsrc, h, NP * 1024, cudaMemcpyHostToDevice));
  CK(cudaMemset(ddst, 0xEE, NP * 1024));
  void **ps, **pd;
  CK(cudaMallocHost((void**)&ps, NP * sizeof(void*)));
  CK(cudaMallocHost((void**)&pd, NP * sizeof(void*)));
  for (int i = 0; i < NP; ++i) {
    ps[i] = dsrc + (size_t)i * 1024 + (i % 3);          /* odd alignments on purpose */
    pd[i] = ddst + (size_t)((i * 7) % NP) * 1024 + (i % 5);
  }
  CK(kvbm_kernels_launch_vectorized_copy(ps, pd, SZ, NP, st));
  CK(cudaStreamSynchronize(st));
  CK(cudaMemcpy(back, ddst, NP * 1024, cudaMemcpyDeviceToHost));
  printf("k1 %016llx\n", (unsigned long long)fnv(back, NP * 1024));
  for (int i = 0; i < NP; ++i)
    if (memcmp(back + (size_t)((i * 7) % NP) * 1024 + (i % 5), h + (size_t)i * 1024 + (i % 3), SZ) != 0) {
      printf("k1 pair %d differs\n", i);
      return 4;
    }
  /* edge cases: zero pairs / zero size succeed before the NULL checks; NULL tables are invalid */
  printf("k1_edges %d %d %d\n", (int)kvbm_kernels_launch_vectorized_copy(NULL, NULL, 16, 0, st),
         (int)kvbm_kernels_launch_vectorized_copy(NULL, NULL, 0, 4, st), (int)kvbm_kernels_launch_vectorized_copy(NULL, pd, 16, 4, st));
  (void)cudaGetLastError();

  /* K4: host pointer tables, every mode */
  CK(cudaMemset(ddst, 0, NP * 1024));
  const void* bs[4];
  void* bd[4];
  for (int i = 0; i < 4; ++i) {
    bs[i] = dsrc + (size_t)i * 4096;
    bd[i] = ddst + (size_t)(3 - i) * 4096;
  }
  for (int mode = 0; mode < 3; ++mode) {
    cudaError_t e = kvbm_kernels_memcpy_batch(bs, bd, 4096, 4, mode, st);
    CK(cudaStreamSynchronize(st));
    CK(cudaMemcpy(back, ddst, 16384, cudaMemcpyDeviceToHost));
    printf("k4 mode%d rc%d %016llx\n", mode, (int)e, (unsigned long long)fnv(back, 16384));
    (void)cudaGetLastError();
  }
  printf("k4_edges %d %d\n", (int)kvbm_kernels_memcpy_batch(NULL, NULL, 16, 0, 0, st), (int)kvbm_kernels_memcpy_batch(NULL, bd, 16, 2, 0, st));
  (void)cudaGetLastError();

  /* K2 / K3: block stack <-> universal, dims (3,2,2,4,5) bf16, NHD (kernel_roundtrip.rs:418-493) */
  enum { NHh = 3, NLl = 2, NOo = 2, NT = 4, HD = 5 };
  const size_t chunk = (size_t)NT * NHh * HD * 2, nchunks = (size_t)NLl * NOo, uni = chunk * nchunks;
  unsigned char *dchunks, *duni, *dback;
  CK(cudaMalloc((void**)&dchunks, uni));
  CK(cudaMalloc((void**)&duni, uni));
  CK(cudaMalloc((void**)&dback, uni));
  CK(cudaMemcpy(dchunks, h, uni, cudaMemcpyHostToDevice));
  void **cp, **up, **cb;
  CK(cudaMallocHost((void**)&cp, nchunks * sizeof(void*)));
  CK(cudaMallocHost((void**)&cb, nchunks * sizeof(void*)));
  CK(cudaMallocHost((void**)&up, sizeof(void*)));
  for (size_t i = 0; i < nchunks; ++i) {
    cp[i] = dchunks + i * chunk;
    cb[i] = dback + i * chunk;
  }
  up[0] = duni;
  CK(kvbm_kernels_launch_universal_from_block((void* const*)up, (const void* const*)cp, 1, NHh, NLl, NOo, NT, HD, 1, 0, st));
  CK(kvbm_kernels_launch_block_from_universal((const void* const*)up, (void* const*)cb, 1, NHh, NLl, NOo, NT, HD, 1, 0, st));
  CK(cudaStreamSynchronize(st));
  CK(cudaMemcpy(back, duni, uni, cudaMemcpyDeviceToHost));
  printf("k2 %016llx\n", (unsigned long long)fnv(back, uni));
  CK(cudaMemcpy(back, dback, uni, cudaMemcpyDeviceToHost));
  printf("k3_roundtrip %d\n", memcmp(back, h, uni) == 0);
  printf("k2_bad_dtype %d\n", (int)kvbm_kernels_launch_universal_from_block((void* const*)up, (const void* const*)cp, 1, NHh, NLl, NOo, NT, HD, 9, 0, st));
  (void)cudaGetLastError();
  puts("done");
  return 0;
}
