// The witness polynomial of KZG10::open on the GPU: the blocked scan of kzg_open.cuh in three kernels, writing the
// quotient as 32-byte scalars straight into the buffer the bucket MSM reads.  Its own object, so that the objects
// of the other kernels do not change.
#include <string.h>

#include "kernels.h"
#include "kzg_open.cuh"

namespace ptau {

#define PTAU_KZG_BLOCK 256
static_assert(kKzgZPow == kKzgZPowCount, "the host fills the table launch_kzg_quotient copies");

struct FrWords {
  uint32_t w[8];
};

__global__ void __launch_bounds__(PTAU_KZG_BLOCK) kzg_quotient_chunk_sums(const uint32_t* __restrict__ c, uint64_t n,
                                                                          uint64_t m, FrWords z, uint32_t* __restrict__ sums,
                                                                          uint32_t* __restrict__ bad) {
  const uint64_t j = (uint64_t)blockIdx.x * PTAU_KZG_BLOCK + threadIdx.x;
  if (j < m) kzg_chunk_sum_item(c, n, kKzgLgChunk, z.w, j, sums, bad);
}

// one block: chunk sums -> the carry entering each chunk, in place
__global__ void __launch_bounds__(1 << kKzgLgCarryThreads) kzg_quotient_carries(uint32_t* __restrict__ sums, uint64_t m,
                                                                                int lg_run, KzgZPow zp) {
  constexpr int T = 1 << kKzgLgCarryThreads;
  __shared__ uint32_t y[T][8];
  const int t = threadIdx.x;
  uint32_t zl[8], mul[8], acc[8];
  for (int w = 0; w < 8; w++) zl[w] = zp.w[kKzgLgChunk][w];
  kzg_run_sum_item(sums, m, lg_run, zl, t, acc);
  for (int s = 0; s < kKzgLgCarryThreads; s++) {
    for (int w = 0; w < 8; w++) y[t][w] = acc[w];
    __syncthreads();
    for (int w = 0; w < 8; w++) mul[w] = zp.w[kKzgLgChunk + lg_run + s][w];
    if (t + (1 << s) < T) kzg_combine_item(acc, y[t + (1 << s)], mul, acc);
    __syncthreads();
  }
  // acc = the carry leaving run t (all runs above it folded in); run t starts from the one leaving run t + 1
  for (int w = 0; w < 8; w++) y[t][w] = acc[w];
  __syncthreads();
  uint32_t cin[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  if (t + 1 < T)
    for (int w = 0; w < 8; w++) cin[w] = y[t + 1][w];
  kzg_run_carry_item(sums, m, lg_run, zl, t, cin);
}

__global__ void __launch_bounds__(PTAU_KZG_BLOCK) kzg_quotient_write(const uint32_t* __restrict__ c, uint64_t n, uint64_t m,
                                                                     FrWords z, const uint32_t* __restrict__ carries,
                                                                     uint32_t* __restrict__ q, uint32_t* __restrict__ value) {
  const uint64_t j = (uint64_t)blockIdx.x * PTAU_KZG_BLOCK + threadIdx.x;
  if (j < m) kzg_write_item(c, n, kKzgLgChunk, z.w, j, carries, q, value);
}

size_t kzg_quotient_sums_bytes(uint64_t n) { return (size_t)((n + (1u << kKzgLgChunk) - 1) >> kKzgLgChunk) * 32 + 16; }

cudaError_t launch_kzg_quotient(const void* d_coeffs, uint64_t n, const uint32_t (*zpow)[8], void* d_sums, void* d_q,
                                void* d_value, uint32_t* d_bad, int* launches, cudaStream_t stream) {
  *launches = 0;
  if (n == 0) return cudaMemsetAsync(d_value, 0, 32, stream);  // p = 0: p(z) = 0 and no quotient
  KzgZPow zp;
  memcpy(zp.w, zpow, sizeof(zp.w));
  FrWords z;
  memcpy(z.w, zpow[0], 32);
  const uint64_t m = (n + (1u << kKzgLgChunk) - 1) >> kKzgLgChunk;
  int lg_run = 0;  // smallest with m <= 2^(kKzgLgCarryThreads + lg_run)
  while ((1ull << (kKzgLgCarryThreads + lg_run)) < m) lg_run++;
  const unsigned grid = (unsigned)((m + PTAU_KZG_BLOCK - 1) / PTAU_KZG_BLOCK);
  const auto c = (const uint32_t*)d_coeffs;
  const auto sums = (uint32_t*)d_sums;
  kzg_quotient_chunk_sums<<<grid, PTAU_KZG_BLOCK, 0, stream>>>(c, n, m, z, sums, d_bad);
  kzg_quotient_carries<<<1, 1 << kKzgLgCarryThreads, 0, stream>>>(sums, m, lg_run, zp);
  kzg_quotient_write<<<grid, PTAU_KZG_BLOCK, 0, stream>>>(c, n, m, z, sums, (uint32_t*)d_q, (uint32_t*)d_value);
  *launches = 3;
  return cudaGetLastError();
}

}  // namespace ptau
