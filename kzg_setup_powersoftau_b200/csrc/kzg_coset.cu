// Coset openings of KZG10 on the GPU: the division by X^k - c of kzg_coset.cuh in three kernels (writing the quotient
// as 32-byte scalars straight into the buffer the bucket MSM reads), the batched radix-2 NTT over Fr, and the scalar
// assembly of the batched coset check.  Its own object, so that the objects of the other kernels do not change.
#include <string.h>

#include "blake2b.h"
#include "kernels.h"
#include "kzg_coset.cuh"

namespace ptau {

#define PTAU_COSET_BLOCK 256
static_assert(kCosetMaxLgK == kCosetLgKMax, "the host fills the per-item tables kzg_coset.cu reads");
static_assert(kKzgZPow == kKzgZPowCount, "the host fills the table launch_coset_quotient copies");

struct CosetFr {
  uint32_t w[8];
};
struct CosetPow {  // w^(2^s) R for s < kCosetMaxLgK
  uint32_t w[kCosetMaxLgK][8];
};
struct CosetKey {
  uint64_t h[8];
};

__global__ void __launch_bounds__(PTAU_COSET_BLOCK) coset_quotient_chunk_sums(const uint32_t* __restrict__ c, uint64_t n,
                                                                              int lg_k, uint64_t mc, CosetFr cm,
                                                                              uint32_t* __restrict__ sums,
                                                                              uint32_t* __restrict__ bad) {
  const uint64_t id = (uint64_t)blockIdx.x * PTAU_COSET_BLOCK + threadIdx.x;
  if (id < (mc << lg_k)) coset_chunk_sum_item(c, n, lg_k, kKzgLgChunk, mc, cm.w, id, sums, bad);
}

// chunk sums -> the carry entering each chunk, in place; each chain is scanned by a segment of 2^lg_seg threads of
// a block of min(1024, k 2^lg_seg) threads (at k = 1: one block, one segment)
__global__ void __launch_bounds__(1 << kKzgLgCarryThreads) coset_quotient_carries(uint32_t* __restrict__ sums, uint64_t mc,
                                                                                  int lg_seg, int lg_run, KzgZPow cp) {
  constexpr int T = 1 << kKzgLgCarryThreads;
  __shared__ uint32_t y[T][8];
  const int tid = threadIdx.x;
  const uint64_t g = (uint64_t)blockIdx.x * blockDim.x + tid, j = g >> lg_seg;
  const int t = (int)(g & ((1u << lg_seg) - 1)), seg = 1 << lg_seg;
  uint32_t* s = sums + j * mc * 8;
  uint32_t zl[8], mul[8], acc[8];
  for (int w = 0; w < 8; w++) zl[w] = cp.w[kKzgLgChunk][w];
  kzg_run_sum_item(s, mc, lg_run, zl, t, acc);
  for (int st = 0; st < lg_seg; st++) {
    for (int w = 0; w < 8; w++) y[tid][w] = acc[w];
    __syncthreads();
    for (int w = 0; w < 8; w++) mul[w] = cp.w[kKzgLgChunk + lg_run + st][w];
    if (t + (1 << st) < seg) kzg_combine_item(acc, y[tid + (1 << st)], mul, acc);
    __syncthreads();
  }
  for (int w = 0; w < 8; w++) y[tid][w] = acc[w];
  __syncthreads();
  uint32_t cin[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  if (t + 1 < seg)
    for (int w = 0; w < 8; w++) cin[w] = y[tid + 1][w];
  kzg_run_carry_item(s, mc, lg_run, zl, t, cin);
}

__global__ void __launch_bounds__(PTAU_COSET_BLOCK) coset_quotient_write(const uint32_t* __restrict__ c, uint64_t n, int lg_k,
                                                                         uint64_t mc, CosetFr cm,
                                                                         const uint32_t* __restrict__ carries,
                                                                         uint32_t* __restrict__ q, uint32_t* __restrict__ rem) {
  const uint64_t id = (uint64_t)blockIdx.x * PTAU_COSET_BLOCK + threadIdx.x;
  if (id < (mc << lg_k)) coset_write_item(c, n, lg_k, kKzgLgChunk, mc, cm.w, id, carries, q, rem);
}

// tw[i] = w^i R for i < k/2
__global__ void __launch_bounds__(PTAU_COSET_BLOCK) ntt_twiddles(uint32_t* __restrict__ tw, int lg_k, CosetPow wp) {
  const uint64_t i = (uint64_t)blockIdx.x * PTAU_COSET_BLOCK + threadIdx.x;
  if (i >= (1ull << lg_k) / 2) return;
  uint32_t v[8];
  fr_pow_bits(v, wp.w, i, lg_k);
  fr_store(tw + i * 8, v);
}

// items x k elements: out[item][bitrev(j)] = in[item][j] h_item^j (hpow: items x kCosetMaxLgK rows, or null)
__global__ void __launch_bounds__(PTAU_COSET_BLOCK) ntt_permute(const uint32_t* __restrict__ in, uint32_t* __restrict__ out,
                                                                uint64_t items, int lg_k, const uint32_t* __restrict__ hpow) {
  const uint64_t g = (uint64_t)blockIdx.x * PTAU_COSET_BLOCK + threadIdx.x;
  if (g >= (items << lg_k)) return;
  const uint64_t it = g >> lg_k, j = g & ((1ull << lg_k) - 1);
  const uint32_t(*hp)[8] = hpow ? (const uint32_t(*)[8])(hpow + it * kCosetMaxLgK * 8) : nullptr;
  ntt_permute_item(in + (it << lg_k) * 8, out + (it << lg_k) * 8, lg_k, hp, j);
}

__global__ void __launch_bounds__(PTAU_COSET_BLOCK) ntt_stage(uint32_t* __restrict__ x, uint64_t items, int lg_k, int s,
                                                              const uint32_t* __restrict__ tw) {
  const uint64_t g = (uint64_t)blockIdx.x * PTAU_COSET_BLOCK + threadIdx.x;
  if (g >= (items << (lg_k - 1))) return;
  const uint64_t it = g >> (lg_k - 1), i = g & ((1ull << (lg_k - 1)) - 1);
  ntt_butterfly_item(x + (it << lg_k) * 8, lg_k, s, tw, i);
}

// item i of a check: rho_i (BLAKE2b keyed with the seed, domain byte kCosetRhoDomain), then
// srm[i] = rho_i k^-1 R, sc[i] = rho_i, sc[m + i] = rho_i c_i, neg[i] = -rho_i
__global__ void __launch_bounds__(PTAU_COSET_BLOCK) coset_check_scalars(CosetKey key, uint64_t m,
                                                                        const uint32_t* __restrict__ cm, CosetFr kinv_r2,
                                                                        uint32_t* __restrict__ srm, uint32_t* __restrict__ sc,
                                                                        uint32_t* __restrict__ neg) {
  const uint64_t i = (uint64_t)blockIdx.x * PTAU_COSET_BLOCK + threadIdx.x;
  if (i >= m) return;
  uint32_t rho[8], v[8], ci[8];
  const uint32_t zero[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  ratio_coeff(key.h, kCosetRhoDomain, i, rho);
  fr_mul(v, rho, kinv_r2.w);
  fr_store(srm + i * 8, v);
  fr_store(sc + i * 8, rho);
  fr_load(ci, cm + i * 8);
  fr_mul(v, rho, ci);
  fr_store(sc + (m + i) * 8, v);
  fr_sub(v, zero, rho);
  fr_store(neg + i * 8, v);
}

__global__ void __launch_bounds__(PTAU_COSET_BLOCK) coset_interp_sum(const uint32_t* __restrict__ x, uint64_t m, int lg_k,
                                                                     const uint32_t* __restrict__ hinv,
                                                                     const uint32_t* __restrict__ srm, uint32_t* __restrict__ out) {
  const uint64_t j = (uint64_t)blockIdx.x * PTAU_COSET_BLOCK + threadIdx.x;
  if (j < (1ull << lg_k)) coset_interp_sum_item(x, m, lg_k, (const uint32_t(*)[8])hinv, srm, j, out);
}

static unsigned blocks(uint64_t threads) { return (unsigned)((threads + PTAU_COSET_BLOCK - 1) / PTAU_COSET_BLOCK); }

// chunks per chain: ceil(ceil(n / k) / L)
static uint64_t coset_chunks(uint64_t n, int lg_k) {
  const uint64_t rows = (n + (1ull << lg_k) - 1) >> lg_k;
  return (rows + (1u << kKzgLgChunk) - 1) >> kKzgLgChunk;
}

size_t coset_quotient_sums_bytes(uint64_t n, int lg_k) { return (size_t)(coset_chunks(n, lg_k) << lg_k) * 32 + 16; }

cudaError_t launch_coset_quotient(const void* d_coeffs, uint64_t n, int lg_k, const uint32_t (*cpow)[8], void* d_sums,
                                  void* d_q, void* d_rem, uint32_t* d_bad, int* launches, cudaStream_t stream) {
  *launches = 0;
  if (n == 0) return cudaMemsetAsync(d_rem, 0, (size_t)32 << lg_k, stream);  // p = 0: r = 0 and no quotient
  KzgZPow cp;
  memcpy(cp.w, cpow, sizeof(cp.w));
  CosetFr cm;
  memcpy(cm.w, cpow[0], 32);
  const uint64_t mc = coset_chunks(n, lg_k), items = mc << lg_k;
  int lg_seg, lg_run;
  coset_carry_shape(mc, kKzgLgCarryThreads, &lg_seg, &lg_run);
  const uint64_t carry_threads = (uint64_t)1 << (lg_k + lg_seg);
  const unsigned carry_block = carry_threads < (1u << kKzgLgCarryThreads) ? (unsigned)carry_threads : 1u << kKzgLgCarryThreads;
  const auto c = (const uint32_t*)d_coeffs;
  const auto sums = (uint32_t*)d_sums;
  coset_quotient_chunk_sums<<<blocks(items), PTAU_COSET_BLOCK, 0, stream>>>(c, n, lg_k, mc, cm, sums, d_bad);
  coset_quotient_carries<<<(unsigned)(carry_threads / carry_block), carry_block, 0, stream>>>(sums, mc, lg_seg, lg_run, cp);
  coset_quotient_write<<<blocks(items), PTAU_COSET_BLOCK, 0, stream>>>(c, n, lg_k, mc, cm, sums, (uint32_t*)d_q,
                                                                       (uint32_t*)d_rem);
  *launches = 3;
  return cudaGetLastError();
}

cudaError_t launch_ntt_twiddles(void* d_tw, int lg_k, const uint32_t (*wpow)[8], cudaStream_t stream) {
  if (lg_k == 0) return cudaSuccess;  // k = 1: no butterflies
  CosetPow wp;
  memset(&wp, 0, sizeof(wp));
  memcpy(wp.w, wpow, (size_t)lg_k * 32);
  ntt_twiddles<<<blocks((1ull << lg_k) / 2), PTAU_COSET_BLOCK, 0, stream>>>((uint32_t*)d_tw, lg_k, wp);
  return cudaGetLastError();
}

cudaError_t launch_ntt(const void* d_in, void* d_out, uint64_t items, int lg_k, const void* d_hpow, const void* d_tw,
                       int* launches, cudaStream_t stream) {
  *launches = 0;
  if (items == 0) return cudaSuccess;
  ntt_permute<<<blocks(items << lg_k), PTAU_COSET_BLOCK, 0, stream>>>((const uint32_t*)d_in, (uint32_t*)d_out, items, lg_k,
                                                                      (const uint32_t*)d_hpow);
  for (int s = 0; s < lg_k; s++)
    ntt_stage<<<blocks(items << (lg_k - 1)), PTAU_COSET_BLOCK, 0, stream>>>((uint32_t*)d_out, items, lg_k, s,
                                                                           (const uint32_t*)d_tw);
  *launches = 1 + lg_k;
  return cudaGetLastError();
}

cudaError_t launch_coset_check_scalars(const uint64_t* key_h, uint64_t m, const void* d_cm, const uint32_t* kinv_r2,
                                       void* d_srm, void* d_sc, void* d_neg, cudaStream_t stream) {
  CosetKey key;
  memcpy(key.h, key_h, sizeof(key.h));
  CosetFr kr;
  memcpy(kr.w, kinv_r2, 32);
  coset_check_scalars<<<blocks(m), PTAU_COSET_BLOCK, 0, stream>>>(key, m, (const uint32_t*)d_cm, kr, (uint32_t*)d_srm,
                                                                  (uint32_t*)d_sc, (uint32_t*)d_neg);
  return cudaGetLastError();
}

cudaError_t launch_coset_interp_sum(const void* d_x, uint64_t m, int lg_k, const void* d_hinv, const void* d_srm,
                                    void* d_out, cudaStream_t stream) {
  coset_interp_sum<<<blocks(1ull << lg_k), PTAU_COSET_BLOCK, 0, stream>>>((const uint32_t*)d_x, m, lg_k,
                                                                          (const uint32_t*)d_hinv, (const uint32_t*)d_srm,
                                                                          (uint32_t*)d_out);
  return cudaGetLastError();
}

}  // namespace ptau
