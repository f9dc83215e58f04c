// Per-item code of the coset openings (kzg_coset.cu): division by X^k - c for k = 2^lg_k and the radix-2 NTT over Fr.
//
// Division.  p = (X^k - c) q + r, deg r < k.  For each residue j < k the chain p_j, p_{j+k}, p_{j+2k}, ... is folded
// from the top, acc <- p_{j+tk} + c acc: the acc after row t >= 1 is q_{j+(t-1)k}, the final acc is r_j.  Every chain
// is the recurrence of kzg_open.cuh with the multiplier c, so it runs as the same exact blocked scan, chain by chain:
//   1. chunk b of chain j = rows [bL, bL + L) has the local sum S_{j,b} (Horner from the top, carry 0);
//   2. the carry entering chunk b is K_{j,b+1}, K_{j,b} = S_{j,b} + c^L K_{j,b+1}: the carry items of kzg_open.cuh over
//      chain j's mc chunk sums, 2^lg_seg threads per chain (one segment of the carry block);
//   3. chunk b re-runs Horner from its carry and writes q straight into the MSM's scalar buffer, and r_j at b = 0.
// Chunk sums are stored chain after chain (sums[j mc + b]) so each chain's are contiguous.  Item id = b k + j: adjacent
// threads read adjacent coefficients.  With k = 1 this is the scan of kzg_open.cuh with z = c.
//
// NTT.  x natural order in and out: a bit-reversing copy (with the coset scale h^j fused in) and lg_k in-place
// Cooley-Tukey butterfly stages whose twiddles are tw[i] = w^i R for i < k/2.
//
// Shared with the host build (tests/host_emul/hostemul_coset.cpp), which runs the same items serially.
#pragma once
#include "kzg_open.cuh"

namespace ptau {

constexpr int kCosetMaxLgK = 20;  // k <= 2^20: powers_of_h[k] stays inside a 2^21 setup

#if defined(__CUDACC__)
#define PTAU_COSET_HOST static __host__ __device__ inline
#else
#define PTAU_COSET_HOST static inline
#endif

// rows of chain j: ceil((n - j) / k) for j < n
PTAU_FR_HD uint64_t coset_chain_rows(uint64_t n, int lg_k, uint64_t j) {
  return j < n ? ((n - j - 1) >> lg_k) + 1 : 0;
}

// Horner over rows [lo, hi) of chain j from the top, starting from acc; q != nullptr: q_{j+(t-1)k} = acc for t >= 1.
// Returns false when a coefficient is not canonical.
PTAU_FR_HD bool coset_horner(const uint32_t* c, int lg_k, uint64_t j, uint64_t lo, uint64_t hi, const uint32_t* cm,
                             uint32_t* acc, uint32_t* q) {
  bool ok = true;
  for (uint64_t t = hi; t-- > lo;) {
    uint32_t ci[8], u[8];
    fr_load(ci, c + (j + (t << lg_k)) * 8);
    ok = ok && fr_is_canonical(ci);
    fr_mul(u, acc, cm);
    fr_add(acc, ci, u);
    if (q && t) fr_store(q + (j + ((t - 1) << lg_k)) * 8, acc);
  }
  return ok;
}

// step 1: S_{j,b} into sums[j mc + b] for id = b k + j; *bad = 1 when a coefficient of the chunk is not canonical
PTAU_FR_HD void coset_chunk_sum_item(const uint32_t* c, uint64_t n, int lg_k, int lg_chunk, uint64_t mc,
                                     const uint32_t* cm, uint64_t id, uint32_t* sums, uint32_t* bad) {
  const uint64_t j = id & ((1ull << lg_k) - 1), b = id >> lg_k, rows = coset_chain_rows(n, lg_k, j);
  const uint64_t lo = b << lg_chunk, hi = lo + (1ull << lg_chunk) < rows ? lo + (1ull << lg_chunk) : rows;
  uint32_t acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  if (!coset_horner(c, lg_k, j, lo, hi, cm, acc, nullptr)) *bad = 1;
  fr_store(sums + (j * mc + b) * 8, acc);
}

// step 3: chunk b of chain j from its incoming carry: quotient coefficients to q, r_j to rem (b = 0)
PTAU_FR_HD void coset_write_item(const uint32_t* c, uint64_t n, int lg_k, int lg_chunk, uint64_t mc, const uint32_t* cm,
                                 uint64_t id, const uint32_t* carries, uint32_t* q, uint32_t* rem) {
  const uint64_t j = id & ((1ull << lg_k) - 1), b = id >> lg_k, rows = coset_chain_rows(n, lg_k, j);
  const uint64_t lo = b << lg_chunk, hi = lo + (1ull << lg_chunk) < rows ? lo + (1ull << lg_chunk) : rows;
  uint32_t acc[8];
  fr_load(acc, carries + (j * mc + b) * 8);
  coset_horner(c, lg_k, j, lo, hi, cm, acc, q);
  if (b == 0) fr_store(rem + j * 8, acc);
}

// the segment of the carry block per chain: lg_seg = smallest with 2^lg_seg >= mc, at most lg_threads; lg_run =
// smallest with mc <= 2^(lg_seg + lg_run)
PTAU_COSET_HOST void coset_carry_shape(uint64_t mc, int lg_threads, int* lg_seg, int* lg_run) {
  int s = 0;
  while (s < lg_threads && (1ull << s) < mc) s++;
  int r = 0;
  while ((1ull << (s + r)) < mc) r++;
  *lg_seg = s;
  *lg_run = r;
}

PTAU_FR_HD uint64_t coset_bitrev(uint64_t j, int bits) {
  uint64_t r = 0;
  for (int s = 0; s < bits; s++) r |= ((j >> s) & 1) << (bits - 1 - s);
  return r;
}

// out[bitrev(j)] = in[j] h^j for one item; hp[s] = h^(2^s) R (nullptr: no scale)
PTAU_FR_HD void ntt_permute_item(const uint32_t* in, uint32_t* out, int lg_k, const uint32_t (*hp)[8], uint64_t j) {
  uint32_t v[8];
  fr_load(v, in + j * 8);
  if (hp) {
    uint32_t w[8];
    fr_pow_bits(w, hp, j, lg_k);
    fr_mul(v, v, w);
  }
  fr_store(out + coset_bitrev(j, lg_k) * 8, v);
}

// butterfly i < k/2 of stage s (half-width 2^s) of one item: (a, b) <- (a + w b, a - w b), w = tw[pos 2^(lg_k-1-s)]
PTAU_FR_HD void ntt_butterfly_item(uint32_t* x, int lg_k, int s, const uint32_t* tw, uint64_t i) {
  const uint64_t pos = i & ((1ull << s) - 1), a = ((i >> s) << (s + 1)) + pos, b = a + (1ull << s);
  uint32_t u[8], v[8], t[8];
  fr_load(u, x + a * 8);
  fr_load(v, x + b * 8);
  fr_mul(t, v, tw + (pos << (lg_k - 1 - s)) * 8);
  fr_add(v, u, t);
  fr_sub(u, u, t);
  fr_store(x + a * 8, v);
  fr_store(x + b * 8, u);
}

// the k-term MSM scalar j of the check: -sum_i x_i[j] h_i^-j (rho_i k^-1), where x_i = the unscaled inverse NTT of
// item i's values; hinv + i kCosetMaxLgK rows: h_i^(-2^s) R; srm[i] = rho_i k^-1 R
PTAU_FR_HD void coset_interp_sum_item(const uint32_t* x, uint64_t m, int lg_k, const uint32_t (*hinv)[8],
                                      const uint32_t* srm, uint64_t j, uint32_t* out) {
  uint32_t acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  for (uint64_t i = 0; i < m; i++) {
    uint32_t w[8], s[8], v[8];
    fr_pow_bits(w, hinv + i * kCosetMaxLgK, j, lg_k);
    fr_load(s, srm + i * 8);
    fr_mul(w, w, s);  // h_i^-j rho_i k^-1 R
    fr_load(v, x + ((i << lg_k) + j) * 8);
    fr_mul(v, v, w);
    fr_add(acc, acc, v);
  }
  const uint32_t zero[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  fr_sub(acc, zero, acc);
  fr_store(out + j * 8, acc);
}

}  // namespace ptau
