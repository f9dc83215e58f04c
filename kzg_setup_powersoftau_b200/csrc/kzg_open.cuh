// Per-item code of the KZG10 witness polynomial (kzg_open.cu): for p = c_0 .. c_{n-1} and a point z,
//   q_{n-2} = c_{n-1},   q_{i-1} = c_i + z q_i,   p(z) = c_0 + z q_0,
// i.e. the carries k_i = c_i + z k_{i+1} (k_n = 0) of synthetic division, q_{i-1} = k_i and p(z) = k_0.
//
// The recurrence is first order and linear, so it is computed as an exact blocked scan:
//   1. chunk j = coefficients [jL, jL + L) has the local sum S_j = sum_i c_{jL+i} z^i (Horner from the top, carry 0);
//   2. the carry entering chunk j from above is K_{j+1}, where K_j = S_j + z^L K_{j+1} (K_m = 0): the same recurrence
//      over the m chunk sums with the constant multiplier z^L.  One block scans it: each thread folds a run of
//      2^lg_run sums, the block combines the runs (Hillis-Steele, multipliers z^(L 2^lg_run 2^s)), and each thread
//      re-runs its sums from its incoming carry, leaving K_{j+1} in place of S_j;
//   3. chunk j re-runs Horner from K_{j+1} and writes its quotient coefficients, and p(z) at index 0.
// Only the top chunk (and the top run) may be short; their incoming carry is 0, so their length never enters a
// multiplier.  Every step is exact arithmetic in Fr: the result does not depend on L, the run length or the grid.
//
// Scalars stay canonical; the multipliers are z^(2^s) in Montgomery form (fr.cuh).  Shared with the host build
// (tests/host_emul/hostemul_open.cpp), which runs the same items serially.
#pragma once
#include "fr.cuh"

namespace ptau {

constexpr int kKzgZPow = 32;          // z^(2^s) for s < 32: lg L + lg_run + 9 <= 30 for any n < 2^31
constexpr int kKzgLgChunk = 5;        // L = 32 coefficients per thread
constexpr int kKzgLgCarryThreads = 10;  // the carry scan is one block of 1024 threads

// the multipliers of one point: w[s] = z^(2^s) R mod r
struct KzgZPow {
  uint32_t w[kKzgZPow][8];
};

// Horner over [lo, hi) from the top, starting from acc; q != nullptr: q_{i-1} = k_i to q for i >= 1 and k_0 to value.
// Returns false when a coefficient is not canonical.
PTAU_FR_HD bool kzg_horner(const uint32_t* c, uint64_t lo, uint64_t hi, const uint32_t* zm, uint32_t* acc, uint32_t* q,
                           uint32_t* value) {
  bool ok = true;
  for (uint64_t i = hi; i-- > lo;) {
    uint32_t ci[8], t[8];
    fr_load(ci, c + i * 8);
    ok = ok && fr_is_canonical(ci);
    fr_mul(t, acc, zm);
    fr_add(acc, ci, t);
    if (q) fr_store(i ? q + (i - 1) * 8 : value, acc);
  }
  return ok;
}

// The items take their multiplier (zm = z R, zl = z^L R, mul) as 8 words: the kernels pass a local copy of the one
// entry of KzgZPow they need rather than the whole table.

// step 1: S_j into sums[j]; *bad = 1 when a coefficient of the chunk is not canonical
PTAU_FR_HD void kzg_chunk_sum_item(const uint32_t* c, uint64_t n, int lg_chunk, const uint32_t* zm, uint64_t j,
                                   uint32_t* sums, uint32_t* bad) {
  const uint64_t lo = j << lg_chunk, hi = lo + (1ull << lg_chunk) < n ? lo + (1ull << lg_chunk) : n;
  uint32_t acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  if (!kzg_horner(c, lo, hi, zm, acc, nullptr, nullptr)) *bad = 1;
  fr_store(sums + j * 8, acc);
}

// step 2a: thread t's fold of the sums [t 2^lg_run, (t + 1) 2^lg_run) with the multiplier z^L
PTAU_FR_HD void kzg_run_sum_item(const uint32_t* sums, uint64_t m, int lg_run, const uint32_t* zl, uint64_t t, uint32_t* acc) {
  const uint64_t lo = t << lg_run, hi = lo + (1ull << lg_run) < m ? lo + (1ull << lg_run) : m;
  for (int w = 0; w < 8; w++) acc[w] = 0;
  for (uint64_t j = hi; j-- > lo;) {
    uint32_t s[8], u[8];
    fr_load(s, sums + j * 8);
    fr_mul(u, acc, zl);
    fr_add(acc, s, u);
  }
}

// step 2b: one Hillis-Steele step at distance 2^s: y_t + mul y_{t + 2^s}, mul = z^(L 2^lg_run 2^s) R
PTAU_FR_HD void kzg_combine_item(const uint32_t* y_t, const uint32_t* y_up, const uint32_t* mul, uint32_t* out) {
  uint32_t u[8];
  fr_mul(u, y_up, mul);
  fr_add(out, y_t, u);
}

// step 2c: thread t re-runs its sums from its incoming carry cin and leaves the carry entering each chunk in place
PTAU_FR_HD void kzg_run_carry_item(uint32_t* sums, uint64_t m, int lg_run, const uint32_t* zl, uint64_t t, const uint32_t* cin) {
  const uint64_t lo = t << lg_run, hi = lo + (1ull << lg_run) < m ? lo + (1ull << lg_run) : m;
  uint32_t acc[8];
  for (int w = 0; w < 8; w++) acc[w] = cin[w];
  for (uint64_t j = hi; j-- > lo;) {
    uint32_t s[8], u[8];
    fr_load(s, sums + j * 8);
    fr_store(sums + j * 8, acc);
    fr_mul(u, acc, zl);
    fr_add(acc, s, u);
  }
}

// step 3: chunk j from its incoming carry: quotient coefficients to q, p(z) to value (chunk 0)
PTAU_FR_HD void kzg_write_item(const uint32_t* c, uint64_t n, int lg_chunk, const uint32_t* zm, uint64_t j,
                               const uint32_t* carries, uint32_t* q, uint32_t* value) {
  const uint64_t lo = j << lg_chunk, hi = lo + (1ull << lg_chunk) < n ? lo + (1ull << lg_chunk) : n;
  uint32_t acc[8];
  fr_load(acc, carries + j * 8);
  kzg_horner(c, lo, hi, zm, acc, q, value);
}

}  // namespace ptau
