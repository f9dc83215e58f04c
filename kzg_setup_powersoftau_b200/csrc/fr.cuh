// BLS12-381 scalar field Fr, 8 x u32 limbs: the Montgomery product (R = 2^256) of the synthetic generator
// (kernels.cu) and what the KZG10 quotient scan (kzg_open.cu) adds to it: addition, the canonical check and 32-byte
// little-endian load / store; the coset openings (kzg_coset.cu) add subtraction and powers from a table of squares.
//
// Scalars in memory stay canonical (< r), not Montgomery: fr_mul(a, bR) = a b mod r, so a canonical value times a
// constant kept in Montgomery form (z R mod r, prepared once on the host) is again canonical.
//
// Compiled for the host too (tests/host_emul/hostemul_open.cpp), with K_FR_MOD as an ordinary array.
#pragma once
#include <stdint.h>

namespace ptau {

#if defined(__CUDACC__)
__constant__ uint32_t K_FR_MOD[8] = {0x00000001u, 0xffffffffu, 0xfffe5bfeu, 0x53bda402u,
                                     0x09a1d805u, 0x3339d808u, 0x299d7d48u, 0x73eda753u};
#define PTAU_FR_MUL static __device__ __noinline__
#define PTAU_FR_HD static __device__ __forceinline__
#else
static const uint32_t K_FR_MOD[8] = {0x00000001u, 0xffffffffu, 0xfffe5bfeu, 0x53bda402u,
                                     0x09a1d805u, 0x3339d808u, 0x299d7d48u, 0x73eda753u};
#define PTAU_FR_MUL static inline
#define PTAU_FR_HD static inline
#endif
#define PTAU_FR_M0 0xffffffffu  // -r^-1 mod 2^32

// Montgomery product in Fr (R = 2^256), plain 64-bit arithmetic: a few dozen calls per point
PTAU_FR_MUL void fr_mul(uint32_t* r, const uint32_t* a, const uint32_t* b) {
  uint32_t t[10];
#pragma unroll
  for (int i = 0; i < 10; i++) t[i] = 0;
#pragma unroll 1
  for (int i = 0; i < 8; i++) {
    uint64_t c = 0;
#pragma unroll
    for (int j = 0; j < 8; j++) {
      c += (uint64_t)a[j] * b[i] + t[j];
      t[j] = (uint32_t)c;
      c >>= 32;
    }
    c += t[8];
    t[8] = (uint32_t)c;
    t[9] = (uint32_t)(c >> 32);
    uint32_t m = t[0] * PTAU_FR_M0;
    c = (uint64_t)m * K_FR_MOD[0] + t[0];
    c >>= 32;
#pragma unroll
    for (int j = 1; j < 8; j++) {
      c += (uint64_t)m * K_FR_MOD[j] + t[j];
      t[j - 1] = (uint32_t)c;
      c >>= 32;
    }
    c += t[8];
    t[7] = (uint32_t)c;
    t[8] = t[9] + (uint32_t)(c >> 32);
  }
  // conditional subtraction
  uint32_t d[8];
  uint32_t bw = 0;
#pragma unroll
  for (int i = 0; i < 8; i++) {
    uint64_t x = (uint64_t)t[i] - K_FR_MOD[i] - bw;
    d[i] = (uint32_t)x;
    bw = (uint32_t)(x >> 63);
  }
  bool ge = t[8] != 0 || bw == 0;
#pragma unroll
  for (int i = 0; i < 8; i++) r[i] = ge ? d[i] : t[i];
}

// r = a + b mod r for canonical a, b (r may alias either)
PTAU_FR_HD void fr_add(uint32_t* r, const uint32_t* a, const uint32_t* b) {
  uint32_t s[8], d[8];
  uint64_t c = 0;
#pragma unroll
  for (int i = 0; i < 8; i++) {
    c += (uint64_t)a[i] + b[i];
    s[i] = (uint32_t)c;
    c >>= 32;
  }
  uint32_t bw = 0;
#pragma unroll
  for (int i = 0; i < 8; i++) {
    uint64_t x = (uint64_t)s[i] - K_FR_MOD[i] - bw;
    d[i] = (uint32_t)x;
    bw = (uint32_t)(x >> 63);
  }
  // a + b < 2r < 2^256: no carry out of the top limb, so a + b >= r exactly when the subtraction does not borrow
  const bool ge = bw == 0;
#pragma unroll
  for (int i = 0; i < 8; i++) r[i] = ge ? d[i] : s[i];
}

// r = a - b mod r for canonical a, b (r may alias either)
PTAU_FR_HD void fr_sub(uint32_t* r, const uint32_t* a, const uint32_t* b) {
  uint32_t d[8], s[8];
  uint32_t bw = 0;
#pragma unroll
  for (int i = 0; i < 8; i++) {
    uint64_t x = (uint64_t)a[i] - b[i] - bw;
    d[i] = (uint32_t)x;
    bw = (uint32_t)(x >> 63);
  }
  // a < b: the difference wrapped by 2^256; adding r brings it back into [0, r)
  uint64_t c = 0;
#pragma unroll
  for (int i = 0; i < 8; i++) {
    c += (uint64_t)d[i] + K_FR_MOD[i];
    s[i] = (uint32_t)c;
    c >>= 32;
  }
#pragma unroll
  for (int i = 0; i < 8; i++) r[i] = bw ? s[i] : d[i];
}

// R mod r: 1 in Montgomery form
PTAU_FR_HD void fr_mont_one(uint32_t* a) {
  a[0] = 0xfffffffeu, a[1] = 0x00000001u, a[2] = 0x00034802u, a[3] = 0x5884b7fau;
  a[4] = 0xecbc4ff5u, a[5] = 0x998c4fefu, a[6] = 0xacc5056fu, a[7] = 0x1824b159u;
}

// out = prod of tbl[s] over the set bits s < bits of x, in Montgomery form (tbl[s] = w^(2^s) R gives w^x R)
PTAU_FR_HD void fr_pow_bits(uint32_t* out, const uint32_t (*tbl)[8], uint64_t x, int bits) {
  fr_mont_one(out);
  for (int s = 0; s < bits; s++)
    if ((x >> s) & 1) fr_mul(out, out, tbl[s]);
}

// a < r
PTAU_FR_HD bool fr_is_canonical(const uint32_t* a) {
  uint32_t bw = 0;
#pragma unroll
  for (int i = 0; i < 8; i++) bw = (uint32_t)(((uint64_t)a[i] - K_FR_MOD[i] - bw) >> 63);
  return bw != 0;
}

// one 32-byte little-endian scalar; p is 16-byte aligned on the device
PTAU_FR_HD void fr_load(uint32_t* a, const uint32_t* p) {
#if defined(__CUDA_ARCH__)
  const uint4 lo = reinterpret_cast<const uint4*>(p)[0], hi = reinterpret_cast<const uint4*>(p)[1];
  a[0] = lo.x, a[1] = lo.y, a[2] = lo.z, a[3] = lo.w, a[4] = hi.x, a[5] = hi.y, a[6] = hi.z, a[7] = hi.w;
#else
  for (int i = 0; i < 8; i++) a[i] = p[i];
#endif
}
PTAU_FR_HD void fr_store(uint32_t* p, const uint32_t* a) {
#if defined(__CUDA_ARCH__)
  reinterpret_cast<uint4*>(p)[0] = make_uint4(a[0], a[1], a[2], a[3]);
  reinterpret_cast<uint4*>(p)[1] = make_uint4(a[4], a[5], a[6], a[7]);
#else
  for (int i = 0; i < 8; i++) p[i] = a[i];
#endif
}

}  // namespace ptau
