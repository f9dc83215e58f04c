// BLS12-381 scalar field Fr on the host, 4 x u64 limbs: the Montgomery arithmetic that prepares the scalars of the
// synthetic generator and of a contribution (capi.cu, contribute.cu) and the host quotient recurrence.  Host code only.
#pragma once
#include <stdint.h>
#include <string.h>

namespace ptau {

typedef unsigned __int128 u128;
struct Fr {
  uint64_t l[4];
};
constexpr uint64_t FR_MOD[4] = {0xffffffff00000001ull, 0x53bda402fffe5bfeull, 0x3339d80809a1d805ull,
                                0x73eda753299d7d48ull};
constexpr uint64_t FR_INV = 0xfffffffeffffffffull;  // -r^-1 mod 2^64
// R^2 mod r, R = 2^256
constexpr uint64_t FR_R2[4] = {0xc999e990f3f29c6dull, 0x2b6cedcb87925c23ull, 0x05d314967254398full,
                               0x0748d9d99f59ff11ull};

inline bool fr_ge_mod(const uint64_t* a) {
  for (int i = 3; i >= 0; --i) {
    if (a[i] > FR_MOD[i]) return true;
    if (a[i] < FR_MOD[i]) return false;
  }
  return true;
}
inline Fr fr_mont_mul(const Fr& a, const Fr& b) {
  uint64_t t[6] = {0, 0, 0, 0, 0, 0};
  for (int i = 0; i < 4; i++) {
    u128 c = 0;
    for (int j = 0; j < 4; j++) {
      c += (u128)a.l[j] * b.l[i] + t[j];
      t[j] = (uint64_t)c;
      c >>= 64;
    }
    c += t[4];
    t[4] = (uint64_t)c;
    t[5] = (uint64_t)(c >> 64);
    uint64_t m = t[0] * FR_INV;
    c = (u128)m * FR_MOD[0] + t[0];
    c >>= 64;
    for (int j = 1; j < 4; j++) {
      c += (u128)m * FR_MOD[j] + t[j];
      t[j - 1] = (uint64_t)c;
      c >>= 64;
    }
    c += t[4];
    t[3] = (uint64_t)c;
    t[4] = t[5] + (uint64_t)(c >> 64);
  }
  Fr r;
  memcpy(r.l, t, 32);
  if (t[4] || fr_ge_mod(r.l)) {
    u128 bw = 0;
    for (int i = 0; i < 4; i++) {
      u128 d = (u128)r.l[i] - FR_MOD[i] - (uint64_t)bw;
      r.l[i] = (uint64_t)d;
      bw = (d >> 64) & 1;
    }
  }
  return r;
}
inline Fr fr_from_le32(const uint8_t* b) {
  Fr r;
  memcpy(r.l, b, 32);
  return r;
}
inline Fr fr_to_mont(const Fr& a) {
  Fr r2;
  memcpy(r2.l, FR_R2, 32);
  return fr_mont_mul(a, r2);
}
// a + b mod r, both canonical
inline Fr fr_add_mod(const Fr& a, const Fr& b) {
  Fr r;
  u128 c = 0;
  for (int i = 0; i < 4; i++) {
    c += (u128)a.l[i] + b.l[i];
    r.l[i] = (uint64_t)c;
    c >>= 64;
  }
  if (c || fr_ge_mod(r.l)) {
    u128 bw = 0;
    for (int i = 0; i < 4; i++) {
      u128 d = (u128)r.l[i] - FR_MOD[i] - (uint64_t)bw;
      r.l[i] = (uint64_t)d;
      bw = (d >> 64) & 1;
    }
  }
  return r;
}

}  // namespace ptau
