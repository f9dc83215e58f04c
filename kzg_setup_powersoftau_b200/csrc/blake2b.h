// BLAKE2b -- written from RFC 7693.  The compression function is host- and device-callable: the streaming
// unkeyed BLAKE2b-512 below (host) is the digest check of the `powersoftau` / `kzg_setup` files that the
// reference does with blake2b_simd (/root/reference/src/bin/preprocess-kgz.rs:33-36,
// /root/reference/src/lib.rs:128-131); verify.cu derives the coefficients of ptau_verify_powers with one
// compression per coefficient on the device.
#pragma once
#include <stddef.h>
#include <stdint.h>
#include <string.h>

#include <string>

#ifdef __CUDACC__
#define PTAU_B2_HD __host__ __device__ __forceinline__
#else
#define PTAU_B2_HD inline
#endif
// the tables are static on the host (the file digest calls the compression once per 128 bytes) and plain locals on the
// device, where the fully unrolled rounds turn every index into a constant
#ifdef __CUDA_ARCH__
#define PTAU_B2_STATIC
#else
#define PTAU_B2_STATIC static
#endif

namespace ptau {

PTAU_B2_HD uint64_t blake2b_rotr(uint64_t x, int n) { return (x >> n) | (x << (64 - n)); }

// h[0..8) = the chaining value (updated in place); m = one 128-byte block as 16 little-endian words;
// (t0, t1) = the byte counter including this block; last = final block
PTAU_B2_HD void blake2b_compress(uint64_t* h, const uint64_t* m, uint64_t t0, uint64_t t1, bool last) {
  PTAU_B2_STATIC const uint8_t sigma[12][16] = {
      {0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15}, {14, 10, 4, 8, 9, 15, 13, 6, 1, 12, 0, 2, 11, 7, 5, 3},
      {11, 8, 12, 0, 5, 2, 15, 13, 10, 14, 3, 6, 7, 1, 9, 4}, {7, 9, 3, 1, 13, 12, 11, 14, 2, 6, 5, 10, 4, 0, 15, 8},
      {9, 0, 5, 7, 2, 4, 10, 15, 14, 1, 11, 12, 6, 8, 3, 13}, {2, 12, 6, 10, 0, 11, 8, 3, 4, 13, 7, 5, 15, 14, 1, 9},
      {12, 5, 1, 15, 14, 13, 4, 10, 0, 7, 6, 3, 9, 2, 8, 11}, {13, 11, 7, 14, 12, 1, 3, 9, 5, 0, 15, 4, 8, 6, 2, 10},
      {6, 15, 14, 9, 11, 3, 0, 8, 12, 2, 13, 7, 1, 4, 10, 5}, {10, 2, 8, 4, 7, 6, 1, 5, 15, 11, 9, 14, 3, 12, 13, 0},
      {0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15}, {14, 10, 4, 8, 9, 15, 13, 6, 1, 12, 0, 2, 11, 7, 5, 3}};
  PTAU_B2_STATIC const uint64_t iv[8] = {0x6a09e667f3bcc908ull, 0xbb67ae8584caa73bull, 0x3c6ef372fe94f82bull,
                                         0xa54ff53a5f1d36f1ull, 0x510e527fade682d1ull, 0x9b05688c2b3e6c1full,
                                         0x1f83d9abfb41bd6bull, 0x5be0cd19137e2179ull};
  uint64_t v[16];
#pragma unroll
  for (int i = 0; i < 8; i++) {
    v[i] = h[i];
    v[i + 8] = iv[i];
  }
  v[12] ^= t0;
  v[13] ^= t1;
  if (last) v[14] = ~v[14];
#define B2G(a, b, c, d, x, y)            \
  v[a] = v[a] + v[b] + (x);              \
  v[d] = blake2b_rotr(v[d] ^ v[a], 32);  \
  v[c] = v[c] + v[d];                    \
  v[b] = blake2b_rotr(v[b] ^ v[c], 24);  \
  v[a] = v[a] + v[b] + (y);              \
  v[d] = blake2b_rotr(v[d] ^ v[a], 16);  \
  v[c] = v[c] + v[d];                    \
  v[b] = blake2b_rotr(v[b] ^ v[c], 63);
#pragma unroll
  for (int r = 0; r < 12; r++) {
    const uint8_t* s = sigma[r];
    B2G(0, 4, 8, 12, m[s[0]], m[s[1]]);
    B2G(1, 5, 9, 13, m[s[2]], m[s[3]]);
    B2G(2, 6, 10, 14, m[s[4]], m[s[5]]);
    B2G(3, 7, 11, 15, m[s[6]], m[s[7]]);
    B2G(0, 5, 10, 15, m[s[8]], m[s[9]]);
    B2G(1, 6, 11, 12, m[s[10]], m[s[11]]);
    B2G(2, 7, 8, 13, m[s[12]], m[s[13]]);
    B2G(3, 4, 9, 14, m[s[14]], m[s[15]]);
  }
#undef B2G
#pragma unroll
  for (int i = 0; i < 8; i++) h[i] ^= v[i] ^ v[i + 8];
}

// Chaining value of BLAKE2b with digest length `outlen` keyed with key[0..keylen) (keylen 1..64) after its first
// block, which holds only the key: what every message of that key starts from
PTAU_B2_HD void blake2b_keyed_start(uint64_t* h, const uint8_t* key, int keylen, int outlen) {
  const uint64_t iv[8] = {0x6a09e667f3bcc908ull, 0xbb67ae8584caa73bull, 0x3c6ef372fe94f82bull, 0xa54ff53a5f1d36f1ull,
                          0x510e527fade682d1ull, 0x9b05688c2b3e6c1full, 0x1f83d9abfb41bd6bull, 0x5be0cd19137e2179ull};
  for (int i = 0; i < 8; i++) h[i] = iv[i];
  h[0] ^= 0x01010000ull ^ ((uint64_t)keylen << 8) ^ (uint64_t)outlen;
  uint64_t m[16] = {0};
  for (int i = 0; i < keylen; i++) m[i >> 3] |= (uint64_t)key[i] << (8 * (i & 7));
  blake2b_compress(h, m, 128, 0, false);
}

// Coefficient rho_{k,i} of ptau_verify_powers as 8 little-endian u32 words:
//   BLAKE2b(key = seed, digest 16 bytes) of the 9 bytes  k || i (u64 little-endian),  read little-endian, low 127 bits.
// h_key: blake2b_keyed_start(seed, 32, 16).  One compression: the 9-byte message is the second and last block.
PTAU_B2_HD void ratio_coeff(const uint64_t* h_key, uint32_t k, uint64_t i, uint32_t* out) {
  uint64_t h[8], m[16];
#pragma unroll
  for (int j = 0; j < 8; j++) h[j] = h_key[j];
#pragma unroll
  for (int j = 0; j < 16; j++) m[j] = 0;
  m[0] = (uint64_t)(k & 0xffu) | (i << 8);
  m[1] = i >> 56;
  blake2b_compress(h, m, 128 + 9, 0, true);
  out[0] = (uint32_t)h[0];
  out[1] = (uint32_t)(h[0] >> 32);
  out[2] = (uint32_t)h[1];
  out[3] = (uint32_t)(h[1] >> 32) & 0x7fffffffu;
  out[4] = out[5] = out[6] = out[7] = 0;
}

class Blake2b {
 public:
  Blake2b() {
    static const uint64_t iv[8] = {0x6a09e667f3bcc908ull, 0xbb67ae8584caa73bull, 0x3c6ef372fe94f82bull,
                                   0xa54ff53a5f1d36f1ull, 0x510e527fade682d1ull, 0x9b05688c2b3e6c1full,
                                   0x1f83d9abfb41bd6bull, 0x5be0cd19137e2179ull};
    memcpy(h_, iv, sizeof(h_));
    h_[0] ^= 0x01010000ull ^ 64ull;  // digest length 64, no key, fanout = depth = 1
    t0_ = t1_ = 0;
    fill_ = 0;
  }
  void update(const void* data, size_t len) {
    const uint8_t* p = (const uint8_t*)data;
    while (len) {
      if (fill_ == 128) {  // buffer full and more input follows: not the last block
        bump(128);
        compress(false);
        fill_ = 0;
      }
      size_t take = 128 - fill_;
      if (take > len) take = len;
      memcpy(buf_ + fill_, p, take);
      fill_ += take;
      p += take;
      len -= take;
    }
  }
  std::string hexdigest() {
    bump(fill_);
    memset(buf_ + fill_, 0, 128 - fill_);
    compress(true);
    static const char* hx = "0123456789abcdef";
    std::string s;
    for (int i = 0; i < 64; i++) {
      uint8_t b = (uint8_t)(h_[i / 8] >> (8 * (i % 8)));
      s.push_back(hx[b >> 4]);
      s.push_back(hx[b & 15]);
    }
    return s;
  }

 private:
  uint64_t h_[8], t0_, t1_;
  uint8_t buf_[128];
  size_t fill_;
  void bump(uint64_t n) {
    t0_ += n;
    if (t0_ < n) t1_++;
  }
  void compress(bool last) {
    uint64_t m[16];
    memcpy(m, buf_, 128);  // little-endian host
    blake2b_compress(h_, m, t0_, t1_, last);
  }
};

}  // namespace ptau
