// Byte layouts of the records and files the library reads and writes: record sizes, the section table of a
// `powersoftau` response and the `kzg_setup` layouts of preprocess-kgz and preprocess-fastkgz
// (preprocess-kgz.rs:128-200, preprocess-fastkgz.rs:129-214).  Host code only.
#pragma once
#include <stdint.h>

#include <array>

#include "../../include/ptau_b200.h"

namespace ptau {

// ARK_MONT_LIMBS records, the form points take on the device: x, y in Montgomery limbs, then the infinity word and
// padding.  The word after a record is where the MSM kernels report a scalar >= r.
constexpr int kMontG1 = 104, kMontG2 = 200;

// bytes of one record, 0 for an unknown (group, format)
constexpr int rec_size(int group, int fmt) {
  if (group != PTAU_G1 && group != PTAU_G2) return 0;
  const bool g1 = group == PTAU_G1;
  switch (fmt) {
    case PTAU_FMT_ZCASH_UNCOMPRESSED:
    case PTAU_FMT_ARK_UNCOMPRESSED:
      return g1 ? 96 : 192;
    case PTAU_FMT_ZCASH_COMPRESSED:
      return g1 ? 48 : 96;
    case PTAU_FMT_ARK_MONT_LIMBS:
      return g1 ? kMontG1 : kMontG2;
  }
  return 0;
}

struct Section {
  int group;
  uint64_t count;
};

// A `powersoftau` response is a 64-byte challenge hash, these sections in compressed records, and the contributor's
// public key; `powersoftau_uncompressed` is the same sections in uncompressed records and nothing else.
constexpr uint64_t kResponseHash = 64, kResponsePubkey = 3 * 192 + 6 * 96;
inline std::array<Section, 5> response_sections(uint64_t n) {
  return {{
      {PTAU_G1, 2 * n - 1},  // tau_g1
      {PTAU_G2, n},          // tau_g2
      {PTAU_G1, n},          // alpha_g1
      {PTAU_G1, n},          // beta_g1
      {PTAU_G2, 1},          // beta_g2
  }};
}
inline uint64_t response_bytes(uint64_t n, int fmt) {
  uint64_t b = 0;
  for (const Section& s : response_sections(n)) b += s.count * rec_size(s.group, fmt);
  return b;
}
// byte offset of section `sec` (0..4) within the sections of a response / accumulator in records of `fmt`
inline uint64_t section_offset(uint64_t n, int fmt, int sec) {
  const auto secs = response_sections(n);
  uint64_t b = 0;
  for (int s = 0; s < sec; s++) b += secs[s].count * rec_size(secs[s].group, fmt);
  return b;
}

// `kzg_setup` in ark uncompressed records: every G1 record, then every G2 record.  Positions are record indices
// within their group; g1() and g2() turn them into byte offsets.
//   G1: powers_of_g (2n - 1) | powers_of_gamma_g (n) | kgz: the VerifierKey's g, gamma_g
//   G2: the VerifierKey's h, beta_h | fastkgz: powers_of_h (n)
struct SetupLayout {
  uint64_t n_g1, n_g2;
  uint64_t gamma_g;      // powers_of_gamma_g[0]; powers_of_g start at 0
  uint64_t vk_g;         // kgz: g, then gamma_g
  uint64_t powers_of_h;  // fastkgz: powers_of_h[0] (G2); h and beta_h are G2 records 0 and 1
  uint64_t g1(uint64_t i) const { return i * rec_size(PTAU_G1, PTAU_FMT_ARK_UNCOMPRESSED); }
  uint64_t g2(uint64_t i) const { return g1(n_g1) + i * rec_size(PTAU_G2, PTAU_FMT_ARK_UNCOMPRESSED); }
  uint64_t bytes() const { return g2(n_g2); }
};
inline SetupLayout setup_layout(int variant, uint64_t n) {
  const bool fast = variant == PTAU_VARIANT_FASTKGZ;
  return {3 * n - 1 + (fast ? 0 : 2), fast ? n + 2 : 2, 2 * n - 1, 3 * n - 1, 2};
}

}  // namespace ptau
