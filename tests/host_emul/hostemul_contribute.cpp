// Host build of the contribution's per-point code (csrc/contribute.cuh: scalar decompositions, signed recoding, the
// joint ladder) and of its public-key code (ChaCha20, Fq::rand, hash_to_g2), for the CPU-only tests of
// tests/test_contribute.py.  TEST VEHICLE ONLY, like hostemul.cpp: libptau_b200.so never links or calls this.
#include <cstring>

#include "../../kzg_setup_powersoftau_b200/csrc/contribute.cuh"
#include "../../kzg_setup_powersoftau_b200/csrc/layout.h"

using namespace ptau;

namespace {
// 48 big-endian bytes <-> Montgomery Fq
Fq fq_in(const uint8_t* be) {
  uint32_t w[12];
  memcpy(w, be, 48);
  return fq_to_mont(fq_from_be_words(w));
}
void fq_out(const Fq& m, uint8_t* be) {
  uint32_t w[12];
  fq_to_be_words(fq_from_mont(m), w);
  memcpy(be, w, 48);
}
}  // namespace

extern "C" {

// byte offset of response section `sec` in records of `fmt` (the offsets ptau_verify_contribution reads at)
uint64_t hostemul_section_offset(uint64_t n, int fmt, int sec) { return section_offset(n, fmt, sec); }

// k (32 bytes LE) -> k0, k1 (16 bytes LE each)
void hostemul_glv_split_g1(const uint8_t* k, uint8_t* k0, uint8_t* k1) {
  uint64_t kk[4], a[2], b[2];
  memcpy(kk, k, 32);
  glv_split_g1(kk, a, b);
  memcpy(k0, a, 16);
  memcpy(k1, b, 16);
}

// k (32 bytes LE) -> d[4] (8 bytes LE each)
void hostemul_zdigits_g2(const uint8_t* k, uint8_t* d) {
  uint64_t kk[4], dd[4];
  memcpy(kk, k, 32);
  zdigits_g2(kk, dd);
  memcpy(d, dd, 32);
}

// s (nlimbs x 8 bytes LE) -> ndig signed digits
void hostemul_recode(const uint8_t* s, int nlimbs, int8_t* e, int ndig) {
  uint64_t v[4] = {0, 0, 0, 0};
  memcpy(v, s, 8 * nlimbs);
  recode_signed4(v, nlimbs, e, ndig);
}

// [k] P for a finite point P = x || y (plain, big-endian 48-byte coordinates; G2: x.c0, x.c1, y.c0, y.c1); out the
// same layout; returns 0 for infinity, 1 otherwise
int hostemul_contrib_mul(int group, const uint8_t* pt, const uint8_t* k, uint8_t* out) {
  uint32_t kw[8];
  memcpy(kw, k, 32);
  if (group == 1) {
    Jac<Fq> r = contrib_mul(fq_in(pt), fq_in(pt + 48), kw);
    Fq x, y;
    if (!jac_to_affine_t(r, x, y)) return 0;
    fq_out(x, out);
    fq_out(y, out + 48);
    return 1;
  }
  Fq2 px, py;
  px.c0 = fq_in(pt);
  px.c1 = fq_in(pt + 48);
  py.c0 = fq_in(pt + 96);
  py.c1 = fq_in(pt + 144);
  Jac<Fq2> r = contrib_mul(px, py, kw);
  Fq2 x, y;
  if (!jac_to_affine_t(r, x, y)) return 0;
  fq_out(x.c0, out);
  fq_out(x.c1, out + 48);
  fq_out(y.c0, out + 96);
  fq_out(y.c1, out + 144);
  return 1;
}

// the first nwords of ChaChaRng::from_seed(key)
void hostemul_chacha(const uint32_t* key, uint32_t* out, int nwords) {
  ChaChaRng rng(key);
  for (int i = 0; i < nwords; i++) out[i] = rng.next_u32();
}

// hash_to_g2(digest) as a zcash uncompressed record; stats[0] = Fq::rand rejections, stats[1] = x without a root
void hostemul_hash_to_g2(const uint8_t* digest, uint8_t* out192, int* stats) {
  Fq2 x, y;
  stats[0] = stats[1] = 0;
  hash_to_g2(digest, x, y, stats);
  zcash_g2_uncompressed(x, y, out192);
}

}  // extern "C"
