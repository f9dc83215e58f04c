// Host build of the product's G2 bucket MSM item code (csrc/msm_g2.cuh) and of the coefficient / digest code of
// csrc/blake2b.h, for the CPU-only tests of ptau_verify_powers and ptau_msm_g2 (tests/test_verify_powers.py).
// TEST VEHICLE ONLY, like hostemul.cpp: libptau_b200.so never links or calls this.
#include <cstring>
#include <string>
#include <vector>

#include "../../kzg_setup_powersoftau_b200/csrc/blake2b.h"
#include "../../kzg_setup_powersoftau_b200/csrc/msm_g2.cuh"

using namespace ptau;

// the G2 bucket MSM with the product's per-item code (csrc/msm_g2.cuh), the kernels' loops run serially
extern "C" void hostemul_msm_g2(const uint8_t* pts8, const uint8_t* sc8, size_t n, uint8_t* out200) {
  std::vector<uint32_t> pts(n * 50 + 1), sc(n * 8 + 1);
  std::memcpy(pts.data(), pts8, n * 200);
  std::memcpy(sc.data(), sc8, n * 32);
  const MsmGeom g = msm_geometry(n);
  const uint32_t m = (uint32_t)g.a * g.NB + (uint32_t)(g.W - g.a) * (g.NB >> 1);
  std::vector<uint32_t> cnt(m + 1, 0), off(m + 1, 0), cur(m + 1, 0), entries(n * (size_t)g.W + 1);
  auto digits = [&](bool scatter) {
    for (size_t i = 0; i < n; i++) {
      if (pts[i * 50 + 48] & 0xffu) continue;
      uint32_t carry = 0, base = 0;
      int bit = 0;
      for (int w = 0; w < g.W; w++) {
        const int cw = w < g.a ? g.c : g.c - 1;
        int d = msm_digit(&sc[i * 8], bit, cw, carry);
        if (d != 0) {
          uint32_t b = base + (uint32_t)(d < 0 ? -d : d) - 1u;
          if (scatter) entries[cur[b]++] = (uint32_t)i | (d < 0 ? 0x80000000u : 0u);
          else cnt[b]++;
        }
        bit += cw;
        base += 1u << (cw - 1);
      }
    }
  };
  digits(false);
  for (uint32_t b = 0; b < m; b++) off[b + 1] = off[b] + cnt[b];
  cur = off;
  digits(true);
  std::vector<uint32_t> buckets((size_t)m * 72), segs(((size_t)m >> g.lgL) * 72), wsum((size_t)g.W * 72);
  for (uint32_t b = 0; b < m; b++) msm_g2_bucket_item(pts.data(), entries.data(), off.data(), b, buckets.data());
  const uint32_t nseg = m >> g.lgL;
  for (uint32_t t = 0; t < nseg; t++) msm_g2_segment_item(buckets.data(), g, t, segs.data());
  for (int w = 0; w < g.W; w++) {
    const uint32_t first = msm_bucket_base(g, w) >> g.lgL, count = (w < g.a ? g.NB : g.NB >> 1) >> g.lgL;
    Jac<Fq2> acc = jac2_infinity();
    for (uint32_t i = 0; i < count; i++) {
      Jac<Fq2> q = jac2_load(segs.data() + (size_t)(first + i) * 72);
      jac_add_complete_t(acc, q);
    }
    msm_g2_window_weight(acc, g, w);
    jac2_store(wsum.data() + (size_t)w * 72, acc);
  }
  uint32_t out[50];
  msm_g2_finish_item(wsum.data(), g.W, out);
  std::memcpy(out200, out, 200);
}

// coefficients rho_{k,i} of ptau_verify_powers (csrc/blake2b.h): n scalars of 32 bytes for i = first .. first + n - 1
extern "C" void hostemul_ratio_coeffs(const uint8_t* seed32, uint32_t k, uint64_t first, size_t n, uint8_t* out) {
  uint64_t h[8];
  blake2b_keyed_start(h, seed32, 32, 16);
  for (size_t j = 0; j < n; j++) {
    uint32_t sc[8];
    ratio_coeff(h, k, first + j, sc);
    std::memcpy(out + j * 32, sc, 32);
  }
}

// the streaming unkeyed BLAKE2b-512 of blake2b.h (the file digest), as 128 hex characters + NUL
extern "C" void hostemul_blake2b_hex(const uint8_t* data, size_t len, char* out129) {
  Blake2b b;
  b.update(data, len);
  std::string hx = b.hexdigest();
  std::memcpy(out129, hx.c_str(), 129);
}
