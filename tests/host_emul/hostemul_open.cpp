// Host build of the product's Fr arithmetic (csrc/fr.cuh) and of the per-item code of the KZG10 quotient scan
// (csrc/kzg_open.cuh), for the CPU-only tests of ptau_kzg_open (tests/test_kzg_open.py).  The kernels' loops run
// serially, with the chunk length and the width of the carry block as parameters.
// TEST VEHICLE ONLY, like hostemul.cpp: libptau_b200.so never links or calls this.
#include <cstring>
#include <vector>

#include "../../kzg_setup_powersoftau_b200/csrc/kzg_open.cuh"

using namespace ptau;

static const uint32_t kR2[8] = {0xf3f29c6du, 0xc999e990u, 0x87925c23u, 0x2b6cedcbu,
                                0x7254398fu, 0x05d31496u, 0x9f59ff11u, 0x0748d9d9u};  // R^2 mod r, R = 2^256

// op 0: fr_mul(a, b), 1: fr_add(a, b), 2: fr_is_canonical(a) in out[0]
extern "C" void hostemul_fr_op(int op, const uint8_t* a8, const uint8_t* b8, uint8_t* out8) {
  uint32_t a[8], b[8], r[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  std::memcpy(a, a8, 32);
  std::memcpy(b, b8, 32);
  if (op == 0) fr_mul(r, a, b);
  if (op == 1) fr_add(r, a, b);
  if (op == 2) r[0] = fr_is_canonical(a) ? 1 : 0;
  std::memcpy(out8, r, 32);
}

// the quotient of launch_kzg_quotient with chunks of 2^lg_chunk coefficients and a carry block of 2^lg_threads
// threads; q_out: n - 1 scalars, value_out: p(z).  Returns 1 when a coefficient is >= r.
extern "C" int hostemul_kzg_quotient(const uint8_t* coeffs, size_t n, const uint8_t* z8, int lg_chunk, int lg_threads,
                                     uint8_t* q_out, uint8_t* value_out) {
  KzgZPow zp;
  uint32_t z[8];
  std::memcpy(z, z8, 32);
  fr_mul(zp.w[0], z, kR2);
  for (int s = 1; s < kKzgZPow; s++) fr_mul(zp.w[s], zp.w[s - 1], zp.w[s - 1]);
  uint32_t value[8] = {0, 0, 0, 0, 0, 0, 0, 0}, bad = 0;
  if (n) {
    std::vector<uint32_t> c(n * 8), q(n * 8);
    std::memcpy(c.data(), coeffs, n * 32);
    const uint64_t m = (n + (1ull << lg_chunk) - 1) >> lg_chunk;
    std::vector<uint32_t> sums(m * 8);
    for (uint64_t j = 0; j < m; j++) kzg_chunk_sum_item(c.data(), n, lg_chunk, zp.w[0], j, sums.data(), &bad);
    const uint64_t T = 1ull << lg_threads;
    int lg_run = 0;
    while ((1ull << (lg_threads + lg_run)) < m) lg_run++;
    std::vector<uint32_t> acc(T * 8), y(T * 8);
    for (uint64_t t = 0; t < T; t++) kzg_run_sum_item(sums.data(), m, lg_run, zp.w[lg_chunk], t, &acc[t * 8]);
    for (int s = 0; s < lg_threads; s++) {
      y = acc;
      for (uint64_t t = 0; t + (1ull << s) < T; t++)
        kzg_combine_item(&y[t * 8], &y[(t + (1ull << s)) * 8], zp.w[lg_chunk + lg_run + s], &acc[t * 8]);
    }
    const uint32_t zero[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    for (uint64_t t = 0; t < T; t++)
      kzg_run_carry_item(sums.data(), m, lg_run, zp.w[lg_chunk], t, t + 1 < T ? &acc[(t + 1) * 8] : zero);
    for (uint64_t j = 0; j < m; j++) kzg_write_item(c.data(), n, lg_chunk, zp.w[0], j, sums.data(), q.data(), value);
    std::memcpy(q_out, q.data(), (n - 1) * 32);
  }
  std::memcpy(value_out, value, 32);
  return bad ? 1 : 0;
}
