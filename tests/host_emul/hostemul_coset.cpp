// Host build of the coset-opening items (csrc/kzg_coset.cuh) and of the Fr helpers they add to csrc/fr.cuh, for the
// CPU-only tests of ptau_kzg_open_cosets / ptau_kzg_check_cosets (tests/test_kzg_cosets.py).  The kernels' loops run
// serially, with the chunk length and the width of the carry block as parameters.
// TEST VEHICLE ONLY, like hostemul.cpp: libptau_b200.so never links or calls this.
#include <cstring>
#include <vector>

#include "../../kzg_setup_powersoftau_b200/csrc/kzg_coset.cuh"

using namespace ptau;

static const uint32_t kR2[8] = {0xf3f29c6du, 0xc999e990u, 0x87925c23u, 0x2b6cedcbu,
                                0x7254398fu, 0x05d31496u, 0x9f59ff11u, 0x0748d9d9u};  // R^2 mod r, R = 2^256
static const uint32_t kOne[8] = {1, 0, 0, 0, 0, 0, 0, 0};

// t[s] = a^(2^s) R for s < count, a canonical
static void square_table(const uint32_t* a, uint32_t (*t)[8], int count) {
  if (!count) return;
  fr_mul(t[0], a, kR2);
  for (int s = 1; s < count; s++) fr_mul(t[s], t[s - 1], t[s - 1]);
}

// op 0: fr_sub(a, b); 1: fr_mont_one(); 2: a^x by fr_pow_bits (x = the low 64 bits of b, 64 table rows), canonical;
// 3: fr_mul(a, b); 4: fr_add(a, b); 5: fr_is_canonical(a) in out[0]
extern "C" void hostemul_coset_fr_op(int op, const uint8_t* a8, const uint8_t* b8, uint8_t* out8) {
  uint32_t a[8], b[8], r[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  std::memcpy(a, a8, 32);
  std::memcpy(b, b8, 32);
  if (op == 0) fr_sub(r, a, b);
  if (op == 3) fr_mul(r, a, b);
  if (op == 4) fr_add(r, a, b);
  if (op == 5) r[0] = fr_is_canonical(a) ? 1 : 0;
  if (op == 1) fr_mont_one(r);
  if (op == 2) {
    uint32_t t[64][8], w[8];
    square_table(a, t, 64);
    fr_pow_bits(w, t, (uint64_t)b[0] | ((uint64_t)b[1] << 32), 64);
    fr_mul(r, w, kOne);
  }
  std::memcpy(out8, r, 32);
}

// launch_coset_quotient with chunks of 2^lg_chunk rows and a carry block of 2^lg_threads threads: q_out n - k
// scalars (n > k), rem_out k scalars.  Returns 1 when a coefficient is >= r.
extern "C" int hostemul_coset_quotient(const uint8_t* coeffs, size_t n, int lg_k, const uint8_t* c8, int lg_chunk,
                                       int lg_threads, uint8_t* q_out, uint8_t* rem_out) {
  const uint64_t k = 1ull << lg_k;
  KzgZPow cp;
  uint32_t c[8];
  std::memcpy(c, c8, 32);
  square_table(c, cp.w, kKzgZPow);
  std::vector<uint32_t> rem(k * 8, 0);
  uint32_t bad = 0;
  if (n) {
    std::vector<uint32_t> p(n * 8), q((n > k ? n - k : 1) * 8);
    std::memcpy(p.data(), coeffs, n * 32);
    const uint64_t rows = (n + k - 1) >> lg_k, mc = (rows + (1ull << lg_chunk) - 1) >> lg_chunk, items = mc << lg_k;
    std::vector<uint32_t> sums(items * 8);
    for (uint64_t id = 0; id < items; id++)
      coset_chunk_sum_item(p.data(), n, lg_k, lg_chunk, mc, cp.w[0], id, sums.data(), &bad);
    int lg_seg, lg_run;
    coset_carry_shape(mc, lg_threads, &lg_seg, &lg_run);
    const uint64_t T = 1ull << lg_seg;
    const uint32_t zero[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    for (uint64_t j = 0; j < k; j++) {  // one segment of the carry block per chain
      uint32_t* s = sums.data() + j * mc * 8;
      std::vector<uint32_t> acc(T * 8), y(T * 8);
      for (uint64_t t = 0; t < T; t++) kzg_run_sum_item(s, mc, lg_run, cp.w[lg_chunk], t, &acc[t * 8]);
      for (int st = 0; st < lg_seg; st++) {
        y = acc;
        for (uint64_t t = 0; t + (1ull << st) < T; t++)
          kzg_combine_item(&y[t * 8], &y[(t + (1ull << st)) * 8], cp.w[lg_chunk + lg_run + st], &acc[t * 8]);
      }
      for (uint64_t t = 0; t < T; t++)
        kzg_run_carry_item(s, mc, lg_run, cp.w[lg_chunk], t, t + 1 < T ? &acc[(t + 1) * 8] : zero);
    }
    for (uint64_t id = 0; id < items; id++)
      coset_write_item(p.data(), n, lg_k, lg_chunk, mc, cp.w[0], id, sums.data(), q.data(), rem.data());
    if (n > k) std::memcpy(q_out, q.data(), (n - k) * 32);
  }
  std::memcpy(rem_out, rem.data(), k * 32);
  return bad ? 1 : 0;
}

// launch_ntt_twiddles + launch_ntt for `items` items of k scalars: out[i] = NTT_k over w (a canonical root of order
// k) of in[i][j] h_i^j; h: items canonical shifts, or null
extern "C" void hostemul_ntt(const uint8_t* in8, size_t items, int lg_k, const uint8_t* w8, const uint8_t* h8,
                             uint8_t* out8) {
  const uint64_t k = 1ull << lg_k;
  uint32_t w[8], wp[kCosetMaxLgK][8];
  std::memcpy(w, w8, 32);
  square_table(w, wp, lg_k);
  std::vector<uint32_t> tw((k / 2 + 1) * 8), in(items * k * 8), out(items * k * 8), hp(items * kCosetMaxLgK * 8);
  for (uint64_t i = 0; i < k / 2; i++) fr_pow_bits(&tw[i * 8], wp, i, lg_k);
  std::memcpy(in.data(), in8, items * k * 32);
  for (size_t it = 0; it < items; it++) {
    uint32_t (*t)[8] = (uint32_t(*)[8]) & hp[it * kCosetMaxLgK * 8];
    if (h8) {
      uint32_t h[8];
      std::memcpy(h, h8 + it * 32, 32);
      square_table(h, t, kCosetMaxLgK);
    }
    for (uint64_t j = 0; j < k; j++) ntt_permute_item(&in[it * k * 8], &out[it * k * 8], lg_k, h8 ? t : nullptr, j);
    for (int s = 0; s < lg_k; s++)
      for (uint64_t i = 0; i < k / 2; i++) ntt_butterfly_item(&out[it * k * 8], lg_k, s, tw.data(), i);
  }
  std::memcpy(out8, out.data(), items * k * 32);
}
