/* cpu_ref.c -- plain-C restatement of the CPU algorithms the reference stack runs
 * for the Powers-of-Tau -> arkworks path.  TEST INFRASTRUCTURE + CPU BASELINE ONLY:
 * nothing in the product (libptau_b200.so / kzg_setup_powersoftau_b200) links,
 * loads or calls this file.  Used by tests/ (as a second oracle, cross-checked
 * against oracle/ptau_oracle.py) and by bench.py's cpu_baseline / --impl reference
 * legs (kind "port": the Rust reference cannot be built here -- no rustc, crates
 * not vendored, no network).
 *
 * PARITY UNPINNED BY THE REFERENCE (see oracle/ptau_oracle.py header): pinned
 * instead on published BLS12-381 generator encodings and known-tau ground truth.
 *
 * Algorithms follow what the reference executes, not what the GPU executes:
 *   - Fq: 6 x u64 Montgomery (ark-ff 0.2 Fp384 / pairing 0.14.2 Fq), no asm
 *     (Cargo.toml:18-24 builds ark-* with default-features = false)
 *   - subgroup check = multiplication by r, Jacobian double + mixed add
 *     (ark-ec 0.2 is_in_correct_subgroup_assuming_on_curve; src/lib.rs:52,78)
 *   - Fq sqrt a^((p+1)/4); Fq2 sqrt Algorithm 9 of eprint 2012/685
 *     (pairing 0.14.2; reached from preprocess-kgz.rs:105-109)
 *   - zcash BE encodings / ark LE encodings with SWFlags (src/lib.rs:41-80,
 *     preprocess-kgz.rs:188-194)
 *   - threads: contiguous index ranges, like powersoftau's crossbeam chunks.
 */
#include <pthread.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

typedef unsigned __int128 u128;
typedef struct { uint64_t l[6]; } fq;
typedef struct { fq c0, c1; } fq2;

static const uint64_t PM[6] = {0xb9feffffffffaaabull, 0x1eabfffeb153ffffull, 0x6730d2a0f6b0f624ull,
                               0x64774b84f38512bfull, 0x4b1ba7b6434bacd7ull, 0x1a0111ea397fe69aull};
static const uint64_t PINV = 0x89f3fffcfffcfffdull; /* -p^-1 mod 2^64 */
static const fq FQ_ONE = {{0x760900000002fffdull, 0xebf4000bc40c0002ull, 0x5f48985753c758baull,
                           0x77ce585370525745ull, 0x5c071a97a256ec6dull, 0x15f65ec3fa80e493ull}};
static const fq FQ_R2 = {{0xf4df1f341c341746ull, 0x0a76e6a609d104f1ull, 0x8de5476c4c95b6d5ull,
                          0x67eb88a9939d83c0ull, 0x9a793e85b519952dull, 0x11988fe592cae3aaull}};
static const uint64_t R_ORDER[4] = {0xffffffff00000001ull, 0x53bda402fffe5bfeull, 0x3339d80809a1d805ull,
                                    0x73eda753299d7d48ull};

/* ---------------- Fq ---------------- */
static int fq_is_zero(const fq* a) { uint64_t t = 0; for (int i = 0; i < 6; i++) t |= a->l[i]; return t == 0; }
static int fq_eq(const fq* a, const fq* b) { uint64_t t = 0; for (int i = 0; i < 6; i++) t |= a->l[i] ^ b->l[i]; return t == 0; }
static int limbs_ge_p(const uint64_t* a) {
  for (int i = 5; i >= 0; --i) { if (a[i] > PM[i]) return 1; if (a[i] < PM[i]) return 0; }
  return 1;
}
static void fq_sub_p(fq* a) {
  uint64_t bw = 0;
  for (int i = 0; i < 6; i++) { u128 d = (u128)a->l[i] - PM[i] - bw; a->l[i] = (uint64_t)d; bw = (uint64_t)(d >> 64) & 1; }
}
static void fq_add(fq* r, const fq* a, const fq* b) {
  uint64_t c = 0;
  for (int i = 0; i < 6; i++) { u128 s = (u128)a->l[i] + b->l[i] + c; r->l[i] = (uint64_t)s; c = (uint64_t)(s >> 64); }
  if (limbs_ge_p(r->l)) fq_sub_p(r);
}
static void fq_sub(fq* r, const fq* a, const fq* b) {
  uint64_t bw = 0;
  for (int i = 0; i < 6; i++) { u128 d = (u128)a->l[i] - b->l[i] - bw; r->l[i] = (uint64_t)d; bw = (uint64_t)(d >> 64) & 1; }
  if (bw) { uint64_t c = 0; for (int i = 0; i < 6; i++) { u128 s = (u128)r->l[i] + PM[i] + c; r->l[i] = (uint64_t)s; c = (uint64_t)(s >> 64); } }
}
static void fq_neg(fq* r, const fq* a) { fq z; memset(&z, 0, sizeof z); fq_sub(r, &z, a); }
static void fq_dbl(fq* r, const fq* a) { fq_add(r, a, a); }
static void fq_mul(fq* r, const fq* a, const fq* b) {
  uint64_t t[8] = {0};
#pragma GCC unroll 6
  for (int i = 0; i < 6; i++) {
    u128 c = 0;
#pragma GCC unroll 6
    for (int j = 0; j < 6; j++) { c += (u128)a->l[j] * b->l[i] + t[j]; t[j] = (uint64_t)c; c >>= 64; }
    c += t[6]; t[6] = (uint64_t)c; t[7] = (uint64_t)(c >> 64);
    uint64_t m = t[0] * PINV;
    c = (u128)m * PM[0] + t[0]; c >>= 64;
#pragma GCC unroll 6
    for (int j = 1; j < 6; j++) { c += (u128)m * PM[j] + t[j]; t[j - 1] = (uint64_t)c; c >>= 64; }
    c += t[6]; t[5] = (uint64_t)c; t[6] = t[7] + (uint64_t)(c >> 64);
  }
  memcpy(r->l, t, 48);
  if (t[6] || limbs_ge_p(r->l)) fq_sub_p(r);
}
static void fq_sqr(fq* r, const fq* a) { fq_mul(r, a, a); }
static void fq_to_mont(fq* r, const fq* plain) { fq_mul(r, plain, &FQ_R2); }
static void fq_from_mont(fq* r, const fq* m) { fq one; memset(&one, 0, sizeof one); one.l[0] = 1; fq_mul(r, m, &one); }
/* r = a^e, e given as nlimbs u64 little-endian */
static void fq_pow(fq* r, const fq* a, const uint64_t* e, int nlimbs) {
  fq acc = FQ_ONE; int started = 0;
  for (int i = nlimbs * 64 - 1; i >= 0; --i) {
    if (started) fq_sqr(&acc, &acc);
    if ((e[i >> 6] >> (i & 63)) & 1) { if (started) fq_mul(&acc, &acc, a); else { acc = *a; started = 1; } }
  }
  *r = acc;
}
static const uint64_t E_P1_4[6] = {0xee7fbfffffffeaabull, 0x07aaffffac54ffffull, 0xd9cc34a83dac3d89ull,
                                   0xd91dd2e13ce144afull, 0x92c6e9ed90d2eb35ull, 0x0680447a8e5ff9a6ull};
static const uint64_t E_P3_4[6] = {0xee7fbfffffffeaaaull, 0x07aaffffac54ffffull, 0xd9cc34a83dac3d89ull,
                                   0xd91dd2e13ce144afull, 0x92c6e9ed90d2eb35ull, 0x0680447a8e5ff9a6ull};
static const uint64_t E_P1_2[6] = {0xdcff7fffffffd555ull, 0x0f55ffff58a9ffffull, 0xb39869507b587b12ull,
                                   0xb23ba5c279c2895full, 0x258dd3db21a5d66bull, 0x0d0088f51cbff34dull};
/* pairing fq.rs sqrt */
static int fq_sqrt(fq* r, const fq* a) {
  fq s, t; fq_pow(&s, a, E_P1_4, 6); fq_sqr(&t, &s);
  *r = s; return fq_eq(&t, a);
}
/* plain (non-Montgomery) y > (p-1)/2  <=>  y > -y */
static int fq_plain_largest(const fq* yp) {
  static const uint64_t H[6] = {0xdcff7fffffffd555ull, 0x0f55ffff58a9ffffull, 0xb39869507b587b12ull,
                                0xb23ba5c279c2895full, 0x258dd3db21a5d66bull, 0x0d0088f51cbff34dull};
  for (int i = 5; i >= 0; --i) { if (yp->l[i] > H[i]) return 1; if (yp->l[i] < H[i]) return 0; }
  return 0;
}

/* ---------------- Fq2 ---------------- */
static void fq2_add(fq2* r, const fq2* a, const fq2* b) { fq_add(&r->c0, &a->c0, &b->c0); fq_add(&r->c1, &a->c1, &b->c1); }
static void fq2_sub(fq2* r, const fq2* a, const fq2* b) { fq_sub(&r->c0, &a->c0, &b->c0); fq_sub(&r->c1, &a->c1, &b->c1); }
static void fq2_neg(fq2* r, const fq2* a) { fq_neg(&r->c0, &a->c0); fq_neg(&r->c1, &a->c1); }
static void fq2_dbl(fq2* r, const fq2* a) { fq2_add(r, a, a); }
static int fq2_is_zero(const fq2* a) { return fq_is_zero(&a->c0) && fq_is_zero(&a->c1); }
static int fq2_eq(const fq2* a, const fq2* b) { return fq_eq(&a->c0, &b->c0) && fq_eq(&a->c1, &b->c1); }
static void fq2_mul(fq2* r, const fq2* a, const fq2* b) {
  fq v0, v1, s, t, u;
  fq_mul(&v0, &a->c0, &b->c0); fq_mul(&v1, &a->c1, &b->c1);
  fq_add(&s, &a->c0, &a->c1); fq_add(&t, &b->c0, &b->c1); fq_mul(&u, &s, &t);
  fq_sub(&r->c0, &v0, &v1); fq_sub(&u, &u, &v0); fq_sub(&r->c1, &u, &v1);
}
static void fq2_sqr(fq2* r, const fq2* a) {
  fq s, d, t;
  fq_add(&s, &a->c0, &a->c1); fq_sub(&d, &a->c0, &a->c1); fq_mul(&t, &a->c0, &a->c1);
  fq_mul(&r->c0, &s, &d); fq_dbl(&r->c1, &t);
}
static void fq2_conj(fq2* r, const fq2* a) { r->c0 = a->c0; fq_neg(&r->c1, &a->c1); }
static void fq2_pow(fq2* r, const fq2* a, const uint64_t* e, int nlimbs) {
  fq2 acc; int started = 0; memset(&acc, 0, sizeof acc); acc.c0 = FQ_ONE;
  for (int i = nlimbs * 64 - 1; i >= 0; --i) {
    if (started) fq2_sqr(&acc, &acc);
    if ((e[i >> 6] >> (i & 63)) & 1) { if (started) fq2_mul(&acc, &acc, a); else { acc = *a; started = 1; } }
  }
  *r = acc;
}
/* pairing fq2.rs sqrt: Algorithm 9, eprint 2012/685 */
static int fq2_sqrt(fq2* r, const fq2* a) {
  if (fq2_is_zero(a)) { *r = *a; return 1; }
  fq2 a1, alpha, a0, neg1, t;
  fq2_pow(&a1, a, E_P3_4, 6);
  fq2_sqr(&alpha, &a1); fq2_mul(&alpha, &alpha, a);
  fq2_conj(&t, &alpha); fq2_mul(&a0, &t, &alpha);
  memset(&neg1, 0, sizeof neg1); fq_neg(&neg1.c0, &FQ_ONE);
  if (fq2_eq(&a0, &neg1)) return 0;
  fq2_mul(&a1, &a1, a);
  if (fq2_eq(&alpha, &neg1)) {
    fq2 u; memset(&u, 0, sizeof u); u.c1 = FQ_ONE; fq2_mul(r, &a1, &u);
  } else {
    fq2 one; memset(&one, 0, sizeof one); one.c0 = FQ_ONE;
    fq2_add(&alpha, &alpha, &one); fq2_pow(&alpha, &alpha, E_P1_2, 6); fq2_mul(r, &a1, &alpha);
  }
  return 1;
}

/* ---------------- curves: generic via macro over the field ---------------- */
#define DEFINE_CURVE(F, P)                                                                        \
  typedef struct { F X, Y, Z; } P##_jac;                                                          \
  static void P##_double(P##_jac* p) {                                                            \
    if (F##_is_zero(&p->Z)) return;                                                               \
    F A, B, C, D, E, FF, t;                                                                       \
    F##_sqr(&A, &p->X); F##_sqr(&B, &p->Y); F##_sqr(&C, &B);                                      \
    F##_add(&t, &p->X, &B); F##_sqr(&D, &t); F##_sub(&D, &D, &A); F##_sub(&D, &D, &C);            \
    F##_dbl(&D, &D);                                                                              \
    F##_dbl(&E, &A); F##_add(&E, &E, &A); F##_sqr(&FF, &E);                                       \
    F##_mul(&t, &p->Z, &p->Y); F##_dbl(&p->Z, &t);                                                \
    F##_dbl(&t, &D); F##_sub(&p->X, &FF, &t);                                                     \
    F##_sub(&t, &D, &p->X); F##_mul(&t, &t, &E);                                                  \
    F##_dbl(&C, &C); F##_dbl(&C, &C); F##_dbl(&C, &C);                                            \
    F##_sub(&p->Y, &t, &C);                                                                       \
  }                                                                                               \
  static void P##_add_mixed(P##_jac* p, const F* x2, const F* y2, const F* one) {                 \
    if (F##_is_zero(&p->Z)) { p->X = *x2; p->Y = *y2; p->Z = *one; return; }                      \
    F Z1Z1, U2, S2, H, HH, I, J, rr, V, t;                                                        \
    F##_sqr(&Z1Z1, &p->Z); F##_mul(&U2, x2, &Z1Z1);                                               \
    F##_mul(&S2, y2, &p->Z); F##_mul(&S2, &S2, &Z1Z1);                                            \
    if (F##_eq(&U2, &p->X) && F##_eq(&S2, &p->Y)) { P##_double(p); return; }                      \
    F##_sub(&H, &U2, &p->X); F##_sqr(&HH, &H); F##_dbl(&I, &HH); F##_dbl(&I, &I);                 \
    F##_mul(&J, &H, &I); F##_sub(&rr, &S2, &p->Y); F##_dbl(&rr, &rr); F##_mul(&V, &p->X, &I);     \
    F X3, Y3, Z3;                                                                                 \
    F##_sqr(&X3, &rr); F##_sub(&X3, &X3, &J); F##_dbl(&t, &V); F##_sub(&X3, &X3, &t);             \
    F##_sub(&t, &V, &X3); F##_mul(&Y3, &rr, &t); F##_mul(&t, &p->Y, &J); F##_dbl(&t, &t);         \
    F##_sub(&Y3, &Y3, &t);                                                                        \
    F##_add(&Z3, &p->Z, &H); F##_sqr(&Z3, &Z3); F##_sub(&Z3, &Z3, &Z1Z1); F##_sub(&Z3, &Z3, &HH); \
    p->X = X3; p->Y = Y3; p->Z = Z3;                                                              \
  }                                                                                               \
  /* ark mul_bits(BitIteratorBE(k)): res = 0; for bits: double; if bit: add_mixed */             \
  static void P##_mul_bits(P##_jac* res, const F* x, const F* y, const F* one, const uint64_t* k, \
                           int nlimbs) {                                                          \
    memset(res, 0, sizeof *res); res->Y = *one;                                                   \
    for (int i = nlimbs * 64 - 1; i >= 0; --i) {                                                  \
      P##_double(res);                                                                            \
      if ((k[i >> 6] >> (i & 63)) & 1) P##_add_mixed(res, x, y, one);                             \
    }                                                                                             \
  }

DEFINE_CURVE(fq, g1)
DEFINE_CURVE(fq2, g2)

static fq FQ_B1; /* 4 in Montgomery form, set by init */
static fq K_BETA, K_PSI_CX1, K_HALF; /* constants of the fast predicates (baseline row 3 only) */
static fq2 K_PSI_CY;
static fq2 FQ2_ONE, FQ2_B2;
static fq G1X, G1Y; static fq2 G2X, G2Y;
static int g_init = 0;
static void fq_from_hex_limbs(fq* r, const uint64_t l[6]) { fq t; memcpy(t.l, l, 48); fq_to_mont(r, &t); }
static void init_consts(void) {
  if (g_init) return;
  fq four; memset(&four, 0, sizeof four); four.l[0] = 4; fq_to_mont(&FQ_B1, &four);
  memset(&FQ2_ONE, 0, sizeof FQ2_ONE); FQ2_ONE.c0 = FQ_ONE;
  FQ2_B2.c0 = FQ_B1; FQ2_B2.c1 = FQ_B1;
  static const uint64_t g1x[6] = {0xfb3af00adb22c6bbull, 0x6c55e83ff97a1aefull, 0xa14e3a3f171bac58ull, 0xc3688c4f9774b905ull, 0x2695638c4fa9ac0full, 0x17f1d3a73197d794ull};
  static const uint64_t g1y[6] = {0x0caa232946c5e7e1ull, 0xd03cc744a2888ae4ull, 0x00db18cb2c04b3edull, 0xfcf5e095d5d00af6ull, 0xa09e30ed741d8ae4ull, 0x08b3f481e3aaa0f1ull};
  static const uint64_t g2x0[6] = {0xd48056c8c121bdb8ull, 0x0bac0326a805bbefull, 0xb4510b647ae3d177ull, 0xc6e47ad4fa403b02ull, 0x260805272dc51051ull, 0x024aa2b2f08f0a91ull};
  static const uint64_t g2x1[6] = {0xe5ac7d055d042b7eull, 0x334cf11213945d57ull, 0xb5da61bbdc7f5049ull, 0x596bd0d09920b61aull, 0x7dacd3a088274f65ull, 0x13e02b6052719f60ull};
  static const uint64_t g2y0[6] = {0xe193548608b82801ull, 0x923ac9cc3baca289ull, 0x6d429a695160d12cull, 0xadfd9baa8cbdd3a7ull, 0x8cc9cdc6da2e351aull, 0x0ce5d527727d6e11ull};
  static const uint64_t g2y1[6] = {0xaaa9075ff05f79beull, 0x3f370d275cec1da1ull, 0x267492ab572e99abull, 0xcb3e287e85a763afull, 0x32acd2b02bc28b99ull, 0x0606c4a02ea734ccull};
  fq_from_hex_limbs(&G1X, g1x); fq_from_hex_limbs(&G1Y, g1y);
  fq_from_hex_limbs(&G2X.c0, g2x0); fq_from_hex_limbs(&G2X.c1, g2x1);
  fq_from_hex_limbs(&G2Y.c0, g2y0); fq_from_hex_limbs(&G2Y.c1, g2y1);
  static const uint64_t beta[6] = {0x2e01fffffffefffeull, 0xde17d813620a0002ull, 0xddb3a93be6f89688ull, 0xba69c6076a0f77eaull, 0x5f19672fdf76ce51ull, 0};
  static const uint64_t cx1[6] = {0x8bfd00000000aaadull, 0x409427eb4f49fffdull, 0x897d29650fb85f9bull, 0xaa0d857d89759ad4ull, 0xec02408663d4de85ull, 0x1a0111ea397fe699ull};
  static const uint64_t cy0[6] = {0xf1ee7b04121bdea2ull, 0x304466cf3e67fa0aull, 0xef396489f61eb45eull, 0x1c3dedd930b1cf60ull, 0xe2e9c448d77a2cd9ull, 0x135203e60180a68eull};
  static const uint64_t cy1[6] = {0xc81084fbede3cc09ull, 0xee67992f72ec05f4ull, 0x77f76e17009241c5ull, 0x48395dabc2d3435eull, 0x6831e36d6bd17ffeull, 0x06af0e0437ff400bull};
  static const uint64_t half[6] = {0xdcff7fffffffd556ull, 0x0f55ffff58a9ffffull, 0xb39869507b587b12ull, 0xb23ba5c279c2895full, 0x258dd3db21a5d66bull, 0x0d0088f51cbff34dull};
  fq_from_hex_limbs(&K_BETA, beta); fq_from_hex_limbs(&K_PSI_CX1, cx1); fq_from_hex_limbs(&K_PSI_CY.c0, cy0);
  fq_from_hex_limbs(&K_PSI_CY.c1, cy1); fq_from_hex_limbs(&K_HALF, half);
  g_init = 1;
}

/* ---------------- the GPU's predicates, on the CPU ----------------
 * Only used for the third baseline row of BASELINE.md (same C code, endomorphism checks and
 * norm-method square root) so that the algorithmic and the hardware speed-up can be told
 * apart.  Selected with CHK_FAST_PREDICATES; never the default, never the parity oracle. */
static const uint64_t Z_ABS[1] = {0xd201000000010000ull};
static void g1_add_jac(g1_jac* p, const g1_jac* q) { /* add-2007-bl, no special cases needed on the ladders */
  fq Z1Z1, Z2Z2, U1, U2, S1, S2, H, I, J, rr, V, t, X3, Y3, Z3;
  fq_sqr(&Z1Z1, &p->Z); fq_sqr(&Z2Z2, &q->Z); fq_mul(&U1, &p->X, &Z2Z2); fq_mul(&U2, &q->X, &Z1Z1);
  fq_mul(&S1, &p->Y, &q->Z); fq_mul(&S1, &S1, &Z2Z2); fq_mul(&S2, &q->Y, &p->Z); fq_mul(&S2, &S2, &Z1Z1);
  fq_sub(&H, &U2, &U1); fq_dbl(&I, &H); fq_sqr(&I, &I); fq_mul(&J, &H, &I); fq_sub(&rr, &S2, &S1); fq_dbl(&rr, &rr);
  fq_mul(&V, &U1, &I); fq_sqr(&X3, &rr); fq_sub(&X3, &X3, &J); fq_dbl(&t, &V); fq_sub(&X3, &X3, &t);
  fq_sub(&t, &V, &X3); fq_mul(&Y3, &rr, &t); fq_mul(&t, &S1, &J); fq_dbl(&t, &t); fq_sub(&Y3, &Y3, &t);
  fq_mul(&Z3, &p->Z, &q->Z); fq_dbl(&Z3, &Z3); fq_mul(&Z3, &Z3, &H);
  p->X = X3; p->Y = Y3; p->Z = Z3;
}
static int g1_in_subgroup_glv(const fq* x, const fq* y) {
  g1_jac q, acc; g1_mul_bits(&q, x, y, &FQ_ONE, Z_ABS, 1);
  if (fq_is_zero(&q.Z)) return 0;
  acc = q;
  for (int i = 62; i >= 0; --i) { g1_double(&acc); if ((Z_ABS[0] >> i) & 1) g1_add_jac(&acc, &q); }
  if (fq_is_zero(&acc.Z)) return 0;
  fq zz, zzz, bx, ny, l, r2; fq_sqr(&zz, &acc.Z); fq_mul(&zzz, &zz, &acc.Z); fq_mul(&bx, x, &K_BETA); fq_neg(&ny, y);
  fq_mul(&l, &bx, &zz); fq_mul(&r2, &ny, &zzz);
  return fq_eq(&acc.X, &l) && fq_eq(&acc.Y, &r2);
}
static int g2_in_subgroup_psi(const fq2* x, const fq2* y) {
  g2_jac q; g2_mul_bits(&q, x, y, &FQ2_ONE, Z_ABS, 1);
  if (fq2_is_zero(&q.Z)) return 0;
  fq2 px, py, cy, zz, zzz, l, r2; fq_mul(&px.c0, &x->c1, &K_PSI_CX1); fq_mul(&px.c1, &x->c0, &K_PSI_CX1);
  fq2_conj(&cy, y); fq2_mul(&py, &cy, &K_PSI_CY); fq2_neg(&py, &py);
  fq2_sqr(&zz, &q.Z); fq2_mul(&zzz, &zz, &q.Z); fq2_mul(&l, &px, &zz); fq2_mul(&r2, &py, &zzz);
  return fq2_eq(&q.X, &l) && fq2_eq(&q.Y, &r2);
}
static int fq2_sqrt_norm(fq2* r, const fq2* a) {
  fq n, t0, s, d, t, x0, chi, w, nx0; fq_sqr(&n, &a->c0); fq_sqr(&t0, &a->c1); fq_add(&n, &n, &t0);
  fq_pow(&s, &n, E_P1_4, 6); fq_add(&d, &a->c0, &s); fq_mul(&d, &d, &K_HALF);
  if (fq_is_zero(&d)) { fq_sub(&d, &a->c0, &s); fq_mul(&d, &d, &K_HALF); }
  fq_pow(&t, &d, E_P3_4, 6); fq_mul(&x0, &d, &t); fq_mul(&chi, &x0, &t); fq_mul(&w, &a->c1, &t); fq_mul(&w, &w, &K_HALF);
  if (fq_eq(&chi, &FQ_ONE) || fq_is_zero(&d)) { r->c0 = x0; r->c1 = w; } else { fq_neg(&nx0, &x0); r->c0 = w; r->c1 = nx0; }
  fq2 chk; fq2_sqr(&chk, r); return fq2_eq(&chk, a);
}

/* ---------------- encodings ---------------- */
enum { FMT_ZU = 1, FMT_ZC = 2, FMT_AU = 3, FMT_ML = 4 };
enum { G1 = 1, G2 = 2 };
enum { CHK_ON_CURVE = 2, CHK_SUBGROUP = 4, CHK_REJECT_INF = 8, CHK_FAST_PREDICATES = 16 };
enum { OK = 0, BAD_NON_CANONICAL = 1, BAD_FLAGS = 2, BAD_INFINITY = 3, BAD_NOT_ON_CURVE = 4, BAD_NOT_IN_SUBGROUP = 5 };

static void be48_to_limbs(fq* r, const uint8_t* b) {
  for (int i = 0; i < 6; i++) { uint64_t v = 0; for (int k = 0; k < 8; k++) v = (v << 8) | b[(5 - i) * 8 + k]; r->l[i] = v; }
}
static void limbs_to_be48(uint8_t* b, const fq* a) {
  for (int i = 0; i < 6; i++) { uint64_t v = a->l[i]; for (int k = 7; k >= 0; --k) { b[(5 - i) * 8 + k] = (uint8_t)v; v >>= 8; } }
}
static void le48_to_limbs(fq* r, const uint8_t* b) { memcpy(r->l, b, 48); }
static void limbs_to_le48(uint8_t* b, const fq* a) { memcpy(b, a->l, 48); }

static int rec_size(int group, int fmt) {
  int g1 = group == G1;
  switch (fmt) { case FMT_ZU: case FMT_AU: return g1 ? 96 : 192; case FMT_ZC: return g1 ? 48 : 96; case FMT_ML: return g1 ? 104 : 200; }
  return 0;
}
static void fq_plain_neg(fq* r, const fq* a) {
  if (fq_is_zero(a)) { *r = *a; return; }
  uint64_t bw = 0;
  for (int i = 0; i < 6; i++) { u128 d = (u128)PM[i] - a->l[i] - bw; r->l[i] = (uint64_t)d; bw = (uint64_t)(d >> 64) & 1; }
}

/* One G1 point.  Returns status.  Semantics identical to the Python oracle's
 * decode functions + read_g1 + serialize (see ptau_oracle.py for the citations). */
static int g1_one(int in_fmt, const uint8_t* in, int out_fmt, uint8_t* out, unsigned checks) {
  fq xp, yp, xm, ym; int inf = 0, st = OK, have_m = 0;
  memset(&yp, 0, sizeof yp);
  if (in_fmt == FMT_ZC) {
    uint8_t b[48]; memcpy(b, in, 48);
    int fl = b[0] >> 5; b[0] &= 0x1f; be48_to_limbs(&xp, b);
    if (!(fl & 4)) st = BAD_FLAGS;
    else if (fl & 2) { if ((fl & 1) || !fq_is_zero(&xp)) st = BAD_FLAGS; inf = 1; yp.l[0] = 1; }
    else if (limbs_ge_p(xp.l)) st = BAD_NON_CANONICAL;
    if (st == OK && !inf) {
      fq rhs; fq_to_mont(&xm, &xp); fq_sqr(&rhs, &xm); fq_mul(&rhs, &rhs, &xm); fq_add(&rhs, &rhs, &FQ_B1);
      if (!fq_sqrt(&ym, &rhs)) st = BAD_NOT_ON_CURVE;
      fq_from_mont(&yp, &ym);
      if (fq_plain_largest(&yp) != (fl & 1)) { fq_neg(&ym, &ym); fq_plain_neg(&yp, &yp); }
      have_m = 1;
    }
  } else if (in_fmt == FMT_ML) { /* in-memory GroupAffine -> serialize direction (preprocess-kgz.rs:188-194) */
    le48_to_limbs(&xm, in); le48_to_limbs(&ym, in + 48); inf = in[96] != 0;
    if (limbs_ge_p(xm.l) || limbs_ge_p(ym.l)) { st = BAD_NON_CANONICAL; memset(&xm, 0, sizeof xm); memset(&ym, 0, sizeof ym); }
    have_m = 1; fq_from_mont(&xp, &xm); fq_from_mont(&yp, &ym);
    if (st == OK && !inf && (checks & CHK_ON_CURVE)) {
      fq l, r; fq_sqr(&l, &ym); fq_sqr(&r, &xm); fq_mul(&r, &r, &xm); fq_add(&r, &r, &FQ_B1);
      if (!fq_eq(&l, &r)) st = BAD_NOT_ON_CURVE;
    }
  } else {
    if (in_fmt == FMT_ZU) { be48_to_limbs(&xp, in); be48_to_limbs(&yp, in + 48); }
    else { le48_to_limbs(&xp, in); le48_to_limbs(&yp, in + 48); }
    int fl = (int)(yp.l[5] >> 62); yp.l[5] &= 0x3fffffffffffffffull;
    if (limbs_ge_p(xp.l)) st = BAD_NON_CANONICAL; else if (fl == 3) st = BAD_FLAGS; else if (limbs_ge_p(yp.l)) st = BAD_NON_CANONICAL;
    inf = fl == 1;
    if (st == OK) { fq_to_mont(&xm, &xp); fq_to_mont(&ym, &yp); have_m = 1; }
    if (st == OK && !inf && (checks & CHK_ON_CURVE)) {
      fq l, r; fq_sqr(&l, &ym); fq_sqr(&r, &xm); fq_mul(&r, &r, &xm); fq_add(&r, &r, &FQ_B1);
      if (!fq_eq(&l, &r)) st = BAD_NOT_ON_CURVE;
    }
  }
  if (st == OK && inf && (checks & CHK_REJECT_INF)) st = BAD_INFINITY;
  if (st == OK && !inf && (checks & CHK_SUBGROUP)) {
    if (checks & CHK_FAST_PREDICATES) { if (!g1_in_subgroup_glv(&xm, &ym)) st = BAD_NOT_IN_SUBGROUP; }
    else { g1_jac t; g1_mul_bits(&t, &xm, &ym, &FQ_ONE, R_ORDER, 4); if (!fq_is_zero(&t.Z)) st = BAD_NOT_IN_SUBGROUP; }
  }
  if (out_fmt == FMT_AU) { limbs_to_le48(out, &xp); limbs_to_le48(out + 48, &yp); if (inf) out[95] |= 0x40; }
  else if (out_fmt == FMT_ZU) {
    if (inf) { memset(out, 0, 96); out[0] = 0x40; } else { limbs_to_be48(out, &xp); limbs_to_be48(out + 48, &yp); }
  } else {
    if (st == OK && !have_m) { fq_to_mont(&xm, &xp); fq_to_mont(&ym, &yp); have_m = 1; }
    if (!have_m) { memset(&xm, 0, sizeof xm); memset(&ym, 0, sizeof ym); }
    memcpy(out, xm.l, 48); memcpy(out + 48, ym.l, 48); memset(out + 96, 0, 8); out[96] = (uint8_t)inf;
  }
  return st;
}

static int fq2_plain_largest(const fq2* yp) { return fq_is_zero(&yp->c1) ? fq_plain_largest(&yp->c0) : fq_plain_largest(&yp->c1); }

static int g2_one(int in_fmt, const uint8_t* in, int out_fmt, uint8_t* out, unsigned checks) {
  fq2 xp, yp, xm, ym; int inf = 0, st = OK, have_m = 0;
  memset(&yp, 0, sizeof yp);
  if (in_fmt == FMT_ZC) {
    uint8_t b[96]; memcpy(b, in, 96);
    int fl = b[0] >> 5; b[0] &= 0x1f; be48_to_limbs(&xp.c1, b); be48_to_limbs(&xp.c0, b + 48);
    if (!(fl & 4)) st = BAD_FLAGS;
    else if (fl & 2) { if ((fl & 1) || !fq2_is_zero(&xp)) st = BAD_FLAGS; inf = 1; yp.c0.l[0] = 1; }
    else if (limbs_ge_p(xp.c1.l) || limbs_ge_p(xp.c0.l)) st = BAD_NON_CANONICAL;
    if (st == OK && !inf) {
      fq2 rhs; fq_to_mont(&xm.c0, &xp.c0); fq_to_mont(&xm.c1, &xp.c1);
      fq2_sqr(&rhs, &xm); fq2_mul(&rhs, &rhs, &xm); fq2_add(&rhs, &rhs, &FQ2_B2);
      if (checks & CHK_FAST_PREDICATES) { if (!fq2_sqrt_norm(&ym, &rhs)) st = BAD_NOT_ON_CURVE; }
      else if (!fq2_sqrt(&ym, &rhs)) st = BAD_NOT_ON_CURVE;
      else { fq2 chk; fq2_sqr(&chk, &ym); if (!fq2_eq(&chk, &rhs)) st = BAD_NOT_ON_CURVE; }
      fq_from_mont(&yp.c0, &ym.c0); fq_from_mont(&yp.c1, &ym.c1);
      if (fq2_plain_largest(&yp) != (fl & 1)) { fq2_neg(&ym, &ym); fq_plain_neg(&yp.c0, &yp.c0); fq_plain_neg(&yp.c1, &yp.c1); }
      have_m = 1;
    }
  } else if (in_fmt == FMT_ML) {
    le48_to_limbs(&xm.c0, in); le48_to_limbs(&xm.c1, in + 48); le48_to_limbs(&ym.c0, in + 96); le48_to_limbs(&ym.c1, in + 144);
    inf = in[192] != 0;
    if (limbs_ge_p(xm.c0.l) || limbs_ge_p(xm.c1.l) || limbs_ge_p(ym.c0.l) || limbs_ge_p(ym.c1.l)) { st = BAD_NON_CANONICAL; memset(&xm, 0, sizeof xm); memset(&ym, 0, sizeof ym); }
    have_m = 1; fq_from_mont(&xp.c0, &xm.c0); fq_from_mont(&xp.c1, &xm.c1); fq_from_mont(&yp.c0, &ym.c0); fq_from_mont(&yp.c1, &ym.c1);
    if (st == OK && !inf && (checks & CHK_ON_CURVE)) {
      fq2 l, r; fq2_sqr(&l, &ym); fq2_sqr(&r, &xm); fq2_mul(&r, &r, &xm); fq2_add(&r, &r, &FQ2_B2);
      if (!fq2_eq(&l, &r)) st = BAD_NOT_ON_CURVE;
    }
  } else {
    if (in_fmt == FMT_ZU) { be48_to_limbs(&xp.c1, in); be48_to_limbs(&xp.c0, in + 48); be48_to_limbs(&yp.c1, in + 96); be48_to_limbs(&yp.c0, in + 144); }
    else { le48_to_limbs(&xp.c0, in); le48_to_limbs(&xp.c1, in + 48); le48_to_limbs(&yp.c0, in + 96); le48_to_limbs(&yp.c1, in + 144); }
    int fl = (int)(yp.c1.l[5] >> 62); yp.c1.l[5] &= 0x3fffffffffffffffull;
    if (limbs_ge_p(xp.c0.l) || limbs_ge_p(xp.c1.l) || limbs_ge_p(yp.c0.l)) st = BAD_NON_CANONICAL;
    else if (fl == 3) st = BAD_FLAGS; else if (limbs_ge_p(yp.c1.l)) st = BAD_NON_CANONICAL;
    inf = fl == 1;
    if (st == OK) { fq_to_mont(&xm.c0, &xp.c0); fq_to_mont(&xm.c1, &xp.c1); fq_to_mont(&ym.c0, &yp.c0); fq_to_mont(&ym.c1, &yp.c1); have_m = 1; }
    if (st == OK && !inf && (checks & CHK_ON_CURVE)) {
      fq2 l, r; fq2_sqr(&l, &ym); fq2_sqr(&r, &xm); fq2_mul(&r, &r, &xm); fq2_add(&r, &r, &FQ2_B2);
      if (!fq2_eq(&l, &r)) st = BAD_NOT_ON_CURVE;
    }
  }
  if (st == OK && inf && (checks & CHK_REJECT_INF)) st = BAD_INFINITY;
  if (st == OK && !inf && (checks & CHK_SUBGROUP)) {
    if (checks & CHK_FAST_PREDICATES) { if (!g2_in_subgroup_psi(&xm, &ym)) st = BAD_NOT_IN_SUBGROUP; }
    else { g2_jac t; g2_mul_bits(&t, &xm, &ym, &FQ2_ONE, R_ORDER, 4); if (!fq2_is_zero(&t.Z)) st = BAD_NOT_IN_SUBGROUP; }
  }
  if (out_fmt == FMT_AU) {
    limbs_to_le48(out, &xp.c0); limbs_to_le48(out + 48, &xp.c1); limbs_to_le48(out + 96, &yp.c0); limbs_to_le48(out + 144, &yp.c1);
    if (inf) out[191] |= 0x40;
  } else if (out_fmt == FMT_ZU) {
    if (inf) { memset(out, 0, 192); out[0] = 0x40; }
    else { limbs_to_be48(out, &xp.c1); limbs_to_be48(out + 48, &xp.c0); limbs_to_be48(out + 96, &yp.c1); limbs_to_be48(out + 144, &yp.c0); }
  } else {
    /* zcash compressed infinity reaches here with the plain ark zero() = (0, 1): its limbs are Montgomery 0 and 1 */
    if (st == OK && !have_m) {
      fq_to_mont(&xm.c0, &xp.c0); fq_to_mont(&xm.c1, &xp.c1); fq_to_mont(&ym.c0, &yp.c0); fq_to_mont(&ym.c1, &yp.c1);
      have_m = 1;
    }
    if (!have_m) { memset(&xm, 0, sizeof xm); memset(&ym, 0, sizeof ym); }
    memcpy(out, xm.c0.l, 48); memcpy(out + 48, xm.c1.l, 48); memcpy(out + 96, ym.c0.l, 48); memcpy(out + 144, ym.c1.l, 48);
    memset(out + 192, 0, 8); out[192] = (uint8_t)inf;
  }
  return st;
}

/* ---------------- batch entry points ---------------- */
typedef struct {
  int group, in_fmt, out_fmt; unsigned checks;
  const uint8_t* in; uint8_t* out; uint8_t* status; size_t lo, hi;
} job_t;
static void* worker(void* arg) {
  job_t* j = (job_t*)arg;
  int ri = rec_size(j->group, j->in_fmt), ro = rec_size(j->group, j->out_fmt);
  for (size_t i = j->lo; i < j->hi; i++) {
    int st = j->group == G1 ? g1_one(j->in_fmt, j->in + i * ri, j->out_fmt, j->out + i * ro, j->checks)
                            : g2_one(j->in_fmt, j->in + i * ri, j->out_fmt, j->out + i * ro, j->checks);
    if (j->status) j->status[i] = (uint8_t)st;
  }
  return NULL;
}
/* status: one byte per point (may be NULL).  nthreads <= 1: in the calling thread. */
int oracle_convert(int group, int in_fmt, const uint8_t* in, int out_fmt, uint8_t* out, size_t n, unsigned checks,
                   uint8_t* status, int nthreads) {
  init_consts();
  if (!rec_size(group, in_fmt) || !rec_size(group, out_fmt) || out_fmt == FMT_ZC) return -2;
  if (nthreads <= 1) { job_t j = {group, in_fmt, out_fmt, checks, in, out, status, 0, n}; worker(&j); return 0; }
  if (nthreads > 256) nthreads = 256;
  pthread_t th[256]; job_t jobs[256];
  for (int t = 0; t < nthreads; t++) {
    job_t j = {group, in_fmt, out_fmt, checks, in, out, status, n * t / nthreads, n * (t + 1) / nthreads};
    jobs[t] = j; pthread_create(&th[t], NULL, worker, &jobs[t]);
  }
  for (int t = 0; t < nthreads; t++) pthread_join(th[t], NULL);
  return 0;
}

/* ---------------- synthetic generator (known tau) ---------------- */
static const uint64_t FR_INV = 0xfffffffeffffffffull;
static const uint64_t FR_R2[4] = {0xc999e990f3f29c6dull, 0x2b6cedcb87925c23ull, 0x05d314967254398full, 0x0748d9d99f59ff11ull};
static void fr_mul(uint64_t* r, const uint64_t* a, const uint64_t* b) {
  uint64_t t[6] = {0};
  for (int i = 0; i < 4; i++) {
    u128 c = 0;
    for (int j = 0; j < 4; j++) { c += (u128)a[j] * b[i] + t[j]; t[j] = (uint64_t)c; c >>= 64; }
    c += t[4]; t[4] = (uint64_t)c; t[5] = (uint64_t)(c >> 64);
    uint64_t m = t[0] * FR_INV;
    c = (u128)m * R_ORDER[0] + t[0]; c >>= 64;
    for (int j = 1; j < 4; j++) { c += (u128)m * R_ORDER[j] + t[j]; t[j - 1] = (uint64_t)c; c >>= 64; }
    c += t[4]; t[3] = (uint64_t)c; t[4] = t[5] + (uint64_t)(c >> 64);
  }
  int ge = t[4] != 0;
  if (!ge) { ge = 1; for (int i = 3; i >= 0; --i) { if (t[i] > R_ORDER[i]) break; if (t[i] < R_ORDER[i]) { ge = 0; break; } } }
  if (ge) { uint64_t bw = 0; for (int i = 0; i < 4; i++) { u128 d = (u128)t[i] - R_ORDER[i] - bw; t[i] = (uint64_t)d; bw = (uint64_t)(d >> 64) & 1; } }
  memcpy(r, t, 32);
}
static void fq_inv(fq* r, const fq* a) {
  static const uint64_t E_PM2[6] = {0xb9feffffffffaaa9ull, 0x1eabfffeb153ffffull, 0x6730d2a0f6b0f624ull,
                                    0x64774b84f38512bfull, 0x4b1ba7b6434bacd7ull, 0x1a0111ea397fe69aull};
  fq_pow(r, a, E_PM2, 6);
}
typedef struct { int group, fmt; const uint64_t* scalars; uint8_t* out; size_t lo, hi; } gen_job_t;
static void* gen_worker(void* arg) {
  gen_job_t* j = (gen_job_t*)arg;
  int ro = rec_size(j->group, j->fmt);
  for (size_t i = j->lo; i < j->hi; i++) {
    const uint64_t* k = j->scalars + 4 * i; uint8_t* o = j->out + i * ro;
    if (j->group == G1) {
      g1_jac t; g1_mul_bits(&t, &G1X, &G1Y, &FQ_ONE, k, 4);
      fq zi, zi2, zi3, xm, ym, xp, yp; fq_inv(&zi, &t.Z); fq_sqr(&zi2, &zi); fq_mul(&zi3, &zi2, &zi);
      fq_mul(&xm, &t.X, &zi2); fq_mul(&ym, &t.Y, &zi3); fq_from_mont(&xp, &xm); fq_from_mont(&yp, &ym);
      limbs_to_be48(o, &xp);
      if (j->fmt == FMT_ZC) { o[0] |= 0x80; if (fq_plain_largest(&yp)) o[0] |= 0x20; } else limbs_to_be48(o + 48, &yp);
    } else {
      g2_jac t; g2_mul_bits(&t, &G2X, &G2Y, &FQ2_ONE, k, 4);
      fq n0, n1, ni; fq_sqr(&n0, &t.Z.c0); fq_sqr(&n1, &t.Z.c1); fq_add(&n0, &n0, &n1); fq_inv(&ni, &n0);
      fq2 zi, zi2, zi3, xm, ym, xp, yp; fq_mul(&zi.c0, &t.Z.c0, &ni); fq_mul(&zi.c1, &t.Z.c1, &ni); fq_neg(&zi.c1, &zi.c1);
      fq2_sqr(&zi2, &zi); fq2_mul(&zi3, &zi2, &zi); fq2_mul(&xm, &t.X, &zi2); fq2_mul(&ym, &t.Y, &zi3);
      fq_from_mont(&xp.c0, &xm.c0); fq_from_mont(&xp.c1, &xm.c1); fq_from_mont(&yp.c0, &ym.c0); fq_from_mont(&yp.c1, &ym.c1);
      limbs_to_be48(o, &xp.c1); limbs_to_be48(o + 48, &xp.c0);
      if (j->fmt == FMT_ZC) { o[0] |= 0x80; if (fq2_plain_largest(&yp)) o[0] |= 0x20; }
      else { limbs_to_be48(o + 96, &yp.c1); limbs_to_be48(o + 144, &yp.c0); }
    }
  }
  return NULL;
}
/* out[i] = [scalar0 * step^(first+i)] G in zcash compressed / uncompressed form */
int oracle_generate(int group, int fmt, const uint8_t scalar0[32], const uint8_t step[32], uint64_t first, size_t n,
                    uint8_t* out, int nthreads) {
  init_consts();
  if ((fmt != FMT_ZC && fmt != FMT_ZU) || !rec_size(group, fmt)) return -2;
  uint64_t s0[4], st[4], r2[4], one[4] = {1, 0, 0, 0}, cur[4], stm[4];
  memcpy(s0, scalar0, 32); memcpy(st, step, 32); memcpy(r2, FR_R2, 32);
  fr_mul(stm, st, r2); fr_mul(cur, s0, r2);
  { uint64_t b[4]; memcpy(b, stm, 32); uint64_t e = first; while (e) { if (e & 1) fr_mul(cur, cur, b); fr_mul(b, b, b); e >>= 1; } }
  uint64_t* sc = (uint64_t*)malloc(n * 32 + 32);
  if (!sc) return -4;
  for (size_t i = 0; i < n; i++) { fr_mul(sc + 4 * i, cur, one); fr_mul(cur, cur, stm); }
  if (nthreads < 1) nthreads = 1;
  if (nthreads > 256) nthreads = 256;
  pthread_t th[256]; gen_job_t jobs[256];
  for (int t = 0; t < nthreads; t++) {
    gen_job_t j = {group, fmt, sc, out, n * t / nthreads, n * (t + 1) / nthreads};
    jobs[t] = j; pthread_create(&th[t], NULL, gen_worker, &jobs[t]);
  }
  for (int t = 0; t < nthreads; t++) pthread_join(th[t], NULL);
  free(sc);
  return 0;
}

/* raw field op for cross-checks against the Python oracle: op 0 mul, 1 sqrt(Fq), 2 fq2 sqrt (a,b = c0,c1 in; out 96 B) */
int oracle_fq_op(int op, const uint8_t* a, const uint8_t* b, uint8_t* out) {
  init_consts();
  fq x, y, r; memcpy(x.l, a, 48); memcpy(y.l, b, 48);
  if (op == 0) { fq_mul(&r, &x, &y); memcpy(out, r.l, 48); return 1; }
  if (op == 1) { int ok = fq_sqrt(&r, &x); memcpy(out, r.l, 48); return ok; }
  if (op == 2) { fq2 v, s; v.c0 = x; v.c1 = y; int ok = fq2_sqrt(&s, &v); if (ok) { memcpy(out, s.c0.l, 48); memcpy(out + 48, s.c1.l, 48); } return ok; }
  return -1;
}
