// A Powers-of-Tau contribution on the GPU (powersoftau `compute`) and its check (powersoftau `verify_transform`):
// the contribution kernel and the C-ABI entry points ptau_challenge_size, ptau_contribute, ptau_verify_contribution.
//
// ptau_contribute streams the challenge through the context's GPUs section by section, each section split into
// contiguous index ranges like ptau_convert.  Per chunk, on one stream: H2D of the uncompressed records, the existing
// conversion ZCASH_UNCOMPRESSED -> ARK_MONT_LIMBS with the caller's checks (it reports bad points exactly as
// ptau_preprocess does), the contribution kernel (scalar formed on the device, [k]P, affine, compressed record), D2H.
// The compressed records are written into the chunk's input buffer, which the conversion has finished with, so device
// memory is the two double buffers of the context's chunk_points only.  A host thread hashes the challenge meanwhile;
// the public key (nine points, ChaCha20 and the h2 multiplication) is computed on the host after that digest.
#include <cuda_runtime.h>
#include <stdint.h>
#include <string.h>
#include <sys/random.h>

#include <chrono>
#include <string>
#include <thread>
#include <type_traits>

#include "../../include/ptau_b200.h"
#include "blake2b.h"
#include "context.h"
#include "contribute.cuh"
#include "fr.cuh"
#include "fr_host.h"
#include "gen_tail.cuh"
#include "kernels.h"
#include "layout.h"

namespace ptau {
namespace {

template <class F>
struct TailInv;
template <>
struct TailInv<Fq> {
  static __device__ __forceinline__ Fq inv(const Fq& a) { return fq_inv_fermat(a); }
};
template <>
struct TailInv<Fq2> {
  static __device__ __forceinline__ Fq2 inv(const Fq2& a) { return fq2_inv(a); }
};

__device__ __forceinline__ void set_one(Fq& a) { a = fq_one(); }
__device__ __forceinline__ void set_one(Fq2& a) { a = fq2_one(); }

// out[i] = compressed record of [s0 step^(first + i)] in[i] for the ARK_MONT_LIMBS records in[0, n).  A point at
// infinity, and a product that is infinity (only possible for a point outside the subgroup), give the compressed
// infinity record.
template <int G>
__global__ void __launch_bounds__(PTAU_BLOCK)
    contribute_kernel(FrParams fp, const uint32_t* __restrict__ in, uint32_t* __restrict__ out, uint64_t first,
                      uint64_t n) {
  using F = typename std::conditional<G == PTAU_G1, Fq, Fq2>::type;
  constexpr int WOUT = record_bytes(G, PTAU_FMT_ZCASH_COMPRESSED) / 4;
  constexpr int WREC = record_bytes(G, PTAU_FMT_ARK_MONT_LIMBS) / 4;
  __shared__ __align__(16) uint32_t sm[PTAU_BLOCK * WOUT];
  const int tid = threadIdx.x;
  const uint64_t blk0 = (uint64_t)blockIdx.x * (PTAU_BLOCK * PTAU_GEN_B);
  // scalar of this thread's first point, s0 * step^(first + blk0 + tid), as the generator forms it
  uint32_t cur[8];
#pragma unroll
  for (int i = 0; i < 8; i++) cur[i] = fp.s0[i];
  {
    const uint64_t e = first + blk0 + tid;
#pragma unroll 1
    for (int j = 0; j < 64; j++)
      if ((e >> j) & 1ull) fr_mul(cur, cur, fp.pw[j]);
  }
  F one;
  set_one(one);
  Jac<F> pts[PTAU_GEN_B];
  F pre[PTAU_GEN_B];
  uint32_t infmask = 0;
#pragma unroll 1
  for (int j = 0; j < PTAU_GEN_B; j++) {
    const uint64_t idx = blk0 + (uint64_t)j * PTAU_BLOCK + tid;
    Jac<F> acc;
    acc.X = one;
    acc.Y = one;
    acc.Z = one;
    if (idx < n) {
      uint32_t k[8];
      {
        const uint32_t unit[8] = {1, 0, 0, 0, 0, 0, 0, 0};
        fr_mul(k, cur, unit);  // out of Montgomery form
      }
      fr_mul(cur, cur, fp.pw[7]);  // next point of this thread is PTAU_BLOCK = 2^7 further
      F x, y;
      bool inf;
      load_rec(in + idx * WREC, x, y, inf);
      if (!inf) {
        const Jac<F> r = contrib_mul(x, y, k);
        if (fis_zero(r.Z))
          inf = true;
        else
          acc = r;
      }
      if (inf) infmask |= 1u << j;
    }
    pts[j] = acc;
    pre[j] = (j == 0) ? acc.Z : fmul(pre[j - 1], acc.Z);
  }
  affine_encode_tail<G, PTAU_FMT_ZCASH_COMPRESSED, TailInv<F>, true>(pts, pre, sm, out, tid, blk0, n, infmask);
}

cudaError_t launch_contribute(int group, const FrParams& fp, const void* d_in, void* d_out, uint64_t first, uint64_t n,
                              cudaStream_t stream) {
  if (n == 0) return cudaSuccess;
  const uint64_t per_block = (uint64_t)PTAU_BLOCK * PTAU_GEN_B;
  const unsigned grid = (unsigned)((n + per_block - 1) / per_block);
  if (group == PTAU_G1)
    contribute_kernel<PTAU_G1><<<grid, PTAU_BLOCK, 0, stream>>>(fp, (const uint32_t*)d_in, (uint32_t*)d_out, first, n);
  else
    contribute_kernel<PTAU_G2><<<grid, PTAU_BLOCK, 0, stream>>>(fp, (const uint32_t*)d_in, (uint32_t*)d_out, first, n);
  return cudaGetLastError();
}

void fr_words(const Fr& a, uint32_t* w) { memcpy(w, a.l, 32); }

bool fr_is_zero(const Fr& a) { return (a.l[0] | a.l[1] | a.l[2] | a.l[3]) == 0; }

void blake2b_bytes(Blake2b& h, uint8_t* out) {
  const std::string hx = h.hexdigest();
  for (int i = 0; i < 64; i++) out[i] = (uint8_t)std::stoi(hx.substr(2 * i, 2), nullptr, 16);
}

// One section of a contribution: in = count uncompressed records, out = count compressed records.
int contribute_section(ptau_ctx* ctx, int group, const uint8_t* in, uint8_t* out, uint64_t count, unsigned checks,
                       const FrParams& fp, uint64_t* bad_index, int* bad_kind) {
  const int ri = rec_size(group, PTAU_FMT_ZCASH_UNCOMPRESSED), rm = rec_size(group, PTAU_FMT_ARK_MONT_LIMBS);
  const int ro = rec_size(group, PTAU_FMT_ZCASH_COMPRESSED);
  const size_t chunk = ctx->chunk_points;
  const int G = count >= (uint64_t)ctx->n_gpus * 4096 ? ctx->n_gpus : 1;  // a few points: one GPU
  ptau_timing& tm = ctx->timing;
  struct Range {
    uint64_t lo, hi, next;
    int issued;
  } rg[kMaxGpus];
  const unsigned long long none = PTAU_STATUS_NONE;
  for (int g = 0; g < G; g++) {
    const Shard sh = shard(count, g, G);
    rg[g] = {sh.lo, sh.hi, sh.lo, 0};
    GpuSlot& s = ctx->gpu[g];
    CUDA_TRY(ctx, cudaSetDevice(s.device));
    const size_t maxpts = sh.hi - sh.lo < chunk ? sh.hi - sh.lo : chunk;
    CUDA_TRY(ctx, ensure_buffers(s.d_in, &s.cap_in, maxpts * ri + 16));
    CUDA_TRY(ctx, ensure_buffers(s.d_out, &s.cap_out, maxpts * rm + 16));
    CUDA_TRY(ctx, cudaMemcpyAsync(s.d_status, &none, sizeof(none), cudaMemcpyHostToDevice, s.stream[0]));
    CUDA_TRY(ctx, cudaEventRecord(s.ev_first, s.stream[0]));
    CUDA_TRY(ctx, cudaStreamWaitEvent(s.stream[1], s.ev_first, 0));
  }
  // breadth-first issue: one chunk per GPU per round, alternating the two streams
  bool more = true;
  while (more) {
    more = false;
    for (int g = 0; g < G; g++) {
      Range& r = rg[g];
      if (r.next >= r.hi) continue;
      GpuSlot& s = ctx->gpu[g];
      CUDA_TRY(ctx, cudaSetDevice(s.device));
      const int b = r.issued % kBufs;
      const size_t npts = r.hi - r.next < chunk ? r.hi - r.next : chunk;
      if (r.issued >= kBufs) {  // the event pair of this buffer is about to be reused: harvest its time
        CUDA_TRY(ctx, cudaEventSynchronize(s.ev_k1[b]));
        float ms = 0;
        CUDA_TRY(ctx, cudaEventElapsedTime(&ms, s.ev_k0[b], s.ev_k1[b]));
        tm.kernel_ms[g] += ms;
      }
      CUDA_TRY(ctx, cudaMemcpyAsync(s.d_in[b], in + r.next * ri, npts * ri, cudaMemcpyHostToDevice, s.stream[b]));
      CUDA_TRY(ctx, cudaEventRecord(s.ev_k0[b], s.stream[b]));
      CUDA_TRY(ctx, launch_convert(group, PTAU_FMT_ZCASH_UNCOMPRESSED, PTAU_FMT_ARK_MONT_LIMBS, s.d_in[b], s.d_out[b], npts,
                                   checks, r.next, s.d_status, s.stream[b]));
      CUDA_TRY(ctx, launch_contribute(group, fp, s.d_out[b], s.d_in[b], r.next, npts, s.stream[b]));
      CUDA_TRY(ctx, cudaEventRecord(s.ev_k1[b], s.stream[b]));
      CUDA_TRY(ctx, cudaMemcpyAsync(out + r.next * ro, s.d_in[b], npts * ro, cudaMemcpyDeviceToHost, s.stream[b]));
      tm.h2d_bytes[g] += npts * ri;
      tm.d2h_bytes[g] += npts * ro;
      tm.kernel_launches += 2;
      r.next += npts;
      r.issued++;
      more = true;
    }
  }
  unsigned long long status = PTAU_STATUS_NONE;
  for (int g = 0; g < G; g++) {
    GpuSlot& s = ctx->gpu[g];
    CUDA_TRY(ctx, cudaSetDevice(s.device));
    CUDA_TRY(ctx, cudaEventRecord(s.ev_last, s.stream[1]));
    CUDA_TRY(ctx, cudaStreamWaitEvent(s.stream[0], s.ev_last, 0));
    unsigned long long st = PTAU_STATUS_NONE;
    CUDA_TRY(ctx, cudaMemcpyAsync(&st, s.d_status, sizeof(st), cudaMemcpyDeviceToHost, s.stream[0]));
    CUDA_TRY(ctx, cudaEventRecord(s.ev_last, s.stream[0]));
    CUDA_TRY(ctx, cudaStreamSynchronize(s.stream[0]));
    CUDA_TRY(ctx, cudaStreamSynchronize(s.stream[1]));
    if (st < status) status = st;
    float ms = 0;
    CUDA_TRY(ctx, cudaEventElapsedTime(&ms, s.ev_first, s.ev_last));
    tm.gpu_ms[g] += ms;
    const int pending = rg[g].issued < kBufs ? rg[g].issued : kBufs;
    for (int b = 0; b < pending; b++) {
      float k = 0;
      CUDA_TRY(ctx, cudaEventElapsedTime(&k, s.ev_k0[b], s.ev_k1[b]));
      tm.kernel_ms[g] += k;
    }
  }
  if (status != PTAU_STATUS_NONE) {
    if (bad_index) *bad_index = status >> 8;
    if (bad_kind) *bad_kind = (int)(status & 0xff);
    return (int)(status & 0xff);
  }
  return PTAU_OK;
}

// powersoftau keypair for given secrets (canonical, non-zero): for (x, s, personalization) in (tau, s_tau, 0),
// (alpha, s_alpha, 1), (beta, s_beta, 2): g1_s = [s]G1, g1_s_x = [x]g1_s, g2_s = hash_to_g2(BLAKE2b(personalization ||
// digest || g1_s || g1_s_x)), key G2 element [x]g2_s.  out: the 1152-byte uncompressed PublicKey.
void public_key(const uint8_t* digest, const Fr* sec, uint8_t* out) {
  uint32_t x[8], s[8];
  for (int i = 0; i < 3; i++) {
    fr_words(sec[i], x);
    fr_words(sec[3 + i], s);
    Jac<Fq> a;
    Fq sx, sy, tx, ty;
    jac_scalar_mul_t(a, k_g1x_mont(), k_g1y_mont(), s, fq_one());
    jac_to_affine_t(a, sx, sy);
    jac_scalar_mul_t(a, sx, sy, x, fq_one());
    jac_to_affine_t(a, tx, ty);
    uint8_t* g1 = out + 2 * i * 96;
    zcash_g1_uncompressed(sx, sy, g1);
    zcash_g1_uncompressed(tx, ty, g1 + 96);
    Blake2b h;
    const uint8_t pers = (uint8_t)i;
    h.update(&pers, 1);
    h.update(digest, 64);
    h.update(g1, 192);
    uint8_t hd[64];
    blake2b_bytes(h, hd);
    Fq2 gx, gy, kx, ky;
    hash_to_g2(hd, gx, gy);
    Jac<Fq2> b;
    jac_scalar_mul_t(b, gx, gy, x, fq2_one());
    jac_to_affine_t(b, kx, ky);
    zcash_g2_uncompressed(kx, ky, out + 6 * 96 + i * 192);
  }
  explicit_bzero(x, sizeof(x));
  explicit_bzero(s, sizeof(s));
}

// a uniformly drawn non-zero scalar < r from getrandom(2)
bool draw_scalar(Fr* out) {
  for (;;) {
    uint8_t b[32];
    size_t got = 0;
    while (got < 32) {
      const ssize_t r = getrandom(b + got, 32 - got, 0);
      if (r <= 0) return false;
      got += (size_t)r;
    }
    b[31] &= 0x7f;  // r < 2^255
    *out = fr_from_le32(b);
    explicit_bzero(b, sizeof(b));
    if (!fr_ge_mod(out->l) && !fr_is_zero(*out)) return true;
  }
}

// ARK_MONT_LIMBS G1 record with y negated (Montgomery limbs: -(yR) = (-y)R)
void neg_g1_rec(const uint8_t* rec, uint8_t* out) {
  Fq x, y;
  bool inf;
  uint32_t w[26];
  memcpy(w, rec, 104);
  load_g1_rec(w, x, y, inf);
  store_rec(w, x, fq_neg(y), inf);
  memcpy(out, w, 104);
}

}  // namespace
}  // namespace ptau

using namespace ptau;

extern "C" uint64_t ptau_challenge_size(uint64_t n) { return kResponseHash + response_bytes(n, PTAU_FMT_ZCASH_UNCOMPRESSED); }

extern "C" int ptau_contribute(ptau_ctx* ctx, const void* challenge, uint64_t challenge_len, uint64_t n,
                               const uint8_t* secrets, unsigned checks, void* response_out, uint64_t response_len,
                               uint64_t* bad_index, int* bad_kind, int* bad_section) {
  if (!ctx || !challenge || !response_out) return PTAU_ERR_ARG;
  if (n < 2 || n > (1ull << 40)) return PTAU_ERR_ARG;
  if (challenge_len != ptau_challenge_size(n) || response_len != ptau_response_size(n)) return PTAU_ERR_SIZE;
  // tau, alpha, beta, s_tau, s_alpha, s_beta
  Fr sec[6];
  FrParams fp;
  int rc = PTAU_OK;
  for (int i = 0; i < 6 && rc == PTAU_OK; i++) {
    if (secrets) {
      sec[i] = fr_from_le32(secrets + 32 * i);
      if (fr_ge_mod(sec[i].l) || fr_is_zero(sec[i])) rc = PTAU_ERR_ARG;
    } else if (!draw_scalar(&sec[i])) {
      rc = PTAU_ERR_IO;
    }
  }
  if (rc != PTAU_OK) {
    explicit_bzero(sec, sizeof(sec));
    return rc;
  }
  const auto t0 = std::chrono::steady_clock::now();
  timing_reset(ctx);
  const uint8_t* in = (const uint8_t*)challenge;
  uint8_t* out = (uint8_t*)response_out;
  uint8_t digest[64];
  std::thread hasher([&] {
    Blake2b h;
    h.update(in, challenge_len);
    blake2b_bytes(h, digest);
  });
  // the sections' scalars s0 * tau^i: tau_g1, tau_g2 (s0 = 1), alpha_g1 (alpha), beta_g1 and beta_g2 (beta; beta_g2 is
  // one point, i = 0)
  Fr p = fr_to_mont(sec[0]);
  for (int j = 0; j < 64; j++) {
    fr_words(p, fp.pw[j]);
    p = fr_mont_mul(p, p);
  }
  Fr one{{1, 0, 0, 0}};
  const Fr* s0[5] = {&one, &one, &sec[1], &sec[2], &sec[2]};
  uint64_t off_in = kResponseHash, off_out = kResponseHash;
  const auto secs = response_sections(n);
  for (int s = 0; s < 5; s++) {
    Fr m = fr_to_mont(*s0[s]);
    fr_words(m, fp.s0);
    explicit_bzero(&m, sizeof(m));
    rc = contribute_section(ctx, secs[s].group, in + off_in, out + off_out, secs[s].count, checks, fp, bad_index,
                            bad_kind);
    if (rc != PTAU_OK) {
      if (rc > 0 && bad_section) *bad_section = s;
      break;
    }
    off_in += secs[s].count * rec_size(secs[s].group, PTAU_FMT_ZCASH_UNCOMPRESSED);
    off_out += secs[s].count * rec_size(secs[s].group, PTAU_FMT_ZCASH_COMPRESSED);
  }
  hasher.join();
  if (rc == PTAU_OK) {
    memcpy(out, digest, 64);
    public_key(digest, sec, out + off_out);
  }
  explicit_bzero(sec, sizeof(sec));
  explicit_bzero(&fp, sizeof(fp));
  explicit_bzero(&p, sizeof(p));
  ctx->timing.wall_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
  return rc;
}

extern "C" int ptau_verify_contribution(ptau_ctx* ctx, const void* challenge, uint64_t challenge_len,
                                        const void* response, uint64_t response_len, uint64_t n, const uint8_t seed[32],
                                        uint64_t* bad_index, int* bad_kind, int* bad_section, int* bad_relation) {
  if (!ctx || !response) return PTAU_ERR_ARG;
  if (n < 2 || n > (1ull << 40)) return PTAU_ERR_ARG;
  if (response_len != ptau_response_size(n)) return PTAU_ERR_SIZE;
  if (challenge && challenge_len != ptau_challenge_size(n)) return PTAU_ERR_SIZE;
  const auto t0 = std::chrono::steady_clock::now();
  const uint8_t* resp = (const uint8_t*)response;
  const uint8_t* chal = (const uint8_t*)challenge;
  const uint8_t* pk = resp + kResponseHash + response_bytes(n, PTAU_FMT_ZCASH_COMPRESSED);
  auto fail_point = [&](int rc, int section, uint64_t index) {
    if (rc > 0) {
      if (bad_section) *bad_section = section;
      if (bad_index) *bad_index = index;
    }
    return rc;
  };
  // ---- the public key's nine points, strict (powersoftau PublicKey::deserialize): section 5, index in key order
  uint8_t key1[6 * kMontG1], key2[3 * kMontG2];
  uint64_t bi = 0;
  int rc = ptau_convert(ctx, PTAU_G1, PTAU_FMT_ZCASH_UNCOMPRESSED, pk, PTAU_FMT_ARK_MONT_LIMBS, key1, 6, PTAU_CHECKS_STRICT,
                        &bi, bad_kind);
  if (rc) return fail_point(rc, 5, bi);
  rc = ptau_convert(ctx, PTAU_G2, PTAU_FMT_ZCASH_UNCOMPRESSED, pk + 6 * 96, PTAU_FMT_ARK_MONT_LIMBS, key2, 3,
                    PTAU_CHECKS_STRICT, &bi, bad_kind);
  if (rc) return fail_point(rc, 5, 6 + bi);
  // ---- the points of the transform relations: tau_g1[1], alpha_g1[0], beta_g1[0], beta_g2 of both accumulators
  const auto secs = response_sections(n);
  uint64_t off_u[5], off_c[5];  // byte offsets of the sections in the challenge and the response (past the hash)
  for (int s = 0; s < 5; s++) {
    off_u[s] = kResponseHash + section_offset(n, PTAU_FMT_ZCASH_UNCOMPRESSED, s);
    off_c[s] = kResponseHash + section_offset(n, PTAU_FMT_ZCASH_COMPRESSED, s);
  }
  const int rsec[4] = {0, 2, 3, 4};
  const uint64_t ridx[4] = {1, 0, 0, 0};
  uint8_t before[4][kMontG2], after[4][kMontG2];
  if (chal) {
    for (int k = 0; k < 4; k++) {
      const int g = secs[rsec[k]].group;
      rc = ptau_convert(ctx, g, PTAU_FMT_ZCASH_UNCOMPRESSED,
                        chal + off_u[rsec[k]] + ridx[k] * rec_size(g, PTAU_FMT_ZCASH_UNCOMPRESSED),
                        PTAU_FMT_ARK_MONT_LIMBS, before[k], 1, PTAU_CHECKS_STRICT, &bi, bad_kind);
      if (rc) return fail_point(rc, 6 + rsec[k], ridx[k]);
    }
  }
  // ---- the response's own points and powers (ptau_verify_powers: bad points as sections 0-4, relations 0-5)
  int rel = -1;
  rc = ptau_verify_powers(ctx, PTAU_POWERS_RESPONSE, response, response_len, n, seed, bad_index, bad_kind, bad_section,
                          &rel, nullptr);
  if (rc == PTAU_BAD_NOT_POWERS && bad_relation) *bad_relation = rel;
  if (rc) return rc;
  const auto not_powers = [&](int relation) {
    if (bad_relation) *bad_relation = relation;
    return PTAU_BAD_NOT_POWERS;
  };
  for (int k = 0; k < 4; k++) {
    const int g = secs[rsec[k]].group;
    rc = ptau_convert(ctx, g, PTAU_FMT_ZCASH_COMPRESSED,
                      resp + off_c[rsec[k]] + ridx[k] * rec_size(g, PTAU_FMT_ZCASH_COMPRESSED), PTAU_FMT_ARK_MONT_LIMBS,
                      after[k], 1, PTAU_CHECKS_STRICT, &bi, bad_kind);
    if (rc) return fail_point(rc, rsec[k], ridx[k]);
  }
  // ---- HASH: the response names the challenge it transformed
  uint8_t digest[64];
  if (chal) {
    Blake2b h;
    h.update(chal, challenge_len);
    blake2b_bytes(h, digest);
    if (memcmp(digest, resp, 64) != 0) return not_powers(PTAU_REL_HASH);
  } else {
    memcpy(digest, resp, 64);
  }
  // ---- g2_s of each proof of knowledge, recomputed from the key's G1 pair
  uint8_t g2s[3][kMontG2];
  for (int i = 0; i < 3; i++) {
    Blake2b h;
    const uint8_t pers = (uint8_t)i;
    h.update(&pers, 1);
    h.update(digest, 64);
    h.update(pk + 2 * i * 96, 192);
    uint8_t hd[64];
    blake2b_bytes(h, hd);
    Fq2 x, y;
    hash_to_g2(hd, x, y);
    uint32_t w[50];
    store_rec(w, x, y, false);
    memcpy(g2s[i], w, kMontG2);
  }
  // ---- same_ratio((a, b), (c, d)): e(a, d) e(-b, c) = 1, one item each, in relation order
  const int items = chal ? 7 : 3;
  uint8_t g1[7][2][kMontG1], g2[7][2][kMontG2];
  for (int i = 0; i < 3; i++) {  // POK: ((s, s x), (g2_s, [x] g2_s))
    memcpy(g1[i][0], key1 + 2 * i * kMontG1, kMontG1);
    neg_g1_rec(key1 + (2 * i + 1) * kMontG1, g1[i][1]);
    memcpy(g2[i][0], key2 + i * kMontG2, kMontG2);
    memcpy(g2[i][1], g2s[i], kMontG2);
  }
  if (chal) {
    for (int i = 0; i < 3; i++) {  // CHAIN: ((before, after), (g2_s, [x] g2_s))
      memcpy(g1[3 + i][0], before[i], kMontG1);
      neg_g1_rec(after[i], g1[3 + i][1]);
      memcpy(g2[3 + i][0], key2 + i * kMontG2, kMontG2);
      memcpy(g2[3 + i][1], g2s[i], kMontG2);
    }
    // CHAIN_BETA_G2: ((before.beta_g1[0], after.beta_g1[0]), (before.beta_g2, after.beta_g2))
    memcpy(g1[6][0], before[2], kMontG1);
    neg_g1_rec(after[2], g1[6][1]);
    memcpy(g2[6][0], after[3], kMontG2);
    memcpy(g2[6][1], before[3], kMontG2);
  }
  uint8_t ok[7];
  rc = ptau_pairing_product2(ctx, g1, g2, items, nullptr, ok);
  if (rc) return rc;
  ctx->timing.wall_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
  for (int i = 0; i < items; i++)
    if (!ok[i]) return not_powers(PTAU_REL_POK_TAU + i);
  return PTAU_OK;
}
