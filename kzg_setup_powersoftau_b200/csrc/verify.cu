// ptau_verify_powers: does a `powersoftau` response or a `kzg_setup` hold powers of ONE tau?
//
// Every point goes through the strict per-point path (launch_convert, PTAU_CHECKS_STRICT) into device-resident
// ARK_MONT_LIMBS records.  A section S of length L (a ratio relation k) is then reduced to two points with the
// coefficients rho_{k,i} (blake2b.h: ratio_coeff, derived on the device):
//     A = sum_{i < L-1} rho_{k,i} S_i,    B = sum_{i < L-1} rho_{k,i} S_{i+1},
// two bucket MSMs over the same records, one shifted by one point.  The relation holds iff e(B, Q0) e(-A, Q1) = 1
// (G1 section, reference pair Q0, Q1 in G2) or e(P0, B) e(-P1, A) = 1 (G2 section, reference pair P0, P1 in G1);
// all relations go through one pairing_product2 launch.
//
// Streaming: a section's pairs are split into contiguous ranges over the context's GPUs, and every range is cut into
// slabs of kSlabChunks * chunk_points pairs.  A slab of pairs [a, b) converts points [a, b + 1): the one point past
// its end is converted again by the next slab, so every pair (S_i, S_{i+1}) is counted by exactly one slab.  Each
// slab's A and B land in a partial-result slot; the partials are summed on GPU 0 by an MSM with unit scalars.
// Device memory per GPU is a function of chunk_points only (see the header), never of n_powers.
#include <cuda_runtime.h>
#include <stdint.h>
#include <string.h>
#include <sys/random.h>

#include <chrono>
#include <string>
#include <vector>

#include "../../include/ptau_b200.h"
#include "blake2b.h"
#include "context.h"
#include "curve.cuh"
#include "kernels.h"
#include "layout.h"

namespace ptau {

constexpr uint64_t kSlabChunks = 16;  // MSM slab = 16 conversion chunks: 2^22 pairs at the default chunk of 2^18

struct B2Key {
  uint64_t h[8];
};

// rho_{k, first + i} for i < n, as 8 x u32 little-endian scalars, straight into the MSM's scalar buffer
__global__ void __launch_bounds__(256) ratio_coeff_kernel(B2Key key, uint32_t k, uint64_t first, uint64_t n,
                                                          uint32_t* __restrict__ out) {
  const uint64_t i = (uint64_t)blockIdx.x * 256 + threadIdx.x;
  if (i >= n) return;
  ratio_coeff(key.h, k, first + i, out + i * 8);
}

// key points, converted into one device buffer on GPU 0: G1 records in 32-word slots first, then G2 records in
// 64-word slots (the conversion kernels store to 16-byte aligned records)
enum { K1_P0, K1_P1, K1_BETA0, K1_G, K1_GAMMA_G, K1_GAMMA0, K1_N };
enum { K2_Q0, K2_Q1, K2_BETA_G2, K2_H, K2_BETA_H, K2_N };
constexpr int kKeyWords = K1_N * 32 + K2_N * 64;
constexpr int kItems = 5;  // pairing items: relations TAU_G1 .. BETA_G2

__device__ bool rec_eq(const uint32_t* a, const uint32_t* b, int coord_words) {
  bool eq = (a[coord_words] & 0xffu) == (b[coord_words] & 0xffu);
  for (int w = 0; w < coord_words; w++) eq = eq && a[w] == b[w];
  return eq;
}
__device__ void rec_copy(uint32_t* d, const uint32_t* s, int words) {
  for (int w = 0; w < words; w++) d[w] = s[w];
}
__device__ void rec_infinity(uint32_t* d, int words) {
  for (int w = 0; w < words; w++) d[w] = 0;
  d[words - 2] = 1;
}
// -P of a G1 record: y -> p - y (an infinity record stays as it is)
__device__ void rec_neg_g1(uint32_t* d, const uint32_t* s) {
  rec_copy(d, s, 26);
  if (s[24] & 0xffu) return;
  Fq y;
  for (int w = 0; w < 12; w++) y.l[w] = s[12 + w];
  y = fq_neg(y);
  for (int w = 0; w < 12; w++) d[12 + w] = y.l[w];
}

// One thread: the pairing items of the ratio relations and BETA_G2 (g1: kItems x 2 x 26 words, g2: kItems x 2 x 50),
// and the record comparisons: flags[0] = GENERATORS holds, flags[1] = KEY holds.  combo: 8 slots of 50 words
// (slot 2k-2 = A_k, 2k-1 = B_k).  rel_mask bit k: relation k applies to the kind.
__global__ void verify_assemble_kernel(const uint32_t* __restrict__ keys, const uint32_t* __restrict__ combo, int kind,
                                       uint32_t rel_mask, uint32_t* __restrict__ g1, uint32_t* __restrict__ g2,
                                       uint32_t* __restrict__ flags) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
#define K1(slot) (keys + (slot) * 32)
#define K2(slot) (keys + K1_N * 32 + (slot) * 64)
  for (int it = 0; it < kItems; it++) {
    const int rel = it + 1;
    uint32_t* a = g1 + it * 52;
    uint32_t* b = g2 + it * 100;
    const uint32_t* A = combo + (2 * rel - 2) * 50;
    const uint32_t* B = combo + (2 * rel - 1) * 50;
    if (!((rel_mask >> rel) & 1u)) {
      rec_infinity(a, 26);
      rec_infinity(a + 26, 26);
      rec_copy(b, K2(K2_Q0), 50);
      rec_copy(b + 50, K2(K2_Q0), 50);
    } else if (rel == PTAU_REL_TAU_G2) {  // e(P0, B) e(-P1, A)
      rec_copy(a, K1(K1_P0), 26);
      rec_neg_g1(a + 26, K1(K1_P1));
      rec_copy(b, B, 50);
      rec_copy(b + 50, A, 50);
    } else if (rel == PTAU_REL_BETA_G2) {  // e(beta_g1[0], H) e(-G, beta_g2)
      rec_copy(a, K1(K1_BETA0), 26);
      rec_neg_g1(a + 26, K1(K1_P0));
      rec_copy(b, K2(K2_Q0), 50);
      rec_copy(b + 50, K2(K2_BETA_G2), 50);
    } else {  // G1 section: e(B, Q0) e(-A, Q1)
      rec_copy(a, B, 26);
      rec_neg_g1(a + 26, A);
      rec_copy(b, K2(K2_Q0), 50);
      rec_copy(b + 50, K2(K2_Q1), 50);
    }
  }
  uint32_t gen1[26], gen2[50];
  const Fq c[6] = {k_g1x_mont(), k_g1y_mont(), k_g2x0_mont(), k_g2x1_mont(), k_g2y0_mont(), k_g2y1_mont()};
  for (int w = 0; w < 12; w++) {
    gen1[w] = c[0].l[w];
    gen1[12 + w] = c[1].l[w];
    for (int j = 0; j < 4; j++) gen2[12 * j + w] = c[2 + j].l[w];
  }
  gen1[24] = gen1[25] = 0;
  gen2[48] = gen2[49] = 0;
  flags[0] = rec_eq(K1(K1_P0), gen1, 24) && rec_eq(K2(K2_Q0), gen2, 48);
  if (kind == PTAU_POWERS_KGZ)
    flags[1] = rec_eq(K1(K1_G), K1(K1_P0), 24) && rec_eq(K1(K1_GAMMA_G), K1(K1_GAMMA0), 24);
  else if (kind == PTAU_POWERS_FASTKGZ)
    flags[1] = rec_eq(K2(K2_H), K2(K2_Q0), 48) && rec_eq(K2(K2_BETA_H), K2(K2_Q1), 48);
  else
    flags[1] = 1;
#undef K1
#undef K2
}

namespace {

// A contiguous run of points of one input section (the unit of error reporting): `rel` = 0 (validated only) or the
// ratio relation whose section it is.
struct Piece {
  int sec;         // index into the section table
  uint64_t first;  // first point, section-relative
  uint64_t count;
  int rel;
};
struct Sec {
  int group;
  const uint8_t* data;  // first byte of the section
  uint64_t count;
};
struct KeyPoint {
  int sec;
  uint64_t index;
  int slot;  // K1_* (G1) or K2_* (G2)
};
// one slab of work on one GPU: points [a, b) of a piece are converted; with a relation, pairs [a, b - 1) are summed
struct Job {
  int gpu, piece;
  uint64_t a, b;
  int part;  // first of its two partial-result slots (A, B) on that GPU; -1 without a relation
};

struct GpuWork {
  void* d_rec = nullptr;
  void* d_sc = nullptr;
  void* d_scratch = nullptr;
  void* d_in[kBufs] = {nullptr, nullptr};
  unsigned long long* d_status = nullptr;  // one word per section
  uint8_t* d_parts = nullptr;              // 256-byte slots: MSM result record + "scalar >= r" word
  int parts = 0;
  cudaEvent_t ev = nullptr;
};

struct Run {
  ptau_ctx* ctx;
  int G = 1;
  GpuWork w[kMaxGpus];
  void *d_keys = nullptr, *d_keys_in = nullptr, *d_combo = nullptr, *d_g1 = nullptr, *d_g2 = nullptr, *d_flags = nullptr,
       *d_one = nullptr;
  unsigned long long* d_key_status = nullptr;
  ~Run() {
    for (int g = 0; g < G; g++) {
      GpuSlot& s = ctx->gpu[g];
      cudaSetDevice(s.device);
      for (int b = 0; b < kBufs; b++) cudaStreamSynchronize(s.stream[b]);
      GpuWork& x = w[g];
      void* ps[] = {x.d_rec, x.d_sc, x.d_scratch, x.d_in[0], x.d_in[1], x.d_status, x.d_parts};
      for (void* p : ps)
        if (p) cudaFree(p);
      if (x.ev) cudaEventDestroy(x.ev);
      if (g == 0) {
        void* qs[] = {d_keys, d_keys_in, d_combo, d_g1, d_g2, d_flags, d_one, d_key_status};
        for (void* p : qs)
          if (p) cudaFree(p);
      }
    }
  }
};

}  // namespace
}  // namespace ptau

using namespace ptau;

extern "C" int ptau_verify_powers(ptau_ctx* ctx, int kind, const void* data, uint64_t len, uint64_t n,
                                  const uint8_t seed[32], uint64_t* bad_index, int* bad_kind, int* bad_section,
                                  int* bad_relation, void* combos_out) {
  if (!ctx || !data) return PTAU_ERR_ARG;
  if (kind != PTAU_POWERS_RESPONSE && kind != PTAU_POWERS_KGZ && kind != PTAU_POWERS_FASTKGZ) return PTAU_ERR_ARG;
  if (n < 2 || n > (1ull << 40)) return PTAU_ERR_ARG;
  const int variant = kind == PTAU_POWERS_KGZ ? PTAU_VARIANT_KGZ : PTAU_VARIANT_FASTKGZ;  // of a setup
  const uint64_t want = kind == PTAU_POWERS_RESPONSE ? ptau_response_size(n) : ptau_setup_size(variant, n);
  if (len != want) return PTAU_ERR_SIZE;
  const auto t0 = std::chrono::steady_clock::now();
  const uint8_t* base = (const uint8_t*)data;

  // ---- layout: sections (the unit of error reporting, as in ptau_preprocess / ptau_load_setup), pieces, key points
  std::vector<Sec> secs;
  std::vector<Piece> pieces;
  std::vector<KeyPoint> keys;
  uint32_t rel_mask = 0;
  int fmt;
  uint64_t g2_index_offset = 0;  // setups report a G2 index in file order over all points
  if (kind == PTAU_POWERS_RESPONSE) {
    fmt = PTAU_FMT_ZCASH_COMPRESSED;
    const uint8_t* p = base + kResponseHash;  // the trailing public key is not read
    for (const Section& s : response_sections(n)) {
      secs.push_back({s.group, p, s.count});
      p += s.count * rec_size(s.group, fmt);
    }
    pieces = {{0, 0, secs[0].count, PTAU_REL_TAU_G1}, {1, 0, n, PTAU_REL_TAU_G2}, {2, 0, n, PTAU_REL_ALPHA_G1},
              {3, 0, n, PTAU_REL_BETA_G1}, {4, 0, 1, 0}};
    keys = {{0, 0, K1_P0}, {0, 1, K1_P1}, {3, 0, K1_BETA0}, {1, 0, K2_Q0}, {1, 1, K2_Q1}, {4, 0, K2_BETA_G2}};
    rel_mask = (1u << PTAU_REL_TAU_G1) | (1u << PTAU_REL_TAU_G2) | (1u << PTAU_REL_ALPHA_G1) | (1u << PTAU_REL_BETA_G1) |
               (1u << PTAU_REL_BETA_G2);
  } else {
    fmt = PTAU_FMT_ARK_UNCOMPRESSED;
    const SetupLayout L = setup_layout(variant, n);
    secs.push_back({PTAU_G1, base, L.n_g1});
    secs.push_back({PTAU_G2, base + L.g2(0), L.n_g2});
    g2_index_offset = L.n_g1;
    // powers_of_g are G1 records [0, gamma_g)
    pieces = {{0, 0, L.gamma_g, PTAU_REL_TAU_G1}, {0, L.gamma_g, n, PTAU_REL_ALPHA_G1}};
    keys = {{0, 0, K1_P0}, {0, 1, K1_P1}, {0, L.gamma_g, K1_GAMMA0}};
    rel_mask = (1u << PTAU_REL_TAU_G1) | (1u << PTAU_REL_ALPHA_G1);
    if (variant == PTAU_VARIANT_FASTKGZ) {
      pieces.push_back({1, 0, 2, 0});
      pieces.push_back({1, L.powers_of_h, n, PTAU_REL_TAU_G2});
      keys.push_back({1, L.powers_of_h, K2_Q0});
      keys.push_back({1, L.powers_of_h + 1, K2_Q1});
      keys.push_back({1, 0, K2_H});
      keys.push_back({1, 1, K2_BETA_H});
      rel_mask |= 1u << PTAU_REL_TAU_G2;
    } else {
      pieces.push_back({0, L.vk_g, 2, 0});
      pieces.push_back({1, 0, 2, 0});
      keys.push_back({0, L.vk_g, K1_G});
      keys.push_back({0, L.vk_g + 1, K1_GAMMA_G});
      keys.push_back({1, 0, K2_Q0});
      keys.push_back({1, 1, K2_Q1});
    }
  }
  const int nsec = (int)secs.size();

  // ---- coefficients: the keyed first block of BLAKE2b is the same for every coefficient
  uint8_t sd[32];
  if (seed) {
    memcpy(sd, seed, 32);
  } else {
    size_t got = 0;
    while (got < 32) {
      ssize_t r = getrandom(sd + got, 32 - got, 0);
      if (r <= 0) return PTAU_ERR_IO;
      got += (size_t)r;
    }
  }
  B2Key key;
  blake2b_keyed_start(key.h, sd, 32, 16);

  // ---- schedule: pairs of every relation piece split over the GPUs, then into slabs
  const size_t chunk = (ctx->chunk_points + 15) & ~(size_t)15;  // keeps every chunk's output record 16-byte aligned
  const uint64_t slab = kSlabChunks * chunk;
  Run run;
  run.ctx = ctx;
  run.G = ctx->n_gpus;
  const int G = run.G;
  std::vector<Job> jobs;
  uint64_t max_pts = 1;
  for (int pi = 0; pi < (int)pieces.size(); pi++) {
    const Piece& pc = pieces[pi];
    if (!pc.rel) {  // a few points: validated on GPU 0
      jobs.push_back({0, pi, 0, pc.count, -1});
      continue;
    }
    const uint64_t P = pc.count - 1;
    const int Gp = P >= (uint64_t)G * 4096 ? G : 1;
    for (int g = 0; g < Gp; g++) {
      const auto [lo, hi] = shard(P, g, Gp);
      for (uint64_t a = lo; a < hi; a += slab) {
        const uint64_t b = a + slab < hi ? a + slab : hi;
        jobs.push_back({g, pi, a, b + 1, run.w[g].parts});
        run.w[g].parts += 2;
        if (b + 1 - a > max_pts) max_pts = b + 1 - a;
      }
    }
  }
  // ---- device buffers (sizes bounded by the slab, i.e. by chunk_points)
  const int rb_max = kMontG2;
  const int ri_max = rec_size(PTAU_G2, fmt);
  ptau::MsmPlan p1, p2;
  msm_g1_plan(max_pts, &p1);
  msm_g2_plan(max_pts, &p2);
  const size_t scratch = p1.scratch_bytes > p2.scratch_bytes ? p1.scratch_bytes : p2.scratch_bytes;
  const size_t conv = chunk < max_pts ? chunk : max_pts;
  const unsigned long long none = PTAU_STATUS_NONE;
  std::vector<unsigned long long> none_v(nsec, none);
  for (int g = 0; g < G; g++) {
    GpuSlot& s = ctx->gpu[g];
    GpuWork& x = run.w[g];
    CUDA_TRY(ctx, cudaSetDevice(s.device));
    CUDA_TRY(ctx, cudaMalloc(&x.d_rec, max_pts * rb_max + 16));
    CUDA_TRY(ctx, cudaMalloc(&x.d_in[0], conv * ri_max + 16));
    CUDA_TRY(ctx, cudaMalloc(&x.d_in[1], conv * ri_max + 16));
    CUDA_TRY(ctx, cudaMalloc((void**)&x.d_status, nsec * 8));
    CUDA_TRY(ctx, cudaEventCreateWithFlags(&x.ev, cudaEventDisableTiming));
    if (x.parts) {
      CUDA_TRY(ctx, cudaMalloc(&x.d_sc, max_pts * 32 + 16));
      CUDA_TRY(ctx, cudaMalloc(&x.d_scratch, scratch));
      CUDA_TRY(ctx, cudaMalloc((void**)&x.d_parts, (size_t)x.parts * 256));
    }
    CUDA_TRY(ctx, cudaMemcpyAsync(x.d_status, none_v.data(), nsec * 8, cudaMemcpyHostToDevice, s.stream[0]));
    // none_v is a local; stream[1] must also see the initialised words
    CUDA_TRY(ctx, cudaStreamSynchronize(s.stream[0]));
  }
  uint64_t launches = 0, h2d = 0;

  // ---- key points on GPU 0 (their checks are the main pass's; this status word is not read)
  {
    GpuSlot& s = ctx->gpu[0];
    CUDA_TRY(ctx, cudaSetDevice(s.device));
    CUDA_TRY(ctx, cudaMalloc(&run.d_keys, kKeyWords * 4));
    CUDA_TRY(ctx, cudaMalloc(&run.d_keys_in, 256));
    CUDA_TRY(ctx, cudaMalloc((void**)&run.d_key_status, 8));
    CUDA_TRY(ctx, cudaMemsetAsync(run.d_keys, 0, kKeyWords * 4, s.stream[0]));
    for (const KeyPoint& kp : keys) {
      const Sec& sc = secs[kp.sec];
      const int ri = rec_size(sc.group, fmt);
      uint32_t* dst = (uint32_t*)run.d_keys + (sc.group == PTAU_G1 ? kp.slot * 32 : K1_N * 32 + kp.slot * 64);
      CUDA_TRY(ctx, cudaMemcpyAsync(run.d_keys_in, sc.data + kp.index * ri, ri, cudaMemcpyHostToDevice, s.stream[0]));
      CUDA_TRY(ctx, launch_convert(sc.group, fmt, PTAU_FMT_ARK_MONT_LIMBS, run.d_keys_in, dst, 1, PTAU_CHECKS_STRICT, 0,
                                   run.d_key_status, s.stream[0]));
      launches++;
    }
  }

  // ---- main pass, breadth-first over the GPUs
  std::vector<size_t> next(G, 0);
  std::vector<std::vector<int>> per_gpu(G);
  for (int j = 0; j < (int)jobs.size(); j++) per_gpu[jobs[j].gpu].push_back(j);
  bool more = true;
  while (more) {
    more = false;
    for (int g = 0; g < G; g++) {
      if (next[g] >= per_gpu[g].size()) continue;
      more = true;
      const Job& jb = jobs[per_gpu[g][next[g]++]];
      const Piece& pc = pieces[jb.piece];
      const Sec& sc = secs[pc.sec];
      const int ri = rec_size(sc.group, fmt), rb = sc.group == PTAU_G1 ? kMontG1 : kMontG2;
      GpuSlot& s = ctx->gpu[g];
      GpuWork& x = run.w[g];
      CUDA_TRY(ctx, cudaSetDevice(s.device));
      // the previous slab's MSMs (stream 0) read d_rec: stream 1 starts converting only after them
      CUDA_TRY(ctx, cudaEventRecord(x.ev, s.stream[0]));
      CUDA_TRY(ctx, cudaStreamWaitEvent(s.stream[1], x.ev, 0));
      int c = 0;
      for (uint64_t o = jb.a; o < jb.b; o += chunk, c++) {
        const uint64_t m = jb.b - o < chunk ? jb.b - o : chunk;
        const uint64_t idx = pc.first + o;  // section-relative
        cudaStream_t st = s.stream[c & 1];
        CUDA_TRY(ctx, cudaMemcpyAsync(x.d_in[c & 1], sc.data + idx * ri, m * ri, cudaMemcpyHostToDevice, st));
        uint8_t* dst = (uint8_t*)x.d_rec + (o - jb.a) * rb;
        CUDA_TRY(ctx, launch_convert(sc.group, fmt, PTAU_FMT_ARK_MONT_LIMBS, x.d_in[c & 1], dst, m, PTAU_CHECKS_STRICT,
                                     idx, x.d_status + pc.sec, st));
        launches++;
        h2d += m * ri;
      }
      CUDA_TRY(ctx, cudaEventRecord(x.ev, s.stream[1]));
      CUDA_TRY(ctx, cudaStreamWaitEvent(s.stream[0], x.ev, 0));
      if (jb.part < 0) continue;
      const uint64_t np = jb.b - 1 - jb.a;
      ratio_coeff_kernel<<<(unsigned)((np + 255) / 256), 256, 0, s.stream[0]>>>(key, (uint32_t)pc.rel, jb.a, np,
                                                                                  (uint32_t*)x.d_sc);
      CUDA_TRY(ctx, cudaGetLastError());
      auto msm = sc.group == PTAU_G1 ? launch_msm_g1 : launch_msm_g2;
      int nl = 0;
      CUDA_TRY(ctx, msm(x.d_rec, x.d_sc, np, x.d_scratch, x.d_parts + (size_t)jb.part * 256, &nl, s.stream[0]));
      launches += nl + 1;
      CUDA_TRY(ctx, msm((uint8_t*)x.d_rec + rb, x.d_sc, np, x.d_scratch, x.d_parts + (size_t)(jb.part + 1) * 256, &nl,
                        s.stream[0]));
      launches += nl;
    }
  }

  // ---- point checks: the first failing section in file order, its lowest index
  std::vector<std::vector<uint8_t>> parts(G);
  unsigned long long st_min[8];
  for (int i = 0; i < nsec; i++) st_min[i] = none;
  for (int g = 0; g < G; g++) {
    GpuSlot& s = ctx->gpu[g];
    GpuWork& x = run.w[g];
    CUDA_TRY(ctx, cudaSetDevice(s.device));
    CUDA_TRY(ctx, cudaStreamSynchronize(s.stream[1]));
    unsigned long long st[8];
    CUDA_TRY(ctx, cudaMemcpyAsync(st, x.d_status, nsec * 8, cudaMemcpyDeviceToHost, s.stream[0]));
    parts[g].resize((size_t)x.parts * 256);
    if (x.parts)
      CUDA_TRY(ctx, cudaMemcpyAsync(parts[g].data(), x.d_parts, parts[g].size(), cudaMemcpyDeviceToHost, s.stream[0]));
    CUDA_TRY(ctx, cudaStreamSynchronize(s.stream[0]));
    for (int i = 0; i < nsec; i++)
      if (st[i] < st_min[i]) st_min[i] = st[i];
  }
  timing_reset(ctx);
  for (int i = 0; i < nsec; i++) {
    if (st_min[i] == none) continue;
    uint64_t idx = st_min[i] >> 8;
    const int k = (int)(st_min[i] & 0xff);
    if (kind != PTAU_POWERS_RESPONSE && secs[i].group == PTAU_G2) idx += g2_index_offset;
    if (bad_index) *bad_index = idx;
    if (bad_kind) *bad_kind = k;
    if (bad_section) *bad_section = kind == PTAU_POWERS_RESPONSE ? i : 0;
    ctx->timing.wall_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    return k;
  }

  // ---- A_k, B_k: the partials of every slab and GPU summed with unit scalars
  std::vector<uint8_t> combo(8 * 200, 0);
  for (int pi = 0; pi < (int)pieces.size(); pi++) {
    const int rel = pieces[pi].rel;
    if (!rel) continue;
    const bool g1 = secs[pieces[pi].sec].group == PTAU_G1;
    const int rb = g1 ? kMontG1 : kMontG2;
    for (int ab = 0; ab < 2; ab++) {
      std::vector<uint8_t> recs;
      for (const Job& jb : jobs) {
        if (jb.piece != pi || jb.part < 0) continue;
        const uint8_t* slot = parts[jb.gpu].data() + (size_t)(jb.part + ab) * 256;
        uint32_t bad;
        memcpy(&bad, slot + rb, 4);
        if (bad) {  // coefficients are < 2^127: cannot happen unless the MSM misread them
          ctx->last_error = "ptau_verify_powers: coefficient rejected by the MSM";
          return PTAU_ERR_CUDA;
        }
        recs.insert(recs.end(), slot, slot + rb);
      }
      uint8_t* out = combo.data() + (size_t)(2 * rel - 2 + ab) * 200;
      const size_t cnt = recs.size() / rb;
      if (cnt == 1) {
        memcpy(out, recs.data(), rb);
        continue;
      }
      std::vector<uint8_t> ones(cnt * 32, 0);
      for (size_t i = 0; i < cnt; i++) ones[i * 32] = 1;
      const int rc = g1 ? ptau_kzg_commit(ctx, recs.data(), ones.data(), cnt, out)
                        : ptau_msm_g2(ctx, recs.data(), ones.data(), cnt, out);
      if (rc) return rc;
    }
  }

  // ---- GENERATORS, KEY and one pairing launch for the ratio relations and BETA_G2
  uint32_t flags[2] = {0, 0};
  uint8_t is_one[kItems];
  {
    GpuSlot& s = ctx->gpu[0];
    CUDA_TRY(ctx, cudaSetDevice(s.device));
    CUDA_TRY(ctx, cudaMalloc(&run.d_combo, combo.size()));
    CUDA_TRY(ctx, cudaMalloc(&run.d_g1, kItems * 2 * kMontG1));
    CUDA_TRY(ctx, cudaMalloc(&run.d_g2, kItems * 2 * kMontG2));
    CUDA_TRY(ctx, cudaMalloc(&run.d_flags, 8));
    CUDA_TRY(ctx, cudaMalloc(&run.d_one, kItems));
    CUDA_TRY(ctx, cudaMemcpyAsync(run.d_combo, combo.data(), combo.size(), cudaMemcpyHostToDevice, s.stream[0]));
    verify_assemble_kernel<<<1, 32, 0, s.stream[0]>>>((const uint32_t*)run.d_keys, (const uint32_t*)run.d_combo, kind,
                                                     rel_mask, (uint32_t*)run.d_g1, (uint32_t*)run.d_g2,
                                                     (uint32_t*)run.d_flags);
    CUDA_TRY(ctx, cudaGetLastError());
    CUDA_TRY(ctx, launch_pairing_product2(run.d_g1, run.d_g2, kItems, nullptr, run.d_one, s.stream[0]));
    launches += 2;
    CUDA_TRY(ctx, cudaMemcpyAsync(flags, run.d_flags, 8, cudaMemcpyDeviceToHost, s.stream[0]));
    CUDA_TRY(ctx, cudaMemcpyAsync(is_one, run.d_one, kItems, cudaMemcpyDeviceToHost, s.stream[0]));
    CUDA_TRY(ctx, cudaStreamSynchronize(s.stream[0]));
  }
  if (combos_out) memcpy(combos_out, combo.data(), combo.size());
  timing_reset(ctx);
  ctx->timing.wall_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
  ctx->timing.kernel_launches = launches;
  ctx->timing.h2d_bytes[0] = h2d;
  int failed = -1;
  if (!flags[0]) {
    failed = PTAU_REL_GENERATORS;
  } else {
    for (int it = 0; it < kItems && failed < 0; it++)
      if (((rel_mask >> (it + 1)) & 1u) && !is_one[it]) failed = it + 1;
    if (failed < 0 && !flags[1]) failed = PTAU_REL_KEY;
  }
  if (failed >= 0) {
    if (bad_relation) *bad_relation = failed;
    return PTAU_BAD_NOT_POWERS;
  }
  return PTAU_OK;
}
