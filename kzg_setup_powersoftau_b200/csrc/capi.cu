// C-ABI host layer of libptau_b200.so (include/ptau_b200.h): context, per-GPU
// streams and double buffers, index-range sharding, status reduction, and the
// whole-file pipelines that reproduce the reference binaries' section tables
// (/root/reference/src/bin/preprocess-kgz.rs:128-200,
//  /root/reference/src/bin/preprocess-fastkgz.rs:129-214,
//  /root/reference/src/lib.rs:82-121, :174-228).
//
// There is no CPU implementation of the point path in this library: without a
// CUDA device every entry point returns PTAU_ERR_CUDA.
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>
#include <sys/random.h>

#include <chrono>
#include <string>
#include <vector>

#include "../../include/ptau_b200.h"
#include <future>

#include "blake2b.h"
#include "context.h"
#include "fr_host.h"
#include "kernels.h"
#include "layout.h"

using namespace ptau;

namespace {

constexpr size_t kEdgePoints = 148 * 2 * 128;  // one wave of convert-kernel blocks on a B200

// device copies of a list of host arrays, freed together
struct DevArgs {
  std::vector<void*> ptrs;
  ~DevArgs() {
    for (void* p : ptrs) cudaFree(p);
  }
  cudaError_t push(const void* host, size_t bytes, cudaStream_t st, void** out) {
    void* d = nullptr;
    cudaError_t e = cudaMalloc(&d, bytes ? bytes : 16);
    if (e != cudaSuccess) return e;
    ptrs.push_back(d);
    if (host && bytes) e = cudaMemcpyAsync(d, host, bytes, cudaMemcpyHostToDevice, st);
    *out = d;
    return e;
  }
};

// A device buffer of launch_once: uploaded from `in` before the launch and/or copied to `out` after it.  With neither,
// nothing is allocated and *dev stays null.
struct LaunchBuf {
  const void* in;
  void* out;
  size_t bytes;
  void** dev;
};
// One launch on the first stream of GPU `gpu` over freshly allocated buffers, their copies back and a synchronise.
// With `timed` the launch is timed and ctx->timing describes the call.
template <class Launch>
int launch_once(ptau_ctx* ctx, int gpu, const char* where, bool timed, std::initializer_list<LaunchBuf> bufs,
                Launch launch) {
  GpuSlot& s = ctx->gpu[gpu];
  const cudaStream_t st = s.stream[0];
  DevArgs a;
  size_t h2d = 0, d2h = 0;
  cudaError_t e = cudaSetDevice(s.device);
  for (const LaunchBuf& b : bufs) {
    if (e == cudaSuccess && (b.in || b.out)) e = a.push(b.in, b.bytes, st, b.dev);
    h2d += b.in ? b.bytes : 0;
  }
  if (e == cudaSuccess && timed) e = cudaEventRecord(s.ev_k0[0], st);
  if (e == cudaSuccess) e = launch(st);
  if (e == cudaSuccess && timed) e = cudaEventRecord(s.ev_k1[0], st);
  for (const LaunchBuf& b : bufs) {
    if (e == cudaSuccess && b.out) e = cudaMemcpyAsync(b.out, *b.dev, b.bytes, cudaMemcpyDeviceToHost, st);
    d2h += b.out ? b.bytes : 0;
  }
  if (e == cudaSuccess) e = cudaStreamSynchronize(st);
  float ms = 0;
  if (e == cudaSuccess && timed) e = cudaEventElapsedTime(&ms, s.ev_k0[0], s.ev_k1[0]);
  if (e != cudaSuccess) return cuda_fail(ctx, where, e);
  if (timed) {
    timing_reset(ctx);
    ctx->timing.kernel_ms[gpu] = ms;
    ctx->timing.gpu_ms[gpu] = ms;
    ctx->timing.kernel_launches = 1;
    ctx->timing.h2d_bytes[gpu] = h2d;
    ctx->timing.d2h_bytes[gpu] = d2h;
  }
  return PTAU_OK;
}

}  // namespace

extern "C" {

int ptau_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) return 0;
  return n;
}

const char* ptau_strerror(int code) {
  switch (code) {
    case PTAU_OK: return "ok";
    case PTAU_BAD_NON_CANONICAL: return "coordinate not canonical (>= p)";
    case PTAU_BAD_FLAGS: return "illegal encoding flag bits";
    case PTAU_BAD_INFINITY: return "point at infinity";
    case PTAU_BAD_NOT_ON_CURVE: return "point not on the curve";
    case PTAU_BAD_NOT_IN_SUBGROUP: return "point not in the prime-order subgroup";
    case PTAU_BAD_NOT_POWERS: return "points are valid but not powers of one tau";
    case PTAU_ERR_CUDA: return "CUDA runtime error (no CPU fallback exists)";
    case PTAU_ERR_ARG: return "invalid argument";
    case PTAU_ERR_SIZE: return "buffer or file size does not match the layout";
    case PTAU_ERR_NOMEM: return "out of memory";
    case PTAU_ERR_IO: return "I/O error";
    case PTAU_ERR_DIGEST: return "BLAKE2b digest mismatch";
    case PTAU_ERR_EXISTS: return "output file already exists";
  }
  return "unknown";
}

int ptau_create(ptau_ctx** out, int n_gpus, const int* device_ids, size_t chunk_points) {
  if (!out || n_gpus < 1 || n_gpus > kMaxGpus) return PTAU_ERR_ARG;
  int have = 0;
  if (cudaGetDeviceCount(&have) != cudaSuccess || have < 1) return PTAU_ERR_CUDA;
  ptau_ctx* ctx = new ptau_ctx();
  ctx->n_gpus = n_gpus;
  ctx->chunk_points = chunk_points ? chunk_points : (size_t)1 << 18;
  memset(&ctx->timing, 0, sizeof(ctx->timing));
  for (int g = 0; g < n_gpus; g++) {
    GpuSlot& s = ctx->gpu[g];
    s.device = device_ids ? device_ids[g] : g;
    if (s.device < 0 || s.device >= have) {
      delete ctx;
      return PTAU_ERR_ARG;
    }
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, s.device) != cudaSuccess || prop.major < 10) {
      delete ctx;
      return PTAU_ERR_CUDA;  // kernels are built for sm_100a only
    }
    bool ok = cudaSetDevice(s.device) == cudaSuccess;
    for (int b = 0; ok && b < kBufs; b++) {
      ok = ok && cudaStreamCreateWithFlags(&s.stream[b], cudaStreamNonBlocking) == cudaSuccess;
      ok = ok && cudaEventCreate(&s.ev_k0[b]) == cudaSuccess && cudaEventCreate(&s.ev_k1[b]) == cudaSuccess;
    }
    ok = ok && cudaEventCreate(&s.ev_first) == cudaSuccess && cudaEventCreate(&s.ev_last) == cudaSuccess;
    ok = ok && cudaMalloc(&s.d_status, sizeof(unsigned long long)) == cudaSuccess;
    if (!ok) {
      ptau_destroy(ctx);
      return PTAU_ERR_CUDA;
    }
  }
  *out = ctx;
  return PTAU_OK;
}

void ptau_destroy(ptau_ctx* ctx) {
  if (!ctx) return;
  for (int g = 0; g < ctx->n_gpus; g++) {
    GpuSlot& s = ctx->gpu[g];
    if (s.device < 0) continue;
    cudaSetDevice(s.device);
    for (int b = 0; b < kBufs; b++) {
      if (s.stream[b]) cudaStreamSynchronize(s.stream[b]);
      if (s.d_in[b]) cudaFree(s.d_in[b]);
      if (s.d_out[b]) cudaFree(s.d_out[b]);
      if (s.ev_k0[b]) cudaEventDestroy(s.ev_k0[b]);
      if (s.ev_k1[b]) cudaEventDestroy(s.ev_k1[b]);
      if (s.stream[b]) cudaStreamDestroy(s.stream[b]);
    }
    if (s.d_status) cudaFree(s.d_status);
    for (int t = 0; t < 2; t++)
      if (s.d_tbl[t]) cudaFree(s.d_tbl[t]);
    if (s.ev_first) cudaEventDestroy(s.ev_first);
    if (s.ev_last) cudaEventDestroy(s.ev_last);
    if (s.d_kzg_tbl) cudaFree(s.d_kzg_tbl);
    if (s.d_msm_pts) cudaFree(s.d_msm_pts);
    if (s.d_msm_sc) cudaFree(s.d_msm_sc);
    if (s.d_msm_scratch) cudaFree(s.d_msm_scratch);
    if (s.d_msm_out) cudaFree(s.d_msm_out);
    if (s.h_msm_sc) cudaFreeHost(s.h_msm_sc);
    if (s.h_msm_out) cudaFreeHost(s.h_msm_out);
    if (s.d_open) cudaFree(s.d_open);
  }
  delete ctx;
}

const char* ptau_last_error(ptau_ctx* ctx) { return ctx ? ctx->last_error.c_str() : ""; }

int ptau_last_timing(ptau_ctx* ctx, ptau_timing* out) {
  if (!ctx || !out) return PTAU_ERR_ARG;
  *out = ctx->timing;
  return PTAU_OK;
}

void* ptau_host_alloc(size_t bytes) {
  void* p = nullptr;
  if (cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocPortable) != cudaSuccess) return nullptr;
  return p;
}
void ptau_host_free(void* p) {
  if (p) cudaFreeHost(p);
}
int ptau_host_register(void* p, size_t bytes) {
  return cudaHostRegister(p, bytes, cudaHostRegisterPortable) == cudaSuccess ? PTAU_OK : PTAU_ERR_CUDA;
}
int ptau_host_unregister(void* p) { return cudaHostUnregister(p) == cudaSuccess ? PTAU_OK : PTAU_ERR_CUDA; }

size_t ptau_record_size(int group, int fmt) { return (size_t)rec_size(group, fmt); }

uint64_t ptau_response_size(uint64_t n) {
  return ptau::kResponseHash + ptau::response_bytes(n, PTAU_FMT_ZCASH_COMPRESSED) + ptau::kResponsePubkey;
}
uint64_t ptau_uncompressed_size(uint64_t n) { return ptau::response_bytes(n, PTAU_FMT_ZCASH_UNCOMPRESSED); }
uint64_t ptau_setup_size(int variant, uint64_t n) {
  if (variant != PTAU_VARIANT_KGZ && variant != PTAU_VARIANT_FASTKGZ) return 0;
  return ptau::setup_layout(variant, n).bytes();
}

int ptau_status_decode(uint64_t status, uint64_t* bad_index) {
  if (status == PTAU_STATUS_NONE) return PTAU_OK;
  if (bad_index) *bad_index = status >> 8;
  return (int)(status & 0xff);
}

int ptau_convert_device(ptau_ctx* ctx, int gpu, int group, int in_fmt, const void* d_in, int out_fmt, void* d_out,
                        size_t n_points, unsigned checks, uint64_t base_index, uint64_t* d_status, void* stream) {
  if (!ctx || gpu < 0 || gpu >= ctx->n_gpus || !d_status) return PTAU_ERR_ARG;
  if (!rec_size(group, in_fmt) || !rec_size(group, out_fmt) || out_fmt == PTAU_FMT_ZCASH_COMPRESSED) return PTAU_ERR_ARG;
  if (((uintptr_t)d_in | (uintptr_t)d_out) & 15) return PTAU_ERR_ARG;
  CUDA_TRY(ctx, cudaSetDevice(ctx->gpu[gpu].device));
  CUDA_TRY(ctx, ptau::launch_convert(group, in_fmt, out_fmt, d_in, d_out, n_points, checks, base_index,
                                     (unsigned long long*)d_status, (cudaStream_t)stream));
  return PTAU_OK;
}

int ptau_convert(ptau_ctx* ctx, int group, int in_fmt, const void* in, int out_fmt, void* out, size_t n_points,
                 unsigned checks, uint64_t* bad_index, int* bad_kind) {
  if (!ctx || (!in && n_points)) return PTAU_ERR_ARG;  // out == NULL: validate only, nothing is copied back
  const int ri = rec_size(group, in_fmt), ro = rec_size(group, out_fmt);
  if (!ri || !ro || out_fmt == PTAU_FMT_ZCASH_COMPRESSED) return PTAU_ERR_ARG;
  auto t0 = std::chrono::steady_clock::now();
  const int G = ctx->n_gpus;
  const size_t chunk = ctx->chunk_points;
  ptau_timing& tm = ctx->timing;
  timing_reset(ctx);

  struct Range {
    size_t lo, hi, next;
    int issued;
  } rg[kMaxGpus];
  const unsigned long long none = PTAU_STATUS_NONE;
  for (int g = 0; g < G; g++) {
    const ptau::Shard sh = shard(n_points, g, G);
    rg[g] = {sh.lo, sh.hi, sh.lo, 0};
    GpuSlot& s = ctx->gpu[g];
    CUDA_TRY(ctx, cudaSetDevice(s.device));
    size_t maxpts = rg[g].hi - rg[g].lo < chunk ? rg[g].hi - rg[g].lo : chunk;
    CUDA_TRY(ctx, ensure_buffers(s.d_in, &s.cap_in, maxpts * ri + 16));
    CUDA_TRY(ctx, ensure_buffers(s.d_out, &s.cap_out, maxpts * ro + 16));
    CUDA_TRY(ctx, cudaMemcpyAsync(s.d_status, &none, sizeof(none), cudaMemcpyHostToDevice, s.stream[0]));
    CUDA_TRY(ctx, cudaEventRecord(s.ev_first, s.stream[0]));
    // stream[1] must not start before the status word is initialised
    CUDA_TRY(ctx, cudaStreamWaitEvent(s.stream[1], s.ev_first, 0));
  }
  // breadth-first issue: one chunk per GPU per round, alternating the two streams
  std::vector<float> kms[kMaxGpus];
  bool more = true;
  while (more) {
    more = false;
    for (int g = 0; g < G; g++) {
      Range& r = rg[g];
      if (r.next >= r.hi) continue;
      GpuSlot& s = ctx->gpu[g];
      CUDA_TRY(ctx, cudaSetDevice(s.device));
      const int b = r.issued % kBufs;
      // The first H2D copy and the last D2H copy of a range have nothing to overlap with, so the first and the
      // last chunk are one wave of blocks (148 SMs x 2 blocks x 128 points) instead of a full chunk.
      const size_t rem = r.hi - r.next;
      size_t npts;
      if (r.issued == 0 && rem > 2 * kEdgePoints && chunk > kEdgePoints)
        npts = kEdgePoints;
      else if (rem > chunk + kEdgePoints || chunk <= kEdgePoints)
        npts = rem < chunk ? rem : chunk;
      else if (rem > 2 * kEdgePoints)
        npts = rem - kEdgePoints;  // at most `chunk`; leaves exactly one wave for the last chunk
      else
        npts = rem < chunk ? rem : chunk;
      if (r.issued >= kBufs) {
        // the event pair of this buffer is about to be reused: harvest its time
        CUDA_TRY(ctx, cudaEventSynchronize(s.ev_k1[b]));
        float ms = 0;
        CUDA_TRY(ctx, cudaEventElapsedTime(&ms, s.ev_k0[b], s.ev_k1[b]));
        tm.kernel_ms[g] += ms;
      }
      const uint8_t* src = (const uint8_t*)in + r.next * (size_t)ri;
      uint8_t* dst = out ? (uint8_t*)out + r.next * (size_t)ro : nullptr;
      CUDA_TRY(ctx, cudaMemcpyAsync(s.d_in[b], src, npts * ri, cudaMemcpyHostToDevice, s.stream[b]));
      CUDA_TRY(ctx, cudaEventRecord(s.ev_k0[b], s.stream[b]));
      CUDA_TRY(ctx, ptau::launch_convert(group, in_fmt, out_fmt, s.d_in[b], s.d_out[b], npts, checks, r.next,
                                         s.d_status, s.stream[b]));
      CUDA_TRY(ctx, cudaEventRecord(s.ev_k1[b], s.stream[b]));
      if (out) {
        CUDA_TRY(ctx, cudaMemcpyAsync(dst, s.d_out[b], npts * ro, cudaMemcpyDeviceToHost, s.stream[b]));
        tm.d2h_bytes[g] += npts * ro;
      }
      tm.h2d_bytes[g] += npts * ri;
      tm.kernel_launches++;
      r.next += npts;
      r.issued++;
      more = true;
    }
  }
  unsigned long long status = PTAU_STATUS_NONE;
  for (int g = 0; g < G; g++) {
    GpuSlot& s = ctx->gpu[g];
    CUDA_TRY(ctx, cudaSetDevice(s.device));
    // join stream[1] into stream[0], read the status word back, stamp the end
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
    tm.gpu_ms[g] = ms;
    int pending = rg[g].issued < kBufs ? rg[g].issued : kBufs;
    for (int b = 0; b < pending; b++) {
      float k = 0;
      CUDA_TRY(ctx, cudaEventElapsedTime(&k, s.ev_k0[b], s.ev_k1[b]));
      tm.kernel_ms[g] += k;
    }
  }
  tm.wall_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
  if (status != PTAU_STATUS_NONE) {
    if (bad_index) *bad_index = status >> 8;
    if (bad_kind) *bad_kind = (int)(status & 0xff);
    return (int)(status & 0xff);
  }
  return PTAU_OK;
}

// ---- generator -------------------------------------------------------------------
// fixed-base table T[w][d-1] = [d * 256^w]G (w < 32, d = 1..255) in ARK_MONT_LIMBS records,
// built once per (context, GPU, group) with the v1 double-and-add kernel
static int ensure_gen_table(ptau_ctx* ctx, GpuSlot& s, int group, cudaStream_t stream) {
  const int gi = group == PTAU_G1 ? 0 : 1;
  if (s.d_tbl[gi]) return PTAU_OK;
  const size_t cnt = 32 * 255;
  const int r_zu = rec_size(group, PTAU_FMT_ZCASH_UNCOMPRESSED), r_ml = rec_size(group, PTAU_FMT_ARK_MONT_LIMBS);
  std::vector<uint32_t> sc(cnt * 8, 0);
  for (int w = 0; w < 32; w++)
    for (int d = 1; d <= 255; d++) {
      uint32_t* k = &sc[(size_t)(w * 255 + d - 1) * 8];
      if (w == 31 && d > 0x73) {
        k[0] = 1;  // digits the top window never takes (k < r < 0x74 * 256^31): any valid scalar
        continue;
      }
      k[w >> 2] = (uint32_t)d << ((w & 3) * 8);
    }
  DevArgs a;
  void *d_sc = nullptr, *d_zu = nullptr, *d_st = nullptr;
  const unsigned long long none = PTAU_STATUS_NONE;
  unsigned long long st = 0;
  cudaError_t e = a.push(sc.data(), cnt * 32, stream, &d_sc);
  if (e == cudaSuccess) e = a.push(nullptr, cnt * r_zu, stream, &d_zu);
  if (e == cudaSuccess) e = a.push(&none, 8, stream, &d_st);
  if (e == cudaSuccess) e = cudaMalloc((void**)&s.d_tbl[gi], cnt * r_ml);
  if (e == cudaSuccess)
    e = ptau::launch_generate(group, PTAU_FMT_ZCASH_UNCOMPRESSED, (const uint32_t*)d_sc, d_zu, cnt, stream);
  if (e == cudaSuccess)
    e = ptau::launch_convert(group, PTAU_FMT_ZCASH_UNCOMPRESSED, PTAU_FMT_ARK_MONT_LIMBS, d_zu, s.d_tbl[gi], cnt, 0, 0,
                             (unsigned long long*)d_st, stream);
  if (e == cudaSuccess) e = cudaMemcpyAsync(&st, d_st, 8, cudaMemcpyDeviceToHost, stream);
  if (e == cudaSuccess) e = cudaStreamSynchronize(stream);
  if (e == cudaSuccess && st == PTAU_STATUS_NONE) return PTAU_OK;
  cudaFree(s.d_tbl[gi]);
  s.d_tbl[gi] = nullptr;
  if (e != cudaSuccess) return cuda_fail(ctx, "ptau_generate_device", e);
  ctx->last_error = "ptau_generate_device: bad generator table point";
  return PTAU_ERR_CUDA;
}

int ptau_generate_device(ptau_ctx* ctx, int gpu, int group, int fmt, const uint8_t scalar0[32], const uint8_t step[32],
                         uint64_t first, size_t n_points, void* d_out, void* stream) {
  if (!ctx || gpu < 0 || gpu >= ctx->n_gpus || !scalar0 || !step) return PTAU_ERR_ARG;
  if (fmt != PTAU_FMT_ZCASH_COMPRESSED && fmt != PTAU_FMT_ZCASH_UNCOMPRESSED) return PTAU_ERR_ARG;
  if (!rec_size(group, fmt)) return PTAU_ERR_ARG;
  if (n_points == 0) return PTAU_OK;
  Fr s0 = fr_from_le32(scalar0), st = fr_from_le32(step);
  if (fr_ge_mod(s0.l) || fr_ge_mod(st.l)) return PTAU_ERR_ARG;
  if ((s0.l[0] | s0.l[1] | s0.l[2] | s0.l[3]) == 0 || (st.l[0] | st.l[1] | st.l[2] | st.l[3]) == 0) return PTAU_ERR_ARG;
  GpuSlot& slot = ctx->gpu[gpu];
  CUDA_TRY(ctx, cudaSetDevice(slot.device));
  int rc = ensure_gen_table(ctx, slot, group, (cudaStream_t)stream);
  if (rc) return rc;
  // host side of the scalars: s0 and step^(2^j) in Montgomery form; the per-point
  // powers are formed on the device
  Fr s0m = fr_to_mont(s0);
  uint32_t pw[64][8];
  Fr p = fr_to_mont(st);
  for (int j = 0; j < 64; j++) {
    memcpy(pw[j], p.l, 32);
    p = fr_mont_mul(p, p);
  }
  CUDA_TRY(ctx, ptau::launch_generate_win(group, fmt, (const uint32_t*)s0m.l, pw, slot.d_tbl[group == PTAU_G1 ? 0 : 1], d_out,
                                          first, n_points, (cudaStream_t)stream));
  return PTAU_OK;
}

int ptau_generate(ptau_ctx* ctx, int group, int fmt, const uint8_t scalar0[32], const uint8_t step[32], uint64_t first,
                  size_t n_points, void* out) {
  if (!ctx || (!out && n_points)) return PTAU_ERR_ARG;
  const int ro = rec_size(group, fmt);
  if (!ro) return PTAU_ERR_ARG;
  // one GPU is plenty for a generator; chunk through that GPU's output buffer
  GpuSlot& s = ctx->gpu[0];
  CUDA_TRY(ctx, cudaSetDevice(s.device));
  const size_t chunk = ctx->chunk_points;
  CUDA_TRY(ctx, ensure_buffers(s.d_in, &s.cap_in, 16));
  CUDA_TRY(ctx, ensure_buffers(s.d_out, &s.cap_out, (n_points < chunk ? n_points : chunk) * ro + 16));
  for (size_t off = 0; off < n_points; off += chunk) {
    size_t n = n_points - off < chunk ? n_points - off : chunk;
    int rc = ptau_generate_device(ctx, 0, group, fmt, scalar0, step, first + off, n, s.d_out[0], s.stream[0]);
    if (rc) return rc;
    CUDA_TRY(ctx, cudaMemcpyAsync((uint8_t*)out + off * ro, s.d_out[0], n * ro, cudaMemcpyDeviceToHost, s.stream[0]));
    CUDA_TRY(ctx, cudaStreamSynchronize(s.stream[0]));
  }
  return PTAU_OK;
}

// ---- whole-file pipelines ----------------------------------------------------------
// out[s] == NULL with process[s] set: the section is validated but nothing is copied back
static int run_sections(ptau_ctx* ctx, const Section* secs, int nsec, int in_fmt, const uint8_t* in, int out_fmt,
                        uint8_t* const* out, unsigned checks, uint64_t* bad_index, int* bad_kind, int* bad_section,
                        const bool* process = nullptr) {
  // Sections are processed in file order and the first failing section wins, so
  // the reported (section, index) is the first bad point in file order.
  ptau_timing total{};
  total.n_gpus = ctx->n_gpus;
  size_t off = 0;
  for (int s = 0; s < nsec; s++) {
    const int ri = rec_size(secs[s].group, in_fmt);
    if (out[s] || (process && process[s])) {
      int rc = ptau_convert(ctx, secs[s].group, in_fmt, in + off, out_fmt, out[s], secs[s].count, checks, bad_index,
                            bad_kind);
      total.wall_ms += ctx->timing.wall_ms;
      total.kernel_launches += ctx->timing.kernel_launches;
      for (int g = 0; g < ctx->n_gpus; g++) {
        total.gpu_ms[g] += ctx->timing.gpu_ms[g];
        total.kernel_ms[g] += ctx->timing.kernel_ms[g];
        total.h2d_bytes[g] += ctx->timing.h2d_bytes[g];
        total.d2h_bytes[g] += ctx->timing.d2h_bytes[g];
      }
      if (rc != PTAU_OK) {
        if (bad_section) *bad_section = s;
        ctx->timing = total;
        return rc;
      }
    }
    off += secs[s].count * (size_t)ri;
  }
  ctx->timing = total;
  return PTAU_OK;
}

static int preprocess_common(ptau_ctx* ctx, int variant, int in_fmt, const uint8_t* body, uint64_t n, uint8_t* setup,
                             unsigned checks, uint64_t* bad_index, int* bad_kind, int* bad_section) {
  if (n < 2) return PTAU_ERR_ARG;
  const bool fast = variant == PTAU_VARIANT_FASTKGZ;
  const auto secs = ptau::response_sections(n);
  const ptau::SetupLayout L = ptau::setup_layout(variant, n);
  // tau_g2: kgz needs only [0], [1] in the output but the reference checks all n
  // (preprocess-kgz.rs:146-148): all n are validated on the GPU without copying the
  // results back, and the first two are converted again for the VerifierKey; fastkgz
  // writes all n in place as powers_of_h.  beta_tau_powers_g1 is read, checked and
  // dropped by fastkgz (preprocess-fastkgz.rs:156-159) and never read by kgz; beta_g2
  // (section 4) is never read by either binary (preprocess-fastkgz.rs:161).
  uint8_t first_g2[384];
  uint8_t* outs[5] = {setup + L.g1(0), fast ? setup + L.g2(L.powers_of_h) : nullptr, setup + L.g1(L.gamma_g), nullptr,
                      nullptr};
  const bool process[5] = {true, true, true, fast, false};
  int rc = run_sections(ctx, secs.data(), 5, in_fmt, body, PTAU_FMT_ARK_UNCOMPRESSED, outs, checks, bad_index, bad_kind,
                        bad_section, process);
  if (rc) return rc;
  // fastkgz: h, beta_h are the first two entries of powers_of_h, which follow them (preprocess-fastkgz.rs:163-208)
  const uint8_t* tau_g2_ark = setup + L.g2(L.powers_of_h);
  if (!fast) {
    const size_t g2_off = secs[0].count * (size_t)rec_size(secs[0].group, in_fmt);
    ptau_timing keep = ctx->timing;
    rc = ptau_convert(ctx, PTAU_G2, in_fmt, body + g2_off, PTAU_FMT_ARK_UNCOMPRESSED, first_g2, 2, checks, bad_index,
                      bad_kind);
    keep.kernel_launches += ctx->timing.kernel_launches;
    ctx->timing = keep;
    if (rc) {
      if (bad_section) *bad_section = 1;
      return rc;
    }
    tau_g2_ark = first_g2;
    // kgz tail: VerifierKey { g = tau_g1[0], gamma_g = alpha_g1[0], h = tau_g2[0], beta_h = tau_g2[1] }
    //   (preprocess-kgz.rs:177-194)
    memcpy(setup + L.g1(L.vk_g), setup + L.g1(0), 96);              // g
    memcpy(setup + L.g1(L.vk_g + 1), setup + L.g1(L.gamma_g), 96);  // gamma_g
  }
  memcpy(setup + L.g2(0), tau_g2_ark, 384);  // h, beta_h
  return PTAU_OK;
}

int ptau_preprocess(ptau_ctx* ctx, int variant, const void* response, uint64_t response_len, uint64_t n_powers,
                    void* setup_out, uint64_t setup_len, void* uncompressed_out, uint64_t uncompressed_len,
                    unsigned checks, uint64_t* bad_index, int* bad_kind, int* bad_section) {
  if (!ctx || !response || !setup_out) return PTAU_ERR_ARG;
  if (variant != PTAU_VARIANT_KGZ && variant != PTAU_VARIANT_FASTKGZ) return PTAU_ERR_ARG;
  // preprocess-kgz.rs:83: the response must have exactly CONTRIBUTION_BYTE_SIZE bytes
  if (response_len != ptau_response_size(n_powers)) return PTAU_ERR_SIZE;
  if (setup_len != ptau_setup_size(variant, n_powers)) return PTAU_ERR_SIZE;
  if (uncompressed_out && uncompressed_len != ptau_uncompressed_size(n_powers)) return PTAU_ERR_SIZE;
  // skip the 64-byte challenge hash (:96-101); the trailing public key is never read
  const uint8_t* body = (const uint8_t*)response + ptau::kResponseHash;
  if (uncompressed_out) {
    // two stages, exactly as the reference: decompress everything into
    // `powersoftau_uncompressed` (:105-124), then read that back (:128-160)
    const auto secs = ptau::response_sections(n_powers);
    uint8_t* outs[5];
    size_t o = 0;
    for (int s = 0; s < 5; s++) {
      outs[s] = (uint8_t*)uncompressed_out + o;
      o += secs[s].count * (size_t)rec_size(secs[s].group, PTAU_FMT_ZCASH_UNCOMPRESSED);
    }
    int rc = run_sections(ctx, secs.data(), 5, PTAU_FMT_ZCASH_COMPRESSED, body, PTAU_FMT_ZCASH_UNCOMPRESSED, outs,
                          PTAU_CHECKS_DECOMPRESS, bad_index, bad_kind, bad_section);
    if (rc) return rc;
    return preprocess_common(ctx, variant, PTAU_FMT_ZCASH_UNCOMPRESSED, (const uint8_t*)uncompressed_out, n_powers,
                             (uint8_t*)setup_out, checks, bad_index, bad_kind, bad_section);
  }
  // fused: compressed -> checked -> ark, no intermediate file
  return preprocess_common(ctx, variant, PTAU_FMT_ZCASH_COMPRESSED, body, n_powers, (uint8_t*)setup_out, checks,
                           bad_index, bad_kind, bad_section);
}

int ptau_preprocess_uncompressed(ptau_ctx* ctx, int variant, const void* uncompressed, uint64_t uncompressed_len,
                                 uint64_t n_powers, void* setup_out, uint64_t setup_len, unsigned checks,
                                 uint64_t* bad_index, int* bad_kind, int* bad_section) {
  if (!ctx || !uncompressed || !setup_out) return PTAU_ERR_ARG;
  if (variant != PTAU_VARIANT_KGZ && variant != PTAU_VARIANT_FASTKGZ) return PTAU_ERR_ARG;
  if (uncompressed_len != ptau_uncompressed_size(n_powers)) return PTAU_ERR_SIZE;
  if (setup_len != ptau_setup_size(variant, n_powers)) return PTAU_ERR_SIZE;
  return preprocess_common(ctx, variant, PTAU_FMT_ZCASH_UNCOMPRESSED, (const uint8_t*)uncompressed, n_powers,
                           (uint8_t*)setup_out, checks, bad_index, bad_kind, bad_section);
}

int ptau_load_setup(ptau_ctx* ctx, int variant, const void* setup, uint64_t setup_len, uint64_t n, unsigned checks,
                    void* g1_out, uint64_t g1_out_len, void* g2_out, uint64_t g2_out_len, uint64_t* bad_index,
                    int* bad_kind) {
  if (!ctx || !setup || !g1_out || !g2_out) return PTAU_ERR_ARG;
  if (variant != PTAU_VARIANT_KGZ && variant != PTAU_VARIANT_FASTKGZ) return PTAU_ERR_ARG;
  if (setup_len != ptau_setup_size(variant, n)) return PTAU_ERR_SIZE;
  const ptau::SetupLayout L = ptau::setup_layout(variant, n);
  if (g1_out_len != L.n_g1 * kMontG1 || g2_out_len != L.n_g2 * kMontG2) return PTAU_ERR_SIZE;
  // both layouts are "all G1 records, then all G2 records" (src/lib.rs:179-192, :202-215)
  const Section secs[2] = {{PTAU_G1, L.n_g1}, {PTAU_G2, L.n_g2}};
  uint8_t* outs[2] = {(uint8_t*)g1_out, (uint8_t*)g2_out};
  int sec = 0;
  int rc = run_sections(ctx, secs, 2, PTAU_FMT_ARK_UNCOMPRESSED, (const uint8_t*)setup, PTAU_FMT_ARK_MONT_LIMBS, outs,
                        checks, bad_index, bad_kind, &sec);
  if (rc > 0 && sec == 1 && bad_index) *bad_index += L.n_g1;  // index in file order over all points
  return rc;
}

int ptau_load_phase1(ptau_ctx* ctx, const void* data, uint64_t len, uint64_t m, unsigned checks, void* g1_out,
                     uint64_t g1_out_len, void* g2_out, uint64_t g2_out_len, uint64_t* bad_index, int* bad_kind) {
  if (!ctx || !data || !g1_out || !g2_out) return PTAU_ERR_ARG;
  // src/lib.rs:92-110: alpha, beta_g1 (G1), beta_g2 (G2), m G1, m G2, m G1, m G1
  if (len != 2 * 96 + 192 + m * 96 + m * 192 + m * 96 + m * 96) return PTAU_ERR_SIZE;
  if (g1_out_len != (2 + 3 * m) * kMontG1 || g2_out_len != (1 + m) * kMontG2) return PTAU_ERR_SIZE;
  const Section secs[5] = {{PTAU_G1, 2}, {PTAU_G2, 1}, {PTAU_G1, m}, {PTAU_G2, m}, {PTAU_G1, 2 * m}};
  uint8_t* g1 = (uint8_t*)g1_out;
  uint8_t* g2 = (uint8_t*)g2_out;
  uint8_t* outs[5] = {g1, g2, g1 + 2 * kMontG1, g2 + kMontG2, g1 + (2 + m) * kMontG1};
  return run_sections(ctx, secs, 5, PTAU_FMT_ZCASH_UNCOMPRESSED, (const uint8_t*)data, PTAU_FMT_ARK_MONT_LIMBS, outs,
                      checks, bad_index, bad_kind, nullptr);
}

namespace {
cudaError_t grow(void** p, size_t* cap, size_t need, bool pinned = false) {
  if (need <= *cap) return cudaSuccess;
  if (*p) {
    cudaError_t e = pinned ? cudaFreeHost(*p) : cudaFree(*p);
    *p = nullptr;
    *cap = 0;
    if (e != cudaSuccess) return e;
  }
  need += need / 8;  // head room: the next slightly larger call does not reallocate
  cudaError_t e = pinned ? cudaHostAlloc(p, need, cudaHostAllocPortable) : cudaMalloc(p, need);
  if (e == cudaSuccess) *cap = need;
  return e;
}
// pageable -> pinned in parallel parts (one thread copies ~10 GB/s; 32 MB of scalars would cost as much as a
// quarter of the kernels)
void copy_parts(void* dst, const void* src, size_t len) {
  const size_t kPart = 4u << 20;
  if (len <= 2 * kPart) {
    memcpy(dst, src, len);
    return;
  }
  const int parts = len / kPart > 4 ? 4 : (int)(len / kPart);
  const size_t each = (len / parts + 63) & ~(size_t)63;
  std::future<void> f[4];
  for (int i = 1; i < parts; i++) {
    const size_t lo = each * i, n = i == parts - 1 ? len - lo : each;
    f[i] = std::async(std::launch::async, [=] { memcpy((uint8_t*)dst + lo, (const uint8_t*)src + lo, n); });
  }
  memcpy(dst, src, each);
  for (int i = 1; i < parts; i++) f[i].get();
}
// One multi-scalar multiplication on one GPU, issued asynchronously on the slot's first stream; result and the
// "scalar >= r" flag land in s.h_msm_out.  pts: host records, or (resident = true) device records on this GPU;
// G1 (104-byte records) or, with g2, G2 (200-byte records).
cudaError_t msm_issue(GpuSlot& s, const void* pts, const void* sc, size_t n, int* launches, bool resident = false,
                      bool g2 = false) {
  cudaError_t e = cudaSetDevice(s.device);
  const size_t rb = g2 ? kMontG2 : kMontG1;
  ptau::MsmPlan plan;
  (g2 ? ptau::msm_g2_plan : ptau::msm_g1_plan)(n, &plan);
  const void* d_pts = pts;
  if (e == cudaSuccess && !resident) {
    e = grow(&s.d_msm_pts, &s.cap_msm_pts, n * rb + 16);
    d_pts = s.d_msm_pts;
  }
  if (e == cudaSuccess) e = grow(&s.d_msm_sc, &s.cap_msm_sc, n * 32 + 16);
  if (e == cudaSuccess) e = grow(&s.d_msm_scratch, &s.cap_msm_scratch, plan.scratch_bytes);
  if (e == cudaSuccess) e = grow(&s.h_msm_sc, &s.cap_h_msm_sc, n * 32 + 16, true);
  if (e == cudaSuccess && !s.d_msm_out) e = cudaMalloc(&s.d_msm_out, 256);
  if (e == cudaSuccess && !s.h_msm_out) e = cudaHostAlloc((void**)&s.h_msm_out, 256, cudaHostAllocPortable);
  if (e != cudaSuccess) return e;
  copy_parts(s.h_msm_sc, sc, n * 32);
  if (!resident) e = cudaMemcpyAsync(s.d_msm_pts, pts, n * rb, cudaMemcpyHostToDevice, s.stream[0]);
  if (e == cudaSuccess) e = cudaMemcpyAsync(s.d_msm_sc, s.h_msm_sc, n * 32, cudaMemcpyHostToDevice, s.stream[0]);
  if (e == cudaSuccess) e = cudaEventRecord(s.ev_k0[0], s.stream[0]);
  if (e == cudaSuccess)
    e = (g2 ? ptau::launch_msm_g2 : ptau::launch_msm_g1)(d_pts, s.d_msm_sc, n, s.d_msm_scratch, s.d_msm_out, launches,
                                                         s.stream[0]);
  if (e == cudaSuccess) e = cudaEventRecord(s.ev_k1[0], s.stream[0]);
  if (e == cudaSuccess) e = cudaMemcpyAsync(s.h_msm_out, s.d_msm_out, rb + 4, cudaMemcpyDeviceToHost, s.stream[0]);
  return e;
}
cudaError_t msm_wait(GpuSlot& s, float* ms) {
  cudaError_t e = cudaSetDevice(s.device);
  if (e == cudaSuccess) e = cudaStreamSynchronize(s.stream[0]);
  if (e == cudaSuccess) e = cudaEventElapsedTime(ms, s.ev_k0[0], s.ev_k1[0]);
  return e;
}
// point indices travel in 31 bits and the bucket lists (n x W entries) are addressed with 32-bit offsets
bool msm_fits(size_t n, bool g2 = false) {
  ptau::MsmPlan plan;
  (g2 ? ptau::msm_g2_plan : ptau::msm_g1_plan)(n, &plan);
  return n < (1ull << 31) && (uint64_t)n * (uint64_t)plan.W < (1ull << 32);
}
}  // namespace

// With several GPUs in the context the terms are sharded by contiguous index range like every other call of the
// library; the per-GPU partial sums (one point each) are added by one more tiny MSM with unit scalars on GPU 0.
struct ptau_kzg_powers {
  ptau_ctx* ctx = nullptr;
  size_t n = 0;
  void* d_pts[kMaxGpus] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
};

static int kzg_commit_impl(ptau_ctx* ctx, const void* powers, const ptau_kzg_powers* res, const void* coeffs, size_t n,
                           void* commitment, bool g2 = false);

int ptau_kzg_commit(ptau_ctx* ctx, const void* powers, const void* coeffs, size_t n, void* commitment) {
  if (!ctx || (!powers && n) || (!coeffs && n) || !commitment) return PTAU_ERR_ARG;
  return kzg_commit_impl(ctx, powers, nullptr, coeffs, n, commitment);
}

int ptau_msm_g2(ptau_ctx* ctx, const void* points, const void* scalars, size_t n, void* out) {
  if (!ctx || (!points && n) || (!scalars && n) || !out) return PTAU_ERR_ARG;
  return kzg_commit_impl(ctx, points, nullptr, scalars, n, out, true);
}

// The powers of a setup are the same for every commitment: keep a copy on every GPU of the context and send only the
// scalars per call.
int ptau_kzg_powers_upload(ptau_ctx* ctx, const void* powers, size_t n, ptau_kzg_powers** out) {
  if (!ctx || !out || (!powers && n)) return PTAU_ERR_ARG;
  ptau_kzg_powers* p = new ptau_kzg_powers;
  p->ctx = ctx;
  p->n = n;
  for (int g = 0; g < ctx->n_gpus; g++) {
    cudaError_t e = cudaSetDevice(ctx->gpu[g].device);
    if (e == cudaSuccess) e = cudaMalloc(&p->d_pts[g], n * kMontG1 + 16);
    if (e == cudaSuccess && n) e = cudaMemcpy(p->d_pts[g], powers, n * kMontG1, cudaMemcpyHostToDevice);
    if (e != cudaSuccess) {
      ptau_kzg_powers_free(p);
      return cuda_fail(ctx, __func__, e);
    }
  }
  *out = p;
  return PTAU_OK;
}

void ptau_kzg_powers_free(ptau_kzg_powers* p) {
  if (!p) return;
  for (int g = 0; g < kMaxGpus; g++)
    if (p->d_pts[g]) cudaFree(p->d_pts[g]);
  delete p;
}

int ptau_kzg_commit_resident(ptau_ctx* ctx, const ptau_kzg_powers* powers, const void* coeffs, size_t n, void* commitment) {
  if (!ctx || !powers || powers->ctx != ctx || n > powers->n || (!coeffs && n) || !commitment) return PTAU_ERR_ARG;
  return kzg_commit_impl(ctx, nullptr, powers, coeffs, n, commitment);
}

static int kzg_commit_impl(ptau_ctx* ctx, const void* powers, const ptau_kzg_powers* res, const void* coeffs, size_t n,
                           void* commitment, bool g2) {
  // scalars must be canonical (< r), like ark's Fr: checked on the device by the kernel that reads them anyway
  const size_t rb = g2 ? kMontG2 : kMontG1;
  if (!msm_fits(n, g2)) return PTAU_ERR_ARG;
  const int G = (ctx->n_gpus > 1 && n >= (size_t)ctx->n_gpus * (1u << 12)) ? ctx->n_gpus : 1;
  timing_reset(ctx);
  cudaError_t e = cudaSuccess;
  int launches[kMaxGpus] = {0};
  for (int g = 0; g < G && e == cudaSuccess; g++) {
    const auto [lo, hi] = shard(n, g, G);
    if (res)
      e = msm_issue(ctx->gpu[g], (const uint8_t*)res->d_pts[g] + lo * kMontG1, (const uint8_t*)coeffs + lo * 32,
                    hi - lo, &launches[g], true);
    else
      e = msm_issue(ctx->gpu[g], (const uint8_t*)powers + lo * rb, (const uint8_t*)coeffs + lo * 32, hi - lo, &launches[g],
                    false, g2);
    ctx->timing.h2d_bytes[g] = (hi - lo) * (res ? 32 : rb + 32);
    ctx->timing.d2h_bytes[g] = rb;
  }
  bool bad_scalar = false;
  uint8_t parts[kMaxGpus * kMontG2];
  for (int g = 0; g < G && e == cudaSuccess; g++) {
    float ms = 0;
    e = msm_wait(ctx->gpu[g], &ms);
    ctx->timing.kernel_ms[g] = ms;
    ctx->timing.gpu_ms[g] = ms;
    ctx->timing.kernel_launches += launches[g];
    if (e == cudaSuccess) {
      memcpy(parts + g * rb, ctx->gpu[g].h_msm_out, rb);
      bad_scalar = bad_scalar || ctx->gpu[g].h_msm_out[rb / 4] != 0;
    }
  }
  if (e == cudaSuccess && bad_scalar) return PTAU_ERR_ARG;
  if (e == cudaSuccess && G > 1) {
    uint8_t ones[kMaxGpus * 32];
    memset(ones, 0, sizeof(ones));
    for (int g = 0; g < G; g++) ones[g * 32] = 1;
    float ms = 0;
    int nl = 0;
    e = msm_issue(ctx->gpu[0], parts, ones, (size_t)G, &nl, false, g2);
    if (e == cudaSuccess) e = msm_wait(ctx->gpu[0], &ms);
    ctx->timing.kernel_ms[0] += ms;
    ctx->timing.gpu_ms[0] += ms;
    ctx->timing.kernel_launches += nl;
    if (e == cudaSuccess) memcpy(commitment, ctx->gpu[0].h_msm_out, rb);
  } else if (e == cudaSuccess) {
    memcpy(commitment, parts, rb);
  }
  return e == cudaSuccess ? PTAU_OK : cuda_fail(ctx, g2 ? "ptau_msm_g2" : "ptau_kzg_commit", e);
}

namespace {
bool scalars_canonical(const void* p, size_t n) {
  for (size_t i = 0; i < n; i++) {
    Fr c = fr_from_le32((const uint8_t*)p + i * 32);
    if (fr_ge_mod(c.l)) return false;
  }
  return true;
}
// error path of a call with work queued on the first stream of GPUs 0..G-1: nothing may still be using its buffers
// when the call returns
int drain_fail(ptau_ctx* ctx, int G, const char* where, cudaError_t e) {
  for (int g = 0; g < G; g++) {
    cudaSetDevice(ctx->gpu[g].device);
    cudaStreamSynchronize(ctx->gpu[g].stream[0]);
  }
  return cuda_fail(ctx, where, e);
}
}  // namespace

int ptau_pairing_product2(ptau_ctx* ctx, const void* g1, const void* g2, size_t n, void* gt_out, uint8_t* is_one) {
  if (!ctx || (n && (!g1 || !g2)) || (!gt_out && !is_one)) return PTAU_ERR_ARG;
  if (n == 0) return PTAU_OK;
  void *d1 = nullptr, *d2 = nullptr, *dgt = nullptr, *dis = nullptr;
  return launch_once(ctx, 0, __func__, true,
                     {{g1, nullptr, n * 2 * kMontG1, &d1},
                      {g2, nullptr, n * 2 * kMontG2, &d2},
                      {nullptr, gt_out, n * 576, &dgt},
                      {nullptr, is_one, n, &dis}},
                     [&](cudaStream_t st) { return ptau::launch_pairing_product2(d1, d2, n, dgt, dis, st); });
}

int ptau_g2_prepare(ptau_ctx* ctx, const void* g2, size_t n, void* coeffs_out, uint8_t* infinity_out) {
  if (!ctx || (n && (!g2 || !coeffs_out || !infinity_out))) return PTAU_ERR_ARG;
  if (n == 0) return PTAU_OK;
  void *d2 = nullptr, *dc = nullptr, *di = nullptr;
  return launch_once(ctx, 0, __func__, true,
                     {{g2, nullptr, n * kMontG2, &d2},
                      {nullptr, coeffs_out, n * PTAU_G2_PREPARED_COEFFS * 288, &dc},
                      {nullptr, infinity_out, n, &di}},
                     [&](cudaStream_t st) { return ptau::launch_g2_prepare(d2, n, dc, di, st); });
}

int ptau_kzg_check(ptau_ctx* ctx, const void* vk_g1, const void* vk_g2, const void* comms, const void* points,
                   const void* values, const void* proofs_w, const void* random_v, size_t n, uint8_t* ok) {
  if (!ctx || !vk_g1 || !vk_g2 || (n && (!comms || !points || !values || !proofs_w || !ok))) return PTAU_ERR_ARG;
  if (n == 0) return PTAU_OK;
  // scalars must be canonical (< r), like ark's Fr
  if (!scalars_canonical(points, n) || !scalars_canonical(values, n) || (random_v && !scalars_canonical(random_v, n)))
    return PTAU_ERR_ARG;
  // openings are independent: contiguous index ranges over the context's GPUs, no exchange
  const int G = (ctx->n_gpus > 1 && n >= (size_t)ctx->n_gpus * 64) ? ctx->n_gpus : 1;
  std::string key((const char*)vk_g1, 2 * kMontG1);
  key.append((const char*)vk_g2, kMontG2);
  timing_reset(ctx);
  DevArgs args[kMaxGpus];
  bool rebuilt[kMaxGpus] = {false};
  cudaError_t e = cudaSuccess;
  for (int g = 0; g < G && e == cudaSuccess; g++) {
    GpuSlot& s = ctx->gpu[g];
    const ptau::Shard sh = shard(n, g, G);
    const size_t lo = sh.lo, cnt = sh.hi - sh.lo;
    cudaStream_t st = s.stream[0];
    DevArgs& a = args[g];
    void *dv1 = nullptr, *dv2 = nullptr, *dc = nullptr, *dz = nullptr, *dv = nullptr, *dw = nullptr, *drv = nullptr, *dok = nullptr;
    e = cudaSetDevice(s.device);
    if (e == cudaSuccess) e = a.push(vk_g1, 2 * kMontG1, st, &dv1);
    if (e == cudaSuccess) e = a.push(vk_g2, 2 * kMontG2, st, &dv2);
    if (e == cudaSuccess) e = a.push((const uint8_t*)comms + lo * kMontG1, cnt * kMontG1, st, &dc);
    if (e == cudaSuccess) e = a.push((const uint8_t*)points + lo * 32, cnt * 32, st, &dz);
    if (e == cudaSuccess) e = a.push((const uint8_t*)values + lo * 32, cnt * 32, st, &dv);
    if (e == cudaSuccess) e = a.push((const uint8_t*)proofs_w + lo * kMontG1, cnt * kMontG1, st, &dw);
    if (e == cudaSuccess && random_v) e = a.push((const uint8_t*)random_v + lo * 32, cnt * 32, st, &drv);
    if (e == cudaSuccess) e = a.push(nullptr, cnt, st, &dok);
    int launches = 1;
    if (e == cudaSuccess) {  // fixed-base tables of g, gamma_g, h: kept while the key stays the same
      if (!s.d_kzg_tbl) e = cudaMalloc(&s.d_kzg_tbl, ptau::kzg_tables_bytes());
      if (e == cudaSuccess && key != s.kzg_tbl_key) {
        // the key is recorded only once the build is known to have completed (below); until then the slot has none
        s.kzg_tbl_key.clear();
        e = ptau::launch_kzg_tables(dv1, dv2, s.d_kzg_tbl, st);
        rebuilt[g] = true;
        launches++;
      }
    }
    if (e == cudaSuccess) e = cudaEventRecord(s.ev_k0[0], st);
    if (e == cudaSuccess) e = ptau::launch_kzg_check(dv1, dv2, dc, dz, dv, dw, drv, s.d_kzg_tbl, cnt, dok, st);
    if (e == cudaSuccess) e = cudaEventRecord(s.ev_k1[0], st);
    if (e == cudaSuccess) e = cudaMemcpyAsync(ok + lo, dok, cnt, cudaMemcpyDeviceToHost, st);
    ctx->timing.kernel_launches += launches;
    ctx->timing.h2d_bytes[g] = 2 * (kMontG1 + kMontG2) + cnt * (kMontG1 + 32 + 32 + kMontG1 + (random_v ? 32 : 0));
    ctx->timing.d2h_bytes[g] = cnt;
  }
  for (int g = 0; g < G && e == cudaSuccess; g++) {
    GpuSlot& s = ctx->gpu[g];
    float ms = 0;
    e = cudaSetDevice(s.device);
    if (e == cudaSuccess) e = cudaStreamSynchronize(s.stream[0]);
    if (e == cudaSuccess) e = cudaEventElapsedTime(&ms, s.ev_k0[0], s.ev_k1[0]);
    if (e == cudaSuccess && rebuilt[g]) s.kzg_tbl_key = key;  // the table kernel ran to completion on this GPU
    ctx->timing.kernel_ms[g] = ms;
    ctx->timing.gpu_ms[g] = ms;
  }
  return e == cudaSuccess ? PTAU_OK : drain_fail(ctx, G, __func__, e);  // before DevArgs frees the buffers
}

// Witness polynomial of KZG10::open: (p(X) - p(z)) / (X - z) by synthetic division, and p(z).  A first-order
// recurrence over Fr (one Montgomery multiplication per coefficient, carry kept canonical by multiplying with z R),
// done on the host like ark-poly's division; the commitment to the result is ptau_kzg_commit.
int ptau_kzg_quotient(const void* coeffs, size_t n, const void* point, void* quotient_out, void* value_out) {
  if ((!coeffs && n) || !point || !value_out || (n > 1 && !quotient_out)) return PTAU_ERR_ARG;
  Fr z = fr_from_le32((const uint8_t*)point);
  if (fr_ge_mod(z.l)) return PTAU_ERR_ARG;
  const Fr zm = fr_to_mont(z);
  Fr carry;
  memset(carry.l, 0, 32);
  for (size_t i = n; i-- > 1;) {
    Fr ci = fr_from_le32((const uint8_t*)coeffs + i * 32);
    if (fr_ge_mod(ci.l)) return PTAU_ERR_ARG;
    carry = fr_add_mod(ci, fr_mont_mul(carry, zm));
    memcpy((uint8_t*)quotient_out + (i - 1) * 32, carry.l, 32);
  }
  Fr c0;
  memset(c0.l, 0, 32);
  if (n) {
    c0 = fr_from_le32((const uint8_t*)coeffs);
    if (fr_ge_mod(c0.l)) return PTAU_ERR_ARG;
  }
  Fr v = fr_add_mod(c0, fr_mont_mul(carry, zm));
  memcpy(value_out, v.l, 32);
  return PTAU_OK;
}

namespace {
size_t up256(size_t v) { return (v + 255) & ~(size_t)255; }
// omega_{2^32} = 7^((r - 1) / 2^32) mod r (ark-bls12-381 Fr TWO_ADIC_ROOT_OF_UNITY), canonical limbs
constexpr uint64_t kFrRootOfUnity[4] = {0x3829971f439f0d2bull, 0xb63683508c2280b9ull, 0xd09b681922c813b4ull,
                                        0x16a2a19edfe81f20ull};
Fr fr_mont_one_host() {
  Fr one{{1, 0, 0, 0}};
  return fr_to_mont(one);
}
// a^e in Montgomery form for a in Montgomery form, e as 4 x u64 limbs
Fr fr_mont_pow(const Fr& a, const uint64_t* e) {
  Fr x = fr_mont_one_host();
  for (int b = 255; b >= 0; b--) {
    x = fr_mont_mul(x, x);
    if ((e[b / 64] >> (b % 64)) & 1) x = fr_mont_mul(x, a);
  }
  return x;
}
// omega_k R for k = 2^lg_k
Fr fr_root_mont(int lg_k) {
  Fr w;
  memcpy(w.l, kFrRootOfUnity, 32);
  w = fr_to_mont(w);
  for (int s = lg_k; s < 32; s++) w = fr_mont_mul(w, w);
  return w;
}
// out[s] = a^(2^s) R for s < count, a R given
void fr_square_table(Fr a, uint32_t (*out)[8], int count) {
  for (int s = 0; s < count; s++) {
    memcpy(out[s], a.l, 32);
    a = fr_mont_mul(a, a);
  }
}
bool fr_is_zero(const Fr& a) { return !(a.l[0] | a.l[1] | a.l[2] | a.l[3]); }
// the shifts: canonical and non-zero
bool shifts_valid(const void* p, size_t m) {
  for (size_t i = 0; i < m; i++) {
    Fr h = fr_from_le32((const uint8_t*)p + i * 32);
    if (fr_ge_mod(h.l) || fr_is_zero(h)) return false;
  }
  return true;
}

// Both openings, per GPU for its contiguous range of the shifts h (the points of ptau_kzg_open, the cosets' shifts of
// ptau_kzg_open_cosets): the coefficients, the blinding coefficients and, for k > 1, the shifts' tables h^(2^s) R are
// uploaded once; then, per shift and on one stream with no host round trip, the quotient kernels write
// q = p div (X^k - h^k) into the MSM's scalar buffer and the remainder r into its slot, and the bucket MSM commits to q
// over the resident powers.  With blinding (only at k = 1) the same follows for b over gamma_powers, and a 2-term MSM
// with unit scalars adds the two results.  For k > 1 one batched NTT of all the GPU's remainders (scaled by h^j) gives
// the values; for k = 1 the remainder is the value p(h) and is written straight into the values.  Values, proofs and
// the "coefficient >= r" word come back once at the end.  `where` names the entry point in the last-error text.
int kzg_open_impl(ptau_ctx* ctx, const char* where, const ptau_kzg_powers* powers, const ptau_kzg_powers* gamma_powers,
                  const void* coeffs, size_t n, const void* blinding, size_t n_b, int log2_k, const void* shifts, size_t m,
                  void* proofs_out, void* values_out, void* random_v_out) {
  auto t0 = std::chrono::steady_clock::now();
  const uint64_t k = 1ull << log2_k;
  const int G = (size_t)ctx->n_gpus < m ? ctx->n_gpus : (int)m;
  const size_t n_max = n > n_b ? n : n_b, nq = n > k ? n - k : 0, nbq = n_b > k ? n_b - k : 0;
  size_t scratch = 0;
  for (size_t len : {nq, nbq, n_b ? (size_t)2 : 0}) {
    ptau::MsmPlan plan;
    ptau::msm_g1_plan(len, &plan);
    scratch = plan.scratch_bytes > scratch ? plan.scratch_bytes : scratch;
  }
  // staging in GPU 0's pinned scalar buffer (portable: every GPU copies from it): coefficients | blinding | 1, 1 |
  // per shift, h^(2^s) R for the NTT's coset scale (k > 1)
  constexpr int kTbl = ptau::kCosetLgKMax;
  const size_t tbl = log2_k ? kTbl * 32 : 0;
  GpuSlot& s0 = ctx->gpu[0];
  const size_t h_b = n * 32, h_one = h_b + n_b * 32, h_tbl = h_one + 64, h_len = h_tbl + m * tbl;
  cudaError_t e = cudaSetDevice(s0.device);
  if (e == cudaSuccess) e = grow(&s0.h_msm_sc, &s0.cap_h_msm_sc, h_len, true);
  if (e != cudaSuccess) return cuda_fail(ctx, where, e);
  uint8_t* stage = (uint8_t*)s0.h_msm_sc;
  if (n) copy_parts(stage, coeffs, n * 32);
  if (n_b) copy_parts(stage + h_b, blinding, n_b * 32);
  memset(stage + h_one, 0, 64);
  stage[h_one] = stage[h_one + 32] = 1;
  std::vector<Fr> hm(m);
  for (size_t i = 0; i < m; i++) {
    hm[i] = fr_to_mont(fr_from_le32((const uint8_t*)shifts + i * 32));
    if (log2_k) fr_square_table(hm[i], (uint32_t(*)[8])(stage + h_tbl + i * tbl), kTbl);
  }
  uint32_t wpow[ptau::kCosetLgKMax][8];
  fr_square_table(fr_root_mont(log2_k), wpow, log2_k);
  // device layout of d_open, per GPU: coefficients | blinding | 1, 1 | chunk sums | MSM results r0, r1 | the pair
  // (r0, r1) as consecutive records | "coefficient >= r" word | twiddles | h tables | remainders | values | random
  // values | proofs.  For k = 1 the remainders take no space: they are the values.
  const size_t d_b = up256(n * 32), d_one = d_b + up256(n_b * 32), d_sums = d_one + 256,
               d_r0 = d_sums + up256(ptau::coset_quotient_sums_bytes(n_max, log2_k)), d_r1 = d_r0 + 256,
               d_pair = d_r1 + 256, d_bad = d_pair + 256, d_tw = d_bad + 256, d_ht = d_tw + up256(k / 2 * 32);
  struct Tail {
    size_t rem, val, rv, pf, len;
  };
  auto tail = [&](size_t cnt) {
    Tail t;
    t.rem = d_ht + up256(cnt * tbl);
    t.val = t.rem + (log2_k ? up256(cnt * k * 32) : 0);
    t.rv = t.val + up256(cnt * k * 32);
    t.pf = t.rv + up256(n_b ? cnt * 32 : 0);
    t.len = t.pf + cnt * kMontG1;
    return t;
  };
  int launches = 0;
  for (int g = 0; g < G && e == cudaSuccess; g++) {
    GpuSlot& s = ctx->gpu[g];
    const ptau::Shard sh = shard(m, g, G);
    const size_t lo = sh.lo, cnt = sh.hi - sh.lo;
    const Tail t = tail(cnt);
    cudaStream_t st = s.stream[0];
    e = cudaSetDevice(s.device);
    if (e == cudaSuccess) e = grow(&s.d_open, &s.cap_open, t.len);
    if (e == cudaSuccess) e = grow(&s.d_msm_sc, &s.cap_msm_sc, n_max * 32 + 16);
    if (e == cudaSuccess) e = grow(&s.d_msm_scratch, &s.cap_msm_scratch, scratch);
    if (e == cudaSuccess && !s.h_msm_out) e = cudaHostAlloc((void**)&s.h_msm_out, 256, cudaHostAllocPortable);
    if (e != cudaSuccess) break;
    uint8_t* d = (uint8_t*)s.d_open;
    uint32_t* bad = (uint32_t*)(d + d_bad);
    e = cudaEventRecord(s.ev_first, st);
    if (e == cudaSuccess && n) e = cudaMemcpyAsync(d, stage, n * 32, cudaMemcpyHostToDevice, st);
    if (e == cudaSuccess && n_b) e = cudaMemcpyAsync(d + d_b, stage + h_b, n_b * 32, cudaMemcpyHostToDevice, st);
    if (e == cudaSuccess && n_b) e = cudaMemcpyAsync(d + d_one, stage + h_one, 64, cudaMemcpyHostToDevice, st);
    if (e == cudaSuccess && log2_k)
      e = cudaMemcpyAsync(d + d_ht, stage + h_tbl + lo * tbl, cnt * tbl, cudaMemcpyHostToDevice, st);
    if (e == cudaSuccess) e = cudaMemsetAsync(bad, 0, 4, st);
    if (e == cudaSuccess) e = cudaEventRecord(s.ev_k0[0], st);
    if (e == cudaSuccess) e = ptau::launch_ntt_twiddles(d + d_tw, log2_k, wpow, st);
    launches += log2_k > 0;
    for (size_t j = 0; j < cnt && e == cudaSuccess; j++) {
      Fr c = hm[lo + j];  // c R = h^k R
      for (int i = 0; i < log2_k; i++) c = fr_mont_mul(c, c);
      uint32_t cp[ptau::kKzgZPowCount][8];
      fr_square_table(c, cp, ptau::kKzgZPowCount);
      int nl = 0;
      e = ptau::launch_coset_quotient(d, n, log2_k, cp, d + d_sums, s.d_msm_sc, d + t.rem + j * k * 32, bad, &nl, st);
      launches += nl;
      if (e == cudaSuccess) e = ptau::launch_msm_g1(powers->d_pts[g], s.d_msm_sc, nq, s.d_msm_scratch, d + d_r0, &nl, st);
      launches += nl;
      if (n_b) {
        if (e == cudaSuccess)
          e = ptau::launch_coset_quotient(d + d_b, n_b, 0, cp, d + d_sums, s.d_msm_sc, d + t.rv + j * 32, bad, &nl, st);
        launches += nl;
        if (e == cudaSuccess)
          e = ptau::launch_msm_g1(gamma_powers->d_pts[g], s.d_msm_sc, nbq, s.d_msm_scratch, d + d_r1, &nl, st);
        launches += nl;
        if (e == cudaSuccess) e = cudaMemcpyAsync(d + d_pair, d + d_r0, kMontG1, cudaMemcpyDeviceToDevice, st);
        if (e == cudaSuccess)
          e = cudaMemcpyAsync(d + d_pair + kMontG1, d + d_r1, kMontG1, cudaMemcpyDeviceToDevice, st);
        if (e == cudaSuccess) e = ptau::launch_msm_g1(d + d_pair, d + d_one, 2, s.d_msm_scratch, d + d_r0, &nl, st);
        launches += nl;
      }
      if (e == cudaSuccess)
        e = cudaMemcpyAsync(d + t.pf + j * kMontG1, d + d_r0, kMontG1, cudaMemcpyDeviceToDevice, st);
    }
    if (log2_k) {
      int nl = 0;
      if (e == cudaSuccess) e = ptau::launch_ntt(d + t.rem, d + t.val, cnt, log2_k, d + d_ht, d + d_tw, &nl, st);
      launches += nl;
    }
    if (e == cudaSuccess) e = cudaEventRecord(s.ev_k1[0], st);
    if (e == cudaSuccess) e = cudaMemcpyAsync(s.h_msm_out, bad, 4, cudaMemcpyDeviceToHost, st);
    ctx->timing.h2d_bytes[g] = (n + n_b) * 32 + (n_b ? 64 : 0) + cnt * tbl;
    ctx->timing.d2h_bytes[g] = cnt * (kMontG1 + k * 32 + (n_b ? 32 : 0)) + 4;
  }
  ctx->timing.kernel_launches = launches;
  // results to the caller's (pageable) memory only once every GPU has its work queued
  bool bad_coeff = false;
  for (int g = 0; g < G && e == cudaSuccess; g++) {
    GpuSlot& s = ctx->gpu[g];
    const ptau::Shard sh = shard(m, g, G);
    const size_t lo = sh.lo, cnt = sh.hi - sh.lo;
    const Tail t = tail(cnt);
    const uint8_t* d = (const uint8_t*)s.d_open;
    cudaStream_t st = s.stream[0];
    e = cudaSetDevice(s.device);
    if (e == cudaSuccess)
      e = cudaMemcpyAsync((uint8_t*)proofs_out + lo * kMontG1, d + t.pf, cnt * kMontG1, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess)
      e = cudaMemcpyAsync((uint8_t*)values_out + lo * k * 32, d + t.val, cnt * k * 32, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess && n_b)
      e = cudaMemcpyAsync((uint8_t*)random_v_out + lo * 32, d + t.rv, cnt * 32, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaEventRecord(s.ev_last, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    float kms = 0, gms = 0;
    if (e == cudaSuccess) e = cudaEventElapsedTime(&kms, s.ev_k0[0], s.ev_k1[0]);
    if (e == cudaSuccess) e = cudaEventElapsedTime(&gms, s.ev_first, s.ev_last);
    ctx->timing.kernel_ms[g] = kms;
    ctx->timing.gpu_ms[g] = gms;
    bad_coeff = bad_coeff || s.h_msm_out[0] != 0;
  }
  if (e != cudaSuccess) return drain_fail(ctx, G, where, e);
  ctx->timing.wall_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
  return bad_coeff ? PTAU_ERR_ARG : PTAU_OK;
}
}  // namespace

// KZG10::open of p at k points: the division by X - z of kzg_open_impl at log2_k = 0, optionally hiding.
int ptau_kzg_open(ptau_ctx* ctx, const ptau_kzg_powers* powers, const ptau_kzg_powers* gamma_powers, const void* coeffs,
                  size_t n, const void* blinding, size_t n_b, const void* points, size_t k, void* proofs_out,
                  void* values_out, void* random_v_out) {
  if (!ctx || !powers || powers->ctx != ctx || (gamma_powers && gamma_powers->ctx != ctx)) return PTAU_ERR_ARG;
  if (n > powers->n || (n_b && (!gamma_powers || n_b > gamma_powers->n))) return PTAU_ERR_ARG;  // TooManyCoefficients
  if ((n && !coeffs) || (n_b && !blinding)) return PTAU_ERR_ARG;
  if (k && (!points || !proofs_out || !values_out || (n_b > 0) != (random_v_out != nullptr))) return PTAU_ERR_ARG;
  if (!msm_fits(n) || !msm_fits(n_b)) return PTAU_ERR_ARG;
  timing_reset(ctx);
  if (k == 0) return PTAU_OK;
  if (!scalars_canonical(points, k)) return PTAU_ERR_ARG;
  return kzg_open_impl(ctx, __func__, powers, gamma_powers, coeffs, n, blinding, n_b, 0, points, k, proofs_out,
                       values_out, random_v_out);
}

// KZG10 openings of p on m cosets h <omega_k>: kzg_open_impl over the shifts, without hiding.
int ptau_kzg_open_cosets(ptau_ctx* ctx, const ptau_kzg_powers* powers, const void* coeffs, size_t n, int log2_k,
                         const void* shifts, size_t m, void* proofs_out, void* values_out) {
  if (!ctx || !powers || powers->ctx != ctx || log2_k < 0 || log2_k > ptau::kCosetLgKMax) return PTAU_ERR_ARG;
  if (n > powers->n || (n && !coeffs) || (m && (!shifts || !proofs_out || !values_out))) return PTAU_ERR_ARG;
  const uint64_t k = 1ull << log2_k;
  if (!msm_fits(n > k ? n - k : 0)) return PTAU_ERR_ARG;
  timing_reset(ctx);
  if (m == 0) return PTAU_OK;
  if (!shifts_valid(shifts, m)) return PTAU_ERR_ARG;
  return kzg_open_impl(ctx, __func__, powers, nullptr, coeffs, n, nullptr, 0, log2_k, shifts, m, proofs_out, values_out,
                       nullptr);
}

// GPU 0, one stream, no host round trip: the inverse NTT of every item's values, the randomizers and scalars, the
// k-term MSM over the resident powers, the 2m-term MSM over the commitments and proofs, their sum (a 2-term MSM with
// unit scalars), the m-term MSM -sum rho_i pi_i, and one pairing_product2 item; only its "is one" byte comes back.
int ptau_kzg_check_cosets(ptau_ctx* ctx, const ptau_kzg_powers* powers, const void* h, const void* tau_k_h, int log2_k,
                          const void* comms, const void* shifts, const void* values, const void* proofs, size_t m,
                          const uint8_t* seed, uint8_t* ok) {
  if (!ctx || !powers || powers->ctx != ctx || !h || !tau_k_h || !ok) return PTAU_ERR_ARG;
  if (log2_k < 0 || log2_k > ptau::kCosetLgKMax || (1ull << log2_k) > powers->n) return PTAU_ERR_ARG;
  if (m && (!comms || !shifts || !values || !proofs)) return PTAU_ERR_ARG;
  const uint64_t k = 1ull << log2_k;
  if (!msm_fits(k) || !msm_fits(2 * m)) return PTAU_ERR_ARG;
  auto t0 = std::chrono::steady_clock::now();
  timing_reset(ctx);
  if (m == 0) {  // nothing to refute
    *ok = 1;
    return PTAU_OK;
  }
  if (!shifts_valid(shifts, m) || !scalars_canonical(values, m * k)) return PTAU_ERR_ARG;
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
  uint64_t key[8];
  blake2b_keyed_start(key, sd, 32, 16);
  constexpr int kTbl = ptau::kCosetLgKMax;
  // per item: h^-1 by one batch inversion, its table h^(-2^s) R and c R = h^k R
  std::vector<Fr> hm(m), pre(m);
  for (size_t i = 0; i < m; i++) {
    hm[i] = fr_to_mont(fr_from_le32((const uint8_t*)shifts + i * 32));
    pre[i] = i ? fr_mont_mul(pre[i - 1], hm[i]) : hm[i];
  }
  uint64_t rm2[4];
  memcpy(rm2, FR_MOD, 32);
  rm2[0] -= 2;  // r - 2: the low limb of r is 0xffffffff00000001
  Fr inv = fr_mont_pow(pre[m - 1], rm2);
  // staging (pinned): values | h^-1 tables | c R | commitments, proofs | h, tau_k_h | 1, 1
  const size_t h_tbl = m * k * 32, h_cm = h_tbl + m * kTbl * 32, h_pts = h_cm + m * 32, h_g2 = h_pts + 2 * m * kMontG1,
               h_one = h_g2 + 2 * kMontG2, h_len = h_one + 64;
  GpuSlot& s = ctx->gpu[0];
  cudaError_t e = cudaSetDevice(s.device);
  if (e == cudaSuccess) e = grow(&s.h_msm_sc, &s.cap_h_msm_sc, h_len, true);
  if (e != cudaSuccess) return cuda_fail(ctx, __func__, e);
  uint8_t* stage = (uint8_t*)s.h_msm_sc;
  copy_parts(stage, values, m * k * 32);
  for (size_t i = m; i-- > 0;) {
    const Fr hinv = i ? fr_mont_mul(inv, pre[i - 1]) : inv;  // inv = (h_0 .. h_i)^-1 R
    inv = fr_mont_mul(inv, hm[i]);
    fr_square_table(hinv, (uint32_t(*)[8])(stage + h_tbl + i * kTbl * 32), kTbl);
    Fr c = hm[i];
    for (int t = 0; t < log2_k; t++) c = fr_mont_mul(c, c);
    memcpy(stage + h_cm + i * 32, c.l, 32);
  }
  memcpy(stage + h_pts, comms, m * kMontG1);
  memcpy(stage + h_pts + m * kMontG1, proofs, m * kMontG1);
  memcpy(stage + h_g2, h, kMontG2);
  memcpy(stage + h_g2 + kMontG2, tau_k_h, kMontG2);
  memset(stage + h_one, 0, 64);
  stage[h_one] = stage[h_one + 32] = 1;
  // inverse twiddles: powers of omega_k^-1 = omega_k^(k - 1); k^-1 R^2 for the unscale
  Fr winv = fr_mont_one_host(), w = fr_root_mont(log2_k);
  for (int t = 0; t < log2_k; t++) {
    if (t) winv = fr_mont_mul(winv, winv);
    winv = fr_mont_mul(winv, w);
  }
  uint32_t wpow[ptau::kCosetLgKMax][8];
  fr_square_table(winv, wpow, log2_k);
  Fr half;  // 2^-1 = (r + 1) / 2
  memcpy(half.l, FR_MOD, 32);
  for (int i = 0; i < 4; i++) half.l[i] = (half.l[i] >> 1) | (i < 3 ? half.l[i + 1] << 63 : 0);
  half.l[0] += 1;  // r is odd: (r + 1) / 2 = (r >> 1) + 1
  Fr kinv = fr_mont_one_host(), hm2 = fr_to_mont(half);
  for (int t = 0; t < log2_k; t++) kinv = fr_mont_mul(kinv, hm2);
  const Fr kinv_r2 = fr_to_mont(kinv);
  // device layout of d_open: values | inverse NTT | twiddles | h^-1 tables | c R | rho k^-1 R | k-term scalars |
  // 2m-term scalars | -rho | points | G2 pair | 1, 1 | MSM results | their pair | pairing G1 input | is one
  const size_t d_x = up256(m * k * 32), d_tw = d_x + up256(m * k * 32), d_ht = d_tw + up256(k / 2 * 32),
               d_cm = d_ht + up256(m * kTbl * 32), d_srm = d_cm + up256(m * 32), d_sa = d_srm + up256(m * 32),
               d_sb = d_sa + up256(k * 32), d_neg = d_sb + up256(2 * m * 32), d_pts = d_neg + up256(m * 32),
               d_g2 = d_pts + up256(2 * m * kMontG1), d_one = d_g2 + up256(2 * kMontG2), d_ra = d_one + 256,
               d_rb = d_ra + 256, d_pair = d_rb + 256, d_g1 = d_pair + 256, d_ok = d_g1 + 512, d_len = d_ok + 256;
  size_t scratch = 0;
  for (size_t t : {(size_t)k, 2 * m, m, (size_t)2}) {
    ptau::MsmPlan plan;
    ptau::msm_g1_plan(t, &plan);
    scratch = plan.scratch_bytes > scratch ? plan.scratch_bytes : scratch;
  }
  if (e == cudaSuccess) e = grow(&s.d_open, &s.cap_open, d_len);
  if (e == cudaSuccess) e = grow(&s.d_msm_scratch, &s.cap_msm_scratch, scratch);
  if (e == cudaSuccess && !s.h_msm_out) e = cudaHostAlloc((void**)&s.h_msm_out, 256, cudaHostAllocPortable);
  if (e != cudaSuccess) return cuda_fail(ctx, __func__, e);
  uint8_t* d = (uint8_t*)s.d_open;
  cudaStream_t st = s.stream[0];
  int launches = 0, nl = 0;
  e = cudaEventRecord(s.ev_first, st);
  if (e == cudaSuccess) e = cudaMemcpyAsync(d, stage, m * k * 32, cudaMemcpyHostToDevice, st);
  if (e == cudaSuccess) e = cudaMemcpyAsync(d + d_ht, stage + h_tbl, m * kTbl * 32, cudaMemcpyHostToDevice, st);
  if (e == cudaSuccess) e = cudaMemcpyAsync(d + d_cm, stage + h_cm, m * 32, cudaMemcpyHostToDevice, st);
  if (e == cudaSuccess) e = cudaMemcpyAsync(d + d_pts, stage + h_pts, 2 * m * kMontG1, cudaMemcpyHostToDevice, st);
  if (e == cudaSuccess) e = cudaMemcpyAsync(d + d_g2, stage + h_g2, 2 * kMontG2, cudaMemcpyHostToDevice, st);
  if (e == cudaSuccess) e = cudaMemcpyAsync(d + d_one, stage + h_one, 64, cudaMemcpyHostToDevice, st);
  if (e == cudaSuccess) e = cudaEventRecord(s.ev_k0[0], st);
  if (e == cudaSuccess) e = ptau::launch_ntt_twiddles(d + d_tw, log2_k, wpow, st);
  launches += log2_k > 0;
  if (e == cudaSuccess) e = ptau::launch_ntt(d, d + d_x, m, log2_k, nullptr, d + d_tw, &nl, st);
  launches += nl;
  if (e == cudaSuccess)
    e = ptau::launch_coset_check_scalars(key, m, d + d_cm, (const uint32_t*)kinv_r2.l, d + d_srm, d + d_sb, d + d_neg, st);
  if (e == cudaSuccess) e = ptau::launch_coset_interp_sum(d + d_x, m, log2_k, d + d_ht, d + d_srm, d + d_sa, st);
  launches += 2;
  // sum rho_i (C_i + [c_i] pi_i) - [sum_j a_j tau^j] G  (the scalars a_j are negated), as the 2-term sum of two MSMs
  if (e == cudaSuccess) e = ptau::launch_msm_g1(powers->d_pts[0], d + d_sa, k, s.d_msm_scratch, d + d_ra, &nl, st);
  launches += nl;
  if (e == cudaSuccess) e = ptau::launch_msm_g1(d + d_pts, d + d_sb, 2 * m, s.d_msm_scratch, d + d_rb, &nl, st);
  launches += nl;
  if (e == cudaSuccess) e = cudaMemcpyAsync(d + d_pair, d + d_ra, kMontG1, cudaMemcpyDeviceToDevice, st);
  if (e == cudaSuccess) e = cudaMemcpyAsync(d + d_pair + kMontG1, d + d_rb, kMontG1, cudaMemcpyDeviceToDevice, st);
  if (e == cudaSuccess) e = ptau::launch_msm_g1(d + d_pair, d + d_one, 2, s.d_msm_scratch, d + d_g1, &nl, st);
  launches += nl;
  // -sum rho_i pi_i second: its result word past the record lands beyond the pairing input
  if (e == cudaSuccess)
    e = ptau::launch_msm_g1(d + d_pts + m * kMontG1, d + d_neg, m, s.d_msm_scratch, d + d_g1 + kMontG1, &nl, st);
  launches += nl;
  if (e == cudaSuccess) e = ptau::launch_pairing_product2(d + d_g1, d + d_g2, 1, nullptr, d + d_ok, st);
  launches += 1;
  if (e == cudaSuccess) e = cudaEventRecord(s.ev_k1[0], st);
  if (e == cudaSuccess) e = cudaMemcpyAsync(s.h_msm_out, d + d_ok, 1, cudaMemcpyDeviceToHost, st);
  if (e == cudaSuccess) e = cudaEventRecord(s.ev_last, st);
  if (e == cudaSuccess) e = cudaStreamSynchronize(st);
  float kms = 0, gms = 0;
  if (e == cudaSuccess) e = cudaEventElapsedTime(&kms, s.ev_k0[0], s.ev_k1[0]);
  if (e == cudaSuccess) e = cudaEventElapsedTime(&gms, s.ev_first, s.ev_last);
  if (e != cudaSuccess) return drain_fail(ctx, 1, __func__, e);
  ctx->timing.kernel_launches = launches;
  ctx->timing.kernel_ms[0] = kms;
  ctx->timing.gpu_ms[0] = gms;
  ctx->timing.h2d_bytes[0] = h_len;
  ctx->timing.d2h_bytes[0] = 1;
  *ok = ((const uint8_t*)s.h_msm_out)[0] != 0;
  ctx->timing.wall_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
  return PTAU_OK;
}

int ptau_selftest_fq_op(ptau_ctx* ctx, int gpu, int op, const void* a, const void* b, void* out, size_t n) {
  if (!ctx || gpu < 0 || gpu >= ctx->n_gpus || !a || !b || !out) return PTAU_ERR_ARG;
  void *da = nullptr, *db = nullptr, *dout = nullptr;
  return launch_once(ctx, gpu, __func__, false,
                     {{a, nullptr, n * 48, &da}, {b, nullptr, n * 48, &db}, {nullptr, out, n * 48, &dout}},
                     [&](cudaStream_t st) { return ptau::launch_fq_op(op, da, db, dout, n, st); });
}

int ptau_microbench(ptau_ctx* ctx, int gpu, int kind, int iters, double* ms, double* ops) {
  if (!ctx || gpu < 0 || gpu >= ctx->n_gpus || !ms || !ops || iters < 1) return PTAU_ERR_ARG;
  GpuSlot& s = ctx->gpu[gpu];
  CUDA_TRY(ctx, cudaSetDevice(s.device));
  cudaDeviceProp prop;
  CUDA_TRY(ctx, cudaGetDeviceProperties(&prop, s.device));
  const int block = 256;
  const int grid = prop.multiProcessorCount * (kind == 2 ? 2 : ((kind == 3 || kind == 4) ? 1 : 4));
  uint32_t* d_out = nullptr;
  CUDA_TRY(ctx, cudaMalloc((void**)&d_out, (size_t)grid * block * 4 * 4));
  double o = 0;
  cudaError_t e = ptau::launch_microbench(kind, iters > 16 ? 16 : iters, d_out, grid, block, &o, s.stream[0]);  // warm-up
  if (e == cudaSuccess) e = cudaEventRecord(s.ev_k0[0], s.stream[0]);
  if (e == cudaSuccess) e = ptau::launch_microbench(kind, iters, d_out, grid, block, &o, s.stream[0]);
  if (e == cudaSuccess) e = cudaEventRecord(s.ev_k1[0], s.stream[0]);
  if (e == cudaSuccess) e = cudaStreamSynchronize(s.stream[0]);
  float t = 0;
  if (e == cudaSuccess) e = cudaEventElapsedTime(&t, s.ev_k0[0], s.ev_k1[0]);
  cudaFree(d_out);
  if (e != cudaSuccess) return cuda_fail(ctx, __func__, e);
  *ms = t;
  *ops = o;
  return PTAU_OK;
}

}  // extern "C"
