// CUDA kernels (sm_100a) of the per-point path and their launch wrappers.
//
// Data movement: a block of PTAU_BLOCK threads owns PTAU_BLOCK consecutive
// records.  The packed record stream is read with coalesced 128-bit loads into
// shared memory, each thread gathers its own record (its 12/24/48 big- or
// little-endian words) from there, and results go back the same way.  HBM traffic
// is exactly record_in + record_out bytes per point; everything between is
// integer multiply-add work on the FMA pipe (IMAD.WIDE chains, see fq.cuh).
#include <cuda_runtime.h>
#include <stdint.h>
#include <string.h>

#include <type_traits>

#include "kernels.h"
#include "point.cuh"
#include "msm.cuh"

namespace ptau {

#ifndef PTAU_BLOCK
#define PTAU_BLOCK 128
#endif
// A/B-measured on B200 (tools/ab_bench.py): G1 ladders with the doubling expanded in place
// (PTAU_G1_DBL_INLINE) run best at 2 blocks/SM (30.1 M pts/s); with calls, 3-4 blocks/SM
// (29.1-29.4 M pts/s).
#ifndef PTAU_MINBLOCKS_G1
#define PTAU_MINBLOCKS_G1 2
#endif
#ifndef PTAU_MINBLOCKS_G2
#define PTAU_MINBLOCKS_G2 2
#endif
// threads per block of the convert kernels, per group (A/B knob; the staging buffer is BLK records)
#ifndef PTAU_BLOCK_G1
#define PTAU_BLOCK_G1 PTAU_BLOCK
#endif
#ifndef PTAU_BLOCK_G2
#define PTAU_BLOCK_G2 PTAU_BLOCK
#endif

__device__ __forceinline__ uint4 ld_stream(const uint4* p) {
  uint4 v;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
               : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w)
               : "l"(p));
  return v;
}

// Shared-memory stride of a record of W words.  Each thread reads / writes its own record with 128-bit accesses, which a
// warp performs in quarter-warps: conflict-free iff (stride / 4) is odd.  24- and 48-word records get one vector of
// padding (28, 52); 12-word records are fine; the 26- / 50-word Montgomery records (8-byte granular) are left alone.
__host__ __device__ constexpr int smem_stride(int w) { return (w % 4 == 0 && ((w / 4) % 2) == 0) ? w + 4 : w; }

// global -> shared: record r of W words lands at sm + r * S (block-cooperative, coalesced 128-bit global accesses)
template <int BLK, int W, int S>
__device__ __forceinline__ void stage_in(const uint32_t* __restrict__ g, uint32_t* sm, int nrec) {
  if (W % 4 == 0) {
    constexpr int VPR = W / 4;
    const uint4* g4 = reinterpret_cast<const uint4*>(g);
    uint4* s4 = reinterpret_cast<uint4*>(sm);
    const int nvec = nrec * VPR;
    for (int i = threadIdx.x; i < nvec; i += BLK) {
      const int r = i / VPR, c = i - r * VPR;
      s4[r * (S / 4) + c] = ld_stream(g4 + i);
    }
  } else {  // S == W: flat copy
    const int nwords = nrec * W, nvec = nwords >> 2;
    const uint4* g4 = reinterpret_cast<const uint4*>(g);
    uint4* s4 = reinterpret_cast<uint4*>(sm);
    for (int i = threadIdx.x; i < nvec; i += BLK) s4[i] = ld_stream(g4 + i);
    for (int i = (nvec << 2) + threadIdx.x; i < nwords; i += BLK) sm[i] = g[i];
  }
}
template <int BLK, int W, int S>
__device__ __forceinline__ void stage_out(uint32_t* __restrict__ g, const uint32_t* sm, int nrec) {
  if (W % 4 == 0) {
    constexpr int VPR = W / 4;
    uint4* g4 = reinterpret_cast<uint4*>(g);
    const uint4* s4 = reinterpret_cast<const uint4*>(sm);
    const int nvec = nrec * VPR;
    for (int i = threadIdx.x; i < nvec; i += BLK) {
      const int r = i / VPR, c = i - r * VPR;
      g4[i] = s4[r * (S / 4) + c];
    }
  } else {
    const int nwords = nrec * W, nvec = nwords >> 2;
    uint4* g4 = reinterpret_cast<uint4*>(g);
    const uint4* s4 = reinterpret_cast<const uint4*>(sm);
    for (int i = threadIdx.x; i < nvec; i += BLK) g4[i] = s4[i];
    for (int i = (nvec << 2) + threadIdx.x; i < nwords; i += BLK) g[i] = sm[i];
  }
}

// shared -> global, flat (the generators: records written at their natural stride)
template <int BLK>
__device__ __forceinline__ void stage_out_flat(uint32_t* __restrict__ g, const uint32_t* sm, int nwords) {
  int nvec = nwords >> 2;
  uint4* g4 = reinterpret_cast<uint4*>(g);
  const uint4* s4 = reinterpret_cast<const uint4*>(sm);
  for (int i = threadIdx.x; i < nvec; i += BLK) g4[i] = s4[i];
  for (int i = (nvec << 2) + threadIdx.x; i < nwords; i += BLK) g[i] = sm[i];
}

// shared memory of one block: the record staging buffer (BLK x max(stride_in, stride_out)) and, for the G2 kernels
// with curve checks, the operand file of the subgroup ladder (PTAU_PARK_WORDS per thread, transposed: conflict-free)
template <int G, int INFMT, int OUTFMT, bool HEAVY>
constexpr int convert_smem_words() {
  constexpr int BLK = G == PTAU_G1 ? PTAU_BLOCK_G1 : PTAU_BLOCK_G2;
  constexpr int SIN = smem_stride(record_bytes(G, INFMT) / 4);
  constexpr int SOUT = smem_stride(record_bytes(G, OUTFMT) / 4);
  return BLK * (SIN > SOUT ? SIN : SOUT) + ((G == PTAU_G2 && HEAVY) ? BLK * PTAU_PARK_WORDS : 0);
}

// blocks per SM of the kernels without curve checks (memory-bound; A/B on B200: 2, 6 and 8 give the same 5.76-5.78 TB/s)
#ifndef PTAU_MINBLOCKS_LIGHT
#define PTAU_MINBLOCKS_LIGHT 2
#endif
template <int G, int INFMT, int OUTFMT, bool HEAVY>
__global__ void __launch_bounds__((G == PTAU_G1 ? PTAU_BLOCK_G1 : PTAU_BLOCK_G2),
                                  (!HEAVY ? PTAU_MINBLOCKS_LIGHT : G == PTAU_G1 ? PTAU_MINBLOCKS_G1 : PTAU_MINBLOCKS_G2))
    convert_kernel(const uint32_t* __restrict__ in, uint32_t* __restrict__ out, uint64_t n, uint32_t checks,
                   uint64_t base_index, unsigned long long* __restrict__ status) {
  constexpr int BLK = G == PTAU_G1 ? PTAU_BLOCK_G1 : PTAU_BLOCK_G2;
  constexpr int WIN = record_bytes(G, INFMT) / 4;
  constexpr int WOUT = record_bytes(G, OUTFMT) / 4;
  constexpr int SIN = smem_stride(WIN), SOUT = smem_stride(WOUT);
  constexpr int SMAX = SIN > SOUT ? SIN : SOUT;
  extern __shared__ __align__(16) uint32_t sm[];

  const uint64_t rec0 = (uint64_t)blockIdx.x * BLK;
  const int nrec = (int)((n - rec0) < (uint64_t)BLK ? (n - rec0) : (uint64_t)BLK);
  const int tid = threadIdx.x;

  stage_in<BLK, WIN, SIN>(in + rec0 * WIN, sm, nrec);
  __syncthreads();

  uint32_t win[WIN];
  if (tid < nrec) {
    if (WIN % 4 == 0) {
      const uint4* s4 = reinterpret_cast<const uint4*>(sm + tid * SIN);
#pragma unroll
      for (int j = 0; j < WIN / 4; j++) {
        uint4 v = s4[j];
        win[4 * j] = v.x;
        win[4 * j + 1] = v.y;
        win[4 * j + 2] = v.z;
        win[4 * j + 3] = v.w;
      }
    } else {  // Montgomery-limb records: 104 / 200 bytes, 8-byte granular
      const uint2* s2 = reinterpret_cast<const uint2*>(sm + tid * SIN);
#pragma unroll
      for (int j = 0; j < WIN / 2; j++) {
        uint2 v = s2[j];
        win[2 * j] = v.x;
        win[2 * j + 1] = v.y;
      }
    }
  }
  __syncthreads();

  if (tid < nrec) {
    uint32_t st;
    if (G == PTAU_G2 && HEAVY) {
      // every input record is in registers now: the thread's slot of the staging buffer takes the output record
      // directly (written before the subgroup ladder starts), and the ladder's base point lives in the operand file
      Park<BLK> pk;
      pk.base = (uint32_t)__cvta_generic_to_shared(sm + BLK * SMAX + tid);
      st = g2_process<INFMT, HEAVY, BLK>(win, OUTFMT, sm + tid * SOUT, checks, pk);
    } else {
      uint32_t wout[WOUT];
      if (G == PTAU_G2) {
        Park<BLK> pk;
        pk.base = 0;  // no ladder in this instance: never touched
        st = g2_process<INFMT, HEAVY, BLK>(win, OUTFMT, wout, checks, pk);
      } else {
        st = g1_process<INFMT, HEAVY>(win, OUTFMT, wout, checks);
      }
      if (WOUT % 4 == 0) {
        uint4* s4 = reinterpret_cast<uint4*>(sm + tid * SOUT);
#pragma unroll
        for (int j = 0; j < WOUT / 4; j++) s4[j] = make_uint4(wout[4 * j], wout[4 * j + 1], wout[4 * j + 2], wout[4 * j + 3]);
      } else {
        uint2* s2 = reinterpret_cast<uint2*>(sm + tid * SOUT);
#pragma unroll
        for (int j = 0; j < WOUT / 2; j++) s2[j] = make_uint2(wout[2 * j], wout[2 * j + 1]);
      }
    }
    if (st != PTAU_OK) atomicMin(status, (unsigned long long)(((base_index + rec0 + tid) << 8) | st));
  }
  __syncthreads();
  stage_out<BLK, WOUT, SOUT>(out + rec0 * WOUT, sm, nrec);
}

template <int G, int INFMT, int OUTFMT, bool HEAVY>
static cudaError_t launch_inst(const void* d_in, void* d_out, uint64_t n, uint32_t checks, uint64_t base_index,
                               unsigned long long* d_status, cudaStream_t stream) {
  constexpr int BLK = G == PTAU_G1 ? PTAU_BLOCK_G1 : PTAU_BLOCK_G2;
  constexpr int SMEM = convert_smem_words<G, INFMT, OUTFMT, HEAVY>() * 4;
  auto kern = convert_kernel<G, INFMT, OUTFMT, HEAVY>;
  if (SMEM > 48 * 1024) {  // per device: cheap, and a context may own several GPUs
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM);
    if (e != cudaSuccess) return e;
  }
  unsigned grid = (unsigned)((n + BLK - 1) / BLK);
  kern<<<grid, BLK, SMEM, stream>>>((const uint32_t*)d_in, (uint32_t*)d_out, n, checks, base_index, d_status);
  return cudaGetLastError();
}

template <int G, int INFMT, int OUTFMT>
static cudaError_t launch_one(const void* d_in, void* d_out, uint64_t n, uint32_t checks, uint64_t base_index,
                              unsigned long long* d_status, cudaStream_t stream) {
  if (n == 0) return cudaSuccess;
  // no curve checks requested on an uncompressed input: the lightweight instance
  // (compressed input is on the curve by construction, so only the subgroup bit matters there)
  const bool light = INFMT == PTAU_FMT_ZCASH_COMPRESSED
                         ? !(checks & PTAU_CHECK_SUBGROUP)
                         : !(checks & (PTAU_CHECK_ON_CURVE | PTAU_CHECK_SUBGROUP));
  if (light) return launch_inst<G, INFMT, OUTFMT, false>(d_in, d_out, n, checks, base_index, d_status, stream);
  return launch_inst<G, INFMT, OUTFMT, true>(d_in, d_out, n, checks, base_index, d_status, stream);
}

template <int G, int INFMT>
static cudaError_t launch_in(int out_fmt, const void* d_in, void* d_out, uint64_t n, uint32_t checks,
                             uint64_t base_index, unsigned long long* d_status, cudaStream_t stream) {
  switch (out_fmt) {
    case PTAU_FMT_ZCASH_UNCOMPRESSED:
      return launch_one<G, INFMT, PTAU_FMT_ZCASH_UNCOMPRESSED>(d_in, d_out, n, checks, base_index, d_status, stream);
    case PTAU_FMT_ARK_UNCOMPRESSED:
      return launch_one<G, INFMT, PTAU_FMT_ARK_UNCOMPRESSED>(d_in, d_out, n, checks, base_index, d_status, stream);
    case PTAU_FMT_ARK_MONT_LIMBS:
      return launch_one<G, INFMT, PTAU_FMT_ARK_MONT_LIMBS>(d_in, d_out, n, checks, base_index, d_status, stream);
  }
  return cudaErrorInvalidValue;
}

template <int G>
static cudaError_t launch_g(int in_fmt, int out_fmt, const void* d_in, void* d_out, uint64_t n, uint32_t checks,
                            uint64_t base_index, unsigned long long* d_status, cudaStream_t stream) {
  switch (in_fmt) {
    case PTAU_FMT_ZCASH_UNCOMPRESSED:
      return launch_in<G, PTAU_FMT_ZCASH_UNCOMPRESSED>(out_fmt, d_in, d_out, n, checks, base_index, d_status, stream);
    case PTAU_FMT_ZCASH_COMPRESSED:
      return launch_in<G, PTAU_FMT_ZCASH_COMPRESSED>(out_fmt, d_in, d_out, n, checks, base_index, d_status, stream);
    case PTAU_FMT_ARK_UNCOMPRESSED:
      return launch_in<G, PTAU_FMT_ARK_UNCOMPRESSED>(out_fmt, d_in, d_out, n, checks, base_index, d_status, stream);
    case PTAU_FMT_ARK_MONT_LIMBS:
      return launch_in<G, PTAU_FMT_ARK_MONT_LIMBS>(out_fmt, d_in, d_out, n, checks, base_index, d_status, stream);
  }
  return cudaErrorInvalidValue;
}

cudaError_t launch_convert(int group, int in_fmt, int out_fmt, const void* d_in, void* d_out, uint64_t n,
                           uint32_t checks, uint64_t base_index, unsigned long long* d_status,
                           cudaStream_t stream) {
  if (group == PTAU_G1) return launch_g<PTAU_G1>(in_fmt, out_fmt, d_in, d_out, n, checks, base_index, d_status, stream);
  if (group == PTAU_G2) return launch_g<PTAU_G2>(in_fmt, out_fmt, d_in, d_out, n, checks, base_index, d_status, stream);
  return cudaErrorInvalidValue;
}

// =============================================================================
// generator v1: out[i] = [k_i] G for host-supplied scalars, plain double-and-add and a
// Fermat inversion per point.  Only used to build the fixed-base table of generator v2.
// =============================================================================
__constant__ uint32_t K_PM2[12] = {0xffffaaa9u, 0xb9feffffu, 0xb153ffffu, 0x1eabfffeu, 0xf6b0f624u, 0x6730d2a0u,
                                   0xf38512bfu, 0x64774b84u, 0x434bacd7u, 0x4b1ba7b6u, 0x397fe69au, 0x1a0111eau};

// a^(p-2) (Fermat inverse), plain square-and-multiply over the constant exponent
static __device__ __noinline__ Fq fq_inv(Fq a) {
  Fq acc = a;  // top bit of p-2 (bit 380)
#pragma unroll 1
  for (int i = 379; i >= 0; --i) {
    acc = fq_sqr(acc);
    if ((K_PM2[i >> 5] >> (i & 31)) & 1u) acc = fq_mul(acc, a);
  }
  return acc;
}

template <int G, int OUTFMT>
__global__ void __launch_bounds__(PTAU_BLOCK)
    generate_kernel(const uint32_t* __restrict__ scalars, uint32_t* __restrict__ out, uint64_t n) {
  constexpr int WOUT = record_bytes(G, OUTFMT) / 4;
  __shared__ __align__(16) uint32_t sm[PTAU_BLOCK * WOUT];
  const uint64_t rec0 = (uint64_t)blockIdx.x * PTAU_BLOCK;
  const int nrec = (int)((n - rec0) < (uint64_t)PTAU_BLOCK ? (n - rec0) : (uint64_t)PTAU_BLOCK);
  const int tid = threadIdx.x;
  if (tid < nrec) {
    uint32_t k[8];
#pragma unroll
    for (int j = 0; j < 8; j++) k[j] = scalars[(rec0 + tid) * 8 + j];
    uint32_t* o = sm + tid * WOUT;
    if (G == PTAU_G1) {
      Fq gx = k_g1x_mont(), gy = k_g1y_mont();
      Jac<Fq> acc;
      acc.X = gx;
      acc.Y = gy;
      acc.Z = fq_one();
      bool started = false;
#pragma unroll 1
      for (int i = 254; i >= 0; --i) {
        bool bit = (k[i >> 5] >> (i & 31)) & 1u;
        if (started) {
          jac_dbl(acc);
          if (bit) jac_madd(acc, gx, gy);
        } else if (bit) {
          started = true;
        }
      }
      // to affine (k != 0 and k < r guarantee a finite result without exceptional cases)
      Fq zi = fq_inv(acc.Z);
      Fq zi2 = fq_sqr(zi);
      Fq xm = fq_mul(acc.X, zi2);
      Fq ym = fq_mul(acc.Y, fq_mul(zi2, zi));
      Fq xp = fq_from_mont(xm), yp = fq_from_mont(ym);
      if (OUTFMT == PTAU_FMT_ZCASH_COMPRESSED) {
        uint32_t fl = 0x80000000u | (fq_plain_is_largest(yp) ? 0x20000000u : 0u);
        xp.l[11] |= fl;
        fq_to_be_words(xp, o);
      } else {
        fq_to_be_words(xp, o);
        fq_to_be_words(yp, o + 12);
      }
    } else {
      Fq2 gx, gy;
      gx.c0 = k_g2x0_mont();
      gx.c1 = k_g2x1_mont();
      gy.c0 = k_g2y0_mont();
      gy.c1 = k_g2y1_mont();
      Jac<Fq2> acc;
      acc.X = gx;
      acc.Y = gy;
      acc.Z = fq2_one();
      bool started = false;
#pragma unroll 1
      for (int i = 254; i >= 0; --i) {
        bool bit = (k[i >> 5] >> (i & 31)) & 1u;
        if (started) {
          jac_dbl(acc);
          if (bit) jac_madd(acc, gx, gy);
        } else if (bit) {
          started = true;
        }
      }
      // 1/Z in Fq2 = conj(Z) / norm(Z)
      Fq nrm = fq_add(fq_sqr(acc.Z.c0), fq_sqr(acc.Z.c1));
      Fq ni = fq_inv(nrm);
      Fq2 zi;
      zi.c0 = fq_mul(acc.Z.c0, ni);
      zi.c1 = fq_neg(fq_mul(acc.Z.c1, ni));
      Fq2 zi2 = fq2_sqr(zi);
      Fq2 xm = fq2_mul(acc.X, zi2);
      Fq2 ym = fq2_mul(acc.Y, fq2_mul(zi2, zi));
      Fq2 xp, yp;
      xp.c0 = fq_from_mont(xm.c0);
      xp.c1 = fq_from_mont(xm.c1);
      yp.c0 = fq_from_mont(ym.c0);
      yp.c1 = fq_from_mont(ym.c1);
      if (OUTFMT == PTAU_FMT_ZCASH_COMPRESSED) {
        bool largest = fq_is_zero(yp.c1) ? fq_plain_is_largest(yp.c0) : fq_plain_is_largest(yp.c1);
        xp.c1.l[11] |= 0x80000000u | (largest ? 0x20000000u : 0u);
        fq_to_be_words(xp.c1, o);
        fq_to_be_words(xp.c0, o + 12);
      } else {
        fq_to_be_words(xp.c1, o);
        fq_to_be_words(xp.c0, o + 12);
        fq_to_be_words(yp.c1, o + 24);
        fq_to_be_words(yp.c0, o + 36);
      }
    }
  }
  __syncthreads();
  stage_out_flat<PTAU_BLOCK>(out + rec0 * WOUT, sm, nrec * WOUT);
}

cudaError_t launch_generate(int group, int fmt, const uint32_t* d_scalars, void* d_out, uint64_t n,
                            cudaStream_t stream) {
  if (n == 0) return cudaSuccess;
  unsigned grid = (unsigned)((n + PTAU_BLOCK - 1) / PTAU_BLOCK);
  if (group == PTAU_G1 && fmt == PTAU_FMT_ZCASH_COMPRESSED)
    generate_kernel<PTAU_G1, PTAU_FMT_ZCASH_COMPRESSED><<<grid, PTAU_BLOCK, 0, stream>>>(d_scalars, (uint32_t*)d_out, n);
  else if (group == PTAU_G1 && fmt == PTAU_FMT_ZCASH_UNCOMPRESSED)
    generate_kernel<PTAU_G1, PTAU_FMT_ZCASH_UNCOMPRESSED><<<grid, PTAU_BLOCK, 0, stream>>>(d_scalars, (uint32_t*)d_out, n);
  else if (group == PTAU_G2 && fmt == PTAU_FMT_ZCASH_COMPRESSED)
    generate_kernel<PTAU_G2, PTAU_FMT_ZCASH_COMPRESSED><<<grid, PTAU_BLOCK, 0, stream>>>(d_scalars, (uint32_t*)d_out, n);
  else if (group == PTAU_G2 && fmt == PTAU_FMT_ZCASH_UNCOMPRESSED)
    generate_kernel<PTAU_G2, PTAU_FMT_ZCASH_UNCOMPRESSED><<<grid, PTAU_BLOCK, 0, stream>>>(d_scalars, (uint32_t*)d_out, n);
  else
    return cudaErrorInvalidValue;
  return cudaGetLastError();
}

// =============================================================================
// generator v2 (SURVEY 8f-1): fixed-base windowed multiplication, scalars formed
// on the device, batch inversion to affine.
//
//   k_i = scalar0 * step^(first+i) mod r        (8 x u32 Montgomery arithmetic in Fr)
//   [k_i]G = sum_w T[w][digit_w(k_i)]           (32 windows of 8 bits, 31 mixed additions)
//   to affine: one field inversion per PTAU_GEN_B points of a thread (Montgomery's
//   trick: B-1 prefix products, one Fermat inversion, 2(B-1) back-multiplications).
//
// T[w][d-1] = [d * 256^w]G as PTAU_FMT_ARK_MONT_LIMBS records, built once per context
// with the v1 kernel.  No exceptional cases: the partial sums are < 256^w <= d*256^w and
// k < r, so an addition never meets equal or opposite points.
// =============================================================================
#define PTAU_GEN_B 8

struct FrParams {
  uint32_t s0[8];         // scalar0, Montgomery form
  uint32_t pw[64][8];     // step^(2^j), Montgomery form
};

}  // namespace ptau
// K_FR_MOD, fr_mul; included here so that the constant bank keeps its layout
#include "fr.cuh"
namespace ptau {

template <class F>
struct FieldInv;
template <>
struct FieldInv<Fq> {
  static __device__ __forceinline__ Fq inv(const Fq& a) { return fq_inv(a); }
};
template <>
struct FieldInv<Fq2> {
  static __device__ __forceinline__ Fq2 inv(const Fq2& a) {
    Fq ni = fq_inv(fq_add(fq_sqr(a.c0), fq_sqr(a.c1)));
    Fq2 r;
    r.c0 = fq_mul(a.c0, ni);
    r.c1 = fq_neg(fq_mul(a.c1, ni));
    return r;
  }
};

template <class F>
__device__ __forceinline__ F load_tbl_field(const uint32_t* p);
template <>
__device__ __forceinline__ Fq load_tbl_field<Fq>(const uint32_t* p) {
  Fq r;
  const uint2* q = reinterpret_cast<const uint2*>(p);
#pragma unroll
  for (int i = 0; i < 6; i++) {
    uint2 v = __ldg(q + i);
    r.l[2 * i] = v.x;
    r.l[2 * i + 1] = v.y;
  }
  return r;
}
template <>
__device__ __forceinline__ Fq2 load_tbl_field<Fq2>(const uint32_t* p) {
  Fq2 r;
  r.c0 = load_tbl_field<Fq>(p);
  r.c1 = load_tbl_field<Fq>(p + 12);
  return r;
}

template <class F>
__device__ __forceinline__ F field_one();
template <>
__device__ __forceinline__ Fq field_one<Fq>() { return fq_one(); }
template <>
__device__ __forceinline__ Fq2 field_one<Fq2>() { return fq2_one(); }

template <int G, int OUTFMT>
__global__ void __launch_bounds__(PTAU_BLOCK)
    generate_win_kernel(FrParams fp, const uint32_t* __restrict__ tbl, uint32_t* __restrict__ out, uint64_t first,
                        uint64_t n) {
  using F = typename std::conditional<G == PTAU_G1, Fq, Fq2>::type;
  constexpr int WOUT = record_bytes(G, OUTFMT) / 4;
  constexpr int WTBL = record_bytes(G, PTAU_FMT_ARK_MONT_LIMBS) / 4;
  constexpr int WF = sizeof(F) / 4;
  __shared__ __align__(16) uint32_t sm[PTAU_BLOCK * WOUT];
  const int tid = threadIdx.x;
  // the block owns PTAU_BLOCK * B consecutive points; thread t owns t + j * PTAU_BLOCK
  const uint64_t blk0 = (uint64_t)blockIdx.x * (PTAU_BLOCK * PTAU_GEN_B);

  // ---- scalar of this thread's first point: s0 * step^(first + blk0 + tid) ----
  uint32_t cur[8];
  {
#pragma unroll
    for (int i = 0; i < 8; i++) cur[i] = fp.s0[i];
    uint64_t e = first + blk0 + tid;
#pragma unroll 1
    for (int j = 0; j < 64; j++)
      if ((e >> j) & 1ull) fr_mul(cur, cur, fp.pw[j]);
  }

  Jac<F> pts[PTAU_GEN_B];
  F pre[PTAU_GEN_B];
#pragma unroll 1
  for (int j = 0; j < PTAU_GEN_B; j++) {
    const uint64_t idx = blk0 + (uint64_t)j * PTAU_BLOCK + tid;
    Jac<F> acc;
    acc.X = field_one<F>();
    acc.Y = field_one<F>();
    acc.Z = field_one<F>();
    if (idx < n) {
      uint32_t k[8];
      {
        uint32_t one[8] = {1, 0, 0, 0, 0, 0, 0, 0};
        fr_mul(k, cur, one);  // out of Montgomery form
      }
      bool started = false;
#pragma unroll 1
      for (int w = 0; w < 32; w++) {
        uint32_t d = (k[w >> 2] >> ((w & 3) * 8)) & 0xffu;
        if (d) {
          const uint32_t* e = tbl + (size_t)(w * 255 + (d - 1)) * WTBL;
          F x = load_tbl_field<F>(e);
          F y = load_tbl_field<F>(e + WF);
          if (started) {
            jac_madd(acc, x, y);
          } else {
            acc.X = x;
            acc.Y = y;
            started = true;
          }
        }
      }
      fr_mul(cur, cur, fp.pw[7]);  // next point of this thread is PTAU_BLOCK = 2^7 further
    }
    pts[j] = acc;
    pre[j] = (j == 0) ? acc.Z : fmul(pre[j - 1], acc.Z);
  }
  // ---- batch inversion (Montgomery's trick) ----
  F inv = FieldInv<F>::inv(pre[PTAU_GEN_B - 1]);
#pragma unroll 1
  for (int j = PTAU_GEN_B - 1; j >= 0; j--) {
    F zi = (j == 0) ? inv : fmul(inv, pre[j - 1]);
    if (j) inv = fmul(inv, pts[j].Z);
    F zi2 = fsqr(zi);
    F xm = fmul(pts[j].X, zi2);
    F ym = fmul(pts[j].Y, fmul(zi2, zi));
    const uint64_t rec0 = blk0 + (uint64_t)j * PTAU_BLOCK;
    uint32_t* o = sm + tid * WOUT;
    if (rec0 + tid < n) {
      if (G == PTAU_G1) {
        const Fq& xq = reinterpret_cast<const Fq&>(xm);
        const Fq& yq = reinterpret_cast<const Fq&>(ym);
        Fq xp = fq_from_mont(xq), yp = fq_from_mont(yq);
        if (OUTFMT == PTAU_FMT_ZCASH_COMPRESSED) {
          xp.l[11] |= 0x80000000u | (fq_plain_is_largest(yp) ? 0x20000000u : 0u);
          fq_to_be_words(xp, o);
        } else {
          fq_to_be_words(xp, o);
          fq_to_be_words(yp, o + 12);
        }
      } else {
        const Fq2& xq = reinterpret_cast<const Fq2&>(xm);
        const Fq2& yq = reinterpret_cast<const Fq2&>(ym);
        Fq2 xp, yp;
        xp.c0 = fq_from_mont(xq.c0);
        xp.c1 = fq_from_mont(xq.c1);
        yp.c0 = fq_from_mont(yq.c0);
        yp.c1 = fq_from_mont(yq.c1);
        if (OUTFMT == PTAU_FMT_ZCASH_COMPRESSED) {
          bool largest = fq_is_zero(yp.c1) ? fq_plain_is_largest(yp.c0) : fq_plain_is_largest(yp.c1);
          xp.c1.l[11] |= 0x80000000u | (largest ? 0x20000000u : 0u);
          fq_to_be_words(xp.c1, o);
          fq_to_be_words(xp.c0, o + 12);
        } else {
          fq_to_be_words(xp.c1, o);
          fq_to_be_words(xp.c0, o + 12);
          fq_to_be_words(yp.c1, o + 24);
          fq_to_be_words(yp.c0, o + 36);
        }
      }
    }
    __syncthreads();
    if (rec0 < n) {
      const int nrec = (int)((n - rec0) < (uint64_t)PTAU_BLOCK ? (n - rec0) : (uint64_t)PTAU_BLOCK);
      stage_out_flat<PTAU_BLOCK>(out + rec0 * WOUT, sm, nrec * WOUT);
    }
    __syncthreads();
  }
}

cudaError_t launch_generate_win(int group, int fmt, const uint32_t* s0_mont, const uint32_t (*pw_mont)[8],
                                const uint32_t* d_tbl, void* d_out, uint64_t first, uint64_t n, cudaStream_t stream) {
  if (n == 0) return cudaSuccess;
  FrParams fp;
  memcpy(fp.s0, s0_mont, 32);
  memcpy(fp.pw, pw_mont, sizeof(fp.pw));
  const uint64_t per_block = (uint64_t)PTAU_BLOCK * PTAU_GEN_B;
  unsigned grid = (unsigned)((n + per_block - 1) / per_block);
  if (group == PTAU_G1 && fmt == PTAU_FMT_ZCASH_COMPRESSED)
    generate_win_kernel<PTAU_G1, PTAU_FMT_ZCASH_COMPRESSED><<<grid, PTAU_BLOCK, 0, stream>>>(fp, d_tbl, (uint32_t*)d_out, first, n);
  else if (group == PTAU_G1 && fmt == PTAU_FMT_ZCASH_UNCOMPRESSED)
    generate_win_kernel<PTAU_G1, PTAU_FMT_ZCASH_UNCOMPRESSED><<<grid, PTAU_BLOCK, 0, stream>>>(fp, d_tbl, (uint32_t*)d_out, first, n);
  else if (group == PTAU_G2 && fmt == PTAU_FMT_ZCASH_COMPRESSED)
    generate_win_kernel<PTAU_G2, PTAU_FMT_ZCASH_COMPRESSED><<<grid, PTAU_BLOCK, 0, stream>>>(fp, d_tbl, (uint32_t*)d_out, first, n);
  else if (group == PTAU_G2 && fmt == PTAU_FMT_ZCASH_UNCOMPRESSED)
    generate_win_kernel<PTAU_G2, PTAU_FMT_ZCASH_UNCOMPRESSED><<<grid, PTAU_BLOCK, 0, stream>>>(fp, d_tbl, (uint32_t*)d_out, first, n);
  else
    return cudaErrorInvalidValue;
  return cudaGetLastError();
}

// =============================================================================
// SURVEY 8f-4: KZG10 commit = multi-scalar multiplication over the loaded powers,
//   C = sum_i [c_i] P_i   (ark-poly-commit 0.2 KZG10::commit, used at /root/reference/src/lib.rs:268-275).
// Bucket (Pippenger) method with signed windows.  The 256 scalar bits are cut into W = ceil(256 / c) windows of
// width c (the low `a` ones) or c - 1 (the rest) that add up to exactly 256, so that no window is partial:
// a partial top window (or a carry-only window) would put n / 2^few points into each of a handful of buckets
// and serialise them in a handful of threads.  The top window ends at bit 255, which is 0 for every scalar < r,
// so its digit never goes negative and never carries out.
//   1. msm_digits<false>  one thread per scalar: signed digits d_w in [-(2^(cw-1)-1), 2^(cw-1)], histogram of
//                   bucket (w, |d_w|) sizes
//   2. msm_scan     exclusive prefix sum of the histogram (one block; <= 2^19 + 1 counters)
//   3. msm_digits<true>  the same digits again, each non-zero one claims a slot of its bucket: a list of
//                   point indices (sign in bit 31) grouped by bucket -- a counting sort without a key array
//   3b. msm_size_hist / msm_size_scan / msm_size_scatter  counting sort of the buckets by size, largest first: thread t
//                   of the next kernel takes the t-th largest bucket, so the 32 lanes of a warp run the same number of
//                   additions (bucket sizes are Poisson around 32: in bucket order a warp waits for its largest lane,
//                   ~1.35 x the mean)
//   4. msm_bucket_sum    one thread per bucket: sum of its points (mixed additions)
//   5. msm_window_segments  per window, runs of L consecutive buckets: sum_j j B_j by running sums
//   6. msm_window_sum    one block per window adds the runs up and applies the window's weight 2^(c w)
//   7. msm_finish   adds the windows, one inversion, ark record
// Complete addition rules everywhere: the inputs are caller data (equal points, opposite points,
// infinity and zero scalars all occur in the tests), not ladders with known-safe scalars.
// =============================================================================

// pts: ARK_MONT_LIMBS records (26 words); scalars: 8 x u32 LE each, < r.  SCATTER = false: histogram
// into cnt[]; SCATTER = true: cnt[] holds the running cursor of every bucket, entries[] receives the indices.
// `bad` (SCATTER = false only): set when a scalar is not canonical (>= r; ark's Fr cannot hold such a value).
template <bool SCATTER>
__global__ void __launch_bounds__(256) msm_digits(const uint32_t* __restrict__ pts, const uint32_t* __restrict__ scalars,
                                                  uint64_t n, MsmGeom g, uint32_t* __restrict__ cnt,
                                                  uint32_t* __restrict__ entries, uint32_t* __restrict__ bad) {
  const uint64_t i = (uint64_t)blockIdx.x * 256 + threadIdx.x;
  if (i >= n) return;
  const uint32_t* k = scalars + i * 8;
  if (!SCATTER) {
    uint32_t bf = 0;  // k - r borrows  <=>  k < r
#pragma unroll
    for (int j = 0; j < 8; j++) {
      uint64_t t = (uint64_t)k[j] - K_R_ORDER_D[j] - bf;
      bf = (uint32_t)(t >> 63);
    }
    if (!bf) *bad = 1u;
  }
  if (pts[i * 26 + 24] & 0xffu) return;  // a point flagged infinity contributes nothing
  uint32_t carry = 0, base = 0;
  int bit = 0;
  for (int w = 0; w < g.W; w++) {
    const int cw = w < g.a ? g.c : g.c - 1;
    int d = msm_digit(k, bit, cw, carry);
    if (d != 0) {
      uint32_t b = base + (uint32_t)(d < 0 ? -d : d) - 1u;
      uint32_t pos = atomicAdd(&cnt[b], 1u);
      if (SCATTER) entries[pos] = (uint32_t)i | (d < 0 ? 0x80000000u : 0u);
    }
    bit += cw;
    base += 1u << (cw - 1);
  }
}

// the same over 50-word G2 records (only the position of the infinity flag differs; kept apart so that the
// G1 kernel keeps its code)
template <bool SCATTER>
__global__ void __launch_bounds__(256) msm_g2_digits(const uint32_t* __restrict__ pts, const uint32_t* __restrict__ scalars,
                                                  uint64_t n, MsmGeom g, uint32_t* __restrict__ cnt,
                                                  uint32_t* __restrict__ entries, uint32_t* __restrict__ bad) {
  const uint64_t i = (uint64_t)blockIdx.x * 256 + threadIdx.x;
  if (i >= n) return;
  const uint32_t* k = scalars + i * 8;
  if (!SCATTER) {
    uint32_t bf = 0;  // k - r borrows  <=>  k < r
#pragma unroll
    for (int j = 0; j < 8; j++) {
      uint64_t t = (uint64_t)k[j] - K_R_ORDER_D[j] - bf;
      bf = (uint32_t)(t >> 63);
    }
    if (!bf) *bad = 1u;
  }
  if (pts[i * 50 + 48] & 0xffu) return;  // a point flagged infinity contributes nothing
  uint32_t carry = 0, base = 0;
  int bit = 0;
  for (int w = 0; w < g.W; w++) {
    const int cw = w < g.a ? g.c : g.c - 1;
    int d = msm_digit(k, bit, cw, carry);
    if (d != 0) {
      uint32_t b = base + (uint32_t)(d < 0 ? -d : d) - 1u;
      uint32_t pos = atomicAdd(&cnt[b], 1u);
      if (SCATTER) entries[pos] = (uint32_t)i | (d < 0 ? 0x80000000u : 0u);
    }
    bit += cw;
    base += 1u << (cw - 1);
  }
}

// exclusive scan of cnt[0..m) into off[0..m], off[m] = total; cur[] = copy of off[] (scatter cursors).
// One block walks the array in coalesced tiles of 1024 x 4 counters (m <= 2^19 + 1: a few hundred tiles).
__global__ void __launch_bounds__(1024) msm_scan(const uint32_t* __restrict__ cnt, uint32_t m, uint32_t* __restrict__ off,
                                                 uint32_t* __restrict__ cur) {
  __shared__ uint32_t wsum[32];
  __shared__ uint32_t carry_s;
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  if (threadIdx.x == 0) carry_s = 0;
  __syncthreads();
  for (uint32_t base = 0; base < m; base += 4096) {
    const uint32_t j = base + threadIdx.x * 4;
    uint32_t v[4];
#pragma unroll
    for (int k = 0; k < 4; k++) v[k] = (j + k < m) ? cnt[j + k] : 0u;
    const uint32_t mine = v[0] + v[1] + v[2] + v[3];
    uint32_t incl = mine;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      uint32_t t = __shfl_up_sync(0xffffffffu, incl, d);
      if (lane >= d) incl += t;
    }
    if (lane == 31) wsum[wid] = incl;
    __syncthreads();
    if (wid == 0) {
      uint32_t w = wsum[lane], wi = w;
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) {
        uint32_t t = __shfl_up_sync(0xffffffffu, wi, d);
        if (lane >= d) wi += t;
      }
      wsum[lane] = wi - w;  // exclusive prefix of the warp totals
    }
    __syncthreads();
    const uint32_t carry = carry_s;
    uint32_t run = carry + wsum[wid] + incl - mine;
#pragma unroll
    for (int k = 0; k < 4; k++) {
      if (j + k < m) {
        off[j + k] = run;
        cur[j + k] = run;
      }
      run += v[k];
    }
    __syncthreads();
    if (threadIdx.x == 1023) carry_s = run;
    __syncthreads();
  }
  if (threadIdx.x == 0) off[m] = carry_s;
}

// Buckets ordered by size, largest first (a counting sort over min(size, PTAU_MSM_BINS - 1)).
//   msm_size_hist: hist[s] = number of buckets of size s;  msm_size_scan: hist[s] <- number of buckets larger than s;
//   msm_size_scatter: order[hist[s]++] = b.  The order inside a size class is not deterministic; the sums do not
//   depend on it (every bucket is still summed by one thread, in list order).
#define PTAU_MSM_BINS 1024
__global__ void __launch_bounds__(PTAU_MSM_BINS) msm_size_hist(const uint32_t* __restrict__ cnt, uint32_t m, uint32_t* __restrict__ hist) {
  __shared__ uint32_t h[PTAU_MSM_BINS];
  h[threadIdx.x] = 0;
  __syncthreads();
  const uint32_t b = blockIdx.x * PTAU_MSM_BINS + threadIdx.x;
  if (b < m) atomicAdd(&h[min(cnt[b], (uint32_t)PTAU_MSM_BINS - 1u)], 1u);
  __syncthreads();
  if (h[threadIdx.x]) atomicAdd(&hist[threadIdx.x], h[threadIdx.x]);
}
__global__ void __launch_bounds__(PTAU_MSM_BINS) msm_size_scan(uint32_t* __restrict__ hist) {
  __shared__ uint32_t wsum[32];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const uint32_t bin = PTAU_MSM_BINS - 1 - threadIdx.x;  // thread 0 owns the largest size
  const uint32_t mine = hist[bin];
  uint32_t incl = mine;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    uint32_t t = __shfl_up_sync(0xffffffffu, incl, d);
    if (lane >= d) incl += t;
  }
  if (lane == 31) wsum[wid] = incl;
  __syncthreads();
  if (wid == 0) {
    uint32_t w = wsum[lane], wi = w;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      uint32_t t = __shfl_up_sync(0xffffffffu, wi, d);
      if (lane >= d) wi += t;
    }
    wsum[lane] = wi - w;
  }
  __syncthreads();
  hist[bin] = wsum[wid] + incl - mine;
}
__global__ void __launch_bounds__(PTAU_MSM_BINS) msm_size_scatter(const uint32_t* __restrict__ cnt, uint32_t m, uint32_t* __restrict__ cursor,
                                                                  uint32_t* __restrict__ order) {
  __shared__ uint32_t h[PTAU_MSM_BINS], base[PTAU_MSM_BINS];
  h[threadIdx.x] = 0;
  __syncthreads();
  const uint32_t b = blockIdx.x * PTAU_MSM_BINS + threadIdx.x;
  uint32_t bin = 0, rank = 0;
  if (b < m) {
    bin = min(cnt[b], (uint32_t)PTAU_MSM_BINS - 1u);
    rank = atomicAdd(&h[bin], 1u);
  }
  __syncthreads();
  if (h[threadIdx.x]) base[threadIdx.x] = atomicAdd(&cursor[threadIdx.x], h[threadIdx.x]);
  __syncthreads();
  if (b < m) order[base[bin] + rank] = b;
}

// one thread per bucket (thread t: the t-th largest): sum of the bucket's points
__global__ void __launch_bounds__(PTAU_BLOCK) msm_bucket_sum(const uint32_t* __restrict__ pts, const uint32_t* __restrict__ entries,
                                                             const uint32_t* __restrict__ off, const uint32_t* __restrict__ order,
                                                             uint32_t m, uint32_t* __restrict__ buckets /* 36 words each */) {
  const uint32_t t = blockIdx.x * PTAU_BLOCK + threadIdx.x;
  if (t >= m) return;
  msm_bucket_item(pts, entries, off, order[t], buckets);
}

// one thread per run of L = 2^lgL consecutive buckets of one window (msm.cuh: msm_segment_item)
__global__ void __launch_bounds__(PTAU_BLOCK) msm_window_segments(const uint32_t* __restrict__ buckets, MsmGeom g, uint32_t nseg_total,
                                                                  uint32_t* __restrict__ seg /* 36 words each */) {
  const uint32_t t_id = blockIdx.x * PTAU_BLOCK + threadIdx.x;
  if (t_id >= nseg_total) return;
  msm_segment_item(buckets, g, t_id, seg);
}

// one block per window: adds the window's runs up (strided per thread, then a shared-memory tree) and applies
// the window's weight 2^bitoff, all windows in parallel
__global__ void __launch_bounds__(PTAU_BLOCK) msm_window_sum(const uint32_t* __restrict__ seg, MsmGeom g,
                                                             uint32_t* __restrict__ wsum /* 36 words per window */) {
  __shared__ uint32_t sm[PTAU_BLOCK * 36];
  const int w = blockIdx.x;
  const uint32_t first = msm_bucket_base(g, w) >> g.lgL;
  const uint32_t count = (w < g.a ? g.NB : g.NB >> 1) >> g.lgL;
  const uint32_t* base = seg + (uint64_t)first * 36;
  Jac<Fq> acc = jac_infinity();
  for (uint32_t i = threadIdx.x; i < count; i += PTAU_BLOCK) {
    Jac<Fq> q = jac_load(base + (uint64_t)i * 36);
    g1_add_complete(acc, q);
  }
  for (int stride = PTAU_BLOCK / 2; stride >= 1; stride >>= 1) {
    jac_store(sm + threadIdx.x * 36, acc);
    __syncthreads();
    if ((int)threadIdx.x < stride) {
      Jac<Fq> q = jac_load(sm + (threadIdx.x + stride) * 36);
      g1_add_complete(acc, q);
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    msm_window_weight(acc, g, w);
    jac_store(wsum + (uint64_t)w * 36, acc);
  }
}

// sum of the weighted window sums, one inversion, one record (msm.cuh: msm_finish_item)
__global__ void msm_finish(const uint32_t* __restrict__ wsum, int W, uint32_t* __restrict__ out) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  msm_finish_item(wsum, W, out);
}

// scratch layout for n terms; jac_bytes = 144 (G1) or 288 (G2) per Jacobian bucket / segment / window record
static void msm_plan(uint64_t n, uint64_t jac_bytes, MsmPlan* p) {
  const MsmGeom g = msm_geometry(n);
  p->c = g.c;
  p->W = g.W;
  p->a = g.a;
  p->NB = g.NB;
  p->lgL = g.lgL;
  p->buckets = (uint64_t)p->a * p->NB + (uint64_t)(p->W - p->a) * (p->NB >> 1);
  p->segments = p->buckets >> p->lgL;
  const uint64_t a256 = 256;
  auto up = [&](uint64_t v) { return (v + a256 - 1) / a256 * a256; };
  p->off_counts = 0;  // bucket sizes (buckets + 1 words), then the histogram of the sizes (1024 words): one memset
  p->off_offsets = up((p->buckets + 1 + 1024) * 4);
  p->off_cursor = p->off_offsets + up((p->buckets + 1) * 4);
  p->off_entries = p->off_cursor + up((p->buckets + 1) * 4);
  p->off_buckets = p->off_entries + up((n ? n : 1) * (uint64_t)p->W * 4);
  p->off_segments = p->off_buckets + up(p->buckets * jac_bytes);
  p->off_wsum = p->off_segments + up(p->segments * jac_bytes);
  p->off_order = p->off_wsum + up((uint64_t)p->W * jac_bytes);
  p->scratch_bytes = p->off_order + up(p->buckets * 4);
}
void msm_g1_plan(uint64_t n, MsmPlan* p) { msm_plan(n, 144, p); }
void msm_g2_plan(uint64_t n, MsmPlan* p) { msm_plan(n, 288, p); }

// steps 1-7 of either group; d_out: the result record (26 / 50 words) followed by the "scalar >= r" word
template <bool G2>
static cudaError_t launch_msm(const void* d_pts, const void* d_scalars, uint64_t n, void* d_scratch, void* d_out,
                              int* launches, cudaStream_t stream) {
  MsmPlan p;
  msm_plan(n, G2 ? 288 : 144, &p);
  MsmGeom g;
  g.c = p.c;
  g.W = p.W;
  g.a = p.a;
  g.lgL = p.lgL;
  g.NB = p.NB;
  uint8_t* base = (uint8_t*)d_scratch;
  uint32_t* counts = (uint32_t*)(base + p.off_counts);
  uint32_t* offsets = (uint32_t*)(base + p.off_offsets);
  uint32_t* cursor = (uint32_t*)(base + p.off_cursor);
  uint32_t* entries = (uint32_t*)(base + p.off_entries);
  uint32_t* buckets = (uint32_t*)(base + p.off_buckets);
  uint32_t* segs = (uint32_t*)(base + p.off_segments);
  uint32_t* wsum = (uint32_t*)(base + p.off_wsum);
  uint32_t* order = (uint32_t*)(base + p.off_order);
  const uint32_t m = (uint32_t)p.buckets;
  uint32_t* size_hist = counts + m + 1;
  const uint32_t* pts = (const uint32_t*)d_pts;
  const uint32_t* sc = (const uint32_t*)d_scalars;
  cudaError_t e = cudaMemsetAsync(counts, 0, (size_t)(m + 1 + PTAU_MSM_BINS) * 4, stream);
  if (e != cudaSuccess) return e;
  uint32_t* bad = (uint32_t*)d_out + (G2 ? 50 : 26);
  e = cudaMemsetAsync(bad, 0, 4, stream);
  if (e != cudaSuccess) return e;
  const unsigned gn = (unsigned)((n + 255) / 256);
  int nl = 0;
  if (gn) {
    if (G2)
      msm_g2_digits<false><<<gn, 256, 0, stream>>>(pts, sc, n, g, counts, nullptr, bad);
    else
      msm_digits<false><<<gn, 256, 0, stream>>>(pts, sc, n, g, counts, nullptr, bad);
    nl++;
  }
  msm_scan<<<1, 1024, 0, stream>>>(counts, m, offsets, cursor);
  if (gn) {
    if (G2)
      msm_g2_digits<true><<<gn, 256, 0, stream>>>(pts, sc, n, g, cursor, entries, nullptr);
    else
      msm_digits<true><<<gn, 256, 0, stream>>>(pts, sc, n, g, cursor, entries, nullptr);
    nl++;
  }
  const unsigned gs = (m + PTAU_MSM_BINS - 1) / PTAU_MSM_BINS;
  msm_size_hist<<<gs, PTAU_MSM_BINS, 0, stream>>>(counts, m, size_hist);
  msm_size_scan<<<1, PTAU_MSM_BINS, 0, stream>>>(size_hist);
  msm_size_scatter<<<gs, PTAU_MSM_BINS, 0, stream>>>(counts, m, size_hist, order);
  nl += 3;
  const uint32_t nseg = (uint32_t)p.segments;
  if (G2) {
    e = launch_msm_g2_sums(pts, entries, offsets, order, m, buckets, g, nseg, segs, wsum, (uint32_t*)d_out, stream);
    if (e != cudaSuccess) return e;
  } else {
    msm_bucket_sum<<<(m + PTAU_BLOCK - 1) / PTAU_BLOCK, PTAU_BLOCK, 0, stream>>>(pts, entries, offsets, order, m, buckets);
    msm_window_segments<<<(nseg + PTAU_BLOCK - 1) / PTAU_BLOCK, PTAU_BLOCK, 0, stream>>>(buckets, g, nseg, segs);
    msm_window_sum<<<p.W, PTAU_BLOCK, 0, stream>>>(segs, g, wsum);
    msm_finish<<<1, 32, 0, stream>>>(wsum, p.W, (uint32_t*)d_out);
  }
  nl += 5;
  if (launches) *launches = nl;
  return cudaGetLastError();
}
cudaError_t launch_msm_g1(const void* d_pts, const void* d_scalars, uint64_t n, void* d_scratch, void* d_out,
                          int* launches, cudaStream_t stream) {
  return launch_msm<false>(d_pts, d_scalars, n, d_scratch, d_out, launches, stream);
}
cudaError_t launch_msm_g2(const void* d_pts, const void* d_scalars, uint64_t n, void* d_scratch, void* d_out,
                          int* launches, cudaStream_t stream) {
  return launch_msm<true>(d_pts, d_scalars, n, d_scratch, d_out, launches, stream);
}

// =============================================================================
// self-test hook: raw field operations on caller-supplied Montgomery limbs, so that the
// PTX carry chains themselves (not only their host emulation) can be checked against big
// integers on carry-propagation stress patterns.  op: 0 mul, 1 add, 2 sub, 3 neg, 4 sqr,
// 5 a^((p-3)/4), 6 inverse
// =============================================================================
__global__ void fq_op_kernel(int op, const Fq* __restrict__ a, const Fq* __restrict__ b, Fq* __restrict__ out, uint64_t n) {
  uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  Fq x = a[i], y = b[i], r;
  switch (op) {
    case 0: r = fq_mul(x, y); break;
    case 1: r = fq_add(x, y); break;
    case 2: r = fq_sub(x, y); break;
    case 3: r = fq_neg(x); break;
    case 4: r = fq_sqr(x); break;
    case 5: r = fq_pow_p34(x); break;
    case 6: r = fq_inv(x); break;
    default: r = fq_zero();
  }
  out[i] = r;
}
cudaError_t launch_fq_op(int op, const void* d_a, const void* d_b, void* d_out, uint64_t n, cudaStream_t stream) {
  if (n == 0) return cudaSuccess;
  fq_op_kernel<<<(unsigned)((n + 127) / 128), 128, 0, stream>>>(op, (const Fq*)d_a, (const Fq*)d_b, (Fq*)d_out, n);
  return cudaGetLastError();
}

// =============================================================================
// microbenchmarks: the measured denominators of the IMAD roofline
// =============================================================================
// kind 0: 32-bit IMAD, 8 independent dependent-chains per thread
__global__ void __launch_bounds__(256) mb_imad(uint32_t* out, int iters, uint32_t seed) {
  uint32_t a0 = seed + threadIdx.x, a1 = a0 * 3, a2 = a0 * 5, a3 = a0 * 7, a4 = a0 * 11, a5 = a0 * 13, a6 = a0 * 17,
           a7 = a0 * 19;
  uint32_t m = seed | 1u;
#pragma unroll 1
  for (int i = 0; i < iters; i++) {
#pragma unroll
    for (int u = 0; u < 8; u++) {
      asm volatile(
          "mad.lo.u32 %0, %0, %8, %0;\n\tmad.lo.u32 %1, %1, %8, %1;\n\t"
          "mad.lo.u32 %2, %2, %8, %2;\n\tmad.lo.u32 %3, %3, %8, %3;\n\t"
          "mad.lo.u32 %4, %4, %8, %4;\n\tmad.lo.u32 %5, %5, %8, %5;\n\t"
          "mad.lo.u32 %6, %6, %8, %6;\n\tmad.lo.u32 %7, %7, %8, %7;"
          : "+r"(a0), "+r"(a1), "+r"(a2), "+r"(a3), "+r"(a4), "+r"(a5), "+r"(a6), "+r"(a7)
          : "r"(m));
    }
  }
  out[blockIdx.x * blockDim.x + threadIdx.x] = a0 ^ a1 ^ a2 ^ a3 ^ a4 ^ a5 ^ a6 ^ a7;
}

// kind 1: IMAD.WIDE.U32 carry chains shaped like one multiplier row pair:
// two independent chains of 6 wide MADs (12 wide MADs per inner step)
__global__ void __launch_bounds__(256) mb_imad_wide(uint32_t* out, int iters, uint32_t seed) {
  uint32_t E[12], X[12], a[12];
#pragma unroll
  for (int i = 0; i < 12; i++) {
    E[i] = seed + i + threadIdx.x;
    X[i] = seed * 3 + i + threadIdx.x;
    a[i] = seed * 7 + i * 5 + threadIdx.x;
  }
  uint32_t bi = seed | 1u;
#pragma unroll 1
  for (int i = 0; i < iters; i++) {
#pragma unroll
    for (int u = 0; u < 8; u++) {
      row_mac_even(E, X[11], a, bi);
      row_mac_even(X, E[11], a + 1 - 1, bi + u);
    }
  }
  uint32_t r = 0;
#pragma unroll
  for (int i = 0; i < 12; i++) r ^= E[i] ^ X[i];
  out[blockIdx.x * blockDim.x + threadIdx.x] = r;
}

// kind 2: dependent Fq Montgomery multiplications through the product's own
// (non-inlined) fq_mul
__global__ void __launch_bounds__(256) mb_fqmul(uint32_t* out, int iters, uint32_t seed) {
  Fq x = fq_one(), y = k_beta_mont();
  x.l[0] ^= (seed + threadIdx.x) & 0xffu;
#pragma unroll 1
  for (int i = 0; i < iters; i++) {
    x = fq_mul(x, y);
    y = fq_mul(y, x);
  }
  uint32_t r = 0;
#pragma unroll
  for (int i = 0; i < 12; i++) r ^= x.l[i] ^ y.l[i];
  out[blockIdx.x * blockDim.x + threadIdx.x] = r;
}

// kind 5: IMAD.WIDE.U32 with no carry in or out: eight dependent chains acc = lo(acc) * hi(acc) (pure
// 32x32->64 products; every product is distinct, so ptxas cannot hoist it and replace the MAD by a
// multiply plus ALU adds, which is what it does to a loop-invariant `mad.wide`).  Measured: 9.25 T/s,
// the same half rate as the carry-chained form: a 64-bit result costs two IMAD slots, carry or not.
__global__ void __launch_bounds__(256) mb_imad_wide_plain(uint32_t* out, int iters, uint32_t seed) {
  unsigned long long c[8];
#pragma unroll
  for (int i = 0; i < 8; i++) c[i] = ((unsigned long long)(seed * (2 * i + 3) + threadIdx.x) << 32) | (seed + i * 7 + threadIdx.x) | 1ull;
#pragma unroll 1
  for (int i = 0; i < iters; i++) {
#pragma unroll
    for (int u = 0; u < 8; u++) {
#pragma unroll
      for (int k = 0; k < 8; k++)
        asm volatile("{.reg .u32 l, h;\n\tmov.b64 {l, h}, %0;\n\tmul.wide.u32 %0, l, h;}" : "+l"(c[k]));
    }
  }
  unsigned long long r = c[0] ^ c[1] ^ c[2] ^ c[3] ^ c[4] ^ c[5] ^ c[6] ^ c[7];
  out[blockIdx.x * blockDim.x + threadIdx.x] = (uint32_t)r ^ (uint32_t)(r >> 32);
}

// kind 6: DFMA, eight independent chains (the FP64 pipe: 17.9 T/s = 64 /clk/SM on B200).
// kind 7: the same block runs DFMA chains in its odd warps and IMAD.WIDE.X rows in its even warps.  Measured:
// the two rates add up to one pipe's worth (DFMA and IMAD share the FMA-heavy datapath), which is why an
// FP64 (48-bit limb) field multiplier run beside the integer one buys nothing (DESIGN.md).
template <bool MIXED>
__global__ void __launch_bounds__(256) mb_dfma(uint32_t* out, int iters, uint32_t seed) {
  uint32_t r = 0;
  if (MIXED && ((threadIdx.x >> 5) & 1) == 0) {
    uint32_t E[12], X[12], a[12];
#pragma unroll
    for (int i = 0; i < 12; i++) {
      E[i] = seed + i + threadIdx.x;
      X[i] = seed * 3 + i + threadIdx.x;
      a[i] = seed * 7 + i * 5 + threadIdx.x;
    }
    uint32_t bi = seed | 1u;
#pragma unroll 1
    for (int i = 0; i < iters; i++) {
#pragma unroll
      for (int u = 0; u < 8; u++) {
        row_mac_even(E, X[11], a, bi);
        row_mac_even(X, E[11], a, bi + u);
      }
    }
#pragma unroll
    for (int i = 0; i < 12; i++) r ^= E[i] ^ X[i];
  } else {
    double d[8];
#pragma unroll
    for (int i = 0; i < 8; i++) d[i] = 1.0 + (double)(threadIdx.x + i) * 1e-3;
    const double m = 1.0000001, c = 1e-9;
#pragma unroll 1
    for (int i = 0; i < iters; i++) {
#pragma unroll
      for (int u = 0; u < 12; u++) {
#pragma unroll
        for (int k = 0; k < 8; k++) d[k] = __fma_rz(d[k], m, c);
      }
    }
    double s = d[0] + d[1] + d[2] + d[3] + d[4] + d[5] + d[6] + d[7];
    r = (uint32_t)__double2hiint(s) ^ (uint32_t)__double2loint(s);
  }
  out[blockIdx.x * blockDim.x + threadIdx.x] = r;
}

// kind 3 / 4: the G1 doubling loop of the subgroup ladders, with the product's non-inlined
// fq_mul/fq_sqr (3) and with everything inlined (4): bounds the cost of the call ABI
template <bool INL>
__device__ __forceinline__ void mb_dbl_step(Jac<Fq>& p) {
  auto MUL = [](const Fq& a, const Fq& b) { return INL ? fq_mul_inl(a, b) : fq_mul(a, b); };
  auto SQR = [](const Fq& a) { return INL ? fq_sqr_inl(a) : fq_sqr(a); };
  Fq B = SQR(p.Y);
  p.Z = fq_dbl(MUL(p.Z, p.Y));
  Fq C = SQR(B);
  Fq t = fq_add(p.X, B);
  Fq A = SQR(p.X);
  Fq D = SQR(t);
  D = fq_sub(fq_sub(D, A), C);
  D = fq_dbl(D);
  Fq E = fq_add(fq_dbl(A), A);
  Fq Fv = SQR(E);
  p.X = fq_sub(Fv, fq_dbl(D));
  C = fq_dbl(fq_dbl(fq_dbl(C)));
  p.Y = fq_sub(MUL(fq_sub(D, p.X), E), C);
}
#ifndef PTAU_MB_MINB
#define PTAU_MB_MINB 3
#endif
template <bool INL>
__global__ void __launch_bounds__(128, PTAU_MB_MINB) mb_dbl(uint32_t* out, int iters, uint32_t seed) {
  Jac<Fq> p;
  p.X = k_g1x_mont();
  p.Y = k_g1y_mont();
  p.Z = fq_one();
  p.X.l[0] ^= (seed + threadIdx.x) & 0xffu;
#pragma unroll 1
  for (int i = 0; i < iters; i++) mb_dbl_step<INL>(p);
  uint32_t r = 0;
#pragma unroll
  for (int i = 0; i < 12; i++) r ^= p.X.l[i] ^ p.Y.l[i] ^ p.Z.l[i];
  out[blockIdx.x * blockDim.x + threadIdx.x] = r;
}

cudaError_t launch_microbench(int kind, int iters, uint32_t* d_out, int grid, int block, double* ops,
                              cudaStream_t stream) {
  double threads = (double)grid * block;
  switch (kind) {
    case 0:
      mb_imad<<<grid, block, 0, stream>>>(d_out, iters, 12345u);
      *ops = threads * iters * 64.0;
      break;
    case 1:
      mb_imad_wide<<<grid, block, 0, stream>>>(d_out, iters, 12345u);
      *ops = threads * iters * 8.0 * 12.0;
      break;
    case 2:
      mb_fqmul<<<grid, block, 0, stream>>>(d_out, iters, 12345u);
      *ops = threads * iters * 2.0;
      break;
    case 5:
      mb_imad_wide_plain<<<grid, block, 0, stream>>>(d_out, iters, 12345u);
      *ops = threads * iters * 64.0;
      break;
    case 6:
      mb_dfma<false><<<grid, block, 0, stream>>>(d_out, iters, 12345u);
      *ops = threads * iters * 96.0;
      break;
    case 7:  // ops = slots of the shared pipe: 96 DFMA per odd-warp thread, 96 wide MADs (2 slots each) per even-warp thread
      mb_dfma<true><<<grid, block, 0, stream>>>(d_out, iters, 12345u);
      *ops = threads * 0.5 * iters * 96.0 + threads * 0.5 * iters * 96.0 * 2.0;
      break;
    case 3:
      mb_dbl<false><<<grid * PTAU_MB_MINB, 128, 0, stream>>>(d_out, iters, 12345u);
      *ops = (double)grid * PTAU_MB_MINB * 128 * iters;
      break;
    case 4:
      mb_dbl<true><<<grid * PTAU_MB_MINB, 128, 0, stream>>>(d_out, iters, 12345u);
      *ops = (double)grid * PTAU_MB_MINB * 128 * iters;
      break;
    default:
      return cudaErrorInvalidValue;
  }
  return cudaGetLastError();
}

}  // namespace ptau
