// The tail shared by the kernels that compute a batch of points per thread and write zcash records: Jacobian ->
// affine with one field inversion per thread (Montgomery's trick), encode, and the block-cooperative store.  Used by
// the synthetic generator (kernels.cu: generate_win_kernel) and the contribution kernel (contribute.cu).
#pragma once
#include "point.cuh"

namespace ptau {

#ifndef PTAU_BLOCK
#define PTAU_BLOCK 128
#endif
#define PTAU_GEN_B 8  // points per thread: thread t of a block owns points t + j * PTAU_BLOCK, j < PTAU_GEN_B

// the scalars s0 * step^i of a batch kernel, formed on the device (8 x u32 Montgomery arithmetic in Fr, fr.cuh)
struct FrParams {
  uint32_t s0[8];         // scalar0, Montgomery form
  uint32_t pw[64][8];     // step^(2^j), Montgomery form
};

// shared -> global, flat (the generators: records written at their natural stride)
template <int BLK>
__device__ __forceinline__ void stage_out_flat(uint32_t* __restrict__ g, const uint32_t* sm, int nwords) {
  int nvec = nwords >> 2;
  uint4* g4 = reinterpret_cast<uint4*>(g);
  const uint4* s4 = reinterpret_cast<const uint4*>(sm);
  for (int i = threadIdx.x; i < nvec; i += BLK) g4[i] = s4[i];
  for (int i = (nvec << 2) + threadIdx.x; i < nwords; i += BLK) g[i] = sm[i];
}

// pts[j]: point blk0 + j * PTAU_BLOCK + tid of the block, Jacobian in Montgomery form with Z != 0; pre[j] = Z_0 ... Z_j.
// Writes the records of the points < n in OUTFMT (ZCASH_COMPRESSED or ZCASH_UNCOMPRESSED) to out + point * WOUT,
// staged through sm (PTAU_BLOCK * WOUT words); tid = threadIdx.x.  Inv::inv(a) = 1 / a in F.
// With INF, bit j of infmask marks point j as the point at infinity: it is written as the zcash infinity record, and
// pts[j] holds any stand-in with Z != 0 so that the shared inversion stays valid.
template <int G, int OUTFMT, class Inv, bool INF = false, class F>
__device__ __forceinline__ void affine_encode_tail(Jac<F> (&pts)[PTAU_GEN_B], F (&pre)[PTAU_GEN_B], uint32_t* sm,
                                                   uint32_t* __restrict__ out, int tid, uint64_t blk0, uint64_t n,
                                                   uint32_t infmask = 0) {
  constexpr int WOUT = record_bytes(G, OUTFMT) / 4;
  F inv = Inv::inv(pre[PTAU_GEN_B - 1]);
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
      if (INF && ((infmask >> j) & 1u)) {
#pragma unroll
        for (int i = 0; i < WOUT; i++) o[i] = 0;
        o[0] = OUTFMT == PTAU_FMT_ZCASH_COMPRESSED ? 0xc0u : 0x40u;  // zcash infinity (compression flag when compressed)
      } else if (G == PTAU_G1) {
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

}  // namespace ptau
