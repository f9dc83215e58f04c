// Per-item code of the G2 bucket MSM: msm.cuh's algorithm over Fq2, with the field-generic complete additions of
// pairing.cuh.  Point records are 50 words (ARK_MONT_LIMBS), bucket / segment / window records 72 words (X | Y | Z,
// c0 then c1).  A header of its own, compiled into msm_g2.cu: kernels.cu does not include pairing.cuh, so the G1
// kernels keep exactly their code.  Host- and device-callable like msm.cuh (tests/host_emul).
#pragma once
#include "msm.cuh"
#include "pairing.cuh"

namespace ptau {

PTAU_HD Jac<Fq2> jac2_infinity() {
  Jac<Fq2> a;
  a.X = fq2_zero();
  a.Y = fq2_one();
  a.Z = fq2_zero();
  return a;
}
PTAU_HD void jac2_store(uint32_t* o, const Jac<Fq2>& a) {
#pragma unroll
  for (int w = 0; w < 12; w++) {
    o[w] = a.X.c0.l[w];
    o[12 + w] = a.X.c1.l[w];
    o[24 + w] = a.Y.c0.l[w];
    o[36 + w] = a.Y.c1.l[w];
    o[48 + w] = a.Z.c0.l[w];
    o[60 + w] = a.Z.c1.l[w];
  }
}
PTAU_HD Jac<Fq2> jac2_load(const uint32_t* s) {
  Jac<Fq2> q;
#pragma unroll
  for (int w = 0; w < 12; w++) {
    q.X.c0.l[w] = s[w];
    q.X.c1.l[w] = s[12 + w];
    q.Y.c0.l[w] = s[24 + w];
    q.Y.c1.l[w] = s[36 + w];
    q.Z.c0.l[w] = s[48 + w];
    q.Z.c1.l[w] = s[60 + w];
  }
  return q;
}

PTAU_HD void msm_g2_bucket_item(const uint32_t* pts, const uint32_t* entries, const uint32_t* off, uint32_t b, uint32_t* buckets) {
  Jac<Fq2> acc = jac2_infinity();
  const uint32_t e1 = off[b + 1];
#pragma unroll 1
  for (uint32_t e = off[b]; e < e1; e++) {
    const uint32_t v = entries[e];
    const uint32_t* rec = pts + (uint64_t)(v & 0x7fffffffu) * 50;
    Fq2 x, y;
    x.c0 = msm_load_fq(rec);
    x.c1 = msm_load_fq(rec + 12);
    y.c0 = msm_load_fq(rec + 24);
    y.c1 = msm_load_fq(rec + 36);
    if (v >> 31) y = fq2_neg(y);
    jac_madd_complete_t(acc, x, y, fq2_one());
  }
  jac2_store(buckets + (uint64_t)b * 72, acc);
}

// msm_segment_item over Fq2
PTAU_HD void msm_g2_segment_item(const uint32_t* buckets, const MsmGeom& g, uint32_t t_id, uint32_t* seg) {
  const uint32_t lo_abs = t_id << g.lgL;
  const uint32_t wide = (uint32_t)g.a * g.NB;
  const uint32_t in_window = lo_abs < wide ? lo_abs % g.NB : (lo_abs - wide) % (g.NB >> 1);
  const uint32_t sidx = in_window >> g.lgL;
  const uint32_t* base = buckets + (uint64_t)lo_abs * 72;
  Jac<Fq2> t = jac2_infinity(), sacc = jac2_infinity();
#pragma unroll 1
  for (int j = (1 << g.lgL) - 1; j >= 0; --j) {
    Jac<Fq2> q = jac2_load(base + (uint64_t)j * 72);
    jac_add_complete_t(t, q);
    jac_add_complete_t(sacc, t);
  }
  if (sidx) {  // sacc += [lo] t = [2^lgL] [sidx] t
    Jac<Fq2> m = jac2_infinity();
    int top = 31;
    while (!((sidx >> top) & 1u)) top--;
#pragma unroll 1
    for (int bit = top; bit >= 0; --bit) {
      if (!fq2_is_zero(m.Z)) jac_dbl(m);
      if ((sidx >> bit) & 1u) jac_add_complete_t(m, t);
    }
#pragma unroll 1
    for (int k = 0; k < g.lgL; k++)
      if (!fq2_is_zero(m.Z)) jac_dbl(m);
    jac_add_complete_t(sacc, m);
  }
  jac2_store(seg + (uint64_t)t_id * 72, sacc);
}

// the window's weight 2^bitoff(w) by plain doublings (Z = 0 stays 0 through dbl-2009-l)
PTAU_HD void msm_g2_window_weight(Jac<Fq2>& acc, const MsmGeom& g, int w) {
  const int nd = msm_bitoff(g, w);
  if (fq2_is_zero(acc.Z)) return;
#pragma unroll 1
  for (int k = 0; k < nd; k++) jac_dbl(acc);
}

// sum of the weighted window sums, then one 50-word ARK_MONT_LIMBS record (affine, or ark zero() = (0, 1, infinity))
PTAU_HD void msm_g2_finish_item(const uint32_t* wsum, int W, uint32_t* out) {
  Jac<Fq2> acc = jac2_infinity();
#pragma unroll 1
  for (int w = 0; w < W; w++) {
    Jac<Fq2> q = jac2_load(wsum + (uint64_t)w * 72);
    jac_add_complete_t(acc, q);
  }
  Fq2 x, y;
  if (jac_to_affine_t(acc, x, y)) {
    store_rec(out, x, y, false);
  } else {
    store_rec(out, fq2_zero(), fq2_one(), false);
    out[48] = 1;
  }
}

}  // namespace ptau
