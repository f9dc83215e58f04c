// Steps 4-7 of the bucket MSM (kernels.cu: launch_msm) over G2: the per-item code of msm_g2.cuh in thin kernels.
// Recoding, bucket lists and the size sort are the scalar-only kernels of kernels.cu, shared with G1.
#include "kernels.h"
#include "msm_g2.cuh"

namespace ptau {

#define PTAU_MSM_G2_BLOCK 128

__global__ void __launch_bounds__(PTAU_MSM_G2_BLOCK) msm_g2_bucket_sum(const uint32_t* __restrict__ pts, const uint32_t* __restrict__ entries,
                                                                const uint32_t* __restrict__ off, const uint32_t* __restrict__ order,
                                                                uint32_t m, uint32_t* __restrict__ buckets /* 72 words each */) {
  const uint32_t t = blockIdx.x * PTAU_MSM_G2_BLOCK + threadIdx.x;
  if (t >= m) return;
  msm_g2_bucket_item(pts, entries, off, order[t], buckets);
}
__global__ void __launch_bounds__(PTAU_MSM_G2_BLOCK) msm_g2_window_segments(const uint32_t* __restrict__ buckets, MsmGeom g,
                                                                     uint32_t nseg_total, uint32_t* __restrict__ seg) {
  const uint32_t t_id = blockIdx.x * PTAU_MSM_G2_BLOCK + threadIdx.x;
  if (t_id >= nseg_total) return;
  msm_g2_segment_item(buckets, g, t_id, seg);
}
// 36 KB of shared memory per block: under the 48 KB a launch gets without opting in
__global__ void __launch_bounds__(PTAU_MSM_G2_BLOCK) msm_g2_window_sum(const uint32_t* __restrict__ seg, MsmGeom g,
                                                                uint32_t* __restrict__ wsum /* 72 words per window */) {
  __shared__ uint32_t sm[PTAU_MSM_G2_BLOCK * 72];
  const int w = blockIdx.x;
  const uint32_t first = msm_bucket_base(g, w) >> g.lgL;
  const uint32_t count = (w < g.a ? g.NB : g.NB >> 1) >> g.lgL;
  const uint32_t* base = seg + (uint64_t)first * 72;
  Jac<Fq2> acc = jac2_infinity();
  for (uint32_t i = threadIdx.x; i < count; i += PTAU_MSM_G2_BLOCK) {
    Jac<Fq2> q = jac2_load(base + (uint64_t)i * 72);
    jac_add_complete_t(acc, q);
  }
  for (int stride = PTAU_MSM_G2_BLOCK / 2; stride >= 1; stride >>= 1) {
    jac2_store(sm + threadIdx.x * 72, acc);
    __syncthreads();
    if ((int)threadIdx.x < stride) {
      Jac<Fq2> q = jac2_load(sm + (threadIdx.x + stride) * 72);
      jac_add_complete_t(acc, q);
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    msm_g2_window_weight(acc, g, w);
    jac2_store(wsum + (uint64_t)w * 72, acc);
  }
}
__global__ void msm_g2_finish(const uint32_t* __restrict__ wsum, int W, uint32_t* __restrict__ out) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  msm_g2_finish_item(wsum, W, out);
}

cudaError_t launch_msm_g2_sums(const uint32_t* pts, const uint32_t* entries, const uint32_t* offsets, const uint32_t* order,
                               uint32_t m, uint32_t* buckets, const MsmGeom& g, uint32_t nseg, uint32_t* segs, uint32_t* wsum,
                               uint32_t* out, cudaStream_t stream) {
  msm_g2_bucket_sum<<<(m + PTAU_MSM_G2_BLOCK - 1) / PTAU_MSM_G2_BLOCK, PTAU_MSM_G2_BLOCK, 0, stream>>>(pts, entries, offsets,
                                                                                                       order, m, buckets);
  msm_g2_window_segments<<<(nseg + PTAU_MSM_G2_BLOCK - 1) / PTAU_MSM_G2_BLOCK, PTAU_MSM_G2_BLOCK, 0, stream>>>(buckets, g,
                                                                                                               nseg, segs);
  msm_g2_window_sum<<<g.W, PTAU_MSM_G2_BLOCK, 0, stream>>>(segs, g, wsum);
  msm_g2_finish<<<1, 32, 0, stream>>>(wsum, g.W, out);
  return cudaGetLastError();
}

}  // namespace ptau
