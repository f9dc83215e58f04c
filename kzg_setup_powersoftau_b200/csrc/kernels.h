// launch wrappers exported by kernels.cu to the C-ABI host layer (capi.cu)
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace ptau {

struct MsmGeom;  // msm_digits.cuh

cudaError_t launch_convert(int group, int in_fmt, int out_fmt, const void* d_in, void* d_out, uint64_t n,
                           uint32_t checks, uint64_t base_index, unsigned long long* d_status,
                           cudaStream_t stream);

// d_scalars: n x 8 u32 little-endian limbs of the scalars (0 < k < r)
cudaError_t launch_generate(int group, int fmt, const uint32_t* d_scalars, void* d_out, uint64_t n,
                            cudaStream_t stream);

// generator v2: scalars formed on the device from s0 (Montgomery Fr) and pw[j] = step^(2^j)
// (Montgomery Fr); d_tbl = 32 x 255 ARK_MONT_LIMBS records of [d * 256^w]G
cudaError_t launch_generate_win(int group, int fmt, const uint32_t* s0_mont, const uint32_t (*pw_mont)[8],
                                const uint32_t* d_tbl, void* d_out, uint64_t first, uint64_t n, cudaStream_t stream);

// sum_i [s_i] P_i over ARK_MONT_LIMBS G1 records and 32-byte LE scalars (< r) by the bucket method;
// msm_g1_plan sizes the device scratch buffer (window width by n); d_out (27 words): one ARK_MONT_LIMBS record and a
// word that is non-zero when some scalar was >= r
struct MsmPlan {
  int c, W, a, lgL;
  uint32_t NB;
  uint64_t buckets, segments;
  uint64_t off_counts, off_offsets, off_cursor, off_entries, off_buckets, off_segments, off_wsum, off_order, scratch_bytes;
};
void msm_g1_plan(uint64_t n, MsmPlan* plan);
cudaError_t launch_msm_g1(const void* d_pts, const void* d_scalars, uint64_t n, void* d_scratch, void* d_out,
                          int* launches, cudaStream_t stream);
// the same over ARK_MONT_LIMBS G2 records (200 B); d_out (51 words): one G2 record and the "scalar >= r" word
void msm_g2_plan(uint64_t n, MsmPlan* plan);
cudaError_t launch_msm_g2(const void* d_pts, const void* d_scalars, uint64_t n, void* d_scratch, void* d_out,
                          int* launches, cudaStream_t stream);
// msm_g2.cu: steps 4-7 of launch_msm_g2 (bucket sums, window segments, window sums, finish)
cudaError_t launch_msm_g2_sums(const uint32_t* pts, const uint32_t* entries, const uint32_t* offsets, const uint32_t* order,
                               uint32_t m, uint32_t* buckets, const MsmGeom& g, uint32_t nseg, uint32_t* segs, uint32_t* wsum,
                               uint32_t* out, cudaStream_t stream);

// kzg.cu: prod_{k<2} e(P_ik, Q_ik) for n items (d_gt: n x 576 bytes or null, d_is_one: n bytes or null), and
// KZG10::check for n openings (d_random_v may be null: no hiding), one item per thread
cudaError_t launch_pairing_product2(const void* d_g1, const void* d_g2, uint64_t n, void* d_gt, void* d_is_one,
                                    cudaStream_t stream);
// d_tbl: kzg_tables_bytes() of fixed-base tables of g, gamma_g, h built by launch_kzg_tables for this key
size_t kzg_tables_bytes();
cudaError_t launch_kzg_tables(const void* d_vk_g1, const void* d_vk_g2, void* d_tbl, cudaStream_t stream);
cudaError_t launch_kzg_check(const void* d_vk_g1, const void* d_vk_g2, const void* d_comms, const void* d_points,
                             const void* d_values, const void* d_proofs, const void* d_random_v, const void* d_tbl,
                             uint64_t n, void* d_ok, cudaStream_t stream);

// kzg_open.cu: the witness polynomial (p - p(z)) / (X - z) of n > 0 canonical 32-byte scalars d_coeffs into d_q (n - 1
// scalars, the layout launch_msm_g1 reads) and p(z) into d_value; zpow[s] = z^(2^s) R mod r for s < kKzgZPowCount; d_sums:
// kzg_quotient_sums_bytes(n) of scratch; *d_bad is set to 1 when a coefficient is >= r.  n == 0: p(z) = 0, no launch.
constexpr int kKzgZPowCount = 32;
size_t kzg_quotient_sums_bytes(uint64_t n);
cudaError_t launch_kzg_quotient(const void* d_coeffs, uint64_t n, const uint32_t (*zpow)[8], void* d_sums, void* d_q,
                                void* d_value, uint32_t* d_bad, int* launches, cudaStream_t stream);

// G2Prepared (ark-ec 0.2): n x 68 x 288 bytes of line coefficients + n infinity bytes
cudaError_t launch_g2_prepare(const void* d_g2, uint64_t n, void* d_coeffs, void* d_infinity, cudaStream_t stream);

cudaError_t launch_fq_op(int op, const void* d_a, const void* d_b, void* d_out, uint64_t n, cudaStream_t stream);

cudaError_t launch_microbench(int kind, int iters, uint32_t* d_out, int grid, int block, double* ops,
                              cudaStream_t stream);

}  // namespace ptau
