// The context behind the opaque ptau_ctx of the C ABI: per-GPU streams, buffers and events.  capi.cu creates and
// destroys it; verify.cu drives the same GPUs.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <string>

#include "../../include/ptau_b200.h"

namespace ptau {

constexpr int kMaxGpus = 8;
constexpr int kBufs = 2;  // double buffering per GPU

struct GpuSlot {
  int device = -1;
  cudaStream_t stream[kBufs] = {nullptr, nullptr};
  void* d_in[kBufs] = {nullptr, nullptr};
  void* d_out[kBufs] = {nullptr, nullptr};
  size_t cap_in = 0, cap_out = 0;
  unsigned long long* d_status = nullptr;
  cudaEvent_t ev_first = nullptr, ev_last = nullptr;
  cudaEvent_t ev_k0[kBufs] = {nullptr, nullptr}, ev_k1[kBufs] = {nullptr, nullptr};
  uint32_t* d_tbl[2] = {nullptr, nullptr};  // fixed-base tables of the generator (G1, G2), built lazily
  // KZG10::check: fixed-base tables of the verifier key's g, gamma_g, h, rebuilt when the key changes
  void* d_kzg_tbl = nullptr;
  std::string kzg_tbl_key;
  // multi-scalar multiplication: device points / scalars / scratch / result and the pinned staging buffer of the
  // scalars, kept between calls and grown on demand (no cudaMalloc / cudaFree inside a commitment)
  void *d_msm_pts = nullptr, *d_msm_sc = nullptr, *d_msm_scratch = nullptr, *d_msm_out = nullptr, *h_msm_sc = nullptr;
  size_t cap_msm_pts = 0, cap_msm_sc = 0, cap_msm_scratch = 0, cap_h_msm_sc = 0;
  uint32_t* h_msm_out = nullptr;  // pinned: the result record (26 or 50 words) + 1 word "a scalar was >= r"
  // KZG10::open: coefficients, points, chunk sums, values and proofs of one call, kept and grown like the MSM buffers
  void* d_open = nullptr;
  size_t cap_open = 0;
};

}  // namespace ptau

struct ptau_ctx {
  int n_gpus = 0;
  size_t chunk_points = 0;
  ptau::GpuSlot gpu[ptau::kMaxGpus];
  ptau_timing timing;
  std::string last_error;
};
