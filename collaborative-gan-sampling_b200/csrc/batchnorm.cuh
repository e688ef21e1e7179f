// Batch-statistic BatchNorm (training mode) over an NHWC activation [rows, C], C a multiple of 4, channel stride C:
// the four streaming kernels of batchnorm.cu and their host launchers.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

#include "conv_gemm.cuh"

namespace cgs {

constexpr double kBnEps = 1e-5;   // nsgan/ops.py:23, the constant cgs/nets.py folds with

// Per-channel state of one batch-BN layer.  stat is [5][C] floats: mean (hi, lo: mean = hi + lo to ~48 bits), rstd,
// and the two backward means, mean(dz^) and mean(dz^ * x^).
struct BnLayer {
  const float* gamma;
  const float* beta;
  long long rows;   // B * H * W (B for an fc layer)
  int C;
  float* stat;
};

// bytes of the FP64 per-CTA partial sums scratch for one [rows, C] reduction (shared by every BN layer of a chain)
size_t bn_partial_bytes(long long rows, int C);

// y -> out = act(gamma * (y - mean) * rstd + beta) through the FWD epilogue `e` (its activation and TF32 rounding);
// the batch statistics are left in L.stat
int bn_forward(const BnLayer& L, const float* y, float* out, const Epilogue& e, double* part, cudaStream_t st);

// dz (gradient w.r.t. the normalised, affine output before the activation) -> dy (w.r.t. y) through the statistics
// of the last bn_forward over the same y; dy may alias dz.  round_out: dy feeds a kind::tf32 MMA.
int bn_backward(const BnLayer& L, const float* y, const float* dz, float* dy, int round_out, double* part,
                cudaStream_t st);

}  // namespace cgs
