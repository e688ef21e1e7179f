// Batch-statistic BatchNorm: the reference refines and scores every sample through D in training mode
// (nsgan/GAN.py:175 `is_training=True`, nsgan/ops.py:19-26): each BN layer of D normalises with the mean and biased
// variance of the batch being refined, and the gradient flows through those statistics.  Over an NHWC [rows, C]:
//   bn_stats_kernel       per-CTA FP64 partial sums of d = y - pivot and d^2 (pivot = row 0: no cancellation)
//   bn_apply_fwd_kernel   out = act(gamma * (y - mean) * rstd + beta)
//   bn_bwd_reduce_kernel  per-CTA FP64 partial sums of dz^ = gamma * dz and dz^ * x^, x^ = (y - mean) * rstd
//   bn_bwd_apply_kernel   dy = rstd * (dz^ - mean(dz^) - x^ * mean(dz^ * x^))
// and bn_merge_kernel, which adds the partial sums of all CTAs in a fixed order.  The CTA count, each CTA's row range and
// every summation order depend on (rows, C) only, so the statistics -- and the bits of everything after them -- do not
// depend on which GEMM lowering produced y.  No atomics.
#include "batchnorm.cuh"
#include "common.h"
#include "ptx.cuh"

namespace cgs {

namespace {

constexpr int kBnQuads = 32;        // threadIdx.x of a reduction CTA: one 4-channel quad each (128 channels per CTA)
constexpr int kBnLanes = 8;         // threadIdx.y: row lanes
constexpr int kBnCtas = 4 * 148;    // CTAs a reduction aims for (four per SM)

struct BnGrid {
  int groups;   // 128-channel column groups (gridDim.y)
  int parts;    // row ranges (gridDim.x)
};

BnGrid bn_grid(long long rows, int C) {
  BnGrid g;
  g.groups = (C / 4 + kBnQuads - 1) / kBnQuads;
  long long parts = (kBnCtas + g.groups - 1) / g.groups;
  const long long cap = (rows + 8 * kBnLanes - 1) / (8 * kBnLanes);   // at least 8 rows per lane
  if (parts > cap) parts = cap;
  g.parts = parts < 1 ? 1 : (int)parts;
  return g;
}

struct BnReduceArgs {
  const float* y;
  const float* dz;      // backward only
  const float* gamma;   // backward only
  const float* stat;    // backward only: mean hi / lo, rstd
  long long rows;
  int C;
  double* part;         // [2][gridDim.x][C]
};

// Partial sums of one CTA: rows [r0, r1) of its 128 channels, lane l taking rows r0 + l, r0 + l + 8, ...; the eight
// lanes are then added in lane order.
template <bool BWD>
__device__ __forceinline__ void bn_partials(const BnReduceArgs& a) {
  __shared__ double red[2][kBnLanes][kBnQuads * 4];
  pdl_launch_dependents();
  pdl_wait();
  const int c = (blockIdx.y * kBnQuads + threadIdx.x) * 4;
  const long long r0 = a.rows * blockIdx.x / gridDim.x, r1 = a.rows * (blockIdx.x + 1) / gridDim.x;
  double s0[4] = {0.0, 0.0, 0.0, 0.0}, s1[4] = {0.0, 0.0, 0.0, 0.0};
  if (c < a.C) {
    float k0[4], k1[4], k2[4], k3[4];
    if (!BWD) {
      const float4 p = __ldg(reinterpret_cast<const float4*>(a.y + c));
      k0[0] = p.x; k0[1] = p.y; k0[2] = p.z; k0[3] = p.w;
    } else {
      const float4 g = __ldg(reinterpret_cast<const float4*>(a.gamma + c));
      const float4 hi = __ldg(reinterpret_cast<const float4*>(a.stat + c));
      const float4 lo = __ldg(reinterpret_cast<const float4*>(a.stat + a.C + c));
      const float4 rs = __ldg(reinterpret_cast<const float4*>(a.stat + 2 * a.C + c));
      k0[0] = g.x; k0[1] = g.y; k0[2] = g.z; k0[3] = g.w;
      k1[0] = hi.x; k1[1] = hi.y; k1[2] = hi.z; k1[3] = hi.w;
      k2[0] = lo.x; k2[1] = lo.y; k2[2] = lo.z; k2[3] = lo.w;
      k3[0] = rs.x; k3[1] = rs.y; k3[2] = rs.z; k3[3] = rs.w;
    }
#pragma unroll 4
    for (long long r = r0 + threadIdx.y; r < r1; r += kBnLanes) {
      const float4 v4 = __ldg(reinterpret_cast<const float4*>(a.y + r * a.C + c));
      const float v[4] = {v4.x, v4.y, v4.z, v4.w};
      if (!BWD) {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const double d = (double)v[j] - (double)k0[j];
          s0[j] += d;
          s1[j] = fma(d, d, s1[j]);
        }
      } else {
        const float4 g4 = __ldg(reinterpret_cast<const float4*>(a.dz + r * a.C + c));
        const float g[4] = {g4.x, g4.y, g4.z, g4.w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const float gh = __fmul_rn(k0[j], g[j]);
          const float xh = __fmul_rn((v[j] - k1[j]) - k2[j], k3[j]);
          s0[j] += (double)gh;
          s1[j] = fma((double)gh, (double)xh, s1[j]);
        }
      }
    }
  }
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    red[0][threadIdx.y][threadIdx.x * 4 + j] = s0[j];
    red[1][threadIdx.y][threadIdx.x * 4 + j] = s1[j];
  }
  __syncthreads();
  const int t = threadIdx.y * kBnQuads + threadIdx.x;          // 256 threads: (sum, channel) pairs
  const int arr = t / (kBnQuads * 4), ch = t % (kBnQuads * 4);
  const int cc = blockIdx.y * kBnQuads * 4 + ch;
  if (cc < a.C) {
    double s = 0.0;
#pragma unroll
    for (int l = 0; l < kBnLanes; ++l) s += red[arr][l][ch];
    a.part[((size_t)arr * gridDim.x + blockIdx.x) * a.C + cc] = s;
  }
}

__global__ void __launch_bounds__(kBnQuads * kBnLanes) bn_stats_kernel(const __grid_constant__ BnReduceArgs a) {
  bn_partials<false>(a);
}

__global__ void __launch_bounds__(kBnQuads * kBnLanes) bn_bwd_reduce_kernel(const __grid_constant__ BnReduceArgs a) {
  bn_partials<true>(a);
}

struct BnMergeArgs {
  const double* part;   // [2][parts][C]
  int parts;
  long long rows;
  int C;
  const float* y;       // forward: the pivot row
  float* stat;
  int bwd;
};

// Per channel: the partial sums of every CTA -> mean (hi + lo) and rstd, or the two backward means.  32 channels per
// CTA; lane l adds the partials of CTAs l, l + 32, ..., then the lanes are added in lane order.
__global__ void __launch_bounds__(1024) bn_merge_kernel(const __grid_constant__ BnMergeArgs a) {
  __shared__ double red[2][32][33];
  pdl_launch_dependents();
  pdl_wait();
  const int c = blockIdx.x * 32 + threadIdx.x;
  double s0 = 0.0, s1 = 0.0;
  if (c < a.C) {
#pragma unroll 4
    for (int p = threadIdx.y; p < a.parts; p += 32) {
      s0 += a.part[(size_t)p * a.C + c];
      s1 += a.part[((size_t)a.parts + p) * a.C + c];
    }
  }
  red[0][threadIdx.y][threadIdx.x] = s0;
  red[1][threadIdx.y][threadIdx.x] = s1;
  __syncthreads();
  if (threadIdx.y != 0 || c >= a.C) return;
  s0 = s1 = 0.0;
  for (int l = 0; l < 32; ++l) {
    s0 += red[0][l][threadIdx.x];
    s1 += red[1][l][threadIdx.x];
  }
  const double n = (double)a.rows;
  if (a.bwd) {
    a.stat[3 * a.C + c] = (float)(s0 / n);
    a.stat[4 * a.C + c] = (float)(s1 / n);
    return;
  }
  const double m = s0 / n;                                   // mean of y - pivot
  double var = s1 / n - m * m;                               // biased variance (tf.nn.moments)
  if (var < 0.0) var = 0.0;
  const double mean = (double)__ldg(a.y + c) + m;
  const float hi = (float)mean;
  a.stat[c] = hi;
  a.stat[a.C + c] = (float)(mean - (double)hi);
  a.stat[2 * a.C + c] = (float)(1.0 / sqrt(var + kBnEps));
}

struct BnApplyArgs {
  const float* y;
  const float* dz;      // backward
  float* out;
  const float* gamma;
  const float* beta;    // forward
  const float* stat;
  long long rows;
  int C;
  Epilogue e;           // forward: activation and TF32 rounding
  int round_out;        // backward
};

// The apply kernels walk the reduction's grid: a thread keeps its four channels' constants in registers and streams
// rows r0 + lane, r0 + lane + 8, ... of its CTA's range (a warp reads 512 contiguous bytes of a row).
__global__ void __launch_bounds__(kBnQuads * kBnLanes) bn_apply_fwd_kernel(const __grid_constant__ BnApplyArgs a) {
  pdl_launch_dependents();
  pdl_wait();
  const int c = (blockIdx.y * kBnQuads + threadIdx.x) * 4;
  if (c >= a.C) return;
  const long long r0 = a.rows * blockIdx.x / gridDim.x, r1 = a.rows * (blockIdx.x + 1) / gridDim.x;
  const float4 zero = make_float4(0.f, 0.f, 0.f, 0.f);
  const float4 g = __ldg(reinterpret_cast<const float4*>(a.gamma + c));
  const float4 b = __ldg(reinterpret_cast<const float4*>(a.beta + c));
  const float4 hi = __ldg(reinterpret_cast<const float4*>(a.stat + c));
  const float4 lo = __ldg(reinterpret_cast<const float4*>(a.stat + a.C + c));
  const float4 rs = __ldg(reinterpret_cast<const float4*>(a.stat + 2 * a.C + c));
#pragma unroll 4
  for (long long r = r0 + threadIdx.y; r < r1; r += kBnLanes) {
    const float4 v = __ldg(reinterpret_cast<const float4*>(a.y + r * a.C + c));
    float4 z;
    z.x = fmaf(g.x, ((v.x - hi.x) - lo.x) * rs.x, b.x);
    z.y = fmaf(g.y, ((v.y - hi.y) - lo.y) * rs.y, b.y);
    z.z = fmaf(g.z, ((v.z - hi.z) - lo.z) * rs.z, b.z);
    z.w = fmaf(g.w, ((v.w - hi.w) - lo.w) * rs.w, b.w);
    *reinterpret_cast<float4*>(a.out + r * a.C + c) = epilogue4_t<EPI_FWD>(a.e, 0, z, zero, zero);
  }
}

__global__ void __launch_bounds__(kBnQuads * kBnLanes) bn_bwd_apply_kernel(const __grid_constant__ BnApplyArgs a) {
  pdl_launch_dependents();
  pdl_wait();
  const int c = (blockIdx.y * kBnQuads + threadIdx.x) * 4;
  if (c >= a.C) return;
  const long long r0 = a.rows * blockIdx.x / gridDim.x, r1 = a.rows * (blockIdx.x + 1) / gridDim.x;
  const float4 g = __ldg(reinterpret_cast<const float4*>(a.gamma + c));
  const float4 hi = __ldg(reinterpret_cast<const float4*>(a.stat + c));
  const float4 lo = __ldg(reinterpret_cast<const float4*>(a.stat + a.C + c));
  const float4 rs = __ldg(reinterpret_cast<const float4*>(a.stat + 2 * a.C + c));
  const float4 m1 = __ldg(reinterpret_cast<const float4*>(a.stat + 3 * a.C + c));
  const float4 m2 = __ldg(reinterpret_cast<const float4*>(a.stat + 4 * a.C + c));
#pragma unroll 4
  for (long long r = r0 + threadIdx.y; r < r1; r += kBnLanes) {
    const float4 v = __ldg(reinterpret_cast<const float4*>(a.y + r * a.C + c));
    const float4 d = *reinterpret_cast<const float4*>(a.dz + r * a.C + c);   // may alias out: no read-only path
    // dz^ and x^ rounded exactly as bn_bwd_reduce_kernel rounded them, so the means subtracted are theirs
    float4 o;
    o.x = rs.x * ((__fmul_rn(g.x, d.x) - m1.x) - __fmul_rn((v.x - hi.x) - lo.x, rs.x) * m2.x);
    o.y = rs.y * ((__fmul_rn(g.y, d.y) - m1.y) - __fmul_rn((v.y - hi.y) - lo.y, rs.y) * m2.y);
    o.z = rs.z * ((__fmul_rn(g.z, d.z) - m1.z) - __fmul_rn((v.z - hi.z) - lo.z, rs.z) * m2.z);
    o.w = rs.w * ((__fmul_rn(g.w, d.w) - m1.w) - __fmul_rn((v.w - hi.w) - lo.w, rs.w) * m2.w);
    if (a.round_out) { o.x = tf32_rn(o.x); o.y = tf32_rn(o.y); o.z = tf32_rn(o.z); o.w = tf32_rn(o.w); }
    *reinterpret_cast<float4*>(a.out + r * a.C + c) = o;
  }
}

template <typename A>
int bn_launch(void (*kernel)(A), const char* name, dim3 grid, dim3 block, cudaStream_t st, const A& args) {
  const cudaError_t e = launch_pdl(kernel, grid, block, (size_t)0, st, args);
  count_launch();
  if (e != cudaSuccess) return set_error(CGS_ERR_CUDA, "%s: %s", name, cudaGetErrorString(e));
  return check_launch(name);
}

int bn_merge(const BnLayer& L, const double* part, int parts, const float* y, int bwd, cudaStream_t st) {
  const BnMergeArgs m{part, parts, L.rows, L.C, y, L.stat, bwd};
  return bn_launch(bn_merge_kernel, "bn_merge_kernel", dim3((unsigned)((L.C + 31) / 32)), dim3(32, 32), st, m);
}

// Batch statistics of y into L.stat (mean hi / lo, rstd).
int bn_stats(const BnLayer& L, const float* y, double* part, cudaStream_t st) {
  const BnGrid g = bn_grid(L.rows, L.C);
  const BnReduceArgs r{y, nullptr, nullptr, nullptr, L.rows, L.C, part};
  if (int rc = bn_launch(bn_stats_kernel, "bn_stats_kernel", dim3((unsigned)g.parts, (unsigned)g.groups),
                         dim3(kBnQuads, kBnLanes), st, r))
    return rc;
  return bn_merge(L, part, g.parts, y, 0, st);
}

}  // namespace

size_t bn_partial_bytes(long long rows, int C) { return 2 * (size_t)bn_grid(rows, C).parts * C * sizeof(double); }

int bn_forward(const BnLayer& L, const float* y, float* out, const Epilogue& e, double* part, cudaStream_t st) {
  if (int rc = bn_stats(L, y, part, st)) return rc;
  const BnGrid g = bn_grid(L.rows, L.C);
  BnApplyArgs a;
  a.y = y; a.dz = nullptr; a.out = out; a.gamma = L.gamma; a.beta = L.beta; a.stat = L.stat;
  a.rows = L.rows; a.C = L.C; a.e = e; a.round_out = 0;
  return bn_launch(bn_apply_fwd_kernel, "bn_apply_fwd_kernel", dim3((unsigned)g.parts, (unsigned)g.groups),
                   dim3(kBnQuads, kBnLanes), st, a);
}

int bn_backward(const BnLayer& L, const float* y, const float* dz, float* dy, int round_out, double* part,
                cudaStream_t st) {
  const BnGrid g = bn_grid(L.rows, L.C);
  const BnReduceArgs r{y, dz, L.gamma, L.stat, L.rows, L.C, part};
  if (int rc = bn_launch(bn_bwd_reduce_kernel, "bn_bwd_reduce_kernel", dim3((unsigned)g.parts, (unsigned)g.groups),
                         dim3(kBnQuads, kBnLanes), st, r))
    return rc;
  if (int rc = bn_merge(L, part, g.parts, nullptr, 1, st)) return rc;
  BnApplyArgs a;
  a.y = y; a.dz = dz; a.out = dy; a.gamma = L.gamma; a.beta = nullptr; a.stat = L.stat;
  a.rows = L.rows; a.C = L.C; a.e = Epilogue(EPI_RAW, ACT_NONE); a.round_out = round_out;
  return bn_launch(bn_bwd_apply_kernel, "bn_bwd_apply_kernel", dim3((unsigned)g.parts, (unsigned)g.groups),
                   dim3(kBnQuads, kBnLanes), st, a);
}

}  // namespace cgs

using namespace cgs;

// ------------------------------------------------------------------------------------------------------------------
// The kernels alone (include/cgs.h): workspace = FP64 partial sums + the [5][C] per-channel state.
// ------------------------------------------------------------------------------------------------------------------
// every kernel moves four channels at a time (float4)
static bool aligned16(const void* p) { return ((uintptr_t)p & 15) == 0; }

static int bn_api_layer(int64_t rows, int C, const float* y, const float* gamma, void* workspace,
                        size_t workspace_bytes, BnLayer& L, double*& part) {
  if (int rc = require_sm100()) return rc;
  if (!y || !gamma) return set_error(CGS_ERR_INVALID, "null argument");
  if (rows <= 0 || C <= 0 || C % 4) return set_error(CGS_ERR_INVALID, "rows %lld / channels %d (a positive multiple of 4)",
                                                     (long long)rows, C);
  if (!aligned16(y) || !aligned16(gamma)) return set_error(CGS_ERR_INVALID, "y / gamma must be 16-byte aligned");
  if (rows * (int64_t)C / 4 >= (1ll << 31)) return set_error(CGS_ERR_UNSUPPORTED, "tensor too large for 32-bit indexing");
  if (!workspace || workspace_bytes < cgs_batchnorm_workspace_bytes(rows, C))
    return set_error(CGS_ERR_WORKSPACE, "workspace too small");
  char* base = (char*)(((uintptr_t)workspace + 255) & ~uintptr_t(255));
  part = (double*)base;
  L.gamma = gamma;
  L.beta = nullptr;
  L.rows = rows;
  L.C = C;
  L.stat = (float*)(base + ((bn_partial_bytes(rows, C) + 255) & ~size_t(255)));
  return CGS_OK;
}

extern "C" size_t cgs_batchnorm_workspace_bytes(int64_t rows, int C) {
  if (rows <= 0 || C <= 0) return 0;
  return ((bn_partial_bytes(rows, C) + 255) & ~size_t(255)) + (size_t)5 * C * sizeof(float) + 256;
}

extern "C" int cgs_batchnorm_forward(int64_t rows, int C, const float* y, const float* gamma, const float* beta, int act,
                                     float* out, float* mean_out, float* rstd_out, void* workspace,
                                     size_t workspace_bytes, cgs_stream_t stream) {
  BnLayer L;
  double* part = nullptr;
  if (int rc = bn_api_layer(rows, C, y, gamma, workspace, workspace_bytes, L, part)) return rc;
  if (!beta || !out) return set_error(CGS_ERR_INVALID, "null argument");
  if (!aligned16(beta) || !aligned16(out)) return set_error(CGS_ERR_INVALID, "beta / out must be 16-byte aligned");
  if (act < CGS_ACT_NONE || act > CGS_ACT_TANH) return set_error(CGS_ERR_INVALID, "unknown activation %d", act);
  L.beta = beta;
  cudaStream_t st = (cudaStream_t)stream;
  if (int rc = bn_forward(L, y, out, Epilogue(EPI_FWD, act), part, st)) return rc;
  if (mean_out) cudaMemcpyAsync(mean_out, L.stat, (size_t)C * 4, cudaMemcpyDeviceToDevice, st);
  if (rstd_out) cudaMemcpyAsync(rstd_out, L.stat + 2 * C, (size_t)C * 4, cudaMemcpyDeviceToDevice, st);
  return check_launch("cgs_batchnorm_forward");
}

extern "C" int cgs_batchnorm_backward(int64_t rows, int C, const float* y, const float* gamma, const float* dz, float* dy,
                                      void* workspace, size_t workspace_bytes, cgs_stream_t stream) {
  BnLayer L;
  double* part = nullptr;
  if (int rc = bn_api_layer(rows, C, y, gamma, workspace, workspace_bytes, L, part)) return rc;
  if (!dz || !dy) return set_error(CGS_ERR_INVALID, "null argument");
  if (!aligned16(dz) || !aligned16(dy)) return set_error(CGS_ERR_INVALID, "dz / dy must be 16-byte aligned");
  cudaStream_t st = (cudaStream_t)stream;
  if (int rc = bn_stats(L, y, part, st)) return rc;
  return bn_backward(L, y, dz, dy, 0, part, st);
}
