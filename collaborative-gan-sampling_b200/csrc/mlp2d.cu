// 2-D synthetic path: discriminator MLP forward + saliency (synthetic/GAN.py:28-37,108-111) and the whole
// K-step data-space refinement of sampling/refiner_cpu.py:19-81 fused into ONE kernel launch.
//
// One thread owns one point for all K steps: ladam state, best-so-far and the point itself live in registers,
// the MLP weights (66 KB FP32 at nhidden=64, nlayers=6) live in shared memory and are read as warp-broadcast
// LDS.128, activations are staged per thread in a conflict-free smem column.  FP32 FMA throughout (the reference's
// TF/Eigen path is FP32); nothing but x in / x out touches HBM.
#include "common.h"
#include "policy.cuh"

namespace cgs {
namespace {

constexpr int H = 64;                 // nhidden of these kernels; every other width runs the cluster form (mlp2d_cluster.cu)
constexpr int kMlpThreads = 128;

struct MlpSmem {
  // layout (floats): w0 [2][H] | b0 [H] | hidden l: w [H][H], b [H] | w_last [H] | b_last | act [H][threads]
  float* w0; float* b0; float* wh; float* bh; float* wl; float bl; float* act;
};

__device__ __forceinline__ size_t mlp_weight_floats(int nlayers) {
  return 2 * H + H + (size_t)(nlayers - 2) * (H * H + H) + H + 4;
}

__device__ void mlp_load_weights(const cgs_mlp_desc& d, float* smem, MlpSmem& s) {
  const int nh = d.nlayers - 2;
  s.w0 = smem;
  s.b0 = s.w0 + 2 * H;
  s.wh = s.b0 + H;
  s.bh = s.wh + (size_t)nh * H * H;
  s.wl = s.bh + (size_t)nh * H;
  s.act = s.wl + H + 4;
  for (int i = threadIdx.x; i < 2 * H; i += blockDim.x) s.w0[i] = d.weights[0][i];
  for (int i = threadIdx.x; i < H; i += blockDim.x) s.b0[i] = d.biases[0][i];
  for (int l = 0; l < nh; ++l) {
    const float* w = d.weights[1 + l];
    const float* b = d.biases[1 + l];
    for (int i = threadIdx.x; i < H * H; i += blockDim.x) s.wh[(size_t)l * H * H + i] = w[i];
    for (int i = threadIdx.x; i < H; i += blockDim.x) s.bh[l * H + i] = b[i];
  }
  for (int i = threadIdx.x; i < H; i += blockDim.x) s.wl[i] = d.weights[d.nlayers - 1][i];
  s.bl = d.biases[d.nlayers - 1][0];
  __syncthreads();
}

// Forward + backward through the MLP for one point.  Returns the logit; (gx, gy) = d logit / d (x, y).
// mask bits of each ReLU are kept in registers (2 words per layer).
template <bool kGrad>
__device__ __forceinline__ float mlp_point(const MlpSmem& s, int nlayers, float x, float y, float& gx, float& gy) {
  const int nh = nlayers - 2;
  const int tid = threadIdx.x;
  const int stride = blockDim.x;
  float* col = s.act + tid;                          // element k of this thread's vector: col[k*stride]
  unsigned int mask[CGS_MLP_MAX_LAYERS][2];
  float out[H];
  // layer 0: 2 -> H                                   synthetic/GAN.py:30-31
#pragma unroll
  for (int u = 0; u < H; ++u) out[u] = fmaf(y, s.w0[H + u], fmaf(x, s.w0[u], s.b0[u]));
  {
    unsigned int m0 = 0, m1 = 0;
#pragma unroll
    for (int u = 0; u < H; ++u) {
      const bool on = out[u] > 0.f;
      if (u < 32) m0 |= (on ? 1u : 0u) << u; else m1 |= (on ? 1u : 0u) << (u - 32);
      col[u * stride] = on ? out[u] : 0.f;
    }
    mask[0][0] = m0; mask[0][1] = m1;
  }
  // hidden layers: H -> H                              synthetic/GAN.py:32-34
  for (int l = 0; l < nh; ++l) {
    const float* w = s.wh + (size_t)l * H * H;
    const float* b = s.bh + l * H;
#pragma unroll
    for (int u = 0; u < H; ++u) out[u] = b[u];
#pragma unroll 2
    for (int k = 0; k < H; ++k) {
      const float a = col[k * stride];
      const float4* wr = reinterpret_cast<const float4*>(w + k * H);
#pragma unroll
      for (int u4 = 0; u4 < H / 4; ++u4) {
        const float4 ww = wr[u4];
        out[4 * u4 + 0] = fmaf(a, ww.x, out[4 * u4 + 0]);
        out[4 * u4 + 1] = fmaf(a, ww.y, out[4 * u4 + 1]);
        out[4 * u4 + 2] = fmaf(a, ww.z, out[4 * u4 + 2]);
        out[4 * u4 + 3] = fmaf(a, ww.w, out[4 * u4 + 3]);
      }
    }
    unsigned int m0 = 0, m1 = 0;
#pragma unroll
    for (int u = 0; u < H; ++u) {
      const bool on = out[u] > 0.f;
      if (u < 32) m0 |= (on ? 1u : 0u) << u; else m1 |= (on ? 1u : 0u) << (u - 32);
      col[u * stride] = on ? out[u] : 0.f;
    }
    mask[l + 1][0] = m0; mask[l + 1][1] = m1;
  }
  // last layer: H -> 1                                 synthetic/GAN.py:35
  float logit = s.bl;
#pragma unroll 8
  for (int k = 0; k < H; ++k) logit = fmaf(col[k * stride], s.wl[k], logit);
  if (!kGrad) return logit;

  // backward: g = d logit / d activation, masked by each ReLU
#pragma unroll
  for (int u = 0; u < H; ++u) {
    const unsigned int bit = u < 32 ? (mask[nh][0] >> u) & 1u : (mask[nh][1] >> (u - 32)) & 1u;
    out[u] = bit ? s.wl[u] : 0.f;
  }
  for (int l = nh - 1; l >= 0; --l) {
    const float* w = s.wh + (size_t)l * H * H;
    // g_in[k] = sum_u w[k][u] * g_out[u], then mask of the layer below
    const unsigned int m0 = mask[l][0], m1 = mask[l][1];
#pragma unroll 2
    for (int k = 0; k < H; ++k) {
      const float4* wr = reinterpret_cast<const float4*>(w + k * H);
      float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
#pragma unroll
      for (int u4 = 0; u4 < H / 4; ++u4) {
        const float4 ww = wr[u4];
        a0 = fmaf(ww.x, out[4 * u4 + 0], a0);
        a1 = fmaf(ww.y, out[4 * u4 + 1], a1);
        a2 = fmaf(ww.z, out[4 * u4 + 2], a2);
        a3 = fmaf(ww.w, out[4 * u4 + 3], a3);
      }
      const unsigned int bit = k < 32 ? (m0 >> k) & 1u : (m1 >> (k - 32)) & 1u;
      col[k * stride] = bit ? (a0 + a1) + (a2 + a3) : 0.f;
    }
#pragma unroll
    for (int u = 0; u < H; ++u) out[u] = col[u * stride];
  }
  float ax = 0.f, ay = 0.f;
#pragma unroll
  for (int u = 0; u < H; ++u) {
    ax = fmaf(s.w0[u], out[u], ax);
    ay = fmaf(s.w0[H + u], out[u], ay);
  }
  gx = ax;
  gy = ay;
  return logit;
}

__global__ void __launch_bounds__(kMlpThreads, 1)
mlp2d_score_kernel(const cgs_mlp_desc d, const float* __restrict__ x, int64_t n, float inv_n,
                   float* __restrict__ sig_out, float* __restrict__ logit_out, float* __restrict__ sal_out) {
  extern __shared__ float smem[];
  MlpSmem s;
  mlp_load_weights(d, smem, s);
  const int64_t nround = (n + blockDim.x - 1) / blockDim.x * blockDim.x;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < nround; i += (int64_t)gridDim.x * blockDim.x) {
    const bool ok = i < n;
    const float px = ok ? x[2 * i] : 0.f, py = ok ? x[2 * i + 1] : 0.f;
    float gx = 0.f, gy = 0.f;
    float logit;
    if (sal_out) logit = mlp_point<true>(s, d.nlayers, px, py, gx, gy);
    else logit = mlp_point<false>(s, d.nlayers, px, py, gx, gy);
    if (ok) {
      const float sg = sigmoid_f32(logit);
      sig_out[i] = sg;
      if (logit_out) logit_out[i] = logit;
      if (sal_out) {
        // d mean_N softplus(-l) / d x = (sigmoid(l) - 1)/N * dl/dx        (synthetic/GAN.py:109-111)
        const float dl = (sg - 1.f) * inv_n;
        sal_out[2 * i] = dl * gx;
        sal_out[2 * i + 1] = dl * gy;
      }
    }
  }
}

__global__ void __launch_bounds__(kMlpThreads, 1)
mlp2d_refine_kernel(const cgs_mlp_desc d, PolicyConsts pc, int steps, float inv_n, float real_mean,
                    const float* __restrict__ x_in, int64_t n, float* __restrict__ best_x_out,
                    float* __restrict__ best_loss_out, float* __restrict__ best_step_out,
                    float* __restrict__ traj) {
  extern __shared__ float smem[];
  MlpSmem s;
  mlp_load_weights(d, smem, s);
  const int64_t nround = (n + blockDim.x - 1) / blockDim.x * blockDim.x;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < nround; i += (int64_t)gridDim.x * blockDim.x) {
    const bool ok = i < n;
    float px = ok ? x_in[2 * i] : 0.f, py = ok ? x_in[2 * i + 1] : 0.f;
    float gx, gy;
    float logit = mlp_point<true>(s, d.nlayers, px, py, gx, gy);
    float sg = sigmoid_f32(logit);
    float dl = (sg - 1.f) * inv_n;
    gx *= dl; gy *= dl;                                        // fake_saliency
    float loss = __fsub_rn(real_mean, sg);                     // refiner_cpu.py:28
    float bx = px, by = py, bloss = loss, bstep = 0.f;         // refiner_cpu.py:31-33
    float mx = 0.f, my = 0.f, vx = 0.f, vy = 0.f, lavg = 0.f;
    float* tr = traj ? traj + (size_t)i * (steps + 1) * 3 : nullptr;
    if (tr && ok) { tr[0] = px; tr[1] = py; tr[2] = loss; }
    for (int it = 0; it < steps; ++it) {                       // refiner_cpu.py:46-66
      const int first = it == 0;
      if (pc.method == CGS_POLICY_SGD) {
        px = sgd_update(pc, px, gx);
        py = sgd_update(pc, py, gy);
      } else if (pc.method == CGS_POLICY_MOMENTUM) {
        px = momentum_update(pc, px, gx, mx, first);
        py = momentum_update(pc, py, gy, my, first);
      } else {
        lavg = ladam_loss_avg(pc, lavg, loss, first);
        px = ladam_update(pc, px, gx, mx, vx, lavg, first, 0);
        py = ladam_update(pc, py, gy, my, vy, lavg, first, 0);
      }
      logit = mlp_point<true>(s, d.nlayers, px, py, gx, gy);   // refiner_cpu.py:52
      sg = sigmoid_f32(logit);
      dl = (sg - 1.f) * inv_n;
      gx *= dl; gy *= dl;
      loss = __fsub_rn(real_mean, sg);                         // refiner_cpu.py:55
      if (__fsub_rn(bloss, loss) > 0.f) {                      // refiner_cpu.py:58-61
        bloss = loss; bx = px; by = py; bstep = (float)(it + 1);
      }
      if (tr && ok) { tr[3 * (it + 1)] = px; tr[3 * (it + 1) + 1] = py; tr[3 * (it + 1) + 2] = loss; }
    }
    if (ok) {
      best_x_out[2 * i] = bx;
      best_x_out[2 * i + 1] = by;
      best_loss_out[i] = bloss;
      best_step_out[i] = bstep;
    }
  }
}

// ------------------------------------------------------------------------------------------------------------
// Split form of the refinement kernel.  N = 10^4 points are 313 warps: with one thread per point every SM holds two
// warps and the run time is the latency of ONE thread's 561 layer passes.  Here FOUR threads (one per warp of a
// 4-warp group, same lane) share a point: each computes a 16-wide slice of every hidden layer's outputs (forward)
// or input gradients (backward) and the slices are exchanged through a ping-pong activation buffer in shared memory
// with one named barrier per layer.  Weight reads stay warp-broadcast LDS.128.  Every output element is accumulated
// in exactly the order of mlp_point, so the results are bit-identical to the one-thread form; the tiny 2 -> 64 and
// 64 -> 1 layers, the policy state and the best-so-far bookkeeping are computed redundantly by all four threads.
// ------------------------------------------------------------------------------------------------------------
constexpr int kParts = 4;
constexpr int kSlice = H / kParts;   // 16

__device__ __forceinline__ void group_sync(int id) { asm volatile("bar.sync %0, 128;" ::"r"(id) : "memory"); }

struct SplitCtx {
  float* buf[2];      // activation ping-pong, [H][P]
  int cur;            // buffer holding the vector to read next
  int P, pt, part, bar;
};

template <bool kGrad>
__device__ __forceinline__ float mlp_point_split(const MlpSmem& s, int nlayers, float x, float y, float& gx, float& gy,
                                                 SplitCtx& c) {
  const int nh = nlayers - 2;
  const int u0 = c.part * kSlice;
  const int P = c.P;
  unsigned int mask[CGS_MLP_MAX_LAYERS];
  float out[kSlice];
  // layer 0: 2 -> H (own slice)                         synthetic/GAN.py:30-31
  {
    float* W = c.buf[c.cur ^ 1] + c.pt;
    unsigned int m = 0;
#pragma unroll
    for (int u = 0; u < kSlice; ++u) {
      const float v = fmaf(y, s.w0[H + u0 + u], fmaf(x, s.w0[u0 + u], s.b0[u0 + u]));
      const bool on = v > 0.f;
      m |= (on ? 1u : 0u) << u;
      W[(u0 + u) * P] = on ? v : 0.f;
    }
    mask[0] = m;
    group_sync(c.bar);
    c.cur ^= 1;
  }
  // hidden layers: H -> H                                synthetic/GAN.py:32-34
  for (int l = 0; l < nh; ++l) {
    const float* w = s.wh + (size_t)l * H * H + u0;
    const float* b = s.bh + l * H + u0;
    const float* R = c.buf[c.cur] + c.pt;
    float* W = c.buf[c.cur ^ 1] + c.pt;
#pragma unroll
    for (int u = 0; u < kSlice; ++u) out[u] = b[u];
#pragma unroll 4
    for (int k = 0; k < H; ++k) {
      const float a = R[k * P];
      const float4* wr = reinterpret_cast<const float4*>(w + k * H);
#pragma unroll
      for (int u4 = 0; u4 < kSlice / 4; ++u4) {
        const float4 ww = wr[u4];
        out[4 * u4 + 0] = fmaf(a, ww.x, out[4 * u4 + 0]);
        out[4 * u4 + 1] = fmaf(a, ww.y, out[4 * u4 + 1]);
        out[4 * u4 + 2] = fmaf(a, ww.z, out[4 * u4 + 2]);
        out[4 * u4 + 3] = fmaf(a, ww.w, out[4 * u4 + 3]);
      }
    }
    unsigned int m = 0;
#pragma unroll
    for (int u = 0; u < kSlice; ++u) {
      const bool on = out[u] > 0.f;
      m |= (on ? 1u : 0u) << u;
      W[(u0 + u) * P] = on ? out[u] : 0.f;
    }
    mask[l + 1] = m;
    group_sync(c.bar);
    c.cur ^= 1;
  }
  // last layer: H -> 1 (every thread of the group)       synthetic/GAN.py:35
  float logit = s.bl;
  {
    const float* R = c.buf[c.cur] + c.pt;
#pragma unroll 8
    for (int k = 0; k < H; ++k) logit = fmaf(R[k * P], s.wl[k], logit);
  }
  if (!kGrad) return logit;

  // backward: g = d logit / d activation, masked by each ReLU
  {
    float* W = c.buf[c.cur ^ 1] + c.pt;
#pragma unroll
    for (int u = 0; u < kSlice; ++u) W[(u0 + u) * P] = ((mask[nh] >> u) & 1u) ? s.wl[u0 + u] : 0.f;
    group_sync(c.bar);
    c.cur ^= 1;
  }
  for (int l = nh - 1; l >= 0; --l) {
    const float* w = s.wh + (size_t)l * H * H;
    const float* R = c.buf[c.cur] + c.pt;
    float* W = c.buf[c.cur ^ 1] + c.pt;
    float g[H];
#pragma unroll
    for (int u = 0; u < H; ++u) g[u] = R[u * P];
    const unsigned int m = mask[l];
    // g_in[k] = sum_u w[k][u] * g_out[u] for the k of the own slice, then the mask of the layer below
#pragma unroll 2
    for (int kk = 0; kk < kSlice; ++kk) {
      const int k = u0 + kk;
      const float4* wr = reinterpret_cast<const float4*>(w + k * H);
      float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
#pragma unroll
      for (int u4 = 0; u4 < H / 4; ++u4) {
        const float4 ww = wr[u4];
        a0 = fmaf(ww.x, g[4 * u4 + 0], a0);
        a1 = fmaf(ww.y, g[4 * u4 + 1], a1);
        a2 = fmaf(ww.z, g[4 * u4 + 2], a2);
        a3 = fmaf(ww.w, g[4 * u4 + 3], a3);
      }
      W[k * P] = ((m >> kk) & 1u) ? (a0 + a1) + (a2 + a3) : 0.f;
    }
    group_sync(c.bar);
    c.cur ^= 1;
  }
  {
    const float* R = c.buf[c.cur] + c.pt;
    float ax = 0.f, ay = 0.f;
#pragma unroll 8
    for (int u = 0; u < H; ++u) {
      const float gu = R[u * P];
      ax = fmaf(s.w0[u], gu, ax);
      ay = fmaf(s.w0[H + u], gu, ay);
    }
    gx = ax;
    gy = ay;
  }
  return logit;
}

__global__ void __launch_bounds__(384, 1)
mlp2d_refine_split_kernel(const cgs_mlp_desc d, PolicyConsts pc, int steps, float inv_n, float real_mean,
                          const float* __restrict__ x_in, int64_t n, int ppb, int64_t chunks,
                          float* __restrict__ best_x_out, float* __restrict__ best_loss_out,
                          float* __restrict__ best_step_out, float* __restrict__ traj) {
  extern __shared__ float smem[];
  MlpSmem s;
  mlp_load_weights(d, smem, s);
  SplitCtx c;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  c.P = blockDim.x / kParts;                       // point slots of the CTA
  c.part = warp & (kParts - 1);
  c.pt = (warp / kParts) * 32 + lane;
  c.bar = 1 + warp / kParts;                       // named barrier of the 4-warp group (0 is __syncthreads)
  c.buf[0] = s.act;
  c.buf[1] = s.act + (size_t)H * c.P;
  c.cur = 0;
  for (int64_t ch = blockIdx.x; ch < chunks; ch += gridDim.x) {
    const int64_t i = ch * ppb + c.pt;
    const bool ok = c.pt < ppb && i < n;
    const bool writer = ok && c.part == 0;
    float px = ok ? x_in[2 * i] : 0.f, py = ok ? x_in[2 * i + 1] : 0.f;
    float gx, gy;
    float logit = mlp_point_split<true>(s, d.nlayers, px, py, gx, gy, c);
    float sg = sigmoid_f32(logit);
    float dl = (sg - 1.f) * inv_n;
    gx *= dl; gy *= dl;                                        // fake_saliency
    float loss = __fsub_rn(real_mean, sg);                     // refiner_cpu.py:28
    float bx = px, by = py, bloss = loss, bstep = 0.f;         // refiner_cpu.py:31-33
    float mx = 0.f, my = 0.f, vx = 0.f, vy = 0.f, lavg = 0.f;
    float* tr = traj ? traj + (size_t)i * (steps + 1) * 3 : nullptr;
    if (tr && writer) { tr[0] = px; tr[1] = py; tr[2] = loss; }
    for (int it = 0; it < steps; ++it) {                       // refiner_cpu.py:46-66
      const int first = it == 0;
      if (pc.method == CGS_POLICY_SGD) {
        px = sgd_update(pc, px, gx);
        py = sgd_update(pc, py, gy);
      } else if (pc.method == CGS_POLICY_MOMENTUM) {
        px = momentum_update(pc, px, gx, mx, first);
        py = momentum_update(pc, py, gy, my, first);
      } else {
        lavg = ladam_loss_avg(pc, lavg, loss, first);
        px = ladam_update(pc, px, gx, mx, vx, lavg, first, 0);
        py = ladam_update(pc, py, gy, my, vy, lavg, first, 0);
      }
      logit = mlp_point_split<true>(s, d.nlayers, px, py, gx, gy, c);   // refiner_cpu.py:52
      sg = sigmoid_f32(logit);
      dl = (sg - 1.f) * inv_n;
      gx *= dl; gy *= dl;
      loss = __fsub_rn(real_mean, sg);                         // refiner_cpu.py:55
      if (__fsub_rn(bloss, loss) > 0.f) {                      // refiner_cpu.py:58-61
        bloss = loss; bx = px; by = py; bstep = (float)(it + 1);
      }
      if (tr && writer) { tr[3 * (it + 1)] = px; tr[3 * (it + 1) + 1] = py; tr[3 * (it + 1) + 2] = loss; }
    }
    if (writer) {
      best_x_out[2 * i] = bx;
      best_x_out[2 * i + 1] = by;
      best_loss_out[i] = bloss;
      best_step_out[i] = bstep;
    }
  }
}

int check_mlp(const cgs_mlp_desc* d) {
  if (!d) return set_error(CGS_ERR_INVALID, "null mlp descriptor");
  if (d->nhidden < 16 || d->nhidden > 256 || d->nhidden % 16)
    return set_error(CGS_ERR_UNSUPPORTED, "nhidden %d: this build runs the multiples of 16 from 16 to 256", d->nhidden);
  if (d->nlayers < 2 || d->nlayers > CGS_MLP_MAX_LAYERS) return set_error(CGS_ERR_UNSUPPORTED, "nlayers %d (2..8)", d->nlayers);   // synthetic/GAN.py:32 range(nlayers-2)
  for (int l = 0; l < d->nlayers; ++l)
    if (!d->weights[l] || !d->biases[l]) return set_error(CGS_ERR_INVALID, "null weights for layer %d", l);
  return CGS_OK;
}

// nhidden == 64 runs the kernels above; every other width, and 64 under CGS_DEBUG_MLP2D_CLUSTER, the cluster form
bool use_cluster_form(const cgs_mlp_desc& d) { return d.nhidden != H || (debug_flags() & CGS_DEBUG_MLP2D_CLUSTER); }

size_t mlp_smem_bytes(int nlayers, int threads) {
  const size_t wf = 2 * H + H + (size_t)(nlayers - 2) * (H * H + H) + H + 4;
  return (wf + (size_t)H * threads) * sizeof(float);
}

struct LaunchShape { int grid, threads; size_t smem; };
LaunchShape mlp_launch_shape(int nlayers, int64_t n) {
  // small batches: 64-thread CTAs so that 10^4 points still cover every SM
  LaunchShape s;
  s.threads = n >= 148 * 128 * 2 ? 128 : 64;
  int64_t g = (n + s.threads - 1) / s.threads;
  if (g > 148 * 4) g = 148 * 4;
  if (g < 1) g = 1;
  s.grid = (int)g;
  s.smem = mlp_smem_bytes(nlayers, s.threads);
  return s;
}

}  // namespace
}  // namespace cgs

using namespace cgs;

extern "C" int cgs_mlp2d_score(const cgs_mlp_desc* d, const float* x, int64_t n, int64_t n_mean, float* sigmoid_out,
                               float* logit_out, float* saliency_out, cgs_stream_t stream) {
  if (int rc = require_sm100()) return rc;
  if (int rc = check_mlp(d)) return rc;
  if (n < 0) return set_error(CGS_ERR_INVALID, "negative n");
  if (n == 0) return CGS_OK;
  if (!x || !sigmoid_out) return set_error(CGS_ERR_INVALID, "null argument");
  if (n_mean <= 0) n_mean = n;
  if (use_cluster_form(*d))
    return mlp2d_cluster_score(*d, x, n, 1.0f / (float)n_mean, sigmoid_out, logit_out, saliency_out, (cudaStream_t)stream);
  const LaunchShape s = mlp_launch_shape(d->nlayers, n);
  cudaError_t e = cudaFuncSetAttribute(mlp2d_score_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)s.smem);
  if (e != cudaSuccess) return set_error(CGS_ERR_CUDA, "cudaFuncSetAttribute: %s", cudaGetErrorString(e));
  mlp2d_score_kernel<<<s.grid, s.threads, s.smem, (cudaStream_t)stream>>>(*d, x, n, 1.0f / (float)n_mean, sigmoid_out,
                                                                         logit_out, saliency_out); count_launch();
  return check_launch("cgs_mlp2d_score");
}

extern "C" int cgs_refine_mlp2d(const cgs_mlp_desc* d, const cgs_refine2d_cfg* cfg, const float* x_in, int64_t n,
                                float* best_x, float* best_loss, float* best_step, float* traj_out,
                                cgs_stream_t stream) {
  if (int rc = require_sm100()) return rc;
  if (int rc = check_mlp(d)) return rc;
  if (!cfg) return set_error(CGS_ERR_INVALID, "null config");
  if (n < 0 || cfg->steps < 0) return set_error(CGS_ERR_INVALID, "negative n / steps");
  if (cfg->policy.method < CGS_POLICY_SGD || cfg->policy.method > CGS_POLICY_LADAM)
    return set_error(CGS_ERR_UNSUPPORTED, "unknown policy method %d (sampling/policy.py:64)", cfg->policy.method);
  if (cfg->policy.method == CGS_POLICY_LADAM && cfg->policy.degree != 2)
    return set_error(CGS_ERR_UNSUPPORTED, "ladam degree %d (only 2)", cfg->policy.degree);
  if (n == 0) return CGS_OK;
  if (!x_in || !best_x || !best_loss || !best_step) return set_error(CGS_ERR_INVALID, "null argument");
  const int64_t n_mean = cfg->n_mean > 0 ? cfg->n_mean : n;
  if (use_cluster_form(*d))
    return mlp2d_cluster_refine(*d, *cfg, 1.0f / (float)n_mean, x_in, n, best_x, best_loss, best_step, traj_out,
                                (cudaStream_t)stream);
  if (!(debug_flags() & CGS_DEBUG_MLP2D_ONE_THREAD)) {
    // split form: four threads per point; the points are dealt evenly over the SMs (at most 96 per CTA round)
    const int sms = device_num_sms();
    int64_t ppb64 = (n + sms - 1) / sms;
    const int ppb = (int)(ppb64 < 1 ? 1 : (ppb64 > 96 ? 96 : ppb64));
    const int pw = (ppb + 31) / 32;
    const int threads = pw * 32 * kParts;
    const int64_t chunks = (n + ppb - 1) / ppb;
    const int grid = (int)(chunks < sms ? chunks : sms);
    const size_t smem = (2 * H + H + (size_t)(d->nlayers - 2) * (H * H + H) + H + 4 + (size_t)2 * H * (pw * 32)) * sizeof(float);
    static DynSmemCache cache;
    cudaError_t e2 = ensure_dyn_smem(mlp2d_refine_split_kernel, smem, cache);
    if (e2 != cudaSuccess) return set_error(CGS_ERR_CUDA, "cudaFuncSetAttribute: %s", cudaGetErrorString(e2));
    mlp2d_refine_split_kernel<<<grid, threads, smem, (cudaStream_t)stream>>>(
        *d, make_policy_consts(cfg->policy), cfg->steps, 1.0f / (float)n_mean, cfg->real_sigmoid_mean, x_in, n, ppb, chunks,
        best_x, best_loss, best_step, traj_out); count_launch();
    return check_launch("cgs_refine_mlp2d");
  }
  const LaunchShape s = mlp_launch_shape(d->nlayers, n);
  cudaError_t e = cudaFuncSetAttribute(mlp2d_refine_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)s.smem);
  if (e != cudaSuccess) return set_error(CGS_ERR_CUDA, "cudaFuncSetAttribute: %s", cudaGetErrorString(e));
  mlp2d_refine_kernel<<<s.grid, s.threads, s.smem, (cudaStream_t)stream>>>(
      *d, make_policy_consts(cfg->policy), cfg->steps, 1.0f / (float)n_mean, cfg->real_sigmoid_mean, x_in, n, best_x,
      best_loss, best_step, traj_out); count_launch();
  return check_launch("cgs_refine_mlp2d");
}
