// Cluster form of the 2-D MLP kernels (mlp2d.cu): discriminator MLPs of any hidden width nh = 16..256 (multiple of
// 16), e.g. the nh = 256 of the 25-Gaussians recipe (synthetic/run_shaping.sh:9), whose 263 K weights (1 MB FP32) no
// single SM can hold.  This is the split kernel with its 4-warp group replaced by a thread-block cluster of
// C = nh / 16 CTAs: CTA rank r owns units [16 r, 16 r + 16) of every layer and keeps in shared memory
//   - the column slice [nh][16] of every hidden layer (forward outputs of its units),
//   - the row slice [16][nh] of every hidden layer (data-gradient of its units),
//   - the full w0 / b0 (2 -> nh) and w_last / b_last (nh -> 1), and its hidden bias slices,
//   - a ping-pong activation buffer [P][nh + 4] for a round of P points.
// Inside a CTA four threads (lanes 4p .. 4p + 3) share point p, each with 4 of the 16 units.  A layer writes each
// thread's 4 outputs into the next activation buffer of EVERY CTA of the cluster (mapa + st.shared::cluster) and ends
// with one cluster barrier; the ping-pong makes that one barrier enough.  Every element is accumulated in the order of
// mlp_point (mlp2d.cu), so at nh = 64 the results are bit-identical to the one-thread and split kernels.  Layer
// nh -> 1, the input gradient, the policy state and the best-so-far bookkeeping are computed redundantly by every
// thread of a point in every CTA; thread 0 of the point in CTA rank 0 writes the outputs.
//
// Every CTA of a cluster runs the same rounds, layers and barriers (padding points are computed, never stored), and
// the kernel ends with a cluster barrier, so no CTA leaves while a peer may still write into its shared memory.
#include <map>
#include <mutex>
#include <tuple>

#include "common.h"
#include "policy.cuh"
#include "ptx.cuh"

namespace cgs {
namespace {

constexpr int kSlice = 16;                    // units owned by one CTA
constexpr int kSub = 4;                       // threads per point, 4 units each
constexpr int kMaxPoints = 128;               // point slots of a CTA round
constexpr int kPointQuantum = 32 / kSub;      // point slots come in whole warps
constexpr int kMaxThreads = kSub * kMaxPoints;
constexpr size_t kSmemLimit = 227 * 1024;     // dynamic shared memory a CTA may opt in to on sm_100

// Shared-memory plan in floats.  Rows of the row slice and of the activation buffers are nh + 4 floats apart, so
// the four rows (or points) a quarter-warp's LDS.128 touch fall into distinct banks.
__host__ __device__ inline size_t cl_weight_floats(int nh, int nlayers) {
  const size_t hid = (size_t)(nlayers - 2);
  return 4 * (size_t)nh + 4 + hid * kSlice + hid * ((size_t)nh * kSlice + (size_t)kSlice * (nh + 4));
}
inline size_t cl_smem_bytes(int nh, int nlayers, int P) {
  return (cl_weight_floats(nh, nlayers) + 2 * (size_t)P * (nh + 4)) * sizeof(float);
}

struct ClSmem {
  // w0 [2][nh] | b0 [nh] | w_last [nh] | pad 4 | bh [nl-2][16] | wc [nl-2][nh][16] | wr [nl-2][16][nh+4] | act 2 x [P][nh+4]
  // wc[l][k][j] = w_l[k][u0 + j];  wr[l][row(kk)][u] = w_l[u0 + kk][u] with row(kk) = (kk & 3) * 4 + (kk >> 2), so that
  // the four threads of a point (kk = 4 sub + j for the same j) read four rows in distinct banks.
  float* w0; float* b0; float* wl; float bl; float* bh; float* wc; float* wr; float* act;
};

__device__ void cl_load_weights(const cgs_mlp_desc& d, int nh, int u0, float* smem, ClSmem& s) {
  const int nhid = d.nlayers - 2;
  const int RS = nh + 4;
  s.w0 = smem;
  s.b0 = s.w0 + 2 * nh;
  s.wl = s.b0 + nh;
  s.bh = s.wl + nh + 4;
  s.wc = s.bh + nhid * kSlice;
  s.wr = s.wc + (size_t)nhid * nh * kSlice;
  s.act = s.wr + (size_t)nhid * kSlice * RS;
  for (int i = threadIdx.x; i < 2 * nh; i += blockDim.x) s.w0[i] = d.weights[0][i];
  for (int i = threadIdx.x; i < nh; i += blockDim.x) s.b0[i] = d.biases[0][i];
  for (int i = threadIdx.x; i < nh; i += blockDim.x) s.wl[i] = d.weights[d.nlayers - 1][i];
  s.bl = d.biases[d.nlayers - 1][0];
  for (int l = 0; l < nhid; ++l) {
    const float* w = d.weights[1 + l];
    const float* b = d.biases[1 + l];
    for (int i = threadIdx.x; i < kSlice; i += blockDim.x) s.bh[l * kSlice + i] = b[u0 + i];
    float* wc = s.wc + (size_t)l * nh * kSlice;
    for (int i = threadIdx.x; i < nh * kSlice; i += blockDim.x) wc[i] = w[(i / kSlice) * nh + u0 + i % kSlice];
    float* wr = s.wr + (size_t)l * kSlice * RS;
    for (int i = threadIdx.x; i < kSlice * nh; i += blockDim.x) {
      const int kk = i / nh, u = i % nh;
      wr[((kk & 3) * 4 + (kk >> 2)) * RS + u] = w[(size_t)(u0 + kk) * nh + u];
    }
  }
}

struct ClCtx {
  float* cur;         // activation ping-pong, [P][nh + 4] each: the buffer holding the vector to read next
  float* nxt;         // and the one the layer writes
  int nh, RS, C;      // width, row stride, CTAs of the cluster
  int pt, sub, v0;    // point slot, quarter of the slice, first own unit (16 rank + 4 sub)
};

// This thread's 4 values go to units v0 .. v0 + 3 of its point in the next buffer of every CTA, then the one barrier.
__device__ __forceinline__ void cl_exchange(ClCtx& c, float4 v) {
  const float* dst = c.nxt + c.pt * c.RS + c.v0;
  for (int q = 0; q < c.C; ++q) st_cluster_v4(dst, (uint32_t)q, v);
  cluster_sync_all();
  float* t = c.cur;
  c.cur = c.nxt;
  c.nxt = t;
}

__device__ __forceinline__ float relu_bit(float v, unsigned int& mask, int bit) {
  const bool on = v > 0.f;
  mask |= (on ? 1u : 0u) << bit;
  return on ? v : 0.f;
}

// Forward + backward through the MLP for one point, as mlp_point.  mask bit 4 l + j = ReLU of unit v0 + j at layer l.
template <bool kGrad>
__device__ __forceinline__ float mlp_point_cluster(const ClSmem& s, int nlayers, float x, float y, float& gx, float& gy,
                                                   ClCtx& c) {
  const int nhid = nlayers - 2;
  const int nh = c.nh, v0 = c.v0;
  unsigned int mask = 0;
  // layer 0: 2 -> nh (own units)                         synthetic/GAN.py:30-31
  {
    float4 o;
    o.x = relu_bit(fmaf(y, s.w0[nh + v0 + 0], fmaf(x, s.w0[v0 + 0], s.b0[v0 + 0])), mask, 0);
    o.y = relu_bit(fmaf(y, s.w0[nh + v0 + 1], fmaf(x, s.w0[v0 + 1], s.b0[v0 + 1])), mask, 1);
    o.z = relu_bit(fmaf(y, s.w0[nh + v0 + 2], fmaf(x, s.w0[v0 + 2], s.b0[v0 + 2])), mask, 2);
    o.w = relu_bit(fmaf(y, s.w0[nh + v0 + 3], fmaf(x, s.w0[v0 + 3], s.b0[v0 + 3])), mask, 3);
    cl_exchange(c, o);
  }
  // hidden layers: nh -> nh                                synthetic/GAN.py:32-34
  for (int l = 0; l < nhid; ++l) {
    const float4* w = reinterpret_cast<const float4*>(s.wc + (size_t)l * nh * kSlice + 4 * c.sub);  // k at w[4 k]
    const float* b = s.bh + l * kSlice + 4 * c.sub;
    const float4* R = reinterpret_cast<const float4*>(c.cur + c.pt * c.RS);
    float o0 = b[0], o1 = b[1], o2 = b[2], o3 = b[3];
#pragma unroll 2
    for (int k4 = 0; k4 < nh / 4; ++k4) {
      const float4 a = R[k4];
      float4 ww = w[4 * (4 * k4 + 0)];
      o0 = fmaf(a.x, ww.x, o0); o1 = fmaf(a.x, ww.y, o1); o2 = fmaf(a.x, ww.z, o2); o3 = fmaf(a.x, ww.w, o3);
      ww = w[4 * (4 * k4 + 1)];
      o0 = fmaf(a.y, ww.x, o0); o1 = fmaf(a.y, ww.y, o1); o2 = fmaf(a.y, ww.z, o2); o3 = fmaf(a.y, ww.w, o3);
      ww = w[4 * (4 * k4 + 2)];
      o0 = fmaf(a.z, ww.x, o0); o1 = fmaf(a.z, ww.y, o1); o2 = fmaf(a.z, ww.z, o2); o3 = fmaf(a.z, ww.w, o3);
      ww = w[4 * (4 * k4 + 3)];
      o0 = fmaf(a.w, ww.x, o0); o1 = fmaf(a.w, ww.y, o1); o2 = fmaf(a.w, ww.z, o2); o3 = fmaf(a.w, ww.w, o3);
    }
    const int bit = 4 * (l + 1);
    float4 o;
    o.x = relu_bit(o0, mask, bit + 0);
    o.y = relu_bit(o1, mask, bit + 1);
    o.z = relu_bit(o2, mask, bit + 2);
    o.w = relu_bit(o3, mask, bit + 3);
    cl_exchange(c, o);
  }
  // last layer: nh -> 1 (every thread)                     synthetic/GAN.py:35
  float logit = s.bl;
  {
    const float4* R = reinterpret_cast<const float4*>(c.cur + c.pt * c.RS);
    const float4* wl = reinterpret_cast<const float4*>(s.wl);
#pragma unroll 4
    for (int k4 = 0; k4 < nh / 4; ++k4) {
      const float4 a = R[k4], ww = wl[k4];
      logit = fmaf(a.x, ww.x, logit);
      logit = fmaf(a.y, ww.y, logit);
      logit = fmaf(a.z, ww.z, logit);
      logit = fmaf(a.w, ww.w, logit);
    }
  }
  if (!kGrad) return logit;

  // backward: g = d logit / d activation, masked by each ReLU
  {
    const int bit = 4 * nhid;
    float4 g;
    g.x = ((mask >> (bit + 0)) & 1u) ? s.wl[v0 + 0] : 0.f;
    g.y = ((mask >> (bit + 1)) & 1u) ? s.wl[v0 + 1] : 0.f;
    g.z = ((mask >> (bit + 2)) & 1u) ? s.wl[v0 + 2] : 0.f;
    g.w = ((mask >> (bit + 3)) & 1u) ? s.wl[v0 + 3] : 0.f;
    cl_exchange(c, g);
  }
  for (int l = nhid - 1; l >= 0; --l) {
    // g_in[k] = sum_u w[k][u] * g_out[u] for k = v0 + j: four interleaved partial sums over float4 groups of u
    const float* w = s.wr + (size_t)l * kSlice * c.RS;
    const float4* W0 = reinterpret_cast<const float4*>(w + (0 * 4 + c.sub) * c.RS);
    const float4* W1 = reinterpret_cast<const float4*>(w + (1 * 4 + c.sub) * c.RS);
    const float4* W2 = reinterpret_cast<const float4*>(w + (2 * 4 + c.sub) * c.RS);
    const float4* W3 = reinterpret_cast<const float4*>(w + (3 * 4 + c.sub) * c.RS);
    const float4* R = reinterpret_cast<const float4*>(c.cur + c.pt * c.RS);
    float4 a0 = make_float4(0.f, 0.f, 0.f, 0.f), a1 = a0, a2 = a0, a3 = a0;
#pragma unroll 2
    for (int u4 = 0; u4 < nh / 4; ++u4) {
      const float4 g = R[u4];
      float4 ww = W0[u4];
      a0.x = fmaf(ww.x, g.x, a0.x); a0.y = fmaf(ww.y, g.y, a0.y); a0.z = fmaf(ww.z, g.z, a0.z); a0.w = fmaf(ww.w, g.w, a0.w);
      ww = W1[u4];
      a1.x = fmaf(ww.x, g.x, a1.x); a1.y = fmaf(ww.y, g.y, a1.y); a1.z = fmaf(ww.z, g.z, a1.z); a1.w = fmaf(ww.w, g.w, a1.w);
      ww = W2[u4];
      a2.x = fmaf(ww.x, g.x, a2.x); a2.y = fmaf(ww.y, g.y, a2.y); a2.z = fmaf(ww.z, g.z, a2.z); a2.w = fmaf(ww.w, g.w, a2.w);
      ww = W3[u4];
      a3.x = fmaf(ww.x, g.x, a3.x); a3.y = fmaf(ww.y, g.y, a3.y); a3.z = fmaf(ww.z, g.z, a3.z); a3.w = fmaf(ww.w, g.w, a3.w);
    }
    const int bit = 4 * l;
    float4 o;
    o.x = ((mask >> (bit + 0)) & 1u) ? (a0.x + a0.y) + (a0.z + a0.w) : 0.f;
    o.y = ((mask >> (bit + 1)) & 1u) ? (a1.x + a1.y) + (a1.z + a1.w) : 0.f;
    o.z = ((mask >> (bit + 2)) & 1u) ? (a2.x + a2.y) + (a2.z + a2.w) : 0.f;
    o.w = ((mask >> (bit + 3)) & 1u) ? (a3.x + a3.y) + (a3.z + a3.w) : 0.f;
    cl_exchange(c, o);
  }
  {
    const float4* R = reinterpret_cast<const float4*>(c.cur + c.pt * c.RS);
    const float4* wx = reinterpret_cast<const float4*>(s.w0);
    const float4* wy = reinterpret_cast<const float4*>(s.w0 + nh);
    float ax = 0.f, ay = 0.f;
#pragma unroll 4
    for (int u4 = 0; u4 < nh / 4; ++u4) {
      const float4 g = R[u4], a = wx[u4], b = wy[u4];
      ax = fmaf(a.x, g.x, ax); ay = fmaf(b.x, g.x, ay);
      ax = fmaf(a.y, g.y, ax); ay = fmaf(b.y, g.y, ay);
      ax = fmaf(a.z, g.z, ax); ay = fmaf(b.z, g.z, ay);
      ax = fmaf(a.w, g.w, ax); ay = fmaf(b.w, g.w, ay);
    }
    gx = ax;
    gy = ay;
  }
  return logit;
}

// Weights into this CTA, the thread's place in the cluster, and a first cluster barrier: every CTA has started and
// holds its weights before any peer writes into its activation buffers.
__device__ __forceinline__ void cl_setup(const cgs_mlp_desc& d, int nh, int P, float* smem, ClSmem& s, ClCtx& c) {
  const int rank = (int)cluster_ctarank();
  cl_load_weights(d, nh, rank * kSlice, smem, s);
  c.nh = nh;
  c.RS = nh + 4;
  c.C = nh / kSlice;
  c.pt = threadIdx.x / kSub;
  c.sub = threadIdx.x % kSub;
  c.v0 = rank * kSlice + kSub * c.sub;
  c.cur = s.act;
  c.nxt = s.act + (size_t)P * c.RS;
  cluster_sync_all();
}

__global__ void __launch_bounds__(kMaxThreads, 1)
mlp2d_cluster_score_kernel(const cgs_mlp_desc d, int nh, int P, const float* __restrict__ x, int64_t n, int ppr,
                           int64_t chunks, float inv_n, float* __restrict__ sig_out, float* __restrict__ logit_out,
                           float* __restrict__ sal_out) {
  extern __shared__ float4 smem4[];
  ClSmem s;
  ClCtx c;
  cl_setup(d, nh, P, reinterpret_cast<float*>(smem4), s, c);
  const int C = nh / kSlice;
  const bool lead = cluster_ctarank() == 0 && c.sub == 0;
  for (int64_t ch = blockIdx.x / C; ch < chunks; ch += gridDim.x / C) {
    const int64_t i = ch * ppr + c.pt;
    const bool ok = c.pt < ppr && i < n;
    const float px = ok ? x[2 * i] : 0.f, py = ok ? x[2 * i + 1] : 0.f;
    float gx = 0.f, gy = 0.f;
    float logit;
    if (sal_out) logit = mlp_point_cluster<true>(s, d.nlayers, px, py, gx, gy, c);
    else logit = mlp_point_cluster<false>(s, d.nlayers, px, py, gx, gy, c);
    if (ok && lead) {
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
  cluster_sync_all();
}

__global__ void __launch_bounds__(kMaxThreads, 1)
mlp2d_cluster_refine_kernel(const cgs_mlp_desc d, int nh, int P, PolicyConsts pc, int steps, float inv_n,
                            float real_mean, const float* __restrict__ x_in, int64_t n, int ppr, int64_t chunks,
                            float* __restrict__ best_x_out, float* __restrict__ best_loss_out,
                            float* __restrict__ best_step_out, float* __restrict__ traj) {
  extern __shared__ float4 smem4[];
  ClSmem s;
  ClCtx c;
  cl_setup(d, nh, P, reinterpret_cast<float*>(smem4), s, c);
  const int C = nh / kSlice;
  const bool lead = cluster_ctarank() == 0 && c.sub == 0;
  for (int64_t ch = blockIdx.x / C; ch < chunks; ch += gridDim.x / C) {
    const int64_t i = ch * ppr + c.pt;
    const bool ok = c.pt < ppr && i < n;
    const bool writer = ok && lead;
    float px = ok ? x_in[2 * i] : 0.f, py = ok ? x_in[2 * i + 1] : 0.f;
    float gx, gy;
    float logit = mlp_point_cluster<true>(s, d.nlayers, px, py, gx, gy, c);
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
      logit = mlp_point_cluster<true>(s, d.nlayers, px, py, gx, gy, c);   // refiner_cpu.py:52
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
  cluster_sync_all();
}

// ------------------------------------------------------------------------------------------------ host side
struct ClusterLaunch {
  int C;            // CTAs per cluster
  int P;            // point slots the shared memory is planned for
  size_t smem;
  int clusters;     // clusters launched
  int ppr;          // points per round
  int64_t chunks;   // rounds of ppr points over the whole batch
};

// How many clusters of this kernel fit on the current device at once (asked once per kernel, device, cluster size,
// block size and shared-memory size).  0 means not even one: the caller refuses instead of launching.
template <typename K>
int resident_clusters(K kernel, int C, int threads, size_t smem, int& clusters) {
  static std::mutex m;
  static std::map<std::tuple<int, int, int, size_t>, int> known;
  const int dev = current_device();
  std::lock_guard<std::mutex> lock(m);
  auto it = known.find(std::make_tuple(dev, C, threads, smem));
  if (it != known.end()) { clusters = it->second; return CGS_OK; }
  cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmemLimit);
  if (e != cudaSuccess) return set_error(CGS_ERR_CUDA, "cudaFuncSetAttribute: %s", cudaGetErrorString(e));
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(C);
  cfg.blockDim = dim3(threads);
  cfg.dynamicSmemBytes = smem;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = (unsigned)C;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  int nc = 0;
  e = cudaOccupancyMaxActiveClusters(&nc, kernel, &cfg);
  if (e != cudaSuccess) return set_error(CGS_ERR_CUDA, "cudaOccupancyMaxActiveClusters: %s", cudaGetErrorString(e));
  known[std::make_tuple(dev, C, threads, smem)] = nc;
  clusters = nc;
  return CGS_OK;
}

// The largest round of points that fits beside the weights, the resident clusters, and the points dealt evenly over
// min(resident clusters, rounds) clusters.
template <typename K>
int plan_launch(K kernel, const cgs_mlp_desc& d, int64_t n, ClusterLaunch& L) {
  const int nh = d.nhidden;
  L.C = nh / kSlice;
  const size_t wbytes = cl_weight_floats(nh, d.nlayers) * sizeof(float);
  const size_t per_point = 2 * (size_t)(nh + 4) * sizeof(float);
  size_t P = wbytes < kSmemLimit ? (kSmemLimit - wbytes) / per_point : 0;
  if (P > (size_t)kMaxPoints) P = kMaxPoints;
  P = P / kPointQuantum * kPointQuantum;
  if (P == 0)
    return set_error(CGS_ERR_UNSUPPORTED,
                     "nhidden %d, nlayers %d: the cluster form keeps %zu bytes of weights per CTA and needs %zu more "
                     "for %d points, above the %zu bytes of shared memory a CTA gets",
                     nh, d.nlayers, wbytes, per_point * kPointQuantum, kPointQuantum, kSmemLimit);
  L.P = (int)P;
  L.smem = cl_smem_bytes(nh, d.nlayers, L.P);
  int resident = 0;
  if (int rc = resident_clusters(kernel, L.C, kSub * L.P, L.smem, resident)) return rc;
  if (resident < 1)
    return set_error(CGS_ERR_UNSUPPORTED,
                     "nhidden %d, nlayers %d: a cluster of %d CTAs with %zu bytes of shared memory each is not "
                     "resident on this device",
                     nh, d.nlayers, L.C, L.smem);
  int64_t ppr = (n + resident - 1) / resident;
  L.ppr = (int)(ppr < 1 ? 1 : (ppr > L.P ? L.P : ppr));
  L.chunks = (n + L.ppr - 1) / L.ppr;
  L.clusters = (int)(L.chunks < resident ? L.chunks : resident);
  return CGS_OK;
}

template <typename... KArgs, typename... Args>
int launch_clusters(void (*kernel)(KArgs...), const ClusterLaunch& L, cudaStream_t st, const char* what, Args... args) {
  const int slots = (L.ppr + kPointQuantum - 1) / kPointQuantum * kPointQuantum;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)(L.clusters * L.C));
  cfg.blockDim = dim3((unsigned)(kSub * slots));
  cfg.dynamicSmemBytes = L.smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = (unsigned)L.C;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  cudaError_t e = cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
  count_launch();
  if (e != cudaSuccess) return set_error(CGS_ERR_CUDA, "%s: %s", what, cudaGetErrorString(e));
  return check_launch(what);
}

}  // namespace

int mlp2d_cluster_score(const cgs_mlp_desc& d, const float* x, int64_t n, float inv_n, float* sig_out,
                        float* logit_out, float* sal_out, cudaStream_t st) {
  ClusterLaunch L;
  if (int rc = plan_launch(mlp2d_cluster_score_kernel, d, n, L)) return rc;
  return launch_clusters(mlp2d_cluster_score_kernel, L, st, "cgs_mlp2d_score", d, d.nhidden, L.P, x, n, L.ppr,
                         L.chunks, inv_n, sig_out, logit_out, sal_out);
}

int mlp2d_cluster_refine(const cgs_mlp_desc& d, const cgs_refine2d_cfg& cfg, float inv_n, const float* x_in, int64_t n,
                         float* best_x, float* best_loss, float* best_step, float* traj, cudaStream_t st) {
  ClusterLaunch L;
  if (int rc = plan_launch(mlp2d_cluster_refine_kernel, d, n, L)) return rc;
  return launch_clusters(mlp2d_cluster_refine_kernel, L, st, "cgs_refine_mlp2d", d, d.nhidden, L.P,
                         make_policy_consts(cfg.policy), cfg.steps, inv_n, cfg.real_sigmoid_mean, x_in, n, L.ppr,
                         L.chunks, best_x, best_loss, best_step, traj);
}

}  // namespace cgs
