// Gathered-A implicit GEMM: the one contraction kernel behind every conv / deconv / fc pass of the
// refinement loop (forward AND data-gradient; weights are frozen so there is no wgrad).
//
//   out[b, j*os+oy0, i*os+ox0, n] = epi( sum_{t<ntaps} sum_{c<Cin} in[b, j*S+dy[t], i*S+dx[t], c] * W[n][k0 + t*Cin + c] )
//
// * stride-2 conv fprop (nsgan/ops.py:41) and deconv-backward: S=2, os=1, one class, taps = all (ky,kx)
// * stride-2 deconv fprop (nsgan/ops.py:55) and conv data-gradient: S=1, os=2, four output-parity classes,
//   each with its own tap subset (k4: 2x2 taps; k5: 3x3/3x2/2x3/2x2) -- no zero-insertion MACs
// * fc (nsgan/ops.py:81): IH=IW=MH=MW=1, one tap
// Rows m = (b, j, i) are gathered (zero-filled outside the image) into 128B-swizzled shared memory;
// W is a plain K-major matrix fetched by TMA.  Pixel mode (Cs == 4) packs 8 taps x 4 channels per K block
// for the 1-/3-channel image layers.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

namespace cgs {

enum : int { ACT_NONE = 0, ACT_RELU = 1, ACT_LRELU = 2, ACT_TANH = 3 };
enum : int {
  EPI_FWD = 0,     // out = act(acc + bias)
  EPI_BWD = 1,     // out = acc * act'(aux)      (aux = forward OUTPUT of the layer being differentiated)
  EPI_UPDATE = 2,  // acc is d loss / d feature: momentum/sgd step fused (sampling/policy.py:27-37)
  EPI_RAW = 3      // out = acc
};

constexpr int kMaxTaps = 32;
constexpr int kMaxClasses = 4;
constexpr int kMaxShifts = 18;

// Class-fused transposed passes (stride-2 deconv forward / conv data-gradient): the output-parity classes of one
// input-grid tile read the SAME shifted input tiles (dy, dx in {-1, 0, 1}), each class with its own weights.  A fused
// tile keeps one TMEM accumulator per class ("slot") and walks the shifts once: the A tile of a shift is fetched once
// and multiplied with the weight tile of every class that has a tap there -- 9 A loads instead of 25 for k = 5.
struct FuseShift {
  signed char dy, dx;
  unsigned char ncls;           // classes with a tap at this shift
  unsigned char slot[4];        // their accumulator slots
  // runs of ADJACENT slots with the same accumulate state: one MMA of N = run_len * BN columns per k-step reads the
  // A tile once for all of them (a 64-wide MMA is otherwise bound by its shared-memory operand reads, 6 KB per 32
  // cycles of tensor work); run_acc = the slots already hold partial sums
  unsigned char nrun, run_slot[4], run_len[4], run_acc[4];
  int katom0[4];                // first K atom (32 floats) of that tap's weights; + channel block
  // CTA pairs: a run's B rows are its atoms back to back, split in the middle between the two CTAs.  Per CTA rank the
  // half-atom boxes to fetch: destination slot (half an atom wide per CTA), which half of the atom, its K atom
  unsigned char pc_slot[2][4], pc_half[2][4];
  int pc_katom[2][4];
};
struct FuseGroup {
  int nshifts, shift0, ncls;    // shifts [shift0, shift0 + nshifts) of shf[]; classes in this group
  int cls[4];                   // class index of each slot (output offsets oy0 / ox0)
};

struct GemmClass {
  int k0;      // first K element of this class inside the packed weight matrix
  int nkb;     // K blocks (32 floats) of this class
  int ntaps;   // taps of this class = nky * nkx, tap t = ty * nkx + tx, dy depends on ty only, dx on tx only
  int nkx;
  int oy0, ox0;
  int cb0;     // first 32-channel block of the A operand read by this class (split-K classes of an fc layer)
  signed char dy[kMaxTaps];
  signed char dx[kMaxTaps];
};

struct ConvGemmParams {
  const float* in;
  float* out;
  const float* bias;
  const float* aux;
  float* mom;
  int IH, IW, Cs;     // input image, channel stride (floats per pixel)
  int cblocks;        // Cin / 32 in block mode; 0 in pixel mode
  int MH, MW, S;      // rows per image = MH*MW; input pixel = (j*S+dy, i*S+dx)
  int M;              // B*MH*MW
  int OH, OW, ON, os; // output image, channel stride, output pixel stride
  int N;              // valid output channels
  int n_tiles;        // ceil(N / BLOCK_N)
  int m_tiles;        // row tiles (see tile geometry)
  // tile geometry (filled by the launcher): a row tile = BB images x BH rows x MW columns of the M-space
  // (<= 128 rows, row r = (bb*BH + hh)*MW + ww), so that the A operand of a K block is ONE TMA box
  int B, BH, BB, hy_tiles, rows_valid;
  int a_tma;          // 1: A tiles fetched by TMA; 0: cp.async gather (pixel mode)
  // window mode (strided pass over a <= 4-channel image stored with a zero-padded row pitch): K block ky of output
  // pixel (j,i) is the 128 contiguous bytes starting at stored pixel (2j + ky - pad_y, 2i + win_x0); taps beyond the
  // kernel width carry zero weights.  One TMA box per K block through an overlapping-window tensor map.
  int window, win_k, win_x0, in_pitch_px;
  int nclasses;
  int epi, act;
  int first, clip, sgd;
  float rate, alpha, vmin, vmax;
  float slope;        // derived from act by the launcher: relu 0, lrelu 0.2, none 1 (branch-free epilogue)
  int act_tanh;       // act == tanh (slow path)
  int round_out;      // round results to TF32 (RN) because the next consumer is a kind::tf32 MMA
  int force_bn;       // 0 = tile-width heuristic, else the BN instance to launch
  // early exit (device-resident batch size): when non-null, only the first *live images are processed -- tiles past
  // them are never scheduled, rows past them never stored.  Grids stay sized for the full batch, so the launch
  // sequence is static (CUDA-graph capturable) and no host synchronisation is needed when samples leave the batch.
  const int* live;
  // class fusion (see FuseShift): 0 = one class per tile, else the launcher filled grp / shf
  int fuse, ngroups;
  // adjacent M tiles per scheduling unit: 2 with M-tile pairs (template MT = 2: the pair shares every weight atom
  // of its K loop) or CTA pairs (CG = 2: one tile per CTA of the cluster), 4 with both, else 1 (0 reads as 1)
  int m2;
  FuseGroup grp[2];
  FuseShift shf[kMaxShifts];
  int debug;          // debug_flags() at launch: the profiling knobs of cgs_debug_flag (CGS_DEBUG_SKIP_*, _TRACE)
  // exact division of the persistent tile index by multiply-shift (filled by the launcher; see fast_div)
  unsigned long long fd_tiles_per_class, fd_n_tiles, fd_hy_tiles;
  GemmClass cls[kMaxClasses];
};

__device__ __forceinline__ float act_apply(float v, int act) {
  switch (act) {
    case ACT_RELU: return fmaxf(v, 0.f);
    case ACT_LRELU: return fmaxf(v, 0.2f * v);   // nsgan/ops.py:69-70
    case ACT_TANH: return tanhf(v);
    default: return v;
  }
}
// derivative expressed through the layer OUTPUT y = act(pre)
__device__ __forceinline__ float act_grad_from_output(float y, int act) {
  switch (act) {
    case ACT_RELU: return y > 0.f ? 1.f : 0.f;
    case ACT_LRELU: return y > 0.f ? 1.f : 0.2f;
    case ACT_TANH: return 1.f - y * y;
    default: return 1.f;
  }
}

// n / d by multiply-high with magic = ceil(2^64 / d) (0 encodes d == 1): with magic * d = 2^64 + e, 0 <= e < d, the
// excess n * e / (d * 2^64) stays below 1 / d for every 32-bit n, so the floor is exact
inline unsigned long long fast_div_magic(unsigned d) { return d <= 1 ? 0ull : (~0ull) / d + 1ull; }
__device__ __forceinline__ int fast_div(int n, unsigned long long magic) {
  return magic ? (int)__umul64hi((unsigned long long)(unsigned)n, magic) : n;
}
__device__ __forceinline__ unsigned long long fast_div_magic_dev(unsigned d) { return d <= 1 ? 0ull : (~0ull) / d + 1ull; }

// Tile counts of a launch for the images that are still in the batch (ConvGemmParams::live).
struct LiveTiles {
  int B, tiles_per_class, total;
  unsigned long long fd_tiles_per_class;
};
__device__ __forceinline__ LiveTiles live_tiles(const ConvGemmParams& p) {
  LiveTiles t;
  if (!p.live) {
    t.B = p.B;
    t.tiles_per_class = (p.m2 > 1 ? (p.m_tiles + p.m2 - 1) / p.m2 : p.m_tiles) * p.n_tiles;
    t.fd_tiles_per_class = p.fd_tiles_per_class;
  } else {
    int b = *reinterpret_cast<const volatile int*>(p.live);
    b = b < 0 ? 0 : (b > p.B ? p.B : b);
    t.B = b;
    const int mt_live = ((b + p.BB - 1) / p.BB) * p.hy_tiles;
    t.tiles_per_class = (p.m2 > 1 ? (mt_live + p.m2 - 1) / p.m2 : mt_live) * p.n_tiles;
    t.fd_tiles_per_class = fast_div_magic_dev((unsigned)t.tiles_per_class);
  }
  t.total = t.tiles_per_class * (p.fuse ? p.ngroups : p.nclasses);
  return t;
}

__device__ __forceinline__ float tf32_rn(float x) {
  uint32_t r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
  return __uint_as_float(r);
}

// Four consecutive output channels.  `off` = element offset in mom; x0 / x1 are the operands the caller has already
// fetched (so that many loads can be in flight): FWD x0 = bias; BWD x0 = forward output of the differentiated layer;
// UPDATE x0 = current feature, x1 = momentum.  EPI is a compile-time constant in the tensor-core kernel (the epilogue
// runs per 64-byte row segment: no run-time mode switches there) and p.epi in the other callers.
template <int EPI>
__device__ __forceinline__ float4 epilogue4_t(const ConvGemmParams& p, int off, float4 a, float4 x0, float4 x1) {
  float4 o = a;
  if (EPI == EPI_FWD) {
    const float vx = a.x + x0.x, vy = a.y + x0.y, vz = a.z + x0.z, vw = a.w + x0.w;
    if (!p.act_tanh) {          // relu / lrelu / none: max(v, slope * v)
      o.x = fmaxf(vx, vx * p.slope); o.y = fmaxf(vy, vy * p.slope);
      o.z = fmaxf(vz, vz * p.slope); o.w = fmaxf(vw, vw * p.slope);
    } else {
      o.x = tanhf(vx); o.y = tanhf(vy); o.z = tanhf(vz); o.w = tanhf(vw);
    }
  } else if (EPI == EPI_BWD) {
    if (!p.act_tanh) {          // derivative through the forward output: 1 where it is positive, slope elsewhere
      o.x = a.x * (x0.x > 0.f ? 1.f : p.slope); o.y = a.y * (x0.y > 0.f ? 1.f : p.slope);
      o.z = a.z * (x0.z > 0.f ? 1.f : p.slope); o.w = a.w * (x0.w > 0.f ? 1.f : p.slope);
    } else {
      o.x = a.x * (1.f - x0.x * x0.x); o.y = a.y * (1.f - x0.y * x0.y);
      o.z = a.z * (1.f - x0.z * x0.z); o.w = a.w * (1.f - x0.w * x0.w);
    }
  } else if (EPI == EPI_UPDATE) {
    // sampling/policy.py:27-37; separately rounded multiplies / adds like the reference's un-fused TF ops
    float4 m;
    m.x = __fmul_rn(p.rate, a.x); m.y = __fmul_rn(p.rate, a.y); m.z = __fmul_rn(p.rate, a.z); m.w = __fmul_rn(p.rate, a.w);
    if (!p.sgd) {
      if (!p.first) {
        m.x = __fadd_rn(__fmul_rn(p.alpha, x1.x), m.x);
        m.y = __fadd_rn(__fmul_rn(p.alpha, x1.y), m.y);
        m.z = __fadd_rn(__fmul_rn(p.alpha, x1.z), m.z);
        m.w = __fadd_rn(__fmul_rn(p.alpha, x1.w), m.w);
      }
      *reinterpret_cast<float4*>(p.mom + off) = m;
    }
    o.x = __fsub_rn(x0.x, m.x); o.y = __fsub_rn(x0.y, m.y); o.z = __fsub_rn(x0.z, m.z); o.w = __fsub_rn(x0.w, m.w);
    if (p.clip) {                                                    // collaborator.py:69-70
      o.x = fminf(fmaxf(o.x, p.vmin), p.vmax); o.y = fminf(fmaxf(o.y, p.vmin), p.vmax);
      o.z = fminf(fmaxf(o.z, p.vmin), p.vmax); o.w = fminf(fmaxf(o.w, p.vmin), p.vmax);
    }
    return o;
  }
  if (p.round_out) { o.x = tf32_rn(o.x); o.y = tf32_rn(o.y); o.z = tf32_rn(o.z); o.w = tf32_rn(o.w); }
  return o;
}

__device__ __forceinline__ float4 epilogue4(const ConvGemmParams& p, int off, float4 a, float4 x0, float4 x1) {
  switch (p.epi) {
    case EPI_FWD: return epilogue4_t<EPI_FWD>(p, off, a, x0, x1);
    case EPI_BWD: return epilogue4_t<EPI_BWD>(p, off, a, x0, x1);
    case EPI_UPDATE: return epilogue4_t<EPI_UPDATE>(p, off, a, x0, x1);
    default: return epilogue4_t<EPI_RAW>(p, off, a, x0, x1);
  }
}

// host launchers (conv_gemm.cu)
int launch_conv_gemm_tc(const ConvGemmParams& p, const float* w, int w_rows, int w_cols, cudaStream_t stream);
int launch_conv_gemm_simt(const ConvGemmParams& p, const float* w, int w_rows, int w_cols, cudaStream_t stream);
// host only: fills p.grp / p.shf the way the class-fused launch would and returns the slots per tile (0 = this pass
// is never class-fused).  No device state is touched (cgs_debug_fusion_plan).
int plan_fusion(ConvGemmParams& p);

}  // namespace cgs
