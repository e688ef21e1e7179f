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
#include <cuda_fp16.h>
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

// What a layer pass does to its accumulator: the one description every pass kernel's epilogue reads (epilogue4 /
// epilogue1 below).  Member order matters: the EPI_UPDATE tensor-core instances sit at the register cap, and their
// allocation follows how these fields pair into 8-byte parameter loads.
struct Epilogue {
  const float* bias;  // EPI_FWD (null = no bias)
  const float* aux;   // EPI_BWD: forward OUTPUT of the layer being differentiated
  float* mom;         // EPI_UPDATE: momentum, same layout as out
  int first, clip, sgd;                 // EPI_UPDATE policy constants (sampling/policy.py:27-37, collaborator.py:69-70)
  float rate, alpha, vmin, vmax;
  float slope;        // relu 0, lrelu 0.2, none 1 (branch-free: max(v, slope * v) and its derivative)
  int act_tanh;       // the activation is tanh (slow path)
  int round_out;      // round results to TF32 (RN) because the next consumer is a kind::tf32 MMA
  int mode;           // EPI_*
  // FP16 operand chains (choose_operand_type in refine_conv.cu):
  int out16;          // FWD / BWD: the output is stored as FP16 (it feeds a kind::f16 MMA); aux is FP16 there too
  const int* gexp;    // UPDATE / RAW: the accumulator is d loss / d x times 2^gexp[b] (head_kernel), null = unscaled

  Epilogue() = default;
  // host: mode `mode_` (EPI_*) through activation `act` (ACT_*), no operands -- the only place an activation becomes
  // slope / act_tanh
  Epilogue(int mode_, int act) : bias(nullptr), aux(nullptr), mom(nullptr), first(0), clip(0), sgd(0), rate(0.f),
                                 alpha(0.f), vmin(0.f), vmax(0.f),
                                 slope(act == ACT_RELU ? 0.f : (act == ACT_LRELU ? 0.2f : 1.f)),
                                 act_tanh(act == ACT_TANH), round_out(0), mode(mode_),
                                 out16(0), gexp(nullptr) {}
};

struct ConvGemmParams {
  const float* in;
  float* out;
  Epilogue ep;
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
  int f16;            // FP16 operands on kind::f16: cblocks / nkb / cb0 count 64-channel atoms (host: to_f16_atoms)
  // exact division of the persistent tile index by multiply-shift (filled by the launcher; see fast_div)
  unsigned long long fd_tiles_per_class, fd_n_tiles, fd_hy_tiles;
  GemmClass cls[kMaxClasses];
};

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

// FP16 operands: four values -> four halves (RN, saturating to +-65504 instead of overflowing to inf), and back
__device__ __forceinline__ uint2 pack_half4(float4 v) {
  uint32_t lo, hi;
  asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(lo) : "f"(v.y), "f"(v.x));
  asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(hi) : "f"(v.w), "f"(v.z));
  return make_uint2(lo, hi);
}
__device__ __forceinline__ float4 unpack_half4(uint2 u) {
  const float2 a = __half22float2(*reinterpret_cast<const __half2*>(&u.x));
  const float2 b = __half22float2(*reinterpret_cast<const __half2*>(&u.y));
  return make_float4(a.x, a.y, b.x, b.y);
}
// 2^-e exactly (0 <= e < 127): removes the per-sample gradient scale of head_kernel
__device__ __forceinline__ float exp2_neg(int e) { return __int_as_float((127 - e) << 23); }

// ---------------------------------------------------------------------------------------------
// The epilogue formulas, once: a vector form (four consecutive output channels) and a scalar form (one channel) with
// the same expressions, so a layer's result does not depend on which lowering ran it.  x0 / x1 are the operands the
// caller has already fetched (so that many loads can be in flight):
//   FWD     out = act(acc + x0)          x0 = bias
//   BWD     out = acc * act'(x0)         x0 = forward output of the differentiated layer (act' through the output)
//   UPDATE  momentum / sgd step          x0 = current feature, x1 = momentum; the new momentum goes to e.mom
//   RAW     out = acc
// FWD / BWD / RAW results are rounded to TF32 when e.round_out.  EPI is a compile-time constant where the epilogue is
// hot (no run-time mode switches there); epilogue4 / epilogue1 dispatch on e.mode.
// ---------------------------------------------------------------------------------------------
// `off` = element offset of the four channels in e.mom
template <int EPI>
__device__ __forceinline__ float4 epilogue4_t(const Epilogue& e, int off, float4 a, float4 x0, float4 x1) {
  float4 o = a;
  if (EPI == EPI_FWD) {
    const float vx = a.x + x0.x, vy = a.y + x0.y, vz = a.z + x0.z, vw = a.w + x0.w;
    if (!e.act_tanh) {          // relu / lrelu / none: max(v, slope * v)
      o.x = fmaxf(vx, vx * e.slope); o.y = fmaxf(vy, vy * e.slope);
      o.z = fmaxf(vz, vz * e.slope); o.w = fmaxf(vw, vw * e.slope);
    } else {
      o.x = tanhf(vx); o.y = tanhf(vy); o.z = tanhf(vz); o.w = tanhf(vw);
    }
  } else if (EPI == EPI_BWD) {
    if (!e.act_tanh) {          // derivative through the forward output: 1 where it is positive, slope elsewhere
      o.x = a.x * (x0.x > 0.f ? 1.f : e.slope); o.y = a.y * (x0.y > 0.f ? 1.f : e.slope);
      o.z = a.z * (x0.z > 0.f ? 1.f : e.slope); o.w = a.w * (x0.w > 0.f ? 1.f : e.slope);
    } else {
      o.x = a.x * (1.f - x0.x * x0.x); o.y = a.y * (1.f - x0.y * x0.y);
      o.z = a.z * (1.f - x0.z * x0.z); o.w = a.w * (1.f - x0.w * x0.w);
    }
  } else if (EPI == EPI_UPDATE) {
    // sampling/policy.py:27-37; separately rounded multiplies / adds like the reference's un-fused TF ops
    float4 m;
    m.x = __fmul_rn(e.rate, a.x); m.y = __fmul_rn(e.rate, a.y); m.z = __fmul_rn(e.rate, a.z); m.w = __fmul_rn(e.rate, a.w);
    if (!e.sgd) {
      if (!e.first) {
        m.x = __fadd_rn(__fmul_rn(e.alpha, x1.x), m.x);
        m.y = __fadd_rn(__fmul_rn(e.alpha, x1.y), m.y);
        m.z = __fadd_rn(__fmul_rn(e.alpha, x1.z), m.z);
        m.w = __fadd_rn(__fmul_rn(e.alpha, x1.w), m.w);
      }
      *reinterpret_cast<float4*>(e.mom + off) = m;
    }
    o.x = __fsub_rn(x0.x, m.x); o.y = __fsub_rn(x0.y, m.y); o.z = __fsub_rn(x0.z, m.z); o.w = __fsub_rn(x0.w, m.w);
    if (e.clip) {                                                    // collaborator.py:69-70
      o.x = fminf(fmaxf(o.x, e.vmin), e.vmax); o.y = fminf(fmaxf(o.y, e.vmin), e.vmax);
      o.z = fminf(fmaxf(o.z, e.vmin), e.vmax); o.w = fminf(fmaxf(o.w, e.vmin), e.vmax);
    }
    return o;
  }
  if (e.round_out) { o.x = tf32_rn(o.x); o.y = tf32_rn(o.y); o.z = tf32_rn(o.z); o.w = tf32_rn(o.w); }
  return o;
}

__device__ __forceinline__ float4 epilogue4(const Epilogue& e, int off, float4 a, float4 x0, float4 x1) {
  switch (e.mode) {
    case EPI_FWD: return epilogue4_t<EPI_FWD>(e, off, a, x0, x1);
    case EPI_BWD: return epilogue4_t<EPI_BWD>(e, off, a, x0, x1);
    case EPI_UPDATE: return epilogue4_t<EPI_UPDATE>(e, off, a, x0, x1);
    default: return epilogue4_t<EPI_RAW>(e, off, a, x0, x1);
  }
}

// The new momentum goes to *m_out instead (the caller stores it with its neighbours).  EPI / TANH / ROUND: -1 = read
// e.mode / e.act_tanh / e.round_out at run time, else known at compile time (kernels with one instance per mode).
// (e.mode is re-read at each test rather than copied once: the copy changed the register allocation of the
// mma.sync edge kernels)
template <int EPI = -1, int TANH = -1, int ROUND = -1>
__device__ __forceinline__ float epilogue1_t(const Epilogue& e, float a, float x0, float x1, float* m_out) {
  float o = a;
  if ((EPI < 0 ? e.mode : EPI) == EPI_FWD) {
    const float v = a + x0;
    o = (TANH < 0 ? e.act_tanh : TANH) ? tanhf(v) : fmaxf(v, v * e.slope);
  } else if ((EPI < 0 ? e.mode : EPI) == EPI_BWD) {
    o = (TANH < 0 ? e.act_tanh : TANH) ? a * (1.f - x0 * x0) : a * (x0 > 0.f ? 1.f : e.slope);
  } else if ((EPI < 0 ? e.mode : EPI) == EPI_UPDATE) {
    float m = __fmul_rn(e.rate, a);
    if (!e.sgd) {
      if (!e.first) m = __fadd_rn(__fmul_rn(e.alpha, x1), m);
      *m_out = m;
    }
    o = __fsub_rn(x0, m);
    if (e.clip) o = fminf(fmaxf(o, e.vmin), e.vmax);
    return o;
  }
  return (ROUND < 0 ? e.round_out : ROUND) ? tf32_rn(o) : o;
}

__device__ __forceinline__ float epilogue1(const Epilogue& e, float a, float x0, float x1, float* m_out) {
  return epilogue1_t<>(e, a, x0, x1, m_out);
}

// The operands of epilogue4 for four output channels at element `off` of out / aux / mom and channel n of the bias,
// for the kernels without a tuned load schedule of their own
__device__ __forceinline__ void epilogue_operands4(const Epilogue& e, const float* out, int off, int n, float4& x0,
                                                   float4& x1) {
  x0 = make_float4(0.f, 0.f, 0.f, 0.f);
  x1 = x0;
  if (e.mode == EPI_FWD) { if (e.bias) x0 = __ldg(reinterpret_cast<const float4*>(e.bias + n)); }
  else if (e.mode == EPI_BWD) x0 = __ldg(reinterpret_cast<const float4*>(e.aux + off));
  else if (e.mode == EPI_UPDATE) {
    x0 = *reinterpret_cast<const float4*>(out + off);
    if (!e.sgd && !e.first) x1 = *reinterpret_cast<const float4*>(e.mom + off);
  }
}

// host launchers (conv_gemm.cu)
// p.f16: FP16 operands (p.in, w and the FP16 outputs of the epilogue are __half; K counted in 64-channel atoms)
int launch_conv_gemm_tc(const ConvGemmParams& p, const void* w, int w_rows, int w_cols, cudaStream_t stream);
int launch_conv_gemm_simt(const ConvGemmParams& p, const float* w, int w_rows, int w_cols, cudaStream_t stream);
// host only: fills p.grp / p.shf the way the class-fused launch would and returns the slots per tile (0 = this pass
// is never class-fused).  No device state is touched (cgs_debug_fusion_plan).
int plan_fusion(ConvGemmParams& p);

}  // namespace cgs
