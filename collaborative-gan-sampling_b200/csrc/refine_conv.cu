// Image-path refinement: layer -> gathered-GEMM parameter mapping, the fused head kernel (logit GEMV +
// BCE gradient + best-of-K select + image keep), and the K-step loop of sampling/collaborator.py:41-88.
#include "batchnorm.cuh"
#include "common.h"
#include "conv_gemm.cuh"
#include "edge_conv.cuh"
#include "ptx.cuh"

#include <cstdlib>
#include <cstring>

namespace cgs {

namespace {

inline int cstride(int c) { return (c + 3) & ~3; }   // NHWC channel stride (floats)

inline int same_pad_before(int in_size, int k) {      // TF SAME, stride 2 (SURVEY App. A8)
  const int out = (in_size + 1) / 2;
  int total = (out - 1) * 2 + k - in_size;
  if (total < 0) total = 0;
  return total / 2;
}

struct LayerShape {
  int hout, wout, cs_out;
};

LayerShape layer_shape(const cgs_layer_desc& L) {
  LayerShape s;
  s.cs_out = cstride(L.cout);
  if (L.type == CGS_LAYER_CONV) {
    s.hout = (L.hin + 1) / 2;
    s.wout = (L.win + 1) / 2;
  } else if (L.type == CGS_LAYER_DECONV) {
    s.hout = L.hin * 2;
    s.wout = L.win * 2;
  } else {
    s.hout = s.wout = 1;
  }
  return s;
}

// The fixed facts of one pass of a layer, forward or data-gradient (the pass that maps the gradient w.r.t. the
// layer's pre-activation output back to its input).  The strided type (conv forward, deconv data-gradient) reads
// input pixels (2j + ky - pad, 2i + kx - pad); the transposed type (deconv forward, conv data-gradient) is its
// adjoint.  Either way the TF SAME pads are those of the stride-2 conv over the finer of the two grids.
struct PassShape {
  int ih, iw, oh, ow;     // input and output grid (fc: 1 x 1)
  int kch, nch;           // reduced (K-side) and produced (N-side) channel counts
  int pad_y, pad_x;       // 0 for fc
  bool strided;           // strided type; else transposed type or fc
  const float* w;         // packed weights of the pass: rows x cols
  int rows, cols;
  const float* bias;      // forward only
};

PassShape pass_shape(const cgs_layer_desc& L, bool backward) {
  const LayerShape s = layer_shape(L);
  PassShape p;
  p.ih = backward ? s.hout : L.hin;
  p.iw = backward ? s.wout : L.win;
  p.oh = backward ? L.hin : s.hout;
  p.ow = backward ? L.win : s.wout;
  if (L.type == CGS_LAYER_FC) p.ih = p.iw = p.oh = p.ow = 1;
  p.kch = backward ? L.cout : L.cin;
  p.nch = backward ? L.cin : L.cout;
  p.strided = (L.type == CGS_LAYER_CONV && !backward) || (L.type == CGS_LAYER_DECONV && backward);
  const bool conv = L.type == CGS_LAYER_CONV;
  p.pad_y = L.type == CGS_LAYER_FC ? 0 : same_pad_before(conv ? L.hin : s.hout, L.k);
  p.pad_x = L.type == CGS_LAYER_FC ? 0 : same_pad_before(conv ? L.win : s.wout, L.k);
  p.w = backward ? L.w_bwd : L.w_fwd;
  p.rows = backward ? L.rows_bwd : L.rows_fwd;
  p.cols = backward ? L.kcols_bwd : L.kcols_fwd;
  p.bias = backward ? nullptr : L.bias;
  return p;
}

int check_layer(const cgs_layer_desc& L) {
  if (L.type == CGS_LAYER_FC) {
    if (L.cin % 32) return set_error(CGS_ERR_UNSUPPORTED, "fc input size %d must be a multiple of 32", L.cin);
    return CGS_OK;
  }
  if (L.k < 2 || L.k > 5) return set_error(CGS_ERR_UNSUPPORTED, "kernel size %d unsupported (2..5)", L.k);
  if ((L.hin & 1) && L.type == CGS_LAYER_CONV)
    return set_error(CGS_ERR_UNSUPPORTED, "odd conv input size %d unsupported", L.hin);
  const bool in_ok = (L.cin % 32 == 0) || L.cin <= 4;
  const bool out_ok = (L.cout % 32 == 0) || L.cout <= 4;
  if (!in_ok || !out_ok)
    return set_error(CGS_ERR_UNSUPPORTED, "channels (%d -> %d) must be <= 4 or multiples of 32", L.cin, L.cout);
  // the transposed-type pass gathers 32-channel blocks of its input
  if (L.type == CGS_LAYER_DECONV && L.cin % 32) return set_error(CGS_ERR_UNSUPPORTED, "deconv cin %d", L.cin);
  if (L.type == CGS_LAYER_CONV && L.cout % 32) return set_error(CGS_ERR_UNSUPPORTED, "conv cout %d", L.cout);
  return CGS_OK;
}

// Strided-type pass ("F"): out pixel (j,i) reads in pixels (2j+ky-p, 2i+kx-p); K order (ky,kx,c).
void fill_strided(ConvGemmParams& p, int k, int pad_y, int pad_x, int cin_k) {
  p.nclasses = 1;
  GemmClass& g = p.cls[0];
  g.k0 = 0;
  g.oy0 = g.ox0 = 0;
  g.ntaps = k * k;
  g.nkx = k;
  for (int ky = 0; ky < k; ++ky)
    for (int kx = 0; kx < k; ++kx) {
      g.dy[ky * k + kx] = (signed char)(ky - pad_y);
      g.dx[ky * k + kx] = (signed char)(kx - pad_x);
    }
  if (cin_k % 32 == 0) {
    p.cblocks = cin_k / 32;
    g.nkb = g.ntaps * p.cblocks;
  } else {
    p.cblocks = 0;                          // pixel mode: 8 taps x 4 channels per K block
    g.nkb = (g.ntaps + 7) / 8;
  }
  p.S = 2;
  p.os = 1;
}

// Transposed-type pass ("T"): output pixel (2j+py, 2i+px) reads in pixels (j+dy, i+dx),
// dy = (py + p - ky)/2 over the ky with matching parity; K order (class, tap, c).  Classes are emitted
// heaviest first so the persistent tile loop tails off on the short ones.
void fill_transposed(ConvGemmParams& p, int k, int pad_y, int pad_x, int cin_k) {
  p.nclasses = 4;
  p.cblocks = cin_k / 32;
  p.S = 1;
  p.os = 2;
  int k0 = 0;
  int ci = 0;
  // order parities by tap count (descending)
  int py_order[2] = {0, 1}, px_order[2] = {0, 1};
  auto ntap = [&](int par, int pad) { int n = 0; for (int kk = 0; kk < k; ++kk) if (((par + pad - kk) & 1) == 0) ++n; return n; };
  if (ntap(1, pad_y) > ntap(0, pad_y)) { py_order[0] = 1; py_order[1] = 0; }
  if (ntap(1, pad_x) > ntap(0, pad_x)) { px_order[0] = 1; px_order[1] = 0; }
  // CANONICAL SHIFT ORDER shared by all classes: a class's taps are enumerated in the order of their input shifts
  // (dy, dx), shifts used by more classes first (ties: dy descending, dx descending).  The class-fused tcgen05 tiles
  // (conv_gemm.cu) walk the shifts in this same order and may merge the classes of a shift into one wide MMA, so every
  // class accumulates its taps in the same order fused or not -- results never depend on the tile choice.
  auto has_tap = [&](int par, int pad, int d) { const int kk = par + pad - 2 * d; return kk >= 0 && kk < k; };
  struct Shift { int dy, dx, users; };
  Shift sh[64];
  int nsh = 0;
  for (int dy = 2; dy >= -2; --dy)
    for (int dx = 2; dx >= -2; --dx) {
      int users = 0;
      for (int py = 0; py < 2; ++py)
        for (int px = 0; px < 2; ++px)
          if (has_tap(py, pad_y, dy) && has_tap(px, pad_x, dx)) ++users;
      if (users) sh[nsh++] = Shift{dy, dx, users};
    }
  for (int a = 1; a < nsh; ++a)                       // stable insertion sort by users, descending
    for (int b = a; b > 0 && sh[b].users > sh[b - 1].users; --b) { const Shift t = sh[b]; sh[b] = sh[b - 1]; sh[b - 1] = t; }
  for (int a = 0; a < 2; ++a)
    for (int b = 0; b < 2; ++b) {
      const int py = py_order[a], px = px_order[b];
      GemmClass& g = p.cls[ci++];
      g.k0 = k0;
      g.oy0 = py;
      g.ox0 = px;
      int t = 0;
      for (int si = 0; si < nsh; ++si) {
        if (!has_tap(py, pad_y, sh[si].dy) || !has_tap(px, pad_x, sh[si].dx)) continue;
        g.dy[t] = (signed char)sh[si].dy;
        g.dx[t] = (signed char)sh[si].dx;
        ++t;
      }
      g.ntaps = t;
      g.nkx = ntap(px, pad_x);
      g.nkb = t * p.cblocks;
      k0 += t * cin_k;
    }
}

}  // namespace

// Gathered-GEMM parameters of one layer pass (forward: x -> y; data-gradient: dy -> dx); the epilogue is the caller's.
int make_pass_params(const cgs_layer_desc& L, bool backward, int64_t B, const float* in, float* out, ConvGemmParams& p) {
  if (int rc = check_layer(L)) return rc;
  if (L.type == CGS_LAYER_FC && backward && L.cout % 32)
    return set_error(CGS_ERR_UNSUPPORTED, "fc output size %d must be a multiple of 32", L.cout);
  std::memset(&p, 0, sizeof(p));
  const PassShape sh = pass_shape(L, backward);
  p.in = in;
  p.out = out;
  p.N = sh.nch;
  p.ON = cstride(sh.nch);
  p.OH = sh.oh;
  p.OW = sh.ow;
  p.IH = sh.ih;
  p.IW = sh.iw;
  p.Cs = cstride(sh.kch);
  if (L.type == CGS_LAYER_FC) {
    p.nclasses = 1;
    p.cls[0].ntaps = 1;
    p.cls[0].nkx = 1;
    p.cblocks = sh.kch / 32;
    p.cls[0].nkb = p.cblocks;
    p.S = 1;
    p.os = 1;
    p.MH = p.MW = 1;
  } else if (sh.strided) {
    fill_strided(p, L.k, sh.pad_y, sh.pad_x, cstride(sh.kch));
    p.MH = sh.oh;
    p.MW = sh.ow;
  } else {
    fill_transposed(p, L.k, sh.pad_y, sh.pad_x, sh.kch);
    p.MH = sh.ih;
    p.MW = sh.iw;
  }
  p.M = (int)(B * p.MH * p.MW);
  return CGS_OK;
}


// ---------------------------------------------------------------------------------------------
// Image-like tensors (<= 4 channels: the generated image and its gradient) live in a PITCHED layout inside the
// chain: [B][H][W + 8][4] with pixel x stored at column x + 2 and zero columns around it.  That lets the strided
// passes over them ("window" lowering below) fetch a whole K block with one TMA box and makes horizontal padding
// free; vertical padding is TMA out-of-bounds zero fill.  The public API stays dense: [B][H][W][4].
// ---------------------------------------------------------------------------------------------
constexpr int IMG_XOFF = 2;
inline int img_pitch(int w) { return w + 8; }
// layout of an image-like tensor handed to / produced by a pass
enum : int { IMG_PITCHED = 0,   // [B][H][W + 8][4] (inside the chain, mma.sync edge kernels / general lowerings)
             IMG_DENSE = 1,     // [B][H][W][4]     (single-layer entry points)
             IMG_S2D = 2 };     // [B][H/2][W/2][16] space-to-depth (inside the chain, tcgen05 edge kernels: edge_tc.cu)
inline size_t tensor_elems(int h, int w, int c) {        // per-sample elements of an activation inside the chain
  return c <= 4 ? (size_t)h * img_pitch(w) * 4 : (size_t)h * w * cstride(c);
}

// Window lowering: strided-type passes whose INPUT is image-like (first conv forward, last deconv data-gradient).
bool use_window(const cgs_layer_desc& L, bool backward) {
  return (L.type == CGS_LAYER_CONV && !backward && L.cin <= 4) || (L.type == CGS_LAYER_DECONV && backward && L.cout <= 4);
}
inline int window_kcols(const cgs_layer_desc& L) { return L.k * 32; }

// in = pitched image-like tensor; K block ky = 8 stored pixels x 4 channels starting at (2j + ky - pad_y, 2i + x0)
int make_window_params(const cgs_layer_desc& L, bool backward, int64_t B, const float* in, float* out,
                       ConvGemmParams& p) {
  if (int rc = check_layer(L)) return rc;
  if (L.k > 8) return set_error(CGS_ERR_UNSUPPORTED, "window lowering needs k <= 8");
  std::memset(&p, 0, sizeof(p));
  const PassShape sh = pass_shape(L, backward);      // image-like input, output grid = M-space
  if (sh.pad_x > IMG_XOFF) return set_error(CGS_ERR_UNSUPPORTED, "horizontal padding %d exceeds the image margin", sh.pad_x);
  p.in = in;
  p.out = out;
  p.N = sh.nch;
  p.ON = cstride(p.N);
  p.OH = sh.oh; p.OW = sh.ow;
  p.IH = sh.ih; p.IW = sh.iw;
  p.Cs = 4;
  p.cblocks = 1;
  p.MH = sh.oh; p.MW = sh.ow;
  p.S = 2; p.os = 1;
  p.nclasses = 1;
  GemmClass& g = p.cls[0];
  g.k0 = 0; g.oy0 = g.ox0 = 0;
  g.ntaps = L.k; g.nkx = 1; g.nkb = L.k;
  for (int ky = 0; ky < L.k; ++ky) { g.dy[ky] = (signed char)(ky - sh.pad_y); g.dx[ky] = 0; }
  p.window = 1;
  p.win_k = L.k;
  p.win_x0 = IMG_XOFF - sh.pad_x;
  p.in_pitch_px = img_pitch(sh.iw);
  p.M = (int)(B * p.MH * p.MW);
  return CGS_OK;
}

// dense [B][H][W][4]  <->  pitched [B][H][W+8][4] (test entry points and API copies only)
__global__ void __launch_bounds__(256) pad_image_kernel(const float4* __restrict__ src, float4* __restrict__ dst, int H,
                                                        int W, long long rows) {
  const int P = W + 8;
  for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < rows * P;
       idx += (long long)gridDim.x * blockDim.x) {
    const int c = (int)(idx % P);
    const long long r = idx / P;
    const int x = c - IMG_XOFF;
    dst[idx] = (x >= 0 && x < W) ? src[r * W + x] : make_float4(0.f, 0.f, 0.f, 0.f);
  }
}
int pad_image(const float* dense, float* pitched, int64_t B, int H, int W, cudaStream_t st) {
  const long long rows = (long long)B * H;
  long long blocks = (rows * (W + 8) + 255) / 256;
  if (blocks > 148 * 16) blocks = 148 * 16;
  pad_image_kernel<<<(int)blocks, 256, 0, st>>>((const float4*)dense, (float4*)pitched, H, W, rows); count_launch();
  return check_launch("pad_image_kernel");
}
int unpad_image(const float* pitched, float* dense, int64_t B, int H, int W, cudaStream_t st) {
  cudaError_t e = cudaMemcpy2DAsync(dense, (size_t)W * 16, pitched + IMG_XOFF * 4, (size_t)img_pitch(W) * 16, (size_t)W * 16,
                                    (size_t)B * H, cudaMemcpyDeviceToDevice, st);
  if (e != cudaSuccess) return set_error(CGS_ERR_CUDA, "cudaMemcpy2DAsync: %s", cudaGetErrorString(e));
  return CGS_OK;
}

// ---------------------------------------------------------------------------------------------
// Scatter formulation for transposed-type passes with <= 4 output channels (deconv -> image, conv1 data-gradient).
// The gather form would re-read every input pixel k^2/4 * 4 times for a 1..3-wide output; instead
//   stage 1  col[b,iy,ix,(ky,kx,c)] = sum_ci in[b,iy,ix,ci] * W[(ky,kx,c)][ci]     one GEMM, input read once
//   stage 2  out[b,y,x,c] = epi( sum_{(ky,kx): y = 2 iy + ky - p, x = 2 ix + kx - p} col[b,iy,ix,(ky,kx,c)] )
// Same MACs as the true-tap count; stage 2 is a small memory-bound kernel with the fused epilogue.
// ---------------------------------------------------------------------------------------------
bool use_scatter(const cgs_layer_desc& L, bool backward) {
  return (L.type == CGS_LAYER_DECONV && !backward && L.cout <= 4) || (L.type == CGS_LAYER_CONV && backward && L.cin <= 4);
}
inline int scatter_cols(const cgs_layer_desc& L) { return L.k * L.k * 4; }      // col row pitch (floats)

// Split-K for the forward pass of a long-K fc layer (d_fc3: 6272 -> 1024): at batch 1024 there are only 8 x 4 tiles of
// 128 x 256, and a CTA pays one pipeline hand-shake per K block whatever the tile width, so narrow tiles over the full
// K (128 tiles of 128 x 64, 98 K blocks each) run at a third of the wide-tile rate.  Instead: 128 x 256 tiles over a
// quarter of K each (the split is a "class" of the gathered GEMM: own K range, own output row), FP32 partial sums in
// the pass scratch buffer, and a small kernel that adds the four partials in a fixed order and applies the epilogue.
constexpr int kFcSplit = 4;
inline int env_int(const char* name, int dflt) { const char* e = getenv(name); return e ? atoi(e) : dflt; }
inline int fc_split(const cgs_layer_desc& L, bool backward) {
  static const int S = env_int("CGS_FC_SPLIT", kFcSplit);      // developer knob
  return (L.type == CGS_LAYER_FC && !backward && L.cin >= 4096 && L.cin % (32 * S) == 0) ? S : 1;
}

inline bool use_fc_split(const cgs_layer_desc& L, bool backward, int64_t B, int math, const float* scratch) {
  return fc_split(L, backward) > 1 && math == CGS_MATH_TF32_TENSOR && scratch && !(debug_flags() & CGS_DEBUG_NO_FC_SPLIT) &&
         ((B + 127) / 128) * ((L.cout + 255) / 256) * fc_split(L, backward) <= 2 * 148;
}

size_t scatter_col_elems(const cgs_layer_desc& L, bool backward) {     // per-sample elements of the pass scratch buffer
  if (fc_split(L, backward) > 1) return (size_t)fc_split(L, backward) * cstride(L.cout);
  if (!use_scatter(L, backward)) return 0;
  const PassShape sh = pass_shape(L, backward);
  return (size_t)sh.ih * sh.iw * scatter_cols(L);          // stage-1 rows (input pixels) per sample
}

// stage 1 as a 1-tap "fc over pixels": rows = B * pixels, K = big channel count, N = k*k*4
int make_scatter_gemm_params(const cgs_layer_desc& L, bool backward, int64_t B, const float* in, float* col,
                             ConvGemmParams& p) {
  if (int rc = check_layer(L)) return rc;
  std::memset(&p, 0, sizeof(p));
  const PassShape sh = pass_shape(L, backward);
  const int kch = sh.kch;                                      // reduced (big) channel count
  const int64_t pixels = (int64_t)sh.ih * sh.iw;
  p.in = in;
  p.out = col;
  p.ep = Epilogue(EPI_RAW, ACT_NONE);
  p.N = scatter_cols(L);
  p.ON = scatter_cols(L);
  p.OH = p.OW = 1;
  p.IH = p.IW = 1;
  p.Cs = kch;
  p.nclasses = 1;
  p.cls[0].ntaps = 1;
  p.cls[0].nkx = 1;
  p.cblocks = kch / 32;
  p.cls[0].nkb = p.cblocks;
  p.S = 1;
  p.os = 1;
  p.MH = p.MW = 1;
  if (B * pixels >= (1ll << 31) / p.ON) return set_error(CGS_ERR_UNSUPPORTED, "batch too large for 32-bit indexing; split the batch");
  p.M = (int)(B * pixels);
  return CGS_OK;
}

struct Col2imParams {
  const float* col;
  float* out;
  Epilogue ep;
  int IH, IW, OH, OW, k, pad_y, pad_x, pitch;
  int out_pitch, out_xoff;   // row pitch (pixels) and first data column of out / aux (dense: OW, 0)
  long long pixels;          // B * OH * out_pitch (pad columns are written as zeros)
  const int* live;           // early exit: images still in the batch (null = all)
};

__global__ void __launch_bounds__(256) col2im_kernel(const Col2imParams p) {
  long long pixels = p.pixels;
  if (p.live) {
    const long long per_img = (long long)p.OH * p.out_pitch;
    pixels = (long long)live_images(p.live, (int)(p.pixels / per_img)) * per_img;
  }
  for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < pixels;
       idx += (long long)gridDim.x * blockDim.x) {
    const int xc = (int)(idx % p.out_pitch);
    const long long t = idx / p.out_pitch;
    const int y = (int)(t % p.OH);
    const long long b = t / p.OH;
    const int x = xc - p.out_xoff;
    if (x < 0 || x >= p.OW) {                       // margin of the pitched layout
      *reinterpret_cast<float4*>(p.out + idx * 4) = make_float4(0.f, 0.f, 0.f, 0.f);
      continue;
    }
    float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int ky = 0; ky < p.k; ++ky) {
      const int ty = y + p.pad_y - ky;
      if (ty < 0 || (ty & 1)) continue;
      const int iy = ty >> 1;
      if (iy >= p.IH) continue;
      for (int kx = 0; kx < p.k; ++kx) {
        const int tx = x + p.pad_x - kx;
        if (tx < 0 || (tx & 1)) continue;
        const int ix = tx >> 1;
        if (ix >= p.IW) continue;
        const float4 v = __ldg(reinterpret_cast<const float4*>(
            p.col + ((b * p.IH + iy) * p.IW + ix) * p.pitch + (ky * p.k + kx) * 4));
        a.x += v.x; a.y += v.y; a.z += v.z; a.w += v.w;
      }
    }
    float4 x0 = make_float4(0.f, 0.f, 0.f, 0.f);     // no policy step in this lowering (run_pass)
    if (p.ep.mode == EPI_FWD && p.ep.bias) x0 = __ldg(reinterpret_cast<const float4*>(p.ep.bias));
    else if (p.ep.mode == EPI_BWD) x0 = __ldg(reinterpret_cast<const float4*>(p.ep.aux + idx * 4));
    *reinterpret_cast<float4*>(p.out + idx * 4) = epilogue4(p.ep, 0, a, x0, x0);
  }
}

int launch_gemm(const ConvGemmParams& p, const float* w, int rows, int cols, int math, cudaStream_t stream) {
  if (math == CGS_MATH_FP32_SIMT) return launch_conv_gemm_simt(p, w, rows, cols, stream);
  if (math == CGS_MATH_TF32_TENSOR) return launch_conv_gemm_tc(p, w, rows, cols, stream);
  return set_error(CGS_ERR_INVALID, "unknown math mode %d", math);
}

// out[b][n] = epi( part[b][0][n] + part[b][1][n] + ... ) in a fixed order; same epilogue code as the GEMM kernels
__global__ void __launch_bounds__(256) splitk_reduce_kernel(const __grid_constant__ ConvGemmParams p,
                                                            const float* __restrict__ part, int S, long long total4) {
  pdl_launch_dependents();
  pdl_wait();
  const int groups = p.ON / 4;
  if (p.live) total4 = (long long)live_images(p.live, (int)(total4 / groups)) * groups;
  for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total4;
       idx += (long long)gridDim.x * blockDim.x) {
    const long long b = idx / groups;
    const int ng = (int)(idx - b * groups);
    const int off = (int)(b * p.ON) + ng * 4;
    float4 a = __ldg(reinterpret_cast<const float4*>(part + (size_t)b * S * p.ON + ng * 4));
    for (int s = 1; s < S; ++s) {
      const float4 v = __ldg(reinterpret_cast<const float4*>(part + ((size_t)b * S + s) * p.ON + ng * 4));
      a.x += v.x; a.y += v.y; a.z += v.z; a.w += v.w;
    }
    float4 x0, x1;
    epilogue_operands4(p.ep, p.out, off, ng * 4, x0, x1);
    *reinterpret_cast<float4*>(p.out + off) = epilogue4(p.ep, off, a, x0, x1);
  }
}

int launch_splitk_reduce(const ConvGemmParams& pe, const float* part, int S, int64_t B, cudaStream_t st) {
  const long long total4 = (long long)B * (pe.ON / 4);
  long long blocks = (total4 + 255) / 256;
  if (blocks > 148 * 8) blocks = 148 * 8;
  cudaError_t le = launch_pdl(splitk_reduce_kernel, dim3((unsigned)blocks), dim3(256), (size_t)0, st, pe, part, S, total4);
  count_launch();
  if (le != cudaSuccess) return set_error(CGS_ERR_CUDA, "splitk_reduce_kernel: %s", cudaGetErrorString(le));
  return check_launch("splitk_reduce_kernel");
}

// The packed weights of a pass are in the layout cgs_pass_layout gives it.
int check_weights(const cgs_layer_desc& L, bool backward) {
  const PassShape sh = pass_shape(L, backward);
  if (!sh.w) return set_error(CGS_ERR_INVALID, "layer has no packed %s weights", backward ? "backward" : "forward");
  if (use_scatter(L, backward) && (sh.rows != scatter_cols(L) || sh.cols != sh.kch))
    return set_error(CGS_ERR_INVALID, "weights of this pass must be in scatter layout (%d x %d)", scatter_cols(L), sh.kch);
  if (use_window(L, backward) && (sh.rows != sh.nch || sh.cols != window_kcols(L)))
    return set_error(CGS_ERR_INVALID, "weights of this pass must be in window layout (%d columns)", window_kcols(L));
  return CGS_OK;
}

// Parameters of the fused image-edge kernels (edge_conv.cuh) for a scatter- (narrow) / window-lowered (wide) pass.
EdgeNarrowParams make_edge_narrow(const cgs_layer_desc& L, bool backward, int64_t B, const float* in, float* out,
                                  const Epilogue& e, const int* live, int img_mode, bool in16 = false) {
  const PassShape sh = pass_shape(L, backward);
  EdgeNarrowParams q;
  std::memset(&q, 0, sizeof(q));
  q.in = in; q.out = out; q.w = sh.w;
  q.B = (int)B; q.K = sh.kch; q.k = L.k; q.cimg = sh.nch;
  q.IH = sh.ih; q.IW = sh.iw; q.OH = sh.oh; q.OW = sh.ow;
  q.pad_y = sh.pad_y; q.pad_x = sh.pad_x;
  q.out_pitch = img_mode == IMG_PITCHED ? img_pitch(q.OW) : q.OW;
  q.out_xoff = img_mode == IMG_PITCHED ? IMG_XOFF : 0;
  q.s2d = img_mode == IMG_S2D;
  q.ep = e;
  q.ep.bias = sh.bias;
  q.live = live;
  q.in16 = in16;
  return q;
}

EdgeWideParams make_edge_wide(const cgs_layer_desc& L, bool backward, int64_t B, const float* in, float* out,
                              const Epilogue& e, const int* live) {
  const PassShape sh = pass_shape(L, backward);
  EdgeWideParams q;
  std::memset(&q, 0, sizeof(q));
  q.in = in; q.out = out; q.w = sh.w;
  q.IH = sh.ih; q.pitch = img_pitch(sh.iw); q.xoff = IMG_XOFF; q.OH = sh.oh; q.OW = sh.ow; q.ON = cstride(sh.nch); q.N = sh.nch;
  q.k = L.k; q.cimg = sh.kch;
  q.pad_y = sh.pad_y; q.pad_x = sh.pad_x;
  q.M = (long long)B * sh.oh * sh.ow;
  q.ep = e;
  q.ep.bias = sh.bias;
  q.live = live;
  return q;
}

// How an image-edge pass (scatter- or window-lowered: the generated image is its output or its input) runs.
enum EdgeRoute : int {
  ROUTE_GENERAL,   // scatter GEMM + col2im_kernel / window GEMM (no route for a wide pass over the s2d image)
  ROUTE_MMA,       // mma.sync: edge_narrow (column buffer) / edge_wide over the pitched image (edge_conv.cu)
  ROUTE_TC,        // tcgen05: edge_narrow_tc / edge_wide_tc, the wide pass over the s2d image (edge_tc.cu)
};

// The route of pass (L, backward) with epilogue e, its image-like tensor in layout img_mode, from the kernels' own
// predicates; the only code that reads CGS_DEBUG_EDGE_GENERAL and the math mode for these passes.
EdgeRoute edge_route(const cgs_layer_desc& L, bool backward, int math, const Epilogue& e, int img_mode) {
  if (math != CGS_MATH_TF32_TENSOR || (debug_flags() & CGS_DEBUG_EDGE_GENERAL)) return ROUTE_GENERAL;
  if (use_scatter(L, backward)) {
    const EdgeNarrowParams q = make_edge_narrow(L, backward, 0, nullptr, nullptr, e, nullptr, img_mode);
    return !edge_narrow_supported(q) ? ROUTE_GENERAL : edge_narrow_tc_supported(q) ? ROUTE_TC : ROUTE_MMA;
  }
  const EdgeWideParams q = make_edge_wide(L, backward, 0, nullptr, nullptr, e, nullptr);
  if (!use_window(L, backward) || !edge_wide_supported(q)) return ROUTE_GENERAL;
  if (img_mode != IMG_S2D) return ROUTE_MMA;
  return edge_wide_tc_supported(q, pass_shape(L, backward).iw) ? ROUTE_TC : ROUTE_GENERAL;
}

// The narrow pass of layer `ln` followed by the wide pass of layer `lw` on its output (forward: G's last deconv + D's
// first conv; backward: their data-gradients in the opposite order) as ONE kernel when both fit a one-image tile.
// Returns 1 when the pair was launched, 0 when the caller should run the two passes separately, < 0 on error.
int try_edge_pair(const cgs_layer_desc& ln, const cgs_layer_desc& lw, bool backward, int64_t B, const float* in,
                  float* mid, float* out, const Epilogue& en, const Epilogue& ew, const int* live, int store_mid, int math,
                  cudaStream_t st) {
  if ((debug_flags() & CGS_DEBUG_NO_EDGE_PAIR) || edge_route(ln, backward, math, en, IMG_PITCHED) == ROUTE_GENERAL ||
      edge_route(lw, backward, math, ew, IMG_PITCHED) == ROUTE_GENERAL)
    return 0;
  const EdgeNarrowParams qn = make_edge_narrow(ln, backward, B, in, mid, en, live, IMG_PITCHED);
  const EdgeWideParams qw = make_edge_wide(lw, backward, B, mid, out, ew, live);
  if (!edge_pair_supported(qn, qw)) return 0;
  if (int rc = check_weights(ln, backward)) return rc;
  if (int rc = check_weights(lw, backward)) return rc;
  if (int rc = launch_edge_pair(qn, qw, store_mid, st)) return rc;
  return 1;
}

// One layer pass (forward or data-gradient) with its fused epilogue `e` (its bias is the layer's, set here); an
// image-edge pass on its route, any other on the gathered GEMM.
// in16: `in` is FP16 (choose_operand_type) -- a GEMM pass runs on kind::f16 over the FP16 copy of its packed weights,
// the narrow image-edge pass takes the FP16 form of edge_narrow_tc
int run_pass(const cgs_layer_desc& L, bool backward, int64_t B, const float* in, float* out, const Epilogue& e,
             const int* live, float* col, int math, cudaStream_t st, int img_mode = IMG_PITCHED, bool defer_reduce = false,
             bool in16 = false) {
  if (int rc = check_weights(L, backward)) return rc;
  const PassShape sh = pass_shape(L, backward);
  const bool scatter = use_scatter(L, backward), window = use_window(L, backward);
  ConvGemmParams p;
  if (scatter) {
    if (!col) return set_error(CGS_ERR_WORKSPACE, "scatter pass needs a column workspace");
    if (e.mode == EPI_UPDATE) return set_error(CGS_ERR_UNSUPPORTED, "the policy step is not fused into a scatter-lowered pass");
  } else if (int rc = window ? make_window_params(L, backward, B, in, out, p) : make_pass_params(L, backward, B, in, out, p)) {
    return rc;
  }
  const EdgeRoute r = edge_route(L, backward, math, e, img_mode);
  if ((scatter || window) && img_mode == IMG_S2D && r != ROUTE_TC)
    return set_error(CGS_ERR_UNSUPPORTED, "s2d image layout needs the tcgen05 edge kernels");
  if (in16 && (scatter || window) && !(scatter && r == ROUTE_TC))
    return set_error(CGS_ERR_UNSUPPORTED, "an FP16 input of an image-edge pass needs the tcgen05 narrow kernel");
  if (r != ROUTE_GENERAL && scatter) {
    const EdgeNarrowParams q = make_edge_narrow(L, backward, B, in, out, e, live, img_mode, in16);
    return r == ROUTE_TC ? launch_edge_narrow_tc(q, st) : launch_edge_narrow(q, st);
  }
  if (r != ROUTE_GENERAL) {
    const EdgeWideParams q = make_edge_wide(L, backward, B, in, out, e, live);
    return r == ROUTE_TC ? launch_edge_wide_tc(q, (int)B, st) : launch_edge_wide(q, st);
  }
  Epilogue ep = e;
  ep.bias = sh.bias;
  if (scatter) {
    if (int rc = make_scatter_gemm_params(L, backward, B, in, col, p)) return rc;
    // (early exit: the 1-tap GEMM over pixels runs over the full batch -- its rows are pixels, not images; the
    //  col2im below stops at the live images)
    if (int rc = launch_gemm(p, sh.w, sh.rows, sh.cols, math, st)) return rc;
    Col2imParams c;
    c.col = col;
    c.out = out;
    c.ep = ep;
    c.k = L.k;
    c.pitch = scatter_cols(L);
    c.IH = sh.ih; c.IW = sh.iw; c.OH = sh.oh; c.OW = sh.ow;   // col over the input grid, out = 2x grid
    c.pad_y = sh.pad_y; c.pad_x = sh.pad_x;
    c.out_pitch = img_mode == IMG_PITCHED ? img_pitch(c.OW) : c.OW;
    c.out_xoff = img_mode == IMG_PITCHED ? IMG_XOFF : 0;
    c.pixels = (long long)B * c.OH * c.out_pitch;
    c.live = live;
    long long blocks = (c.pixels + 255) / 256;
    if (blocks > 148 * 16) blocks = 148 * 16;
    col2im_kernel<<<(int)blocks, 256, 0, st>>>(c); count_launch();
    return check_launch("col2im_kernel");
  }
  if (const int S = fc_split(L, backward); use_fc_split(L, backward, B, math, col)) {
    ConvGemmParams pe = p;                    // epilogue description of the real output
    p.out = col;
    pe.ep = ep;
    pe.live = live;
    p.ep = Epilogue(EPI_RAW, ACT_NONE);
    p.live = live;
    p.nclasses = S;
    p.cblocks = L.cin / 32 / S;
    for (int c = 0; c < S; ++c) {
      GemmClass& g = p.cls[c];
      std::memset(&g, 0, sizeof(g));
      g.k0 = c * p.cblocks * 32;
      g.nkb = p.cblocks;
      g.ntaps = 1;
      g.nkx = 1;
      g.oy0 = c;                              // partial sums of split c land in row (b * S + c) of the scratch buffer
      g.cb0 = c * p.cblocks;
    }
    p.OH = S;
    { static const int bn = env_int("CGS_FC_BN", 256); p.force_bn = bn; }
    if (int rc = launch_gemm(p, sh.w, sh.rows, sh.cols, math, st)) return rc;
    if (defer_reduce) return CGS_OK;          // the head kernel adds the partial sums itself (head_takes_partials)
    return launch_splitk_reduce(pe, col, S, B, st);
  }
  p.ep = ep;
  p.live = live;
  if (in16) {
    const __half* w16 = (const __half*)(backward ? L.w16_bwd : L.w16_fwd);
    if (!w16) return set_error(CGS_ERR_INVALID, "layer has no FP16 copy of its packed %s weights", backward ? "backward" : "forward");
    if (math != CGS_MATH_TF32_TENSOR || p.cblocks % 2) return set_error(CGS_ERR_UNSUPPORTED, "FP16 operands need 64-channel blocks");
    p.f16 = 1;                                // K counted in 64-channel atoms
    p.cblocks /= 2;
    for (int c = 0; c < p.nclasses; ++c) { p.cls[c].nkb /= 2; p.cls[c].cb0 /= 2; }
    return launch_conv_gemm_tc(p, w16, sh.rows, sh.cols, st);
  }
  return launch_gemm(p, sh.w, sh.rows, sh.cols, math, st);
}

// ---------------------------------------------------------------------------------------------
// Head kernel: final linear (-> 1 logit), BCE-with-ones gradient, selection, image keep.
//   logit_b = <feat_b, w> + bias                                   (nsgan/ops.py:81, GAN.py:68)
//   d pre_k = (sigmoid(logit_b) - 1) * w_k * act'(feat_bk)         (GAN.py:176-177, collaborator.py:30-31)
//   deterministic: update iff logit > best (strict)                (collaborator.py:79-83)
//   probabilistic: update iff prob_indices[b] == step_index        (collaborator.py:77)
// One CTA per sample; the dot product is reduced in a fixed order that depends only on K (never on B).
// ---------------------------------------------------------------------------------------------
struct HeadParams {
  const float* feat;    // [B, K]  output of the last hidden layer (post activation)
  const float* w;       // [K]
  const float* bias;    // [1] device scalar (folded)
  int K;
  float* dpre;          // [B, K] or nullptr (no backward wanted)
  const float* img;     // [B, img_elems] current image
  float* best_img;      // [B, img_elems]
  const float* feature; // [B, feat_elems] current feature (only if best_feature wanted)
  float* best_feature;
  int img_elems, feat_elems;   // dense per-sample sizes (what the caller sees)
  int img_h, img_w4, img_pitch4, img_xoff4;   // chain-side image layout in float4 units (pitched if <= 4 channels)
  int img_s2d;          // chain-side image is in the space-to-depth layout [H/2][W/2][16] (tcgen05 edge kernels)
  float* cur_logit;     // [B]
  float* best_logit;    // [B]
  float* best_step;     // [B]
  float* default_logit; // [B] or nullptr
  const int* prob_indices;
  int step;             // -1 = initial evaluation (collaborator.py:49-60), else loop index i
  int mode;
  unsigned char* done;  // early-exit flags [B] or nullptr
  const int* orig;      // compact row -> original sample index (early-exit compaction) or nullptr (identity)
  float* final_feature; // [B_orig, feat_elems]: state of a sample at the step it exits (early-exit) or nullptr
  float exit_logit;
  int round_out;        // round dpre to TF32 (RN): it feeds a kind::tf32 MMA
  int dpre16;           // dpre is FP16, scaled per sample by 2^gexp[b] (it feeds a kind::f16 MMA)
  int* gexp;            // [B] that exponent: |dl| * 2^gexp in [1, 2), 0 where dl == 0
  // split-K producer (fc_split): feat is not materialised; feat[b][k] = act(sum_s part[b][s][k] + bias[k])
  const float* part;    // [B][S][K] partial sums or nullptr
  int S;
  // the forward epilogue of the producer of feat (its activation; its bias when feat is given as partial sums)
  Epilogue feat_ep;
  const int* live;      // early exit: device-resident count of the rows still in the batch (null = gridDim.x)
};

// Input of the head for elements k..k+3 of sample b: the stored activation, or the split-K partial sums added in
// a fixed order with the fc layer's bias and activation applied (what splitk_reduce_kernel would have stored).
__device__ __forceinline__ float4 head_feat4(const HeadParams& p, const float* f, int b, int k) {
  if (!p.part) return *reinterpret_cast<const float4*>(f + k);
  const float* pr = p.part + (size_t)b * p.S * p.K + k;
  float4 a = __ldg(reinterpret_cast<const float4*>(pr));
  for (int s = 1; s < p.S; ++s) {
    const float4 v = __ldg(reinterpret_cast<const float4*>(pr + (size_t)s * p.K));
    a.x += v.x; a.y += v.y; a.z += v.z; a.w += v.w;
  }
  const float4 bb = p.feat_ep.bias ? __ldg(reinterpret_cast<const float4*>(p.feat_ep.bias + k)) : make_float4(0.f, 0.f, 0.f, 0.f);
  return epilogue4_t<EPI_FWD>(p.feat_ep, 0, a, bb, bb);
}

__global__ void __launch_bounds__(256) head_kernel(const HeadParams p) {
  __shared__ float red[8];
  __shared__ float s_logit;
  __shared__ int s_update;
  pdl_launch_dependents();
  pdl_wait();
  const int b = blockIdx.x;
  if (p.live && b >= *reinterpret_cast<const volatile int*>(p.live)) return;   // row left the batch (early exit)
  const int ob = p.orig ? p.orig[b] : b;           // where this sample's results live
  const float* f = p.feat + (size_t)b * p.K;
  float acc = 0.f;
  float4 a_first = make_float4(0.f, 0.f, 0.f, 0.f);   // this thread's first four inputs, reused by the gradient pass
  for (int k = threadIdx.x * 4; k < p.K; k += 256 * 4) {
    const float4 a = head_feat4(p, f, b, k);
    if (k < 256 * 4) a_first = a;
    const float4 ww = __ldg(reinterpret_cast<const float4*>(p.w + k));
    acc = fmaf(a.x, ww.x, acc);
    acc = fmaf(a.y, ww.y, acc);
    acc = fmaf(a.z, ww.z, acc);
    acc = fmaf(a.w, ww.w, acc);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    float t = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) t += red[i];
    const float logit = t + (p.bias ? __ldg(p.bias) : 0.f);
    s_logit = logit;
    p.cur_logit[b] = logit;
    int upd;
    if (p.step < 0) {
      upd = 1;
      p.best_logit[ob] = logit;
      p.best_step[ob] = 1.0f;                                  // collaborator.py:60 (sic)
      if (p.default_logit) p.default_logit[ob] = logit;        // collaborator.py:52
    } else {
      const bool frozen = p.done && p.done[b];
      if (p.mode == CGS_MODE_PROBABILISTIC) upd = (p.prob_indices[ob] == p.step);
      else upd = logit > p.best_logit[ob];
      if (frozen) upd = 0;
      if (upd) {
        p.best_logit[ob] = logit;
        p.best_step[ob] = (float)(p.step + 1);
      }
    }
    int exit_now = 0;
    if (p.done && !p.done[b] && logit >= p.exit_logit) {       // opt-in early exit (README.md:13)
      p.done[b] = 1;
      exit_now = 1;
    }
    s_update = upd | (exit_now << 1);
  }
  __syncthreads();
  const float logit = s_logit;
  if (p.dpre) {
    // d softplus(-l)/dl = sigmoid(l) - 1
    float dl = 1.f / (1.f + expf(-logit)) - 1.f;
    if (p.dpre16) {
      // The data-gradient chain is linear and homogeneous in dl per sample (masks and tanh' from the forward pass, no
      // bias), so a power of two set here and removed by the policy step changes no FP32 value.  dl is 0 or at least
      // 2^-24 in magnitude; scaled to [1, 2) it keeps the whole chain inside FP16's normal range (DESIGN §2).
      int e = 0;
      if (dl != 0.f) { (void)frexpf(dl, &e); e = 1 - e; }
      dl = ldexpf(dl, e);
      if (threadIdx.x == 0) p.gexp[b] = e;
    }
    float* d = p.dpre + (size_t)b * p.K;
    for (int k = threadIdx.x * 4; k < p.K; k += 256 * 4) {
      const float4 a = (k < 256 * 4) ? a_first : head_feat4(p, f, b, k);
      const float4 ww = __ldg(reinterpret_cast<const float4*>(p.w + k));
      float4 o = epilogue4_t<EPI_BWD>(p.feat_ep, 0, make_float4(dl * ww.x, dl * ww.y, dl * ww.z, dl * ww.w), a, a);
      if (p.dpre16) {
        *reinterpret_cast<uint2*>(reinterpret_cast<__half*>(p.dpre) + (size_t)b * p.K + k) = pack_half4(o);
        continue;
      }
      if (p.round_out) { o.x = tf32_rn(o.x); o.y = tf32_rn(o.y); o.z = tf32_rn(o.z); o.w = tf32_rn(o.w); }
      *reinterpret_cast<float4*>(d + k) = o;
    }
  }
  if (s_update & 1) {
    // chain-side image rows (possibly pitched) -> dense best_img
    float4* dst = reinterpret_cast<float4*>(p.best_img + (size_t)ob * p.img_elems);
    if (p.img_s2d) {
      // s2d pixel (y/2, x/2), sub-pixel (y & 1, x & 1) -> dense pixel (y, x); img_w4 = W here (one float4 per pixel)
      const float4* src = reinterpret_cast<const float4*>(p.img) + (size_t)b * p.img_h * p.img_w4;
      const int W = p.img_w4;
      for (int i = threadIdx.x; i < p.img_h * W; i += 256) {
        const int y = i / W, x = i - y * W;
        dst[i] = src[((size_t)(y >> 1) * (W >> 1) + (x >> 1)) * 4 + ((y & 1) * 2 + (x & 1))];
      }
    } else {
      const float4* src = reinterpret_cast<const float4*>(p.img) + (size_t)b * p.img_h * p.img_pitch4 + p.img_xoff4;
      for (int i = threadIdx.x; i < p.img_h * p.img_w4; i += 256) {
        const int y = i / p.img_w4;
        dst[i] = src[(size_t)y * p.img_pitch4 + (i - y * p.img_w4)];
      }
    }
    if (p.best_feature) {
      const float4* fs = reinterpret_cast<const float4*>(p.feature + (size_t)b * p.feat_elems);
      float4* fd = reinterpret_cast<float4*>(p.best_feature + (size_t)ob * p.feat_elems);
      for (int i = threadIdx.x; i < p.feat_elems / 4; i += 256) fd[i] = fs[i];
    }
  }
  if ((s_update & 2) && p.final_feature) {                    // the sample leaves the batch: keep its final state
    const float4* fs = reinterpret_cast<const float4*>(p.feature + (size_t)b * p.feat_elems);
    float4* fd = reinterpret_cast<float4*>(p.final_feature + (size_t)ob * p.feat_elems);
    for (int i = threadIdx.x; i < p.feat_elems / 4; i += 256) fd[i] = fs[i];
  }
}

// ---------------------------------------------------------------------------------------------
// Early exit (README.md:13; opt-in, the reference itself always runs K steps: collaborator.py:63-83), device side.
// After every fused policy step the rows D already classifies as real leave the batch: ONE single-CTA kernel turns the
// per-row exit flags into the ordered list of the rows that stay and their count (ballot + warp-sum scan), ONE kernel
// gathers feature / momentum / row-map rows through that list.  The count lives in device memory and every later
// launch of the step reads it (ConvGemmParams::live and friends), so there is no host synchronisation, the launch
// sequence is static and the whole K loop can be captured in a CUDA graph.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(1024) live_compact_kernel(unsigned char* __restrict__ done, const int* __restrict__ live_in,
                                                            int B, int* __restrict__ idx, int* __restrict__ live_out) {
  __shared__ int warp_sums[32];
  __shared__ int s_base;
  const int live = min(max(*live_in, 0), B);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (threadIdx.x == 0) s_base = 0;
  __syncthreads();
  for (int i0 = 0; i0 < B; i0 += 1024) {
    const int i = i0 + threadIdx.x;
    const bool keep = i < live && !done[i];
    if (i < B) done[i] = 0;                               // rows are renumbered: the flags start afresh
    const unsigned m = __ballot_sync(0xffffffffu, keep);
    if (lane == 0) warp_sums[warp] = __popc(m);
    __syncthreads();
    int before = s_base;
    for (int w2 = 0; w2 < warp; ++w2) before += warp_sums[w2];
    if (keep) idx[before + __popc(m & ((1u << lane) - 1u))] = i;
    __syncthreads();
    if (threadIdx.x == 0) {
      int t = s_base;
      for (int w2 = 0; w2 < 32; ++w2) t += warp_sums[w2];
      s_base = t;
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) *live_out = s_base;
}

// rows idx[0 .. *count) of (feature, momentum, row map) -> rows 0 .. *count of the partner buffers (ordered)
__global__ void __launch_bounds__(256) live_gather_kernel(const float4* __restrict__ feat_src, float4* __restrict__ feat_dst,
                                                          const float4* __restrict__ mom_src, float4* __restrict__ mom_dst,
                                                          const int* __restrict__ orig_src, int* __restrict__ orig_dst,
                                                          const int* __restrict__ idx, const int* __restrict__ count,
                                                          int elems4) {
  const int rows = *count;
  for (int r = blockIdx.x; r < rows; r += gridDim.x) {
    const int s = idx[r];
    const float4* fs = feat_src + (size_t)s * elems4;
    float4* fd = feat_dst + (size_t)r * elems4;
    for (int i = threadIdx.x; i < elems4; i += blockDim.x) fd[i] = fs[i];
    if (mom_src) {
      const float4* ms = mom_src + (size_t)s * elems4;
      float4* md = mom_dst + (size_t)r * elems4;
      for (int i = threadIdx.x; i < elems4; i += blockDim.x) md[i] = ms[i];
    }
    if (threadIdx.x == 0) orig_dst[r] = orig_src[s];
  }
}
// feature rows of the samples that never exited -> their slot in the caller's buffer
__global__ void scatter_active_kernel(const float4* __restrict__ feat, const int* __restrict__ orig,
                                      const unsigned char* __restrict__ done, const int* __restrict__ live,
                                      float4* __restrict__ out, int elems4) {
  const int b = blockIdx.x;
  if (b >= *live || done[b]) return;
  const float4* s = feat + (size_t)b * elems4;
  float4* d = out + (size_t)orig[b] * elems4;
  for (int i = threadIdx.x; i < elems4; i += blockDim.x) d[i] = s[i];
}
__global__ void iota_kernel(int* p, int n, int* live) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) p[i] = i;
  if (live && blockIdx.x == 0 && threadIdx.x == 0) *live = n;
}

// ---------------------------------------------------------------------------------------------
// Chain executor
// ---------------------------------------------------------------------------------------------
struct Chain {
  int n;                         // GEMM layers (G-tail + D without the 1-logit head)
  cgs_layer_desc layers[2 * CGS_MAX_LAYERS];
  size_t act_elems[2 * CGS_MAX_LAYERS + 1];   // per-sample elements of act[i] (act[0] = feature)
  int n_gtail;
  cgs_layer_desc head;
  size_t max_elems;
  size_t col_elems;              // per-sample elements of the scatter column buffer (0 if unused)
  int img_mode;                  // layout of the image-like tensors: IMG_S2D or IMG_PITCHED (choose_image_layout)
  int f16;                       // MMA operands of the GEMM layers are FP16 on kind::f16 (choose_operand_type)
  // batch-statistic BN after layer i's GEMM (D layers only; null = none); batch_bn: any layer has it
  const float* bn_gamma[2 * CGS_MAX_LAYERS];
  const float* bn_beta[2 * CGS_MAX_LAYERS];
  int batch_bn;
};

// G's last deconv / D's first conv: the passes that produce or read the image (edge kernels / general lowerings)
static bool edge_layer(const cgs_layer_desc& L) { return use_scatter(L, false) || use_window(L, false); }

// Every pass of every other layer can take FP16 operands: plain gathered GEMMs (no split-K) whose reduced channel
// count fills whole 64-channel atoms, with FP16 copies of both packed weight matrices in the descriptor.
static bool f16_capable(const Chain& c) {
  for (int i = 0; i < c.n; ++i) {
    const cgs_layer_desc& L = c.layers[i];
    if (edge_layer(L)) continue;
    if (!L.w16_fwd || !L.w16_bwd) return false;
    for (int bw = 0; bw < 2; ++bw)
      if (use_scatter(L, bw != 0) || use_window(L, bw != 0) || fc_split(L, bw != 0) > 1 || pass_shape(L, bw != 0).kch % 64)
        return false;
  }
  return true;
}

// In an FP16 chain every 64-channel tensor a pass reads is FP16, with two exceptions:
//  - the refined feature (layer 0's forward input) stays FP32, because momentum integrates steps below its last TF32
//    bit; layer 0's forward pass keeps kind::tf32 over it (the narrow edge kernel's TF32 form when layer 0 is G's last
//    deconv, as in the one-layer G tails);
//  - the generated image act[n_gtail] (returned to the caller) and its gradient stay FP32 in the s2d layout.
// So both image-edge kernels take FP16 on their 64-channel side, except the narrow forward pass of layer 0.
// fwd16(i): layer i's forward input act[i] is FP16.  bwd16(j): the tensor layer j's data-gradient pass reduces,
// d loss / d act[j + 1], is FP16 (and so is act[j + 1], the derivative operand of the pass that produces it).
static bool fwd16(const Chain& c, int i) { return c.f16 && i > 0 && i < c.n && i != c.n_gtail; }
static bool bwd16(const Chain& c, int j) { return c.f16 && j >= 0 && j < c.n && j + 1 != c.n_gtail; }

static int build_chain(const cgs_net_desc* gtail, const cgs_net_desc* d, const cgs_batchnorm_desc* bn, Chain& c) {
  if (!gtail || !d) return set_error(CGS_ERR_INVALID, "null network descriptor");
  if (gtail->n_layers < 1 || gtail->n_layers > CGS_MAX_LAYERS || d->n_layers < 2 || d->n_layers > CGS_MAX_LAYERS)
    return set_error(CGS_ERR_INVALID, "bad layer counts (%d, %d)", gtail->n_layers, d->n_layers);
  c.n = 0;
  c.f16 = 0;
  c.batch_bn = 0;
  for (int i = 0; i < 2 * CGS_MAX_LAYERS; ++i) c.bn_gamma[i] = c.bn_beta[i] = nullptr;
  for (int i = 0; i < gtail->n_layers; ++i) c.layers[c.n++] = gtail->layers[i];
  c.n_gtail = gtail->n_layers;
  for (int i = 0; i < d->n_layers - 1; ++i) c.layers[c.n++] = d->layers[i];
  c.head = d->layers[d->n_layers - 1];
  if (c.head.type != CGS_LAYER_FC || c.head.cout != 1)
    return set_error(CGS_ERR_UNSUPPORTED, "discriminator must end in a linear layer with one logit");
  const cgs_layer_desc& L0 = c.layers[0];
  if (L0.cin <= 4) return set_error(CGS_ERR_UNSUPPORTED, "the refined feature map must have >= 32 channels");
  c.act_elems[0] = (size_t)L0.hin * L0.win * cstride(L0.cin);
  c.max_elems = c.act_elems[0];
  c.col_elems = 0;
  for (int i = 0; i < c.n; ++i) {
    if (int rc = check_layer(c.layers[i])) return rc;
    for (int bw = 0; bw < 2; ++bw) {
      const size_t ce = scatter_col_elems(c.layers[i], bw != 0);
      if (ce > c.col_elems) c.col_elems = ce;
    }
    const LayerShape s = layer_shape(c.layers[i]);
    c.act_elems[i + 1] = tensor_elems(s.hout, s.wout, c.layers[i].cout);
    if (c.act_elems[i + 1] > c.max_elems) c.max_elems = c.act_elems[i + 1];
    if (i + 1 < c.n) {
      const cgs_layer_desc& Ln = c.layers[i + 1];
      const size_t expect = (Ln.type == CGS_LAYER_FC) ? (size_t)Ln.cin : tensor_elems(Ln.hin, Ln.win, Ln.cin);
      if (expect != c.act_elems[i + 1])
        return set_error(CGS_ERR_INVALID, "layer %d output (%zu) does not feed layer %d input (%zu)", i,
                         c.act_elems[i + 1], i + 1, expect);
    }
  }
  if ((size_t)c.head.cin != c.act_elems[c.n]) return set_error(CGS_ERR_INVALID, "head input size mismatch");
  if (c.head.cin % 4) return set_error(CGS_ERR_UNSUPPORTED, "head input size must be a multiple of 4");
  if (!bn) return CGS_OK;
  if (bn->n_layers != d->n_layers)
    return set_error(CGS_ERR_INVALID, "batchnorm descriptor has %d layers, the discriminator %d", bn->n_layers, d->n_layers);
  for (int j = 0; j < d->n_layers; ++j) {
    if (!bn->gamma[j]) continue;
    if (!bn->beta[j]) return set_error(CGS_ERR_INVALID, "batch BN of D layer %d has gamma but no beta", j);
    if (((uintptr_t)bn->gamma[j] | (uintptr_t)bn->beta[j]) & 15)
      return set_error(CGS_ERR_INVALID, "gamma / beta of D layer %d must be 16-byte aligned", j);
    if (j == d->n_layers - 1) return set_error(CGS_ERR_UNSUPPORTED, "batch BN on the 1-logit head is not built");
    const int i = c.n_gtail + j;
    if (edge_layer(c.layers[i])) return set_error(CGS_ERR_UNSUPPORTED, "batch BN on the image-edge layer %d of D is not built", j);
    if (c.layers[i].cout % 4) return set_error(CGS_ERR_UNSUPPORTED, "batch BN needs a multiple of 4 channels (%d)", c.layers[i].cout);
    c.bn_gamma[i] = bn->gamma[j];
    c.bn_beta[i] = bn->beta[j];
    c.batch_bn = 1;
  }
  return CGS_OK;
}

// Forward pass i.  TF32 path: activations that feed another MMA are rounded to TF32 (RN) where they are produced, so
// the tensor core's operand truncation is exact; the image (returned to the caller) and the head input stay FP32.
static Epilogue forward_epi(const Chain& c, int i, int math) {
  Epilogue e(EPI_FWD, c.layers[i].act);
  e.out16 = fwd16(c, i + 1);
  e.round_out = (math == CGS_MATH_TF32_TENSOR) && !e.out16 && (i != c.n_gtail - 1) && (i != c.n - 1);
  return e;
}

// Epilogue of data-gradient pass i: times the derivative of the activation that produced its input x, the policy
// step `upd` or nothing (i = 0).
static Epilogue backward_epi(const Chain& c, int i, int math, const Epilogue* upd, const float* x) {
  if (i == 0) return upd ? *upd : Epilogue(EPI_RAW, ACT_NONE);
  Epilogue e(EPI_BWD, c.layers[i - 1].act);
  e.aux = x;
  e.out16 = bwd16(c, i - 1);
  // a batch-BN layer's gradient feeds bn_backward, not an MMA: it is rounded after that instead
  e.round_out = (math == CGS_MATH_TF32_TENSOR) && !e.out16 && !c.bn_gamma[i - 1];
  return e;
}

// The image-like tensors of the chain are in the s2d layout exactly when all four image-edge passes (G's last deconv
// and D's first conv, forward and data-gradient, with the epilogues of a refinement step) take the tcgen05 route over
// it; pitched otherwise.
static void choose_image_layout(Chain& c, int math) {
  Epilogue upd(EPI_UPDATE, ACT_NONE);
  c.img_mode = IMG_S2D;
  for (int i = c.n_gtail - 1; i <= c.n_gtail; ++i)
    if (edge_route(c.layers[i], false, math, forward_epi(c, i, math), IMG_S2D) != ROUTE_TC ||
        edge_route(c.layers[i], true, math, backward_epi(c, i, math, &upd, nullptr), IMG_S2D) != ROUTE_TC)
      c.img_mode = IMG_PITCHED;
}

// FP16 operands (half the bytes of the TF32-rounded FP32 ones, same 10-bit mantissa; kind::f16 at twice the kind::tf32
// rate) for the DCGAN-shaped chains: s2d image layout, every other layer a plain tcgen05 GEMM with 64-channel atoms.
// CGS_DEBUG_TF32_OPERANDS keeps the TF32 path for A/B comparisons; the gather-mode knob has no FP16 form.  A batch-BN
// chain keeps TF32 operands: the per-sample gradient scale relies on the data-gradient chain being linear per sample,
// and the BN backward mixes the samples.
static void choose_operand_type(Chain& c, int math) {
  c.f16 = math == CGS_MATH_TF32_TENSOR && c.img_mode == IMG_S2D && f16_capable(c) && !c.batch_bn &&
          !(debug_flags() & (CGS_DEBUG_TF32_OPERANDS | CGS_DEBUG_GATHER_A));
}

static inline size_t align256(size_t x) { return (x + 255) & ~size_t(255); }

struct Workspace {
  float* act[2 * CGS_MAX_LAYERS + 1];
  float* g[2];
  float* mom;
  float* col;
  float* cur_logit;
  unsigned char* done;
  // early-exit compaction: ping-pong feature / momentum buffers, row maps, index list, the two live-row counters
  float* feat2;
  float* feat3;
  float* mom2;
  int* orig[2];
  int* idx;
  int* count;            // count[0], count[1]: live rows, ping-pong per step
  int* gexp;             // FP16 operand chains: per-sample gradient scale (head_kernel)
  // batch-BN layers: their pre-BN output y (act[i + 1]'s layout), per-channel state, the FP64 partial sums
  float* pre[2 * CGS_MAX_LAYERS];
  float* bn_stat[2 * CGS_MAX_LAYERS];
  double* bn_part;
  size_t total;
};

// rows of the [rows, C] tensor a batch-BN layer normalises over
static long long bn_rows(const Chain& c, int i, int64_t B) { return (long long)B * (long long)(c.act_elems[i + 1] / cstride(c.layers[i].cout)); }

// act[0] is the caller's feature buffer; everything else is carved out of the workspace.
static void carve(const Chain& c, int64_t B, void* base, Workspace& w) {
  size_t off = 0;
  auto take = [&](size_t bytes) { void* p = base ? (char*)base + off : nullptr; off += align256(bytes); return p; };
  w.act[0] = nullptr;
  for (int i = 1; i <= c.n; ++i) w.act[i] = (float*)take((size_t)B * c.act_elems[i] * 4);
  w.g[0] = (float*)take((size_t)B * c.max_elems * 4);
  w.g[1] = (float*)take((size_t)B * c.max_elems * 4);
  w.mom = (float*)take((size_t)B * c.act_elems[0] * 4);
  w.col = c.col_elems ? (float*)take((size_t)B * c.col_elems * 4) : nullptr;
  w.cur_logit = (float*)take((size_t)B * 4);
  w.done = (unsigned char*)take((size_t)B);
  w.feat2 = (float*)take((size_t)B * c.act_elems[0] * 4);
  w.feat3 = (float*)take((size_t)B * c.act_elems[0] * 4);
  w.mom2 = (float*)take((size_t)B * c.act_elems[0] * 4);
  w.orig[0] = (int*)take((size_t)B * 4);
  w.orig[1] = (int*)take((size_t)B * 4);
  w.idx = (int*)take((size_t)B * 4);
  w.count = (int*)take(16);
  w.gexp = (int*)take((size_t)B * 4);
  size_t part_bytes = 0;
  for (int i = 0; i < c.n; ++i) {
    w.pre[i] = nullptr;
    w.bn_stat[i] = nullptr;
    if (!c.bn_gamma[i]) continue;
    w.pre[i] = (float*)take((size_t)B * c.act_elems[i + 1] * 4);
    w.bn_stat[i] = (float*)take((size_t)5 * c.layers[i].cout * 4);
    const size_t pb = bn_partial_bytes(bn_rows(c, i, B), c.layers[i].cout);
    if (pb > part_bytes) part_bytes = pb;
  }
  w.bn_part = part_bytes ? (double*)take(part_bytes) : nullptr;
  w.total = off;
}

// The last hidden layer runs split-K and nothing but the head reads its output: the head kernel then adds the partial
// sums itself and the activation is never written (CGS_DEBUG_NO_HEAD_PARTIALS keeps the separate reduce kernel).
// (A batch-BN layer's output needs the statistics of the whole sum first.)
static bool head_takes_partials(const Chain& c, const Workspace& w, int64_t B, int math) {
  const cgs_layer_desc& L = c.layers[c.n - 1];
  return use_fc_split(L, false, B, math, w.col) && !(debug_flags() & CGS_DEBUG_NO_HEAD_PARTIALS) &&
         cstride(L.cout) == c.head.cin && !c.bn_gamma[c.n - 1];
}

static BnLayer bn_layer(const Chain& c, const Workspace& w, int i, int64_t B) {
  return BnLayer{c.bn_gamma[i], c.bn_beta[i], bn_rows(c, i, B), c.layers[i].cout, w.bn_stat[i]};
}

static int run_forward(const Chain& c, const Workspace& w, int64_t B, int math, cudaStream_t st,
                       const int* live = nullptr) {
  auto epi = [&](int i) { return forward_epi(c, i, math); };
  for (int i = 0; i < c.n; ++i) {
    if (i == c.n_gtail - 1 && i + 1 < c.n && c.img_mode == IMG_PITCHED) {
      // generator's last deconv + discriminator's first conv on the same image: one kernel when the shapes allow
      const int rc = try_edge_pair(c.layers[i], c.layers[i + 1], false, B, w.act[i], w.act[i + 1], w.act[i + 2], epi(i),
                                   epi(i + 1), live, 1, math, st);
      if (rc < 0) return rc;
      if (rc == 1) { ++i; continue; }
    }
    const bool defer = (i == c.n - 1) && head_takes_partials(c, w, B, math);
    if (c.bn_gamma[i]) {
      // batch BN: the GEMM stores y = conv(x) + b unrounded, the BN kernels normalise it into act[i + 1]
      if (int rc = run_pass(c.layers[i], false, B, w.act[i], w.pre[i], Epilogue(EPI_FWD, ACT_NONE), live, w.col, math, st,
                            c.img_mode))
        return rc;
      if (int rc = bn_forward(bn_layer(c, w, i, B), w.pre[i], w.act[i + 1], epi(i), w.bn_part, st)) return rc;
      continue;
    }
    if (int rc = run_pass(c.layers[i], false, B, w.act[i], w.act[i + 1], epi(i), live, w.col, math, st, c.img_mode, defer,
                          fwd16(c, i)))
      return rc;
  }
  return CGS_OK;
}

// Backward from dpre[c.n-1] (already in w.g[0]) down to the feature.  `upd` != null is the policy step fused into
// the last pass's epilogue; otherwise the raw gradient is written to grad_out.
static int run_backward(const Chain& c, const Workspace& w, int64_t B, int math, const Epilogue* upd,
                        float* grad_out, cudaStream_t st, const int* live = nullptr) {
  auto epi = [&](int i) { return backward_epi(c, i, math, upd, w.act[i]); };
  int cur = 0;
  for (int i = c.n - 1; i >= 0; --i) {
    float* dst = (i == 0) ? (upd ? w.act[0] : grad_out) : w.g[cur ^ 1];
    if (c.bn_gamma[i]) {
      // g[cur] is d loss / d (the BN output before the activation): through the batch statistics to d loss / d y, in place
      if (int rc = bn_backward(bn_layer(c, w, i, B), w.pre[i], w.g[cur], w.g[cur], math == CGS_MATH_TF32_TENSOR, w.bn_part, st))
        return rc;
    }
    if (i == c.n_gtail && i >= 1 && c.img_mode == IMG_PITCHED) {
      // data-gradients of D's first conv and G's last deconv: one kernel, the image gradient never leaves the SM
      float* dst2 = (i - 1 == 0) ? (upd ? w.act[0] : grad_out) : w.g[cur ^ 1];
      // the intermediate (image gradient) buffer is only described, never written: any valid pointer of that size
      const int rc = try_edge_pair(c.layers[i], c.layers[i - 1], true, B, w.g[cur], w.g[cur ^ 1], dst2, epi(i), epi(i - 1),
                                   live, 0, math, st);
      if (rc < 0) return rc;
      if (rc == 1) { --i; cur ^= 1; continue; }
    }
    Epilogue e = epi(i);
    if (i == 0 && c.f16) e.gexp = w.gexp;    // the policy step / raw gradient removes the head's per-sample scale
    if (int rc = run_pass(c.layers[i], true, B, w.g[cur], dst, e, live, w.col, math, st, c.img_mode, false, bwd16(c, i)))
      return rc;
    cur ^= 1;
  }
  return CGS_OK;
}

}  // namespace cgs

using namespace cgs;

// Largest batch one call can take (rows are indexed with 32 bits); larger batches are refined in chunks by the caller.
extern "C" int64_t cgs_refine_max_batch(const cgs_net_desc* gtail, const cgs_net_desc* d) {
  Chain c;
  if (int rc = build_chain(gtail, d, nullptr, c)) return rc;
  const size_t per = c.max_elems > c.col_elems ? c.max_elems : c.col_elems;
  return (int64_t)(((1ull << 31) - 1) / per) - 1;
}

extern "C" size_t cgs_refine_workspace_bytes_bn(const cgs_net_desc* gtail, const cgs_net_desc* d,
                                                 const cgs_batchnorm_desc* bn, int64_t B) {
  Chain c;
  if (build_chain(gtail, d, bn, c) != CGS_OK || B < 0) return 0;
  Workspace w;
  carve(c, B, nullptr, w);
  return w.total + 256;
}

extern "C" size_t cgs_refine_workspace_bytes(const cgs_net_desc* gtail, const cgs_net_desc* d, int64_t B) {
  return cgs_refine_workspace_bytes_bn(gtail, d, nullptr, B);
}

static int head_launch(const Chain& c, const Workspace& w, int64_t B, HeadParams hp, int math, cudaStream_t st) {
  hp.feat = w.act[c.n];
  if (head_takes_partials(c, w, B, math)) {          // run_forward left the split-K partial sums in the scratch buffer
    const cgs_layer_desc& L = c.layers[c.n - 1];
    hp.part = w.col;
    hp.S = fc_split(L, false);
  }
  hp.feat_ep = Epilogue(EPI_FWD, c.layers[c.n - 1].act);
  hp.feat_ep.bias = hp.part ? c.layers[c.n - 1].bias : nullptr;
  hp.w = c.head.w_fwd;
  hp.bias = c.head.bias;
  hp.K = c.head.cin;
  hp.img = w.act[c.n_gtail];
  {
    const cgs_layer_desc& Li = c.layers[c.n_gtail - 1];          // producer of the image
    const LayerShape si = layer_shape(Li);
    const int c4 = si.cs_out / 4;
    const bool pitched = Li.cout <= 4;
    hp.img_h = si.hout;
    hp.img_w4 = si.wout * c4;
    hp.img_pitch4 = (pitched ? img_pitch(si.wout) : si.wout) * c4;
    hp.img_xoff4 = pitched ? IMG_XOFF * c4 : 0;
    hp.img_elems = si.hout * si.wout * si.cs_out;
    hp.img_s2d = c.img_mode == IMG_S2D;
  }
  hp.feature = w.act[0];
  hp.feat_elems = (int)c.act_elems[0];
  hp.cur_logit = w.cur_logit;
  hp.dpre16 = bwd16(c, c.n - 1);
  if (c.bn_gamma[c.n - 1]) hp.round_out = 0;           // dpre feeds bn_backward, which rounds its own output
  hp.gexp = w.gexp;
  cudaError_t le = launch_pdl(head_kernel, dim3((unsigned)B), dim3(256), (size_t)0, st, hp);
  count_launch();
  if (le != cudaSuccess) return set_error(CGS_ERR_CUDA, "head_kernel: %s", cudaGetErrorString(le));
  return check_launch("head_kernel");
}

extern "C" int cgs_refine_conv_bn(const cgs_net_desc* gtail, const cgs_net_desc* d, const cgs_batchnorm_desc* bn,
                                  const cgs_refine_cfg* cfg, int64_t B, float* feature, float* best_img, float* best_logit,
                                  float* best_step, float* default_logit, const int32_t* prob_indices, float* best_feature,
                                  void* workspace, size_t workspace_bytes, cgs_stream_t stream) {
  if (int rc = require_sm100()) return rc;
  if (!cfg || !feature || !best_img || !best_logit || !best_step) return set_error(CGS_ERR_INVALID, "null argument");
  if (B <= 0) return B == 0 ? CGS_OK : set_error(CGS_ERR_INVALID, "negative batch");
  if (cfg->method != CGS_POLICY_SGD && cfg->method != CGS_POLICY_MOMENTUM)
    return set_error(CGS_ERR_UNSUPPORTED, "graph refiner supports sgd / momentum only (sampling/policy.py:51)");
  if (cfg->mode == CGS_MODE_PROBABILISTIC && !prob_indices)
    return set_error(CGS_ERR_INVALID, "probabilistic mode needs prob_indices");
  if (cfg->mode != CGS_MODE_PROBABILISTIC && cfg->mode != CGS_MODE_DETERMINISTIC)
    return set_error(CGS_ERR_UNSUPPORTED, "unknown mode %d", cfg->mode);
  Chain c;
  if (int rc = build_chain(gtail, d, bn, c)) return rc;
  if (c.batch_bn && cfg->early_exit)
    return set_error(CGS_ERR_UNSUPPORTED, "early exit with batch BN: leaving rows would change the batch statistics");
  choose_image_layout(c, cfg->math);
  choose_operand_type(c, cfg->math);
  // programmatic dependent launch for this call's kernels when the average pass is large (common.h launch_pdl):
  // forward + data-gradient FLOPs of one iteration over its 2 n + 1 launches
  double macs = 0.0;
  for (int i = 0; i < c.n; ++i) {
    const cgs_layer_desc& L = c.layers[i];
    const double taps = L.type == CGS_LAYER_FC ? 1.0 : (double)L.k * L.k;
    const double px = L.type == CGS_LAYER_FC ? 1.0 : (L.type == CGS_LAYER_CONV ? (double)((L.hin + 1) / 2) * ((L.win + 1) / 2)
                                                                              : (double)L.hin * L.win);
    macs += px * taps * L.cin * L.cout;
  }
  const PdlScope pdl_scope(4.0 * macs * (double)B / (2.0 * c.n + 1.0) >= 12e9);     // MNIST B=1024: 7.3 GFLOP (off), DCGAN-32: 18 (on), DCGAN-64: 78 (on)
  Workspace w;
  carve(c, B, (void*)(((uintptr_t)workspace + 255) & ~uintptr_t(255)), w);
  if (!workspace || w.total + 256 > workspace_bytes) return set_error(CGS_ERR_WORKSPACE, "workspace too small");
  if (B > cgs_refine_max_batch(gtail, d))
    return set_error(CGS_ERR_UNSUPPORTED, "batch too large for 32-bit row indexing; split it (cgs_refine_max_batch)");
  w.act[0] = feature;
  cudaStream_t st = (cudaStream_t)stream;
  HeadParams hp;
  std::memset(&hp, 0, sizeof(hp));
  hp.best_img = best_img;
  hp.best_logit = best_logit;
  hp.best_step = best_step;
  hp.default_logit = default_logit;
  hp.best_feature = best_feature;
  hp.prob_indices = prob_indices;
  hp.mode = cfg->mode;
  hp.exit_logit = cfg->exit_logit;
  hp.round_out = (cfg->math == CGS_MATH_TF32_TENSOR);
  if (cfg->early_exit) {
    hp.done = w.done;
    cudaMemsetAsync(w.done, 0, (size_t)B, st);
  }
  const int K = cfg->steps;
  const bool compacting = cfg->early_exit != 0;
  if (compacting && cfg->mode != CGS_MODE_DETERMINISTIC)
    return set_error(CGS_ERR_UNSUPPORTED, "early exit is defined for the deterministic mode only");
  float* feature_out = feature;             // the caller's buffer: final state of every sample ends up here
  float* mom_cur = w.mom;
  float* mom_alt = w.mom2;
  const int* live = nullptr;                // device-resident count of the rows still in the batch (early exit)
  int cur = 0;                              // which orig[] map / live counter is current
  if (compacting) {
    // work on a private copy so that exited samples can be dropped and the rest compacted (ping-pong feat2 / feat3)
    cudaMemcpyAsync(w.feat2, feature, (size_t)B * c.act_elems[0] * 4, cudaMemcpyDeviceToDevice, st);
    w.act[0] = w.feat2;
    iota_kernel<<<148, 256, 0, st>>>(w.orig[0], (int)B, w.count); count_launch();
    hp.orig = w.orig[0];
    hp.final_feature = feature_out;
    live = w.count;
    hp.live = live;
  }
  // initial evaluation: collaborator.py:48-60
  if (int rc = run_forward(c, w, B, cfg->math, st, live)) return rc;
  hp.step = -1;
  hp.dpre = K > 0 ? w.g[0] : nullptr;
  if (int rc = head_launch(c, w, B, hp, cfg->math, st)) return rc;
  Epilogue upd(EPI_UPDATE, ACT_NONE);
  upd.sgd = cfg->method == CGS_POLICY_SGD;
  upd.rate = cfg->rate;
  upd.alpha = cfg->alpha;
  upd.clip = cfg->clip;
  upd.vmin = cfg->vmin;
  upd.vmax = cfg->vmax;
  const int elems4 = (int)(c.act_elems[0] / 4);
  for (int i = 0; i < K; ++i) {                       // collaborator.py:63-83
    upd.first = (i == 0);
    upd.mom = mom_cur;
    if (int rc = run_backward(c, w, B, cfg->math, &upd, nullptr, st, live)) return rc;   // grad + policy step (:66-70)
    if (compacting) {
      // drop the samples D already classifies as real (README.md:13): ordered compaction of the rows that stay.
      // Only the feature map, its momentum and the row map are live here (activations / gradients are dead).
      // Everything is sized by the device-side counter: no host read-back, static launch sequence.
      int* live_next = w.count + (cur ^ 1);
      live_compact_kernel<<<1, 1024, 0, st>>>(w.done, live, (int)B, w.idx, live_next); count_launch();
      float* feat_src = w.act[0];
      float* feat_dst = (feat_src == w.feat2) ? w.feat3 : w.feat2;
      const int grid = (int)(B < 148 * 8 ? B : 148 * 8);
      live_gather_kernel<<<grid, 256, 0, st>>>((const float4*)feat_src, (float4*)feat_dst,
                                               upd.sgd ? nullptr : (const float4*)mom_cur, (float4*)mom_alt,
                                               w.orig[cur], w.orig[cur ^ 1], w.idx, live_next, elems4); count_launch();
      if (int rc = check_launch("early-exit compaction")) return rc;
      w.act[0] = feat_dst;
      float* t = mom_cur; mom_cur = mom_alt; mom_alt = t;
      cur ^= 1;
      hp.orig = w.orig[cur];
      live = live_next;
      hp.live = live;
    }
    if (int rc = run_forward(c, w, B, cfg->math, st, live)) return rc;                   // :73
    hp.step = i;
    hp.dpre = (i + 1 < K) ? w.g[0] : nullptr;         // the gradient after the last step is never consumed
    if (int rc = head_launch(c, w, B, hp, cfg->math, st)) return rc;                          // :76-83
  }
  if (compacting) {
    scatter_active_kernel<<<(unsigned)B, 128, 0, st>>>((const float4*)w.act[0], hp.orig, w.done, live, (float4*)feature_out,
                                                       elems4); count_launch();
    if (int rc = check_launch("scatter_active_kernel")) return rc;
  }
  return CGS_OK;
}

extern "C" int cgs_refine_conv(const cgs_net_desc* gtail, const cgs_net_desc* d, const cgs_refine_cfg* cfg,
                               int64_t B, float* feature, float* best_img, float* best_logit, float* best_step,
                               float* default_logit, const int32_t* prob_indices, float* best_feature,
                               void* workspace, size_t workspace_bytes, cgs_stream_t stream) {
  return cgs_refine_conv_bn(gtail, d, nullptr, cfg, B, feature, best_img, best_logit, best_step, default_logit,
                            prob_indices, best_feature, workspace, workspace_bytes, stream);
}

extern "C" int cgs_forward_logits_and_grad_bn(const cgs_net_desc* gtail, const cgs_net_desc* d,
                                              const cgs_batchnorm_desc* bn, int math, int64_t B, const float* feature,
                                              float* logit_out, float* grad_out, float* img_out, void* workspace,
                                              size_t workspace_bytes, cgs_stream_t stream) {
  if (int rc = require_sm100()) return rc;
  if (!feature || !logit_out) return set_error(CGS_ERR_INVALID, "null argument");
  if (B <= 0) return B == 0 ? CGS_OK : set_error(CGS_ERR_INVALID, "negative batch");
  Chain c;
  if (int rc = build_chain(gtail, d, bn, c)) return rc;
  choose_image_layout(c, math);
  choose_operand_type(c, math);
  Workspace w;
  carve(c, B, (void*)(((uintptr_t)workspace + 255) & ~uintptr_t(255)), w);
  if (!workspace || w.total + 256 > workspace_bytes) return set_error(CGS_ERR_WORKSPACE, "workspace too small");
  if (B > cgs_refine_max_batch(gtail, d))
    return set_error(CGS_ERR_UNSUPPORTED, "batch too large for 32-bit row indexing; split it (cgs_refine_max_batch)");
  w.act[0] = const_cast<float*>(feature);
  cudaStream_t st = (cudaStream_t)stream;
  if (int rc = run_forward(c, w, B, math, st)) return rc;
  HeadParams hp;
  std::memset(&hp, 0, sizeof(hp));
  // selection outputs are not wanted here: point them at scratch so the kernel stays branch-free
  hp.best_img = w.g[1];
  hp.best_logit = w.cur_logit;
  hp.best_step = w.mom;          // scratch (>= B floats)
  hp.step = -1;
  hp.round_out = (math == CGS_MATH_TF32_TENSOR);
  hp.dpre = grad_out ? w.g[0] : nullptr;
  if (int rc = head_launch(c, w, B, hp, math, st)) return rc;
  cudaMemcpyAsync(logit_out, w.cur_logit, (size_t)B * 4, cudaMemcpyDeviceToDevice, st);
  if (img_out) {
    const cgs_layer_desc& Li = c.layers[c.n_gtail - 1];
    const LayerShape si = layer_shape(Li);
    if (Li.cout > 4) {
      cudaMemcpyAsync(img_out, w.act[c.n_gtail], (size_t)B * c.act_elems[c.n_gtail] * 4, cudaMemcpyDeviceToDevice, st);
    } else if (int rc = c.img_mode == IMG_S2D ? s2d_to_image(w.act[c.n_gtail], img_out, B, si.hout, si.wout, st)
                                              : unpad_image(w.act[c.n_gtail], img_out, B, si.hout, si.wout, st)) {
      return rc;
    }
  }
  if (grad_out) {
    if (int rc = run_backward(c, w, B, math, nullptr, grad_out, st)) return rc;
  }
  return check_launch("cgs_forward_logits_and_grad");
}

extern "C" int cgs_forward_logits_and_grad(const cgs_net_desc* gtail, const cgs_net_desc* d, int math, int64_t B,
                                           const float* feature, float* logit_out, float* grad_out, float* img_out,
                                           void* workspace, size_t workspace_bytes, cgs_stream_t stream) {
  return cgs_forward_logits_and_grad_bn(gtail, d, nullptr, math, B, feature, logit_out, grad_out, img_out, workspace,
                                        workspace_bytes, stream);
}

// Host-only introspection (include/cgs.h): dtype and layout of every tensor of the chain, from the chain's own
// decisions (build_chain, choose_image_layout, choose_operand_type, fwd16 / bwd16).
extern "C" int64_t cgs_debug_chain_layout(const cgs_net_desc* gtail, const cgs_net_desc* d, int math, int32_t* out,
                                          int64_t capacity) {
  Chain c;
  if (int rc = build_chain(gtail, d, nullptr, c)) return rc;
  choose_image_layout(c, math);
  choose_operand_type(c, math);
  const int64_t need = 4 + (int64_t)(2 * c.n + 1) * 8;
  if (!out) return need;
  if (capacity < need) return set_error(CGS_ERR_INVALID, "capacity too small");
  enum { DENSE = 0, S2D = 1, PITCHED = 2 };
  const int img = c.img_mode == IMG_S2D ? S2D : PITCHED;
  int32_t* o = out;
  *o++ = c.n; *o++ = c.n_gtail; *o++ = img; *o++ = c.f16;
  auto put = [&](int i, bool f16) {          // act[i] (or the gradient in its place): H, W, channels as produced
    const cgs_layer_desc& Lp = c.layers[i == 0 ? 0 : i - 1];
    const LayerShape s = layer_shape(Lp);
    const int h = i == 0 ? Lp.hin : s.hout, w = i == 0 ? Lp.win : s.wout, ch = i == 0 ? Lp.cin : Lp.cout;
    const int lay = ch <= 4 ? img : DENSE;
    *o++ = f16; *o++ = lay; *o++ = h; *o++ = w; *o++ = ch;
    *o++ = lay == DENSE ? cstride(ch) : lay == S2D ? 16 : 4;                 // values per stored pixel
    *o++ = lay == DENSE ? w : lay == S2D ? w / 2 : img_pitch(w);             // stored pixels per row
    *o++ = lay == S2D ? h * w * 4 : (int32_t)c.act_elems[i];                 // s2d samples lie back to back
  };
  for (int i = 0; i <= c.n; ++i) put(i, fwd16(c, i));
  for (int i = 1; i <= c.n; ++i) put(i, bwd16(c, i - 1));
  return need;
}

// Developer entry point (include/cgs.h): one pass of the chain, launched exactly as run_forward / run_backward /
// head_launch launch it, but unpaired (try_edge_pair is not taken) and with the head reading a stored act[n] rather
// than split-K partial sums.
extern "C" int cgs_debug_chain_pass(const cgs_net_desc* gtail, const cgs_net_desc* d, int math, int64_t B, int layer,
                                    int backward, const void* in, void* out, void* aux, int32_t* gexp,
                                    const cgs_refine_cfg* step_cfg, float* mom, int first, void* workspace,
                                    size_t workspace_bytes, cgs_stream_t stream) {
  if (int rc = require_sm100()) return rc;
  if (!in || !out) return set_error(CGS_ERR_INVALID, "null argument");
  if (B <= 0) return B == 0 ? CGS_OK : set_error(CGS_ERR_INVALID, "negative batch");
  Chain c;
  if (int rc = build_chain(gtail, d, nullptr, c)) return rc;
  choose_image_layout(c, math);
  choose_operand_type(c, math);
  if (layer < 0 || layer > c.n || (layer == c.n && !backward))
    return set_error(CGS_ERR_INVALID, "pass %d (%s) is not in the chain", layer, backward ? "data-gradient" : "forward");
  Workspace w;
  carve(c, B, (void*)(((uintptr_t)workspace + 255) & ~uintptr_t(255)), w);
  if (!workspace || w.total + 256 > workspace_bytes) return set_error(CGS_ERR_WORKSPACE, "workspace too small");
  if (B > cgs_refine_max_batch(gtail, d))
    return set_error(CGS_ERR_UNSUPPORTED, "batch too large for 32-bit row indexing; split it (cgs_refine_max_batch)");
  cudaStream_t st = (cudaStream_t)stream;
  const bool scaled = layer == 0 && backward && c.f16;       // the pass that removes the head's per-sample scale
  if (gexp && !scaled && layer != c.n)
    return set_error(CGS_ERR_INVALID, "only layer 0's data-gradient pass of an FP16 chain takes a gradient scale");
  if (layer == c.n) {
    if (!aux || (bwd16(c, c.n - 1) && !gexp)) return set_error(CGS_ERR_INVALID, "the head needs logit / exponent outputs");
    HeadParams hp;
    std::memset(&hp, 0, sizeof(hp));
    w.act[0] = w.feat2;
    w.act[c.n] = (float*)in;
    w.cur_logit = (float*)aux;
    if (gexp) w.gexp = gexp;
    w.col = nullptr;                                         // no split-K partials: the head reads `in`
    hp.best_img = w.g[1];                                    // selection outputs to scratch, as cgs_forward_logits_and_grad
    hp.best_logit = w.cur_logit;
    hp.best_step = w.mom;
    hp.step = -1;
    hp.round_out = (math == CGS_MATH_TF32_TENSOR);
    hp.dpre = (float*)out;
    return head_launch(c, w, B, hp, math, st);
  }
  const cgs_layer_desc& L = c.layers[layer];
  if (!backward)
    return run_pass(L, false, B, (const float*)in, (float*)out, forward_epi(c, layer, math), nullptr, w.col, math, st,
                    c.img_mode, false, fwd16(c, layer));
  Epilogue upd(EPI_UPDATE, ACT_NONE);
  if (step_cfg) {
    if (layer != 0) return set_error(CGS_ERR_INVALID, "the policy step is fused into layer 0's data-gradient pass only");
    if (!mom && step_cfg->method != CGS_POLICY_SGD) return set_error(CGS_ERR_INVALID, "momentum step without momentum");
    upd.sgd = step_cfg->method == CGS_POLICY_SGD;
    upd.rate = step_cfg->rate;
    upd.alpha = step_cfg->alpha;
    upd.clip = step_cfg->clip;
    upd.vmin = step_cfg->vmin;
    upd.vmax = step_cfg->vmax;
    upd.first = first != 0;
    upd.mom = mom;
  }
  if (layer > 0 && !aux) return set_error(CGS_ERR_INVALID, "a data-gradient pass needs the forward output it differentiates");
  Epilogue e = backward_epi(c, layer, math, step_cfg ? &upd : nullptr, (const float*)aux);
  if (scaled) e.gexp = gexp;
  return run_pass(L, true, B, (const float*)in, (float*)out, e, nullptr, w.col, math, st, c.img_mode, false,
                  bwd16(c, layer));
}

static size_t layer_stage_elems(const cgs_layer_desc& L, bool backward) {   // pitched copy of an image-like input
  if (!use_window(L, backward)) return 0;
  const PassShape sh = pass_shape(L, backward);
  return tensor_elems(sh.ih, sh.iw, sh.kch);
}

extern "C" size_t cgs_layer_workspace_bytes(const cgs_layer_desc* L, int64_t B) {
  if (!L || B < 0) return 0;
  size_t ce = scatter_col_elems(*L, false);
  if (scatter_col_elems(*L, true) > ce) ce = scatter_col_elems(*L, true);
  size_t se = layer_stage_elems(*L, false);
  if (layer_stage_elems(*L, true) > se) se = layer_stage_elems(*L, true);
  return (ce + se) * (size_t)B * 4 + 512;
}

// The single-layer entry points take and return DENSE tensors; image-like inputs of window-lowered passes are
// re-laid out into the workspace first (inside the refinement chain they are produced pitched, no copy).
static int layer_pass_dense(const cgs_layer_desc& L, bool backward, int math, int64_t B, const float* in, float* out,
                            const Epilogue& e, void* workspace, size_t workspace_bytes, cudaStream_t st) {
  const bool needs_ws = use_scatter(L, backward) || use_window(L, backward);
  if (needs_ws && (!workspace || workspace_bytes < cgs_layer_workspace_bytes(&L, B)))
    return set_error(CGS_ERR_WORKSPACE, "workspace too small");
  float* base = (float*)(((uintptr_t)workspace + 255) & ~uintptr_t(255));
  float* col = (workspace && workspace_bytes >= cgs_layer_workspace_bytes(&L, B)) ? base : nullptr;
  size_t ce = scatter_col_elems(L, false);
  if (scatter_col_elems(L, true) > ce) ce = scatter_col_elems(L, true);
  float* stage = base + ((ce * (size_t)B + 63) & ~size_t(63));
  int img_mode = IMG_DENSE;
  if (use_window(L, backward)) {
    // the image-like input is re-laid out first (inside the chain it is produced in that layout: no copy there)
    const PassShape sh = pass_shape(L, backward);
    img_mode = edge_route(L, backward, math, e, IMG_S2D) == ROUTE_TC ? IMG_S2D : IMG_PITCHED;
    if (int rc = img_mode == IMG_S2D ? image_to_s2d(in, stage, B, sh.ih, sh.iw, st) : pad_image(in, stage, B, sh.ih, sh.iw, st))
      return rc;
    in = stage;
  }
  return run_pass(L, backward, B, in, out, e, nullptr, col, math, st, img_mode);
}

extern "C" int cgs_layer_forward(const cgs_layer_desc* L, int math, int64_t B, const float* x, float* y,
                                 void* workspace, size_t workspace_bytes, cgs_stream_t stream) {
  if (int rc = require_sm100()) return rc;
  if (!L || !x || !y) return set_error(CGS_ERR_INVALID, "null argument");
  return layer_pass_dense(*L, false, math, B, x, y, Epilogue(EPI_FWD, L->act), workspace, workspace_bytes,
                          (cudaStream_t)stream);
}

extern "C" int cgs_layer_backward(const cgs_layer_desc* L, int math, int64_t B, const float* dy, float* dx,
                                  const float* x_fwd, int prev_act, void* workspace, size_t workspace_bytes,
                                  cgs_stream_t stream) {
  if (int rc = require_sm100()) return rc;
  if (!L || !dy || !dx) return set_error(CGS_ERR_INVALID, "null argument");
  Epilogue e(EPI_RAW, ACT_NONE);
  if (x_fwd && prev_act != CGS_ACT_NONE) {
    e = Epilogue(EPI_BWD, prev_act);
    e.aux = x_fwd;
  }
  return layer_pass_dense(*L, true, math, B, dy, dx, e, workspace, workspace_bytes, (cudaStream_t)stream);
}

// Host-only: 0 = the pass uses the gather layout described by cgs_pack_map, 1 = scatter layout
// (rows = (ky*k + kx)*4 + small channel, K = the large channel count; see "Scatter formulation" above),
// 2 = window layout (rows = large channel, K index = ky*32 + kx*4 + small channel, zero elsewhere).
extern "C" int cgs_pass_layout(const cgs_layer_desc* L, int backward) {
  if (!L) return set_error(CGS_ERR_INVALID, "null layer");
  if (use_window(*L, backward != 0)) return 2;
  return use_scatter(*L, backward != 0) ? 1 : 0;
}

// Host-only: the K ordering of a layer's packed weight matrix, so the packer (cgs/pack.py) never has to
// re-derive the class / tap enumeration.  For K index q: ky[q], kx[q] = filter tap (or -1 for zero padding),
// ch[q] = reduced channel.  Returns the K length (multiple of 32), or a negative status.
extern "C" int64_t cgs_pack_map(const cgs_layer_desc* L, int backward, int32_t* ky, int32_t* kx, int32_t* ch,
                                int64_t capacity) {
  if (!L) return set_error(CGS_ERR_INVALID, "null layer");
  ConvGemmParams p;
  if (int rc = make_pass_params(*L, backward != 0, 1, nullptr, nullptr, p)) return rc;
  int64_t total = 0;
  for (int c = 0; c < p.nclasses; ++c) total += (int64_t)p.cls[c].nkb * 32;
  if (!ky || !kx || !ch) return total;
  if (capacity < total) return set_error(CGS_ERR_INVALID, "pack map capacity too small");
  if (L->type == CGS_LAYER_FC) {
    for (int64_t q = 0; q < total; ++q) { ky[q] = 0; kx[q] = 0; ch[q] = (int32_t)q; }
    return total;
  }
  // recover (ky,kx) from (dy,dx): strided pass dy = ky - pad ; transposed pass dy = (py + pad - ky)/2
  const PassShape sh = pass_shape(*L, backward != 0);
  const bool strided = sh.strided;
  const int pad_y = sh.pad_y, pad_x = sh.pad_x;
  for (int c = 0; c < p.nclasses; ++c) {
    const GemmClass& g = p.cls[c];
    const int cin_k = p.cblocks ? p.cblocks * 32 : 4;
    const int64_t klen = (int64_t)g.nkb * 32;
    for (int64_t q = 0; q < klen; ++q) {
      const int t = (int)(q / cin_k);
      const int cc = (int)(q % cin_k);
      const int64_t o = g.k0 + q;
      if (t >= g.ntaps) { ky[o] = -1; kx[o] = -1; ch[o] = cc; continue; }
      if (strided) {
        ky[o] = g.dy[t] + pad_y;
        kx[o] = g.dx[t] + pad_x;
      } else {
        ky[o] = g.oy0 + pad_y - 2 * g.dy[t];
        kx[o] = g.ox0 + pad_x - 2 * g.dx[t];
      }
      ch[o] = cc;
    }
  }
  return total;
}

// Host-only introspection (no GPU needed): the gathered-GEMM parameters a layer pass is lowered to, flattened to
// int32 so tests can replay the exact gather on the CPU.  Layout: [IH, IW, Cs, cblocks, MH, MW, S, M, OH, OW, ON,
// os, N, nclasses, window, win_k, win_x0, in_pitch_px] then per class [k0, nkb, ntaps, oy0, ox0, dy[32], dx[32]].  Returns the number of ints.
// Host-only introspection of the class-fused lowering (include/cgs.h).
extern "C" int64_t cgs_debug_fusion_plan(const cgs_layer_desc* L, int backward, int64_t B, int32_t* out, int64_t capacity) {
  if (!L) return set_error(CGS_ERR_INVALID, "null layer");
  if (use_window(*L, backward != 0) || use_scatter(*L, backward != 0)) return 0;
  ConvGemmParams p;
  if (int rc = make_pass_params(*L, backward != 0, B, nullptr, nullptr, p)) return rc;
  const int ns = plan_fusion(p);
  if (!ns) return 0;
  int nshf = 0;
  for (int g = 0; g < p.ngroups; ++g) nshf += p.grp[g].nshifts;
  const int64_t need = 2 + (int64_t)p.ngroups * 7 + (int64_t)nshf * 48;
  if (!out) return need;
  if (capacity < need) return set_error(CGS_ERR_INVALID, "capacity too small");
  int32_t* o = out;
  *o++ = ns; *o++ = p.ngroups;
  for (int g = 0; g < p.ngroups; ++g) {
    const FuseGroup& G = p.grp[g];
    *o++ = G.nshifts; *o++ = G.shift0; *o++ = G.ncls;
    for (int q = 0; q < 4; ++q) *o++ = G.cls[q];
  }
  for (int i = 0; i < nshf; ++i) {
    const FuseShift& s = p.shf[i];
    *o++ = s.dy; *o++ = s.dx; *o++ = s.ncls; *o++ = s.nrun;
    for (int q = 0; q < 4; ++q) *o++ = s.slot[q];
    for (int q = 0; q < 4; ++q) *o++ = s.katom0[q];
    for (int q = 0; q < 4; ++q) *o++ = s.run_slot[q];
    for (int q = 0; q < 4; ++q) *o++ = s.run_len[q];
    for (int q = 0; q < 4; ++q) *o++ = s.run_acc[q];
    for (int r = 0; r < 2; ++r) for (int q = 0; q < 4; ++q) *o++ = s.pc_slot[r][q];
    for (int r = 0; r < 2; ++r) for (int q = 0; q < 4; ++q) *o++ = s.pc_half[r][q];
    for (int r = 0; r < 2; ++r) for (int q = 0; q < 4; ++q) *o++ = s.pc_katom[r][q];
  }
  return need;
}

extern "C" int64_t cgs_debug_gemm_params(const cgs_layer_desc* L, int backward, int64_t B, int32_t* out,
                                         int64_t capacity) {
  if (!L) return set_error(CGS_ERR_INVALID, "null layer");
  ConvGemmParams p;
  int rc = use_window(*L, backward != 0) ? make_window_params(*L, backward != 0, B, nullptr, nullptr, p)
           : use_scatter(*L, backward != 0) ? make_scatter_gemm_params(*L, backward != 0, B, nullptr, nullptr, p)
           : make_pass_params(*L, backward != 0, B, nullptr, nullptr, p);
  if (rc) return rc;
  const int64_t need = 18 + (int64_t)p.nclasses * (5 + 2 * kMaxTaps);
  if (!out) return need;
  if (capacity < need) return set_error(CGS_ERR_INVALID, "capacity too small");
  int32_t* o = out;
  const int head[18] = {p.IH, p.IW, p.Cs, p.cblocks, p.MH, p.MW, p.S, p.M, p.OH, p.OW, p.ON, p.os, p.N, p.nclasses,
                        p.window, p.win_k, p.win_x0, p.in_pitch_px};
  for (int i = 0; i < 18; ++i) *o++ = head[i];
  for (int c = 0; c < p.nclasses; ++c) {
    const GemmClass& g = p.cls[c];
    *o++ = g.k0; *o++ = g.nkb; *o++ = g.ntaps; *o++ = g.oy0; *o++ = g.ox0;
    for (int t = 0; t < kMaxTaps; ++t) *o++ = g.dy[t];
    for (int t = 0; t < kMaxTaps; ++t) *o++ = g.dx[t];
  }
  return need;
}
