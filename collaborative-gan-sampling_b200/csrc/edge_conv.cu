// Image-edge passes (see edge_conv.cuh): fused im2col / col2im + mma.sync TF32 + epilogue streaming kernels.
//
// Reference semantics: nsgan/ops.py:41 (conv2d, k x k, stride 2, SAME), nsgan/ops.py:55 (deconv2d) and their
// tf.gradients data-gradients (sampling/collaborator.py:31); epilogues as in conv_gemm.cuh.
#include "edge_conv.cuh"

#include <cstdint>

#include "common.h"
#include "conv_gemm.cuh"
#include "ptx.cuh"

namespace cgs {

namespace {

// D(16x8, fp32) += A(16x8, tf32, row) * B(8x8, tf32, col); g = lane / 4, t = lane % 4:
//   a0 (g, t)  a1 (g+8, t)  a2 (g, t+4)  a3 (g+8, t+4);  b0 (k = t, n = g)  b1 (k = t+4, n = g)
//   c0 (g, 2t) c1 (g, 2t+1) c2 (g+8, 2t) c3 (g+8, 2t+1)
__device__ __forceinline__ void mma_tf32(float (&c)[4], uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t b0,
                                         uint32_t b1) {
  asm volatile(
      "mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
      : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
      : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
}

// ---------------------------------------------------------------------------------------------
// edge_wide: per tile (image b, band of RO output rows <= 256 pixels) the input rows the band needs are staged in
// shared memory by cp.async (rows outside the image zero-filled), double-buffered so the next tile's rows arrive
// while this tile computes; the im2col gather of the A fragments is then plain LDS with no bounds tests.
// N = 64, K = k*k*cimg.  CTA = 8 warps; a warp takes 16 pixels x 64 channels at a time (8 mma tiles per k-step,
// 32 accumulator registers) so that four CTAs fit an SM: the kernel is latency bound, warps in flight are what
// buys bandwidth.  Weights live in shared memory in fragment order (one LDS.64 per B fragment).
// ---------------------------------------------------------------------------------------------
constexpr int EW_THREADS = 256;
constexpr int EW_NT = 8;            // N = 64
constexpr int EW_KMAX = 104;        // k <= 5, cimg <= 4
constexpr int EW_TILE_PX = EW_THREADS;   // 32 pixels per warp

// Epilogue modes compiled into the kernel (the per-element code must stay a handful of instructions: it runs 64
// times per thread and tile): slope-type forward / derivative, the policy step, and a generic fallback (tanh, raw).
enum : int { EM_FWD_SLOPE = 0, EM_BWD_SLOPE = 1, EM_UPDATE = 2, EM_GENERIC = 3 };

template <int MODE, bool ROUND>
__device__ __forceinline__ float epi_fast(const Epilogue& e, float a, float x0, float x1, float* m_out) {
  if (MODE == EM_FWD_SLOPE) return epilogue1_t<EPI_FWD, 0, ROUND>(e, a, x0, x1, m_out);
  if (MODE == EM_BWD_SLOPE) return epilogue1_t<EPI_BWD, 0, ROUND>(e, a, x0, x1, m_out);
  return epilogue1(e, a, x0, x1, m_out);
}

// One-time set-up of an edge_wide CTA: k -> patch offset table, bias, weights in mma fragment order.
__device__ __forceinline__ void wide_setup(const EdgeWideParams& p, int ksteps, float2* bfrag, int* koff_s, float* bias_s) {
  const int tid = threadIdx.x;
  const int CI = p.cimg;
  const int kreal = p.k * p.k * CI;
  const int prow = p.pitch * 4;              // floats per staged row
  for (int kk = tid; kk < ksteps * 8; kk += EW_THREADS) {
    int off = 0;                             // padding k slots read a valid word and multiply a zero weight
    if (kk < kreal) {
      const int tap = kk / CI, c = kk - tap * CI;
      const int ky = tap / p.k, kx = tap - ky * p.k;
      off = ky * prow + (kx - p.pad_x + p.xoff) * 4 + c;
    }
    koff_s[kk] = off;
  }
  if (tid < EW_NT * 8) bias_s[tid] = (p.ep.mode == EPI_FWD && p.ep.bias && tid < p.N) ? __ldg(p.ep.bias + tid) : 0.f;
  for (int idx = tid; idx < ksteps * EW_NT * 32; idx += EW_THREADS) {
    const int l = idx & 31, nt = (idx >> 5) % EW_NT, ks = idx / (EW_NT * 32);
    const int n = nt * 8 + (l >> 2);
    float b[2];
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int kk = ks * 8 + (l & 3) + 4 * h;
      b[h] = 0.f;
      if (kk < kreal && n < p.N) {
        const int tap = kk / CI, c = kk - tap * CI;
        const int ky = tap / p.k, kx = tap - ky * p.k;
        b[h] = __ldg(p.w + (size_t)n * (p.k * 32) + ky * 32 + kx * 4 + c);
      }
    }
    bfrag[idx] = make_float2(b[0], b[1]);
  }
}

// The band's GEMM + epilogue: `patch` holds the staged input rows ([rows][pitch][4] floats, row 0 = image row
// 2*oy0 - pad_y), npx output pixels starting at global pixel m0.  Each warp takes 16 pixels x 64 channels at a time.
template <int MODE, bool ROUND>
__device__ __forceinline__ void wide_band(const EdgeWideParams& p, int ksteps, const float* patch, const float2* bfrag,
                                          const int* koff_s, const float* bias_s, int npx, int m0,
                                          unsigned long long fd_ow) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int g = lane >> 2, t = lane & 3;
  const int prow = p.pitch * 4;
  for (int mt = warp; mt * 16 < npx; mt += EW_THREADS / 32) {
    // the two pixels (rows g, g+8 of the m16 tile) this thread gathers for and stores
    int base[2], mloc[2];
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int ml = mt * 16 + h * 8 + g;
      const int oyr = fast_div(ml, fd_ow), ox = ml - oyr * p.OW;
      const bool ok = ml < npx;
      base[h] = ok ? (2 * oyr * prow + 2 * ox * 4) : 0;
      mloc[h] = ok ? ml : -1;
    }
    float acc[EW_NT][4];
#pragma unroll
    for (int nt = 0; nt < EW_NT; ++nt)
#pragma unroll
      for (int i = 0; i < 4; ++i) acc[nt][i] = 0.f;
#pragma unroll 2
    for (int ks = 0; ks < ksteps; ++ks) {
      const int o0 = koff_s[ks * 8 + t];
      const int o1 = koff_s[ks * 8 + t + 4];
      const uint32_t a0 = __float_as_uint(patch[base[0] + o0]);
      const uint32_t a1 = __float_as_uint(patch[base[1] + o0]);
      const uint32_t a2 = __float_as_uint(patch[base[0] + o1]);
      const uint32_t a3 = __float_as_uint(patch[base[1] + o1]);
#pragma unroll
      for (int nt = 0; nt < EW_NT; ++nt) {
        const float2 bq = bfrag[(ks * EW_NT + nt) * 32 + lane];
        mma_tf32(acc[nt], a0, a1, a2, a3, __float_as_uint(bq.x), __float_as_uint(bq.y));
      }
    }
    // epilogue: thread owns columns nt*8 + 2t, +1 of its two rows; a quad writes one 32-byte sector
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      if (mloc[h] < 0) continue;
      const size_t ro = (size_t)(m0 + mloc[h]) * p.ON + 2 * t;
      float* orow = p.out + ro;
#pragma unroll
      for (int half = 0; half < 2; ++half) {
        float2 x0[EW_NT / 2], x1[EW_NT / 2];
#pragma unroll
        for (int q = 0; q < EW_NT / 2; ++q) {
          const int nt = half * (EW_NT / 2) + q;
          x1[q] = make_float2(0.f, 0.f);
          if (MODE == EM_FWD_SLOPE) {
            x0[q] = *reinterpret_cast<const float2*>(bias_s + nt * 8 + 2 * t);
          } else if (MODE == EM_BWD_SLOPE) {
            x0[q] = __ldg(reinterpret_cast<const float2*>(p.ep.aux + ro + nt * 8));
          } else {
            x0[q] = *reinterpret_cast<const float2*>(bias_s + nt * 8 + 2 * t);
            if (p.ep.mode == EPI_BWD) {
              x0[q] = __ldg(reinterpret_cast<const float2*>(p.ep.aux + ro + nt * 8));
            } else if (p.ep.mode == EPI_UPDATE) {
              x0[q] = *reinterpret_cast<const float2*>(orow + nt * 8);
              if (!p.ep.sgd && !p.ep.first) x1[q] = *reinterpret_cast<const float2*>(p.ep.mom + ro + nt * 8);
            }
          }
        }
#pragma unroll
        for (int q = 0; q < EW_NT / 2; ++q) {
          const int nt = half * (EW_NT / 2) + q;
          float2 m2 = make_float2(0.f, 0.f), o;
          o.x = epi_fast<MODE, ROUND>(p.ep, acc[nt][2 * h], x0[q].x, x1[q].x, &m2.x);
          o.y = epi_fast<MODE, ROUND>(p.ep, acc[nt][2 * h + 1], x0[q].y, x1[q].y, &m2.y);
          if (MODE >= EM_UPDATE && p.ep.mode == EPI_UPDATE && !p.ep.sgd) *reinterpret_cast<float2*>(p.ep.mom + ro + nt * 8) = m2;
          *reinterpret_cast<float2*>(orow + nt * 8) = o;
        }
      }
    }
  }
}

template <int MODE, bool ROUND>
__global__ void __launch_bounds__(EW_THREADS, 4) edge_wide_kernel(const EdgeWideParams p, int ksteps, int ntiles, int RO,
                                                                  int bands, unsigned long long fd_bands,
                                                                  unsigned long long fd_ow) {
  extern __shared__ float4 ew_smem4[];
  const int PR = 2 * RO + p.k - 2;           // staged input rows per band
  const int patch_px = PR * p.pitch;         // pixels (float4) per patch buffer
  float2* bfrag = reinterpret_cast<float2*>(ew_smem4);                          // [ksteps][8][32]
  float4* patch4 = ew_smem4 + ksteps * EW_NT * 32 / 2;                          // [2][PR][pitch]
  __shared__ int koff_s[EW_KMAX];
  __shared__ float bias_s[EW_NT * 8];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  wide_setup(p, ksteps, bfrag, koff_s, bias_s);

  // async copy of the input rows of one tile into patch buffer `buf`
  auto stage_patch = [&](int tile, int buf) {
    const int b = fast_div(tile, fd_bands);
    const int iy0 = 2 * (tile - b * bands) * RO - p.pad_y;       // image row of staged row 0
    const uint32_t dst0 = smem_u32(patch4 + buf * patch_px);
    for (int pr = warp; pr < PR; pr += EW_THREADS / 32) {
      const int iy = iy0 + pr;
      const bool ok = (unsigned)iy < (unsigned)p.IH;
      const float4* src = reinterpret_cast<const float4*>(p.in) + (size_t)(b * p.IH + (ok ? iy : 0)) * p.pitch;
      for (int x = lane; x < p.pitch; x += 32)
        cp_async_16(dst0 + (pr * p.pitch + x) * 16, src + x, ok ? 16u : 0u);
    }
  };

  pdl_launch_dependents();
  pdl_wait();                                // tables and weights above are constants; activations from here on
  if (p.live) ntiles = min(ntiles, live_images(p.live, ntiles / bands) * bands);
  int tile = blockIdx.x;
  if (tile < ntiles) stage_patch(tile, 0);
  cp_async_commit();
  for (int it = 0; tile < ntiles; tile += gridDim.x, ++it) {
    const int cur = it & 1;
    const int b = fast_div(tile, fd_bands);
    const int oy0 = (tile - b * bands) * RO;
    const int npx = min(RO, p.OH - oy0) * p.OW;
    const int m0 = (b * p.OH + oy0) * p.OW;                      // first output pixel of the band
    if (tile + (int)gridDim.x < ntiles) stage_patch(tile + gridDim.x, cur ^ 1);
    cp_async_commit();
    cp_async_wait<1>();                      // this tile's input rows have landed
    __syncthreads();
    wide_band<MODE, ROUND>(p, ksteps, reinterpret_cast<const float*>(patch4 + cur * patch_px), bfrag, koff_s, bias_s, npx,
                           m0, fd_ow);
    __syncthreads();                         // patch[cur] may be overwritten from here on
  }
  cp_async_wait<0>();
}

// ---------------------------------------------------------------------------------------------
// edge_narrow: per tile (image b, band of R input rows + halo) compute col[pixel][(ky,kx,c)] = in[pixel][:] . W with
// mma.sync (A fragments straight from global memory as 16-byte loads, K permuted so that a float4 feeds two k-steps),
// park col in shared memory, then every output pixel of the band sums its taps in a fixed order (ky, kx ascending)
// and applies the epilogue.  K = 64.
// ---------------------------------------------------------------------------------------------
constexpr int EN_THREADS = 256;
constexpr int EN_ROWS = 256;        // col rows (input pixels incl. halo) per tile
constexpr int EN_KSTEPS = 8;        // K = 64

// Weights of an edge_narrow pass in mma fragment order: [8 k-steps][NT][32 lanes] float2.
template <int NT, int CI>
__device__ __forceinline__ void narrow_setup(const EdgeNarrowParams& p, float2* bfrag) {
  const int nreal = p.k * p.k * CI;
  for (int idx = threadIdx.x; idx < EN_KSTEPS * NT * 32; idx += EN_THREADS) {
    const int l = idx & 31, nt = (idx >> 5) % NT, ks = idx / (NT * 32);
    const int n = nt * 8 + (l >> 2);
    // logical k slots (t, t+4) of k-step ks are input channels 16*(ks/2) + 4t + 2*(ks%2) + {0, 1}
    const int ch = 16 * (ks >> 1) + 4 * (l & 3) + 2 * (ks & 1);
    float2 b = make_float2(0.f, 0.f);
    if (n < nreal) {
      const int tap = n / CI, c = n - tap * CI;
      b = __ldg(reinterpret_cast<const float2*>(p.w + (size_t)(tap * 4 + c) * p.K + ch));
    }
    bfrag[idx] = b;
  }
}

// col[pixel][(ky,kx,c)] = in[pixel][:] . W for the mt_rows input pixels starting at src; result in shared memory.
template <int NT>
__device__ __forceinline__ void narrow_mma(const float* src, int K, int mt_rows, const float2* bfrag, float* col_s) {
  constexpr int CP = NT * 8 + 4;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int g = lane >> 2, t = lane & 3;
  const int nmt = (mt_rows + 15) >> 4;
  for (int mt = warp; mt < nmt; mt += EN_THREADS / 32) {
    const int ra = mt * 16 + g, rb = ra + 8;
    float4 va[4], vb[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      va[j] = ra < mt_rows ? __ldg(reinterpret_cast<const float4*>(src + (size_t)ra * K + 16 * j + 4 * t))
                           : make_float4(0.f, 0.f, 0.f, 0.f);
      vb[j] = rb < mt_rows ? __ldg(reinterpret_cast<const float4*>(src + (size_t)rb * K + 16 * j + 4 * t))
                           : make_float4(0.f, 0.f, 0.f, 0.f);
    }
    float acc[NT][4];
#pragma unroll
    for (int nt = 0; nt < NT; ++nt)
#pragma unroll
      for (int i = 0; i < 4; ++i) acc[nt][i] = 0.f;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
#pragma unroll
      for (int nt = 0; nt < NT; ++nt) {
        const float2 be = bfrag[((2 * j) * NT + nt) * 32 + lane];
        mma_tf32(acc[nt], __float_as_uint(va[j].x), __float_as_uint(vb[j].x), __float_as_uint(va[j].y),
                 __float_as_uint(vb[j].y), __float_as_uint(be.x), __float_as_uint(be.y));
        const float2 bo = bfrag[((2 * j + 1) * NT + nt) * 32 + lane];
        mma_tf32(acc[nt], __float_as_uint(va[j].z), __float_as_uint(vb[j].z), __float_as_uint(va[j].w),
                 __float_as_uint(vb[j].w), __float_as_uint(bo.x), __float_as_uint(bo.y));
      }
    }
#pragma unroll
    for (int nt = 0; nt < NT; ++nt) {
      *reinterpret_cast<float2*>(col_s + ra * CP + nt * 8 + 2 * t) = make_float2(acc[nt][0], acc[nt][1]);
      *reinterpret_cast<float2*>(col_s + rb * CP + nt * 8 + 2 * t) = make_float2(acc[nt][2], acc[nt][3]);
    }
  }
}

// col2im + epilogue over output rows [y_lo, y_hi) of image b (margins of the pitched layout are written as zeros): one
// warp per output row, so the ky taps are warp-uniform; only taps of the right parity are visited, in a fixed order.
// The result goes to global memory (unless `out` is null) and, if `patch` is given, into a shared-memory copy of the
// pitched image whose row 0 is image row -patch_row0 (the consumer's staged input, fused pair kernels).
template <int NT, int CI>
__device__ __forceinline__ void narrow_col2im(const EdgeNarrowParams& p, const float* col_s, int b, int iy_lo, int rows_in,
                                              int y_lo, int y_hi, float* out, float4* patch, int patch_row0) {
  constexpr int CP = NT * 8 + 4;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const float4 bias4 = (p.ep.mode == EPI_FWD && p.ep.bias) ? __ldg(reinterpret_cast<const float4*>(p.ep.bias))
                                                          : make_float4(0.f, 0.f, 0.f, 0.f);
  for (int y = y_lo + warp; y < y_hi; y += EN_THREADS / 32) {
    const int ky0 = (y + p.pad_y) & 1;
    const size_t grow = ((size_t)b * p.OH + y) * p.out_pitch * 4;
    for (int xc = lane; xc < p.out_pitch; xc += 32) {
      const int x = xc - p.out_xoff;
      float o[4] = {0.f, 0.f, 0.f, 0.f};
      if (x >= 0 && x < p.OW) {
        float a[CI];
#pragma unroll
        for (int c = 0; c < CI; ++c) a[c] = 0.f;
        const int kx0 = (x + p.pad_x) & 1;
        for (int ky = ky0; ky < p.k; ky += 2) {
          const int lr = ((y + p.pad_y - ky) >> 1) - iy_lo;      // negative (above the image / tile) -> skipped
          if ((unsigned)lr >= (unsigned)rows_in) continue;
          for (int kx = kx0; kx < p.k; kx += 2) {
            const int ix = (x + p.pad_x - kx) >> 1;
            if ((unsigned)ix >= (unsigned)p.IW) continue;
            const float* cp = col_s + (lr * p.IW + ix) * CP + (ky * p.k + kx) * CI;
#pragma unroll
            for (int c = 0; c < CI; ++c) a[c] += cp[c];
          }
        }
        float4 x0 = bias4;
        if (p.ep.mode == EPI_BWD) x0 = __ldg(reinterpret_cast<const float4*>(p.ep.aux + grow + xc * 4));
        const float xs[3] = {x0.x, x0.y, x0.z};
        float unused;
#pragma unroll
        for (int c = 0; c < CI; ++c) o[c] = epilogue1(p.ep, a[c], xs[c], 0.f, &unused);
      }
      const float4 v = make_float4(o[0], o[1], o[2], o[3]);
      if (out) *reinterpret_cast<float4*>(out + grow + xc * 4) = v;
      if (patch) patch[(y + patch_row0) * p.out_pitch + xc] = v;
    }
  }
}

template <int NT, int CI>
__global__ void __launch_bounds__(EN_THREADS) edge_narrow_kernel(const EdgeNarrowParams p, int ntiles) {
  extern __shared__ float2 en_smem[];
  float2* bfrag = en_smem;                                              // [8][NT][32]
  float* col_s = reinterpret_cast<float*>(en_smem + EN_KSTEPS * NT * 32);   // [EN_ROWS][CP]
  narrow_setup<NT, CI>(p, bfrag);
  __syncthreads();
  pdl_launch_dependents();
  pdl_wait();                                // weights above are constants; activations from here on
  if (p.live) ntiles = min(ntiles, live_images(p.live, p.B) * p.bands);

  for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const int b = tile / p.bands;
    const int r0 = (tile - b * p.bands) * p.R;
    const int iy_lo = max(0, r0 - p.halo_lo);
    const int iy_hi = min(p.IH, r0 + p.R + p.halo_hi);
    narrow_mma<NT>(p.in + ((size_t)b * p.IH + iy_lo) * p.IW * p.K, p.K, (iy_hi - iy_lo) * p.IW, bfrag, col_s);
    __syncthreads();
    narrow_col2im<NT, CI>(p, col_s, b, iy_lo, iy_hi - iy_lo, 2 * r0, min(p.OH, 2 * (r0 + p.R)), p.out, nullptr, 0);
    __syncthreads();
  }
}

// ---------------------------------------------------------------------------------------------
// edge_pair: the narrow pass of one layer followed by the wide pass of the next on the same image, in one kernel:
// forward   G's last deconv (-> image, tanh) + D's first conv (-> 64 channels, LeakyReLU)
// backward  D's first conv data-gradient (x tanh') + G's last deconv data-gradient (x ReLU' / policy step)
// The image (or its gradient) goes from the col2im of the first pass straight into the staged-input buffer of the
// second; the forward image is also written to global memory (best-of-K keep, derivative operand), its gradient is
// not.  One image per tile: used when a whole image fits one tile of both passes (MNIST-sized nets).
// ---------------------------------------------------------------------------------------------
template <int NT, int CI, int MODE, bool ROUND>
__global__ void __launch_bounds__(EN_THREADS, 4) edge_pair_kernel(const EdgeNarrowParams pn, const EdgeWideParams pw,
                                                                  int ksteps_w, int store_image,
                                                                  unsigned long long fd_ow) {
  static_assert(EN_THREADS == EW_THREADS, "both passes use the same CTA shape");
  extern __shared__ float4 ep_smem4[];
  const int PR = 2 * pw.OH + pw.k - 2;                                   // staged rows of the wide pass (whole image)
  float2* bfrag_n = reinterpret_cast<float2*>(ep_smem4);                 // [8][NT][32]
  float2* bfrag_w = bfrag_n + EN_KSTEPS * NT * 32;                       // [ksteps_w][8][32]
  float4* patch4 = reinterpret_cast<float4*>(bfrag_w + ksteps_w * EW_NT * 32);   // [PR][pitch]
  float* col_s = reinterpret_cast<float*>(patch4 + PR * pw.pitch);       // [IH*IW rounded to 16][CP]
  __shared__ int koff_s[EW_KMAX];
  __shared__ float bias_s[EW_NT * 8];
  narrow_setup<NT, CI>(pn, bfrag_n);
  wide_setup(pw, ksteps_w, bfrag_w, koff_s, bias_s);
  // rows of the staged image outside the image stay zero for the whole kernel
  for (int idx = threadIdx.x; idx < PR * pw.pitch; idx += EN_THREADS) {
    const int iy = idx / pw.pitch - pw.pad_y;
    if ((unsigned)iy >= (unsigned)pw.IH) patch4[idx] = make_float4(0.f, 0.f, 0.f, 0.f);
  }
  __syncthreads();
  pdl_launch_dependents();
  pdl_wait();
  const int npx = pw.OH * pw.OW;
  const int B_live = live_images(pw.live, pn.B);
  for (int b = blockIdx.x; b < B_live; b += gridDim.x) {
    narrow_mma<NT>(pn.in + (size_t)b * pn.IH * pn.IW * pn.K, pn.K, pn.IH * pn.IW, bfrag_n, col_s);
    __syncthreads();
    narrow_col2im<NT, CI>(pn, col_s, b, 0, pn.IH, 0, pn.OH, store_image ? pn.out : nullptr, patch4, pw.pad_y);
    __syncthreads();
    wide_band<MODE, ROUND>(pw, ksteps_w, reinterpret_cast<const float*>(patch4), bfrag_w, koff_s, bias_s, npx, b * npx, fd_ow);
    __syncthreads();
  }
}

int num_sms() { return device_num_sms(); }

template <int NT, int CI>
int launch_narrow_nt(const EdgeNarrowParams& p, cudaStream_t st) {
  constexpr int CP = NT * 8 + 4;
  constexpr size_t smem = (size_t)EN_KSTEPS * NT * 32 * sizeof(float2) + (size_t)EN_ROWS * CP * sizeof(float);
  int ctas_per_sm = 0;
  {
    static DynSmemCache smem_cache;
    cudaError_t e = ensure_dyn_smem(edge_narrow_kernel<NT, CI>, smem, smem_cache);
    if (e != cudaSuccess) return set_error(CGS_ERR_CUDA, "cudaFuncSetAttribute(edge_narrow): %s", cudaGetErrorString(e));
    e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ctas_per_sm, edge_narrow_kernel<NT, CI>, EN_THREADS, smem);
    if (e != cudaSuccess || ctas_per_sm < 1) return set_error(CGS_ERR_CUDA, "edge_narrow occupancy query failed");
  }
  const long long tiles = (long long)p.B * p.bands;
  if (tiles >= (1ll << 31)) return set_error(CGS_ERR_UNSUPPORTED, "batch too large; split the batch");
  long long grid = (long long)num_sms() * ctas_per_sm;
  if (grid > tiles) grid = tiles;
  cudaError_t le = launch_pdl(edge_narrow_kernel<NT, CI>, dim3((unsigned)grid), dim3(EN_THREADS), smem, st, p, (int)tiles);
  count_launch();
  if (le != cudaSuccess) return set_error(CGS_ERR_CUDA, "edge_narrow_kernel: %s", cudaGetErrorString(le));
  return check_launch("edge_narrow_kernel");
}

}  // namespace

bool edge_wide_supported(const EdgeWideParams& p) {
  return p.N == 64 && p.ON == p.N && p.k >= 1 && p.k <= 5 && p.cimg >= 1 && p.cimg <= 4;
}

bool edge_narrow_supported(const EdgeNarrowParams& p) {
  return p.K == 64 && (p.k == 4 || p.k == 5) && (p.cimg == 1 || p.cimg == 3) && p.IW <= EN_ROWS / 4;
}

template <int MODE, bool ROUND>
int launch_wide_mode(const EdgeWideParams& p, int B, cudaStream_t st) {
  const int ksteps = (p.k * p.k * p.cimg + 7) / 8;
  const int RO = (p.OH * p.OW <= EW_TILE_PX) ? p.OH : EW_TILE_PX / p.OW;   // whole image per tile when it fits
  const int bands = (p.OH + RO - 1) / RO;
  const long long tiles_ll = (long long)B * bands;
  if (tiles_ll >= (1ll << 31)) return set_error(CGS_ERR_UNSUPPORTED, "batch too large; split the batch");
  const int tiles = (int)tiles_ll;
  const int PR = 2 * RO + p.k - 2;
  size_t smem = (size_t)ksteps * EW_NT * 32 * sizeof(float2) + (size_t)2 * PR * p.pitch * sizeof(float4);
  if (smem > 200 * 1024) return set_error(CGS_ERR_UNSUPPORTED, "edge_wide: image band does not fit shared memory");
  {
    static DynSmemCache smem_cache;
    cudaError_t e = ensure_dyn_smem(edge_wide_kernel<MODE, ROUND>, smem, smem_cache);
    if (e != cudaSuccess) return set_error(CGS_ERR_CUDA, "cudaFuncSetAttribute(edge_wide): %s", cudaGetErrorString(e));
  }
  int per_sm = 0;
  cudaError_t e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, edge_wide_kernel<MODE, ROUND>, EW_THREADS, smem);
  if (e != cudaSuccess || per_sm < 1) return set_error(CGS_ERR_CUDA, "edge_wide occupancy query failed");
  long long grid = (long long)num_sms() * per_sm;
  if (grid > tiles) grid = tiles;
  cudaError_t le = launch_pdl(edge_wide_kernel<MODE, ROUND>, dim3((unsigned)grid), dim3(EW_THREADS), smem, st, p, ksteps, tiles, RO,
                              bands, fast_div_magic((unsigned)bands), fast_div_magic((unsigned)p.OW));
  count_launch();
  if (le != cudaSuccess) return set_error(CGS_ERR_CUDA, "edge_wide_kernel: %s", cudaGetErrorString(le));
  return check_launch("edge_wide_kernel");
}

int launch_edge_wide(const EdgeWideParams& p, cudaStream_t st) {
  if (p.M <= 0) return CGS_OK;
  if (p.M * p.ON >= (1ll << 31)) return set_error(CGS_ERR_UNSUPPORTED, "batch too large for 32-bit indexing; split the batch");
  if (p.OW > EW_TILE_PX) return set_error(CGS_ERR_UNSUPPORTED, "edge_wide: output row wider than a tile");
  const int B = (int)(p.M / ((long long)p.OH * p.OW));
  const bool rnd = p.ep.round_out != 0;
  if (p.ep.mode == EPI_FWD && !p.ep.act_tanh)
    return rnd ? launch_wide_mode<EM_FWD_SLOPE, true>(p, B, st) : launch_wide_mode<EM_FWD_SLOPE, false>(p, B, st);
  if (p.ep.mode == EPI_BWD && !p.ep.act_tanh)
    return rnd ? launch_wide_mode<EM_BWD_SLOPE, true>(p, B, st) : launch_wide_mode<EM_BWD_SLOPE, false>(p, B, st);
  if (p.ep.mode == EPI_UPDATE) return launch_wide_mode<EM_UPDATE, false>(p, B, st);
  return launch_wide_mode<EM_GENERIC, false>(p, B, st);
}

namespace {
int narrow_geometry(EdgeNarrowParams& p) {
  // rows of the input needed above / below a band of R input rows (its 2R output rows gather taps
  // iy = (y + pad_y - ky) / 2): brute force over a sample band, the answer does not depend on R or r0
  int lo = 0, hi = 0;
  {
    const int Rs = 8;
    for (int y = 0; y < 2 * Rs; ++y)
      for (int ky = 0; ky < p.k; ++ky) {
        const int ty = y + p.pad_y - ky;
        if (ty & 1) continue;
        const int iy = ty >= 0 ? ty / 2 : -((-ty) / 2);
        if (-iy > lo) lo = -iy;
        if (iy - (Rs - 1) > hi) hi = iy - (Rs - 1);
      }
  }
  p.halo_lo = lo;
  p.halo_hi = hi;
  const int rows_max = EN_ROWS / p.IW;
  if (p.IH <= rows_max) {
    p.R = p.IH;
  } else {
    p.R = rows_max - lo - hi;
    if (p.R < 1) return set_error(CGS_ERR_UNSUPPORTED, "edge_narrow: image row too wide for the tile");
  }
  p.bands = (p.IH + p.R - 1) / p.R;
  return CGS_OK;
}

template <int NT, int CI, int MODE, bool ROUND>
int launch_pair_inst(const EdgeNarrowParams& pn, const EdgeWideParams& pw, int store_image, cudaStream_t st) {
  constexpr int CP = NT * 8 + 4;
  const int ksteps_w = (pw.k * pw.k * pw.cimg + 7) / 8;
  const int PR = 2 * pw.OH + pw.k - 2;
  const int col_rows = ((pn.IH * pn.IW + 15) / 16) * 16;
  const size_t smem = (size_t)EN_KSTEPS * NT * 32 * sizeof(float2) + (size_t)ksteps_w * EW_NT * 32 * sizeof(float2) +
                      (size_t)PR * pw.pitch * sizeof(float4) + (size_t)col_rows * CP * sizeof(float);
  {
    static DynSmemCache smem_cache;
    cudaError_t e = ensure_dyn_smem(edge_pair_kernel<NT, CI, MODE, ROUND>, smem, smem_cache);
    if (e != cudaSuccess) return set_error(CGS_ERR_CUDA, "cudaFuncSetAttribute(edge_pair): %s", cudaGetErrorString(e));
  }
  int per_sm = 0;
  cudaError_t e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, edge_pair_kernel<NT, CI, MODE, ROUND>, EN_THREADS, smem);
  if (e != cudaSuccess || per_sm < 1) return set_error(CGS_ERR_CUDA, "edge_pair occupancy query failed");
  long long grid = (long long)num_sms() * per_sm;
  if (grid > pn.B) grid = pn.B;
  e = launch_pdl(edge_pair_kernel<NT, CI, MODE, ROUND>, dim3((unsigned)grid), dim3(EN_THREADS), smem, st, pn, pw, ksteps_w,
                 store_image, fast_div_magic((unsigned)pw.OW));
  count_launch();
  if (e != cudaSuccess) return set_error(CGS_ERR_CUDA, "edge_pair_kernel: %s", cudaGetErrorString(e));
  return check_launch("edge_pair_kernel");
}

template <int NT, int CI>
int launch_pair_mode(const EdgeNarrowParams& pn, const EdgeWideParams& pw, int store_image, cudaStream_t st) {
  const bool rnd = pw.ep.round_out != 0;
  if (pw.ep.mode == EPI_FWD && !pw.ep.act_tanh)
    return rnd ? launch_pair_inst<NT, CI, EM_FWD_SLOPE, true>(pn, pw, store_image, st)
               : launch_pair_inst<NT, CI, EM_FWD_SLOPE, false>(pn, pw, store_image, st);
  if (pw.ep.mode == EPI_BWD && !pw.ep.act_tanh)
    return rnd ? launch_pair_inst<NT, CI, EM_BWD_SLOPE, true>(pn, pw, store_image, st)
               : launch_pair_inst<NT, CI, EM_BWD_SLOPE, false>(pn, pw, store_image, st);
  if (pw.ep.mode == EPI_UPDATE) return launch_pair_inst<NT, CI, EM_UPDATE, false>(pn, pw, store_image, st);
  return launch_pair_inst<NT, CI, EM_GENERIC, false>(pn, pw, store_image, st);
}
}  // namespace

// Of two passes edge_route gives a fused kernel: one image per tile in both, single-channel image, same pitched layout
// on both sides; the shared-memory footprint (column buffer + staged image + two weights) leaves room for 3 CTAs / SM.
bool edge_pair_supported(const EdgeNarrowParams& pn, const EdgeWideParams& pw) {
  if (pn.cimg != 1 || pw.cimg != 1) return false;
  if (pn.IH * pn.IW > EN_ROWS || pw.OH * pw.OW > EW_TILE_PX) return false;
  if (pn.OH != pw.IH || pn.out_pitch != pw.pitch || pn.out_xoff != pw.xoff) return false;
  return true;
}

int launch_edge_pair(EdgeNarrowParams pn, const EdgeWideParams& pw, int store_image, cudaStream_t st) {
  if (pn.B <= 0) return CGS_OK;
  if ((long long)pn.B * pw.OH * pw.OW * pw.ON >= (1ll << 31)) return set_error(CGS_ERR_UNSUPPORTED, "batch too large for 32-bit indexing; split the batch");
  if (int rc = narrow_geometry(pn)) return rc;
  if (pn.k == 4) return launch_pair_mode<2, 1>(pn, pw, store_image, st);
  if (pn.k == 5) return launch_pair_mode<4, 1>(pn, pw, store_image, st);
  return set_error(CGS_ERR_UNSUPPORTED, "edge_pair: unsupported kernel size");
}

int launch_edge_narrow(EdgeNarrowParams p, cudaStream_t st) {
  if (p.B <= 0) return CGS_OK;
  if (int rc = narrow_geometry(p)) return rc;
  if (p.k == 4 && p.cimg == 1) return launch_narrow_nt<2, 1>(p, st);
  if (p.k == 5 && p.cimg == 1) return launch_narrow_nt<4, 1>(p, st);
  if (p.k == 4 && p.cimg == 3) return launch_narrow_nt<6, 3>(p, st);
  if (p.k == 5 && p.cimg == 3) return launch_narrow_nt<10, 3>(p, st);
  return set_error(CGS_ERR_UNSUPPORTED, "edge_narrow: unsupported k / channel combination");
}

}  // namespace cgs
