// Image-edge passes: the four layer passes that touch the generated image (<= 3 channels) -- the generator's last
// deconv forward, the discriminator's first conv forward and the data-gradients of both.  They carry ~5 % of the
// FLOPs of a refinement step but move as many bytes as the big layers (K or N is only k*k*C_img), so they are
// HBM-bound streaming kernels, not tcgen05 work: plain many-CTA kernels with mma.sync TF32 fragments, operands
// straight from global memory / L1, and everything around the GEMM (im2col, col2im, bias, activation, derivative,
// policy step) fused so each activation byte is read or written exactly once.
//
//   edge_wide   : image-like input [B][IH][pitch][4] -> [B][OH][OW][64]   (conv forward / deconv data-gradient)
//   edge_narrow : [B][IH][IW][64] -> image-like output [B][2IH][pitch][4] (deconv forward / conv data-gradient)
#pragma once
#include <cuda_runtime.h>

#include "conv_gemm.cuh"

namespace cgs {

// images a kernel of the chain has to process (grids stay sized for the full batch; see ConvGemmParams::live)
__device__ __forceinline__ int live_images(const int* live, int B) {
  if (!live) return B;
  const int b = *reinterpret_cast<const volatile int*>(live);
  return b < 0 ? 0 : (b > B ? B : b);
}

struct EdgeWideParams {
  const float* in;    // pitched image-like tensor
  float* out;         // [M][ON]
  const float* w;     // window layout: [N][k*32], element (n, ky*32 + kx*4 + c)
  int IH, pitch, xoff, OH, OW, ON, N, k, cimg, pad_y, pad_x;
  long long M;        // B*OH*OW
  Epilogue ep;
  const int* live;    // early exit: device-resident number of images still in the batch (null = all of them)
};

struct EdgeNarrowParams {
  const float* in;    // [B][IH][IW][K]
  float* out;         // image-like [B][OH][out_pitch][4]
  const float* w;     // scatter layout: [k*k*4][K], row (ky*k + kx)*4 + c
  int B, IH, IW, K, OH, OW, k, cimg, pad_y, pad_x, out_pitch, out_xoff;
  int R, halo_lo, halo_hi, bands;   // input rows per tile, extra rows read above / below, tiles per image
  int s2d;            // 1: out (and ep.aux) are in the space-to-depth image layout [B][IH][IW][16] (see edge_tc.cu)
  Epilogue ep;
  const int* live;    // early exit: device-resident number of images still in the batch (null = all of them)
  int in16;           // in is FP16 (it was stored for a kind::f16 MMA): only the tcgen05 kernel takes it (edge_tc.cu)
};

bool edge_wide_supported(const EdgeWideParams& p);
bool edge_narrow_supported(const EdgeNarrowParams& p);
int launch_edge_wide(const EdgeWideParams& p, cudaStream_t st);
int launch_edge_narrow(EdgeNarrowParams p, cudaStream_t st);
// the same pass on tcgen05 with the input patch resident in shared memory (edge_tc.cu)
bool edge_narrow_tc_supported(const EdgeNarrowParams& p);
int launch_edge_narrow_tc(const EdgeNarrowParams& p, cudaStream_t st);
// the wide pass (image-like input -> 64 channels, stride-2 strided type) on tcgen05 over the SPACE-TO-DEPTH image
// layout [B][H/2][W/2][16], channel (ry * 2 + rx) * 4 + c = image pixel (2j + ry, 2i + rx, c): the k x k stride-2 conv
// becomes a 3 x 3 stride-1 conv over 16 channels, which the resident-patch / shifted-descriptor scheme covers
bool edge_wide_tc_supported(const EdgeWideParams& p, int image_w);   // image_w: width of the image-like input
int launch_edge_wide_tc(const EdgeWideParams& p, int B, cudaStream_t st);
// dense [B][H][W][4] <-> space-to-depth [B][H/2][W/2][16]
int image_to_s2d(const float* dense, float* s2d, long long B, int H, int W, cudaStream_t st);
int s2d_to_image(const float* s2d, float* dense, long long B, int H, int W, cudaStream_t st);
// narrow pass + the wide pass that consumes its output, one image per tile, in one kernel (edge_pair_kernel);
// store_image = 0 keeps the intermediate image-like tensor out of global memory (backward pair)
bool edge_pair_supported(const EdgeNarrowParams& pn, const EdgeWideParams& pw);
int launch_edge_pair(EdgeNarrowParams pn, const EdgeWideParams& pw, int store_image, cudaStream_t st);

}  // namespace cgs
