// edge_narrow_tc: the narrow image-edge pass (64 channels -> image-like output, stride-2 transposed type: the
// generator's last deconv forward, nsgan/ops.py:55, and the data-gradient of the discriminator's first conv,
// sampling/collaborator.py:31) on the 5th-generation tensor cores, with the input PATCH RESIDENT in shared memory.
//
// Gather form: output pixel (2j + py, 2i + px) sums the taps (ky, kx) of matching parity; tap ky reads input row
// j + dy with dy = (py + pad - ky) / 2 in {-1, 0, 1} (pad = 1 for k = 4 and k = 5 under TF SAME), likewise dx.  So for
// the input-grid point (j, i) the 4 output-parity classes x 4 padded channels are 16 GEMM columns and the reduction
// runs over (dy, dx, 64 channels):
//     acc[(j, i)][(py, px, c)] += in[j + dy][i + dx][:] . Wshift[dy][dx][:][(py, px, c)],
// with Wshift zero where a class has no tap at that shift.  mma.sync is throughput-bound on this part (one
// HMMA.1688.TF32 per ~23 cycles per SM sub-partition, ~100 TFLOP/s chip-wide: profiles/round2_ncu_summary.md), so the
// 9x MMA inflation of the gather form made an mma.sync version of it 4x slower than the HBM floor (it was removed).  tcgen05 has the rate, and its shared-memory descriptors make the
// nine shifted A operands FREE: a band of input rows (+ one halo row / column each side, zero-filled by TMA) is loaded
// once as [pixel][32 channels] 128-byte rows (SWIZZLE_128B, two channel halves); the A tile of shift (dy, dx) for the
// 128 "virtual pixels" v .. v+127 is the same memory starting (1 + dy) * pitch + (1 + dx) rows later -- a descriptor
// whose start address is simply advanced by a multiple of 128 bytes (the hardware swizzles on absolute address bits:
// tools/probes/umma_shift_probe.cu).  Virtual pixels run over the halo columns too; those rows are never stored.
//
// CTA = 14 warps, persistent over (image, band) tiles: warp 0 TMA producer (one box per channel half into a ring of
// half-patch stages), warp 1 MMA issuer (tcgen05.mma kind::tf32, M = 128, N = 16, accumulators in TMEM, double-buffered
// per band), warps 2-13 epilogue (tcgen05.ld, bias + tanh or x tanh', pitched float4 stores).  HBM-bound by design:
// every input byte is read once (+ 2 halo rows per band, L2 hits), every output byte written once.
//
// FP16 form (EdgeNarrowParams::in16: the input was stored as FP16 by the pass before it, in an FP16 operand chain): a
// 128-byte row holds all 64 channels, so one TMA box {64 ch, PW, PR, 1} is a whole band and one ring stage; the
// weights are [9 shifts][16 rows][64 k] FP16 (18 KB) and each shift is 4 kind::f16 MMAs (M 128, N 16, K 16) -- half
// the MMAs and half the shared-memory operand reads of the TF32 form over the same row pitch, so the shifted
// descriptors are unchanged.  The epilogue is the same.
#include "edge_conv.cuh"

#include <cuda.h>
#include <cstdint>
#include <cstring>

#include "common.h"
#include "conv_gemm.cuh"
#include "ptx.cuh"

namespace cgs {

namespace {

constexpr int TC_EPI_WARPS = 12;                // three groups of four epilogue warps (one TMEM lane quarter each)
constexpr int TC_THREADS = (2 + TC_EPI_WARPS) * 32;
constexpr int TC_MAX_MT = 4;                   // M tiles (128 virtual pixels) per band
constexpr int TC_B_BYTES = 9 * 2 * 16 * 128;   // weights: [shift][channel half][16 columns][32 k] = 36 KB
constexpr int TC_B16_BYTES = 9 * 16 * 128;     // FP16 form: [shift][16 columns][64 k] = 18 KB
constexpr int TC_SLACK_BYTES = 16 * 1024;      // rows a (never stored) virtual pixel past the band may read

struct NarrowTcParams {
  EdgeNarrowParams p;
  int R, bands, MT, PW, PR;                    // rows per band, bands per image, M tiles per band, patch pitch / rows
  int stage_bytes, nstages, ntiles;
};
// the FP16 form's kernel parameter: an overload of the same kernel, so the TF32 instances stay exactly what they were
struct NarrowTc16Params { NarrowTcParams q; };

// PW (patch pitch = IW + 2) is a template parameter so that every per-MMA descriptor offset is an immediate: the
// single MMA-issuing thread is the serial resource of this kernel (216 MMAs per band), and with run-time offsets each
// MMA cost ~50 cycles of 64-bit address arithmetic and register -> uniform-register moves (11 k cycles per band).
// F16: FP16 input and weights on kind::f16 (one stage per band, 108 MMAs per band).
template <int PW, bool F16>
__device__ __forceinline__ void edge_narrow_tc_body(const NarrowTcParams& q, const CUtensorMap& tmap_in) {
  constexpr int NH = F16 ? 1 : 2;                            // ring stages (channel halves) per band
  constexpr int B_BYTES = F16 ? TC_B16_BYTES : TC_B_BYTES;
  const EdgeNarrowParams& p = q.p;
  extern __shared__ uint8_t tc_smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(tc_smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* smem_b = smem;                                    // [9][NH][16 rows][128 B], swizzled
  uint8_t* smem_a = smem + B_BYTES;                          // ring of (half-)patch stages (+ slack behind the last)
  __shared__ uint64_t full_bar[8], empty_bar[8], tmem_full_bar[2], tmem_empty_bar[2];
  __shared__ uint32_t tmem_ptr_smem;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  // weights -> SWIZZLE_128B K-major tiles: tile (shift, half), row n = (py * 2 + px) * 4 + c, k = channel in the half
  // (FP16: tile (shift), k = channel; converted RN here, like every FP16 operand of the chain)
  for (int idx = threadIdx.x; idx < 9 * NH * 16 * 8; idx += TC_THREADS) {
    const int ck = idx & 7, n = (idx >> 3) & 15, h = F16 ? 0 : (idx >> 7) & 1, sh = idx >> (F16 ? 7 : 8);
    const int dy = sh / 3 - 1, dx = sh % 3 - 1;
    const int py = n >> 3, px = (n >> 2) & 1, c = n & 3;
    const int ky = py + p.pad_y - 2 * dy, kx = px + p.pad_x - 2 * dx;
    const bool tap = c < p.cimg && ky >= 0 && ky < p.k && kx >= 0 && kx < p.k;
    const float* src = p.w + (size_t)((ky * p.k + kx) * 4 + c) * p.K;
    uint8_t* dst = smem_b + ((sh * NH + h) * 16 + n) * 128 + ((ck ^ (n & 7)) << 4);
    if (F16) {
      uint4 v = make_uint4(0u, 0u, 0u, 0u);
      if (tap) {
        const uint2 lo = pack_half4(__ldg(reinterpret_cast<const float4*>(src + ck * 8)));
        const uint2 hi = pack_half4(__ldg(reinterpret_cast<const float4*>(src + ck * 8 + 4)));
        v = make_uint4(lo.x, lo.y, hi.x, hi.y);
      }
      *reinterpret_cast<uint4*>(dst) = v;
    } else {
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (tap) v = __ldg(reinterpret_cast<const float4*>(src + h * 32 + ck * 4));
      *reinterpret_cast<float4*>(dst) = v;
    }
  }
  if (threadIdx.x == 0) {
    for (int s = 0; s < q.nstages; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
    for (int a = 0; a < 2; ++a) { mbar_init(&tmem_full_bar[a], 1); mbar_init(&tmem_empty_bar[a], TC_EPI_WARPS); }
    fence_barrier_init();
  }
  fence_proxy_async_smem();                                  // generic-proxy weight stores -> tensor-core reads
  if (warp == 1) tmem_alloc(&tmem_ptr_smem, 2 * TC_MAX_MT * 16);
  if (warp == 0 && lane == 0) tma_prefetch_desc(&tmap_in);
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem_base = tmem_ptr_smem;
  pdl_launch_dependents();
  pdl_wait();
  int ntiles = q.ntiles;
  if (p.live) ntiles = min(ntiles, live_images(p.live, p.B) * q.bands);

  if (warp == 0) {
    // ------------------------------------------------------------------ TMA producer
    if (elect_one()) {
      uint32_t stage = 0, phase = 0;
      const uint32_t bytes = (uint32_t)q.PR * q.PW * 128u;
      for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const int b = tile / q.bands;
        const int j0 = (tile - b * q.bands) * q.R;
        for (int h = 0; h < NH; ++h) {
          const uint32_t s = stage, ph = phase;
          if (++stage == (uint32_t)q.nstages) { stage = 0; phase ^= 1u; }
          mbar_wait(&empty_bar[s], ph ^ 1);
          mbar_arrive_expect_tx(&full_bar[s], bytes);
          // box {32 channels (FP16: 64), PW pixels from x = -1, PR rows from y = j0 - 1, 1 image}; outside the image
          // reads zeros
          tma_load_4d(smem_u32(smem_a) + s * q.stage_bytes, &tmap_in, &full_bar[s], h * 32, -1, j0 - 1, b);
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------------ MMA issuer
    if (elect_one()) {
      constexpr uint32_t idesc = F16 ? make_idesc_f16(128, 16) : make_idesc_tf32(128, 16);
      const uint64_t da0 = make_smem_desc_sw128(smem_u32(smem_a));
      const uint64_t db0 = make_smem_desc_sw128(smem_u32(smem_b));
      uint32_t stage = 0, phase = 0, tile_count = 0;
      for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x, ++tile_count) {
        const uint32_t acc = tile_count & 1, acc_ph = (tile_count >> 1) & 1;
        mbar_wait(&tmem_empty_bar[acc], acc_ph ^ 1);
        for (int h = 0; h < NH; ++h) {
          const uint32_t s = stage;
          mbar_wait(&full_bar[s], phase);
          if (++stage == (uint32_t)q.nstages) { stage = 0; phase ^= 1u; }
          tcgen05_fence_after();
          const uint64_t da_stage = da0 + (uint64_t)((s * (uint32_t)q.stage_bytes) >> 4);
          const uint64_t db_half = db0 + (uint64_t)(h * ((16 * 128) >> 4));
          // FP16: the stage holds both channel halves; they are still reduced half after half, in the TF32 form's order
#pragma unroll
          for (int hh = 0; hh < (F16 ? 2 : 1); ++hh) {
            for (int mt = 0; mt < q.MT; ++mt) {
              const uint32_t tmem_d = tmem_base + (acc * TC_MAX_MT + mt) * 16;
              const uint64_t da_mt = da_stage + (uint64_t)(mt * ((128 * 128) >> 4));
#pragma unroll
              for (int sh = 0; sh < 9; ++sh) {
                // rows of the A tile = stored pixels 128 mt + dyi * PW + dxi ..: descriptor start in 16-byte units
                constexpr int kRow = 128 >> 4;
                const uint64_t da = da_mt + (uint64_t)(((sh / 3) * PW + (sh % 3)) * kRow);
                const uint64_t db = db_half + (uint64_t)(sh * ((NH * 16 * 128) >> 4));
#pragma unroll
                for (int k = 0; k < (F16 ? 2 : 4); ++k) {      // 32 bytes of the 128-byte row per MMA: K = 8 / 16
                  const uint32_t accum = (h > 0 || hh > 0 || sh > 0 || k > 0) ? 1u : 0u;
                  const int ko = 2 * (hh * 2 + k);              // 16-byte units; a channel half is 64 bytes
                  if (F16) umma_f16_ss(tmem_d, da + ko, db + ko, idesc, accum);
                  else umma_tf32_ss(tmem_d, da + ko, db + ko, idesc, accum);
                }
              }
            }
          }
          umma_commit(&empty_bar[s]);                          // stage reusable once these MMAs have read it
        }
        umma_commit(&tmem_full_bar[acc]);                      // all accumulators of the band complete
      }
    }
  } else {
    // ------------------------------------------------------------------ epilogue: 12 warps (TMEM lane quarter = warp % 4);
    // the three groups of four take the band's M tiles in turn -- the per-pixel epilogue (12 tanh, stores) is a long
    // dependent instruction stream, so warps in flight are what buys throughput here
    const int quarter = warp & 3;
    const int group = (warp - 2) >> 2;
    constexpr int NGROUPS = TC_EPI_WARPS / 4;
    const bool bwd = p.ep.mode == EPI_BWD;
    const float4 bias4 = (p.ep.mode == EPI_FWD && p.ep.bias) ? __ldg(reinterpret_cast<const float4*>(p.ep.bias))
                                                            : make_float4(0.f, 0.f, 0.f, 0.f);
    // the scalar epilogue without the policy step, which no scatter-lowered pass carries (run_pass refuses it)
    auto epi = [&](float v, float x0) {
      float unused;
      return bwd ? epilogue1_t<EPI_BWD>(p.ep, v, x0, 0.f, &unused)
                 : p.ep.mode == EPI_FWD ? epilogue1_t<EPI_FWD>(p.ep, v, x0, 0.f, &unused)
                                        : epilogue1_t<EPI_RAW>(p.ep, v, x0, 0.f, &unused);
    };
    uint32_t tile_count = 0;
    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x, ++tile_count) {
      const int b = tile / q.bands;
      const int j0 = (tile - b * q.bands) * q.R;
      const int j1 = min(p.IH, j0 + q.R);
      const uint32_t acc = tile_count & 1, acc_ph = (tile_count >> 1) & 1;
      bool waited = false;
      for (int mt = group; mt < q.MT; mt += NGROUPS) {
        const int v = 128 * mt + quarter * 32 + lane;          // virtual pixel of this lane
        const int jr = v / q.PW, i = v - jr * q.PW, j = j0 + jr;
        const bool valid = i < p.IW && j < j1;
        // s2d layout: the 16 accumulator columns (py, px, c) of a lane ARE one 64-byte s2d pixel (coalesced rows)
        float* obase = p.s2d ? p.out + (((size_t)b * p.IH + j) * p.IW + i) * 16
                             : p.out + ((size_t)b * p.OH + 2 * j) * p.out_pitch * 4 + (size_t)(2 * i + p.out_xoff) * 4;
        const size_t py_stride = p.s2d ? 8 : (size_t)p.out_pitch * 4;      // floats between the py = 0 and py = 1 pixels
        // derivative operand (the forward image at the four output pixels): in flight while the MMAs still run
        float4 aux[2][2];
        if (bwd && valid) {
          const float* abase = p.ep.aux + (obase - p.out);
#pragma unroll
          for (int py = 0; py < 2; ++py)
#pragma unroll
            for (int px = 0; px < 2; ++px) aux[py][px] = __ldg(reinterpret_cast<const float4*>(abase + py * py_stride + px * 4));
        }
        if (!waited) {
          mbar_wait(&tmem_full_bar[acc], acc_ph);
          tcgen05_fence_after();
          waited = true;
        }
        uint32_t a[16];
        tmem_ld_32x32b_x16(tmem_base + (acc * TC_MAX_MT + mt) * 16 + (static_cast<uint32_t>(quarter * 32) << 16), a);
        tmem_ld_wait();
        if (mt + NGROUPS >= q.MT) {                            // this warp's last accumulator read of the band
          tcgen05_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(&tmem_empty_bar[acc]);
        }
        if (valid) {
#pragma unroll
          for (int py = 0; py < 2; ++py) {
            float* orow = obase + py * py_stride;
#pragma unroll
            for (int px = 0; px < 2; ++px) {
              const int n0 = (py * 2 + px) * 4;
              const float4 x0 = bwd ? aux[py][px] : bias4;
              float4 o;
              o.x = epi(__uint_as_float(a[n0]), x0.x);
              o.y = p.cimg > 1 ? epi(__uint_as_float(a[n0 + 1]), x0.y) : 0.f;
              o.z = p.cimg > 2 ? epi(__uint_as_float(a[n0 + 2]), x0.z) : 0.f;
              o.w = 0.f;
              *reinterpret_cast<float4*>(orow + px * 4) = o;
            }
            if (!p.s2d) {
              // margins of the pitched layout are zeros: written by the lanes at the two ends of the row
              if (i == 0)
                for (int c = 0; c < p.out_xoff; ++c) *reinterpret_cast<float4*>(orow - (size_t)(p.out_xoff - c) * 4) = make_float4(0.f, 0.f, 0.f, 0.f);
              if (i == p.IW - 1)
                for (int c = p.out_xoff + p.OW; c < p.out_pitch; ++c)
                  *reinterpret_cast<float4*>(orow + (size_t)(c - p.out_xoff - 2 * i) * 4) = make_float4(0.f, 0.f, 0.f, 0.f);
            }
          }
        }
      }
      if (group >= q.MT) {                                     // no M tile for this group in the band: arrive all the same
        mbar_wait(&tmem_full_bar[acc], acc_ph);
        tcgen05_fence_after();
        tcgen05_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&tmem_empty_bar[acc]);
      }
    }
  }
  tcgen05_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, 2 * TC_MAX_MT * 16);
}

template <int PW>
__global__ void __launch_bounds__(TC_THREADS, 1)
edge_narrow_tc_kernel(const __grid_constant__ NarrowTcParams q, const __grid_constant__ CUtensorMap tmap_in) {
  edge_narrow_tc_body<PW, false>(q, tmap_in);
}
template <int PW>
__global__ void __launch_bounds__(TC_THREADS, 1)
edge_narrow_tc_kernel(const __grid_constant__ NarrowTc16Params q, const __grid_constant__ CUtensorMap tmap_in) {
  edge_narrow_tc_body<PW, true>(q.q, tmap_in);
}

typedef CUresult (*PFN_encodeTiledTc)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                      const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                      CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
PFN_encodeTiledTc encode_fn() {
  static PFN_encodeTiledTc fn = nullptr;
  if (!fn) {
    void* ptr = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &qres) != cudaSuccess ||
        qres != cudaDriverEntryPointSuccess)
      return nullptr;
    fn = reinterpret_cast<PFN_encodeTiledTc>(ptr);
  }
  return fn;
}

}  // namespace

static bool edge_tc_width_supported(int w) { return w == 16 || w == 32 || w == 64; }   // s2d grid row widths

bool edge_narrow_tc_supported(const EdgeNarrowParams& p) {
  return p.K == 64 && p.pad_y == 1 && p.pad_x == 1 && edge_tc_width_supported(p.IW) && (p.k == 4 || p.k == 5) &&
         p.OW == 2 * p.IW && p.OH == 2 * p.IH && p.cimg >= 1 && p.cimg <= 3;
}

int launch_edge_narrow_tc(const EdgeNarrowParams& p, cudaStream_t st) {
  if (p.B <= 0) return CGS_OK;
  NarrowTcParams q;
  std::memset(&q, 0, sizeof(q));
  q.p = p;
  q.PW = p.IW + 2;
  // rows per band: the largest R <= 16 whose virtual pixels ((R - 1) * PW + IW) fill their 128-row M tiles best
  int bestR = 1;
  double best = -1.0;
  for (int R = 1; R <= 16 && R <= p.IH; ++R) {
    const int valid = (R - 1) * q.PW + p.IW;
    const int mt = (valid + 127) / 128;
    if (mt > TC_MAX_MT) break;
    const int bands = (p.IH + R - 1) / R;
    // cost model: M tiles per image (epilogue work) + a small charge per band (two halo rows re-read)
    const int last = p.IH - (bands - 1) * R;
    const int mt_last = ((last - 1) * q.PW + p.IW + 127) / 128;
    const double cost = (bands - 1) * mt + mt_last + 0.15 * bands;
    const double score = 1.0 / cost;
    if (score > best) { best = score; bestR = R; }
  }
  q.R = bestR;
  q.bands = (p.IH + q.R - 1) / q.R;
  q.PR = q.R + 2;
  q.MT = ((q.R - 1) * q.PW + p.IW + 127) / 128;
  q.stage_bytes = ((q.PR * q.PW * 128 + 1023) / 1024) * 1024;      // 128-byte rows: 32 FP32 or 64 FP16 channels
  const int b_bytes = p.in16 ? TC_B16_BYTES : TC_B_BYTES;
  const int budget = 227 * 1024 - b_bytes - TC_SLACK_BYTES - 2048;
  q.nstages = budget / q.stage_bytes;
  if (q.nstages > 8) q.nstages = 8;
  if (q.nstages < 2) return set_error(CGS_ERR_UNSUPPORTED, "edge_narrow_tc: band does not fit shared memory");
  // a virtual pixel past the band may read up to 128 * MT + 2 * PW + 2 rows from the stage start
  if ((128 * q.MT + 2 * q.PW + 2) * 128 > q.stage_bytes + TC_SLACK_BYTES)
    return set_error(CGS_ERR_UNSUPPORTED, "edge_narrow_tc: slack too small");
  const long long tiles = (long long)p.B * q.bands;
  if (tiles >= (1ll << 31)) return set_error(CGS_ERR_UNSUPPORTED, "batch too large; split the batch");
  q.ntiles = (int)tiles;
  PFN_encodeTiledTc enc = encode_fn();
  if (!enc) return set_error(CGS_ERR_CUDA, "cuTensorMapEncodeTiled entry point not available");
  CUtensorMap tmap;
  const cuuint64_t esz = p.in16 ? 2 : 4;
  cuuint64_t gdim[4] = {64, (cuuint64_t)p.IW, (cuuint64_t)p.IH, (cuuint64_t)p.B};
  cuuint64_t gstr[3] = {64 * esz, (cuuint64_t)p.IW * 64 * esz, (cuuint64_t)p.IH * p.IW * 64 * esz};
  cuuint32_t box[4] = {p.in16 ? 64u : 32u, (cuuint32_t)q.PW, (cuuint32_t)q.PR, 1};   // one 128-byte row per pixel
  cuuint32_t estr[4] = {1, 1, 1, 1};
  CUresult r = enc(&tmap, p.in16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4,
                   const_cast<float*>(p.in), gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return set_error(CGS_ERR_CUDA, "cuTensorMapEncodeTiled (edge_narrow_tc) failed (%d)", (int)r);
  const size_t smem = (size_t)b_bytes + (size_t)q.nstages * q.stage_bytes + TC_SLACK_BYTES + 1024;
  long long grid = tiles < device_num_sms() ? tiles : device_num_sms();
  cudaError_t e = cudaSuccess, le = cudaSuccess;
#define CGS_NARROW_TC_CASE(PWV)                                                                                          \
  case PWV: {                                                                                                            \
    void (*const k32)(NarrowTcParams, CUtensorMap) = edge_narrow_tc_kernel<PWV>;                                         \
    void (*const k16)(NarrowTc16Params, CUtensorMap) = edge_narrow_tc_kernel<PWV>;                                       \
    static DynSmemCache smem_cache, smem_cache16;                                                                        \
    e = p.in16 ? ensure_dyn_smem(k16, smem, smem_cache16) : ensure_dyn_smem(k32, smem, smem_cache);                      \
    if (e == cudaSuccess)                                                                                                \
      le = p.in16 ? launch_pdl(k16, dim3((unsigned)grid), dim3(TC_THREADS), smem, st, NarrowTc16Params{q}, tmap)         \
                  : launch_pdl(k32, dim3((unsigned)grid), dim3(TC_THREADS), smem, st, q, tmap);                          \
  } break;
  switch (q.PW) {
    CGS_NARROW_TC_CASE(18)
    CGS_NARROW_TC_CASE(34)
    CGS_NARROW_TC_CASE(66)
    default: return set_error(CGS_ERR_UNSUPPORTED, "edge_narrow_tc: row width %d", p.IW);
  }
#undef CGS_NARROW_TC_CASE
  if (e != cudaSuccess) return set_error(CGS_ERR_CUDA, "cudaFuncSetAttribute(edge_narrow_tc): %s", cudaGetErrorString(e));
  count_launch();
  if (le != cudaSuccess) return set_error(CGS_ERR_CUDA, "edge_narrow_tc_kernel: %s", cudaGetErrorString(le));
  return check_launch("edge_narrow_tc_kernel");
}


// =====================================================================================================================
// edge_wide_tc: image-like input (s2d layout) -> 64 channels; D's first conv forward (nsgan/ops.py:41) and the
// data-gradient of G's last deconv (sampling/collaborator.py:31), both stride-2 "strided type" passes over the image.
//
// In the s2d layout the k x k stride-2 window of output pixel (oy, ox) is the 3 x 3 neighbourhood of s2d pixel (oy, ox):
//   tap ky reads image row 2 oy + ky - pad = 2 (oy + dy) + ry  with  ky = 2 dy + ry + pad, dy in {-1, 0, 1}, ry in {0, 1}
// so out[(oy, ox)][n] = sum_{dy, dx} s2d[oy + dy][ox + dx][0..15] . W'[dy][dx][0..15][n], W' zero where (ky, kx) falls
// outside the kernel: K = 9 x 16.  The s2d band (+ halo) is resident in shared memory as 64-byte rows (SWIZZLE_64B), the
// A tile of shift (dy, dx) is a descriptor start advanced by (dyi * pitch + dxi) * 64 bytes; 18 MMAs (M 128, N 64, K 8)
// per 128 virtual pixels.  Output rows are transposed through shared memory so global traffic is 64-byte segments.
// =====================================================================================================================
namespace {

constexpr int WT_EPI_WARPS = 12;                 // three groups of four (one TMEM lane quarter each)
constexpr int WT_THREADS = (2 + WT_EPI_WARPS) * 32;
constexpr int WT_B_BYTES = 5 * 64 * 128;          // 18 k-steps of 8 floats -> five [64][32] SWIZZLE_128B tiles
constexpr int WT_PITCH = 20;                      // floats per staged row of the epilogue transpose
constexpr int WT_EPI_BYTES = WT_EPI_WARPS * 2 * 32 * WT_PITCH * 4;   // two staging tiles per warp

// CTA-0 event trace (CGS_DEBUG_TRACE): g_tc_trace[role][tile] = clock; dumped by cgs_debug_trace_tc
__device__ long long g_tc_trace[8][64];
__device__ __forceinline__ void tc_trace(int debug, int role, unsigned tile) {
  if ((debug & CGS_DEBUG_TRACE) && blockIdx.x == 0 && tile < 64) g_tc_trace[role][tile] = clock64();
}

struct WideTcParams {
  const float* in;
  const float* w;
  int B, H2, W2, k, cimg, pad;
  int R, bands, MT, PW, PR, stage_bytes, nstages, ntiles;
  const int* live;
  float* out;              // [B][H2][W2][64], FP16 when ep.out16 (it feeds a kind::f16 MMA; ep.aux is FP16 then too)
  Epilogue ep;
  int debug;               // debug_flags() at launch: CGS_DEBUG_SKIP_*, _NO_PREFETCH, _TRACE
};

__device__ __forceinline__ uint64_t make_smem_desc_sw64(uint32_t smem_addr) {
  const uint32_t lo = (smem_addr >> 4) & 0x3FFFu;
  const uint32_t hi = (512u >> 4) | (1u << 14) | (4u << 29);   // SBO = 512 B (8 rows x 64 B), version 1, SWIZZLE_64B
  return (static_cast<uint64_t>(hi) << 32) | lo;
}

__device__ __forceinline__ void sts_f4(uint32_t addr, float4 v) {
  asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}
__device__ __forceinline__ float4 lds_f4(uint32_t addr) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr) : "memory");
  return v;
}

// PW: patch pitch (see edge_narrow_tc_kernel); EPI: epilogue mode compiled in (the per-element epilogue is a dependent
// instruction stream -- a run-time mode switch per float4 doubled its length); AUX16: the data-gradient pass of an FP16
// operand chain, whose derivative operand is FP16 like its output (Epilogue::out16)
template <int PW, int EPI, bool AUX16>
__device__ __forceinline__ void edge_wide_tc_body(const WideTcParams& q, const CUtensorMap& tmap_in) {
  extern __shared__ uint8_t wt_smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(wt_smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* smem_b = smem;
  float* smem_epi = reinterpret_cast<float*>(smem + WT_B_BYTES);
  uint8_t* smem_a = smem + WT_B_BYTES + ((WT_EPI_BYTES + 1023) / 1024) * 1024;
  __shared__ uint64_t full_bar[8], empty_bar[8], tmem_full_bar[2], tmem_empty_bar[2];
  __shared__ uint32_t tmem_ptr_smem;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  // weights -> [tile = ks / 4][n][32 floats], SWIZZLE_128B; k-step ks = shift * 2 + h holds s2d channels h*8 .. h*8+7
  for (int idx = threadIdx.x; idx < 5 * 64 * 8; idx += WT_THREADS) {
    const int ck = idx & 7, n = (idx >> 3) & 63, tile = idx >> 9;
    float v[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int kk = tile * 32 + ck * 4 + u;            // global k index = shift * 16 + s2d channel
      const int sh = kk >> 4, ch = kk & 15;
      v[u] = 0.f;
      if (sh < 9) {
        const int dy = sh / 3 - 1, dx = sh % 3 - 1;
        const int ry = ch >> 3, rx = (ch >> 2) & 1, c = ch & 3;
        const int ky = 2 * dy + ry + q.pad, kx = 2 * dx + rx + q.pad;
        if (c < q.cimg && ky >= 0 && ky < q.k && kx >= 0 && kx < q.k) v[u] = __ldg(q.w + (size_t)n * (q.k * 32) + ky * 32 + kx * 4 + c);
      }
    }
    *reinterpret_cast<float4*>(smem_b + (tile * 64 + n) * 128 + ((ck ^ (n & 7)) << 4)) = make_float4(v[0], v[1], v[2], v[3]);
  }
  if (threadIdx.x == 0) {
    for (int s = 0; s < q.nstages; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
    for (int a = 0; a < 2; ++a) { mbar_init(&tmem_full_bar[a], 1); mbar_init(&tmem_empty_bar[a], WT_EPI_WARPS); }
    fence_barrier_init();
  }
  fence_proxy_async_smem();
  if (warp == 1) tmem_alloc(&tmem_ptr_smem, 512);
  if (warp == 0 && lane == 0) tma_prefetch_desc(&tmap_in);
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem_base = tmem_ptr_smem;
  pdl_launch_dependents();
  pdl_wait();
  int ntiles = q.ntiles;
  if (q.live) ntiles = min(ntiles, live_images(q.live, q.B) * q.bands);

  if (warp == 0) {
    if (elect_one()) {                                          // TMA producer: one box per (image, band)
      uint32_t stage = 0, phase = 0;
      const uint32_t bytes = (uint32_t)q.PR * q.PW * 64u;
      for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const int b = tile / q.bands;
        const int j0 = (tile - b * q.bands) * q.R;
        const uint32_t s = stage, ph = phase;
        if (++stage == (uint32_t)q.nstages) { stage = 0; phase ^= 1u; }
        mbar_wait(&empty_bar[s], ph ^ 1);
        tc_trace(q.debug, 0, (unsigned)((tile - blockIdx.x) / gridDim.x));
        if (q.debug & CGS_DEBUG_SKIP_A_TMA) { mbar_arrive(&full_bar[s]); continue; }   // profiling knob: no loads
        mbar_arrive_expect_tx(&full_bar[s], bytes);
        tma_load_4d(smem_u32(smem_a) + s * q.stage_bytes, &tmap_in, &full_bar[s], 0, -1, j0 - 1, b);
      }
    }
  } else if (warp == 1) {
    if (elect_one()) {                                          // MMA issuer
      constexpr uint32_t idesc = make_idesc_tf32(128, 64);
      const uint64_t da0 = make_smem_desc_sw64(smem_u32(smem_a));
      const uint64_t db0 = make_smem_desc_sw128(smem_u32(smem_b));
      uint32_t stage = 0, phase = 0, tile_count = 0;
      for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x, ++tile_count) {
        const uint32_t acc = tile_count & 1, acc_ph = (tile_count >> 1) & 1;
        mbar_wait(&tmem_empty_bar[acc], acc_ph ^ 1);
        tc_trace(q.debug, 1, tile_count);
        const uint32_t s = stage;
        mbar_wait(&full_bar[s], phase);
        tc_trace(q.debug, 2, tile_count);
        if (++stage == (uint32_t)q.nstages) { stage = 0; phase ^= 1u; }
        tcgen05_fence_after();
        const uint64_t da_stage = da0 + (uint64_t)((s * (uint32_t)q.stage_bytes) >> 4);
        const bool no_mma = (q.debug & CGS_DEBUG_SKIP_MMA) != 0;             // profiling knob
        for (int mt = 0; mt < q.MT; ++mt) {
          const uint32_t tmem_d = tmem_base + (acc * TC_MAX_MT + mt) * 64;
          const uint64_t da_mt = da_stage + (uint64_t)(mt * ((128 * 64) >> 4));
          if (no_mma) continue;
#pragma unroll
          for (int ks = 0; ks < 18; ++ks) {
            constexpr int kRow = 64 >> 4;
            const int sh = ks >> 1;
            const uint64_t da = da_mt + (uint64_t)(((sh / 3) * PW + (sh % 3)) * kRow + (ks & 1) * 2);
            const uint64_t db = db0 + (uint64_t)((ks >> 2) * (8192 >> 4) + (ks & 3) * 2);
            umma_tf32_ss(tmem_d, da, db, idesc, ks > 0 ? 1u : 0u);
          }
        }
        umma_commit(&empty_bar[s]);
        umma_commit(&tmem_full_bar[acc]);
        tc_trace(q.debug, 3, tile_count);
      }
    }
  } else {
    // ------------------------------------------------------------------ epilogue: 12 warps, three groups take M tiles in turn
    const int ew = warp - 2;
    const int quarter = warp & 3;                  // TMEM lane quarter this warp may read
    const int group = ew >> 2;                     // warps 2-5 / 6-9 / 10-13: each group covers the four quarters
    constexpr int NGROUPS = WT_EPI_WARPS / 4;
    const uint32_t stg = smem_u32(smem_epi) + (uint32_t)ew * (2 * 32 * WT_PITCH * 4);
    const int c4 = lane & 3, rsub = lane >> 2;     // transposed access: 8 rows x 4 float4 per pass
    uint32_t tile_count = 0;
    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x, ++tile_count) {
      const int b = tile / q.bands;
      const int j0 = (tile - b * q.bands) * q.R;
      const int j1 = min(q.H2, j0 + q.R);
      const uint32_t acc = tile_count & 1, acc_ph = (tile_count >> 1) & 1;
      bool waited = false;
      for (int mt = group; mt < q.MT; mt += NGROUPS) {
        const bool last_mt = mt + NGROUPS >= q.MT;
        // output offsets of the 4 rows this lane stores per chunk (rows ps * 8 + rsub of the warp's 32)
        int ro[4];
#pragma unroll
        for (int ps = 0; ps < 4; ++ps) {
          const int v = 128 * mt + quarter * 32 + ps * 8 + rsub;
          const int jr = v / q.PW, i = v - jr * q.PW, j = j0 + jr;
          ro[ps] = (i < q.W2 && j < j1) ? (((b * q.H2 + j) * q.W2 + i) * 64) : -1;
        }
        // epilogue operands of all four 16-channel chunks, fetched before the accumulator wait (their latency hides
        // behind the MMAs of this tile): forward output (derivative; FP16 in the AUX16 form) / feature + momentum
        // (policy step) / bias
        float4 x0[4][4];
        uint2 x0h[4][4];
#pragma unroll
        for (int ch = 0; ch < 4; ++ch) {
          const int n = ch * 16 + c4 * 4;
          if (EPI == EPI_BWD) {
#pragma unroll
            for (int ps = 0; ps < 4; ++ps)
              if (AUX16)                                        // kept packed until used: the loads stay in flight
                x0h[ch][ps] = (ro[ps] >= 0 && !(q.debug & CGS_DEBUG_NO_PREFETCH))
                                  ? __ldg(reinterpret_cast<const uint2*>(reinterpret_cast<const __half*>(q.ep.aux) + ro[ps] + n))
                                  : make_uint2(0x3C003C00u, 0x3C003C00u);
              else
                x0[ch][ps] = (ro[ps] >= 0 && !(q.debug & CGS_DEBUG_NO_PREFETCH)) ? __ldg(reinterpret_cast<const float4*>(q.ep.aux + ro[ps] + n))
                                                                : make_float4(1.f, 1.f, 1.f, 1.f);   // knob 2048: no operand loads
          } else if (EPI == EPI_FWD) {
            x0[ch][0] = q.ep.bias ? __ldg(reinterpret_cast<const float4*>(q.ep.bias + n)) : make_float4(0.f, 0.f, 0.f, 0.f);
          }
        }
        if (!waited) {
          if (warp == 2 && lane == 0) tc_trace(q.debug, 4, tile_count);
          mbar_wait(&tmem_full_bar[acc], acc_ph);
          tcgen05_fence_after();
          waited = true;
          if (warp == 2 && lane == 0) tc_trace(q.debug, 5, tile_count);
        }
        const uint32_t taddr = tmem_base + (acc * TC_MAX_MT + mt) * 64 + (static_cast<uint32_t>(quarter * 32) << 16);
        // policy step / raw gradient of an FP16 operand chain: remove the head's scale 2^gexp[b] of this image
        const float gscale = ((EPI == EPI_UPDATE || EPI == EPI_RAW) && q.ep.gexp) ? exp2_neg(__ldg(q.ep.gexp + b)) : 1.f;
#pragma unroll
        for (int cp = 0; cp < 2; ++cp) {                        // two 16-channel chunks per round
          uint32_t a[2][16];
          tmem_ld_32x32b_x16(taddr + (2 * cp) * 16, a[0]);
          tmem_ld_32x32b_x16(taddr + (2 * cp + 1) * 16, a[1]);
          tmem_ld_wait();
          if (cp == 1 && last_mt) {                             // this warp's last accumulator read of the tile
            tcgen05_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&tmem_empty_bar[acc]);
          }
#pragma unroll
          for (int u = 0; u < 2; ++u)
#pragma unroll
            for (int q4 = 0; q4 < 4; ++q4)
              sts_f4(stg + ((u * 32 + lane) * WT_PITCH + q4 * 4) * 4,
                     make_float4(__uint_as_float(a[u][4 * q4]), __uint_as_float(a[u][4 * q4 + 1]), __uint_as_float(a[u][4 * q4 + 2]),
                                 __uint_as_float(a[u][4 * q4 + 3])));
          __syncwarp();
#pragma unroll
          for (int u = 0; u < 2; ++u) {
            const int ch = 2 * cp + u;
            const int n = ch * 16 + c4 * 4;
#pragma unroll
            for (int ps = 0; ps < 4; ++ps) {
              float4 v = lds_f4(stg + ((u * 32 + ps * 8 + rsub) * WT_PITCH + c4 * 4) * 4);
              if (EPI == EPI_UPDATE || EPI == EPI_RAW) { v.x *= gscale; v.y *= gscale; v.z *= gscale; v.w *= gscale; }
              if (ro[ps] >= 0) {
                float4 xa = EPI == EPI_FWD ? x0[ch][0] : AUX16 ? unpack_half4(x0h[ch][ps]) : x0[ch][ps];
                float4 xb = make_float4(0.f, 0.f, 0.f, 0.f);
                if (EPI == EPI_UPDATE) {         // policy step (only when the G tail is this single layer): not prefetched
                  xa = *reinterpret_cast<const float4*>(q.out + ro[ps] + n);
                  if (!q.ep.sgd && !q.ep.first) xb = *reinterpret_cast<const float4*>(q.ep.mom + ro[ps] + n);
                }
                const float4 o = epilogue4_t<EPI>(q.ep, ro[ps] + n, v, xa, xb);
                if (q.debug & CGS_DEBUG_SKIP_STORES) continue;
                if ((EPI == EPI_FWD || EPI == EPI_BWD) && q.ep.out16)
                  *reinterpret_cast<uint2*>(reinterpret_cast<__half*>(q.out) + ro[ps] + n) = pack_half4(o);
                else
                  *reinterpret_cast<float4*>(q.out + ro[ps] + n) = o;
              }
            }
          }
          __syncwarp();
        }
      }
      if (warp == 2 && lane == 0) tc_trace(q.debug, 6, tile_count);
      if (!waited || group >= q.MT) {
        // a group without an M tile in this band still owes the buffer its arrivals
        if (!waited) { mbar_wait(&tmem_full_bar[acc], acc_ph); tcgen05_fence_after(); }
        tcgen05_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&tmem_empty_bar[acc]);
      }
    }
  }
  tcgen05_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, 512);
}

template <int PW, int EPI>
__global__ void __launch_bounds__(WT_THREADS, 1)
edge_wide_tc_kernel(const __grid_constant__ WideTcParams q, const __grid_constant__ CUtensorMap tmap_in) {
  edge_wide_tc_body<PW, EPI, false>(q, tmap_in);
}
// the FP16-derivative form (EPI_BWD only): an overload of the same kernel, so the other instances stay what they were
struct WideTc16Params { WideTcParams q; };
template <int PW, int EPI>
__global__ void __launch_bounds__(WT_THREADS, 1)
edge_wide_tc_kernel(const __grid_constant__ WideTc16Params q, const __grid_constant__ CUtensorMap tmap_in) {
  edge_wide_tc_body<PW, EPI, true>(q.q, tmap_in);
}

// dense [B][H][W][4] <-> s2d [B][H/2][W/2][16]: one float4 (pixel) per thread
__global__ void __launch_bounds__(256) s2d_convert_kernel(const float4* __restrict__ src, float4* __restrict__ dst, int H, int W,
                                                          long long pixels, int to_s2d) {
  for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < pixels; idx += (long long)gridDim.x * blockDim.x) {
    const int x = (int)(idx % W);
    const long long t = idx / W;
    const int y = (int)(t % H);
    const long long b = t / H;
    const long long sidx = ((b * (H / 2) + (y >> 1)) * (W / 2) + (x >> 1)) * 4 + ((y & 1) * 2 + (x & 1));
    if (to_s2d) dst[sidx] = src[idx]; else dst[idx] = src[sidx];
  }
}

}  // namespace

int image_to_s2d(const float* dense, float* s2d, long long B, int H, int W, cudaStream_t st) {
  const long long px = B * H * W;
  long long blocks = (px + 255) / 256;
  if (blocks > 148 * 16) blocks = 148 * 16;
  if (px > 0) { s2d_convert_kernel<<<(int)blocks, 256, 0, st>>>((const float4*)dense, (float4*)s2d, H, W, px, 1); count_launch(); }
  return check_launch("image_to_s2d");
}
int s2d_to_image(const float* s2d, float* dense, long long B, int H, int W, cudaStream_t st) {
  const long long px = B * H * W;
  long long blocks = (px + 255) / 256;
  if (blocks > 148 * 16) blocks = 148 * 16;
  if (px > 0) { s2d_convert_kernel<<<(int)blocks, 256, 0, st>>>((const float4*)s2d, (float4*)dense, H, W, px, 0); count_launch(); }
  return check_launch("s2d_to_image");
}

int debug_trace_tc(long long* out_host) {
  cudaDeviceSynchronize();
  return cudaMemcpyFromSymbol(out_host, g_tc_trace, sizeof(long long) * 8 * 64) == cudaSuccess ? 8 * 64 : -1;
}

bool edge_wide_tc_supported(const EdgeWideParams& p, int image_w) {
  return p.N == 64 && p.ON == 64 && (p.k == 4 || p.k == 5) && p.cimg >= 1 && p.cimg <= 3 && p.pad_y == 1 && p.pad_x == 1 &&
         p.OH * 2 == p.IH && p.OW * 2 == image_w && edge_tc_width_supported(p.OW);
}

// p.in must be the s2d form of the image-like input; p.pitch / p.xoff are ignored
int launch_edge_wide_tc(const EdgeWideParams& p, int B, cudaStream_t st) {
  if (B <= 0) return CGS_OK;
  WideTcParams q;
  std::memset(&q, 0, sizeof(q));
  q.in = p.in; q.w = p.w; q.B = B; q.H2 = p.OH; q.W2 = p.OW; q.k = p.k; q.cimg = p.cimg; q.pad = p.pad_y;
  q.live = p.live;
  q.PW = q.W2 + 2;
  int bestR = 1;
  double best = 1e30;
  for (int R = 1; R <= 16 && R <= q.H2; ++R) {
    const int mt = ((R - 1) * q.PW + q.W2 + 127) / 128;
    if (mt > TC_MAX_MT) break;
    const int bands = (q.H2 + R - 1) / R;
    const int last = q.H2 - (bands - 1) * R;
    const double cost = (bands - 1) * mt + ((last - 1) * q.PW + q.W2 + 127) / 128 + 0.15 * bands;
    if (cost < best) { best = cost; bestR = R; }
  }
  q.R = bestR;
  q.bands = (q.H2 + q.R - 1) / q.R;
  q.PR = q.R + 2;
  q.MT = ((q.R - 1) * q.PW + q.W2 + 127) / 128;
  q.stage_bytes = ((q.PR * q.PW * 64 + 1023) / 1024) * 1024;
  const int fixed = WT_B_BYTES + ((WT_EPI_BYTES + 1023) / 1024) * 1024 + TC_SLACK_BYTES + 2048;
  q.nstages = (227 * 1024 - fixed) / q.stage_bytes;
  if (q.nstages > 6) q.nstages = 6;
  if (q.nstages < 2) return set_error(CGS_ERR_UNSUPPORTED, "edge_wide_tc: band does not fit shared memory");
  if ((128 * q.MT + 2 * q.PW + 2) * 64 > q.stage_bytes + TC_SLACK_BYTES) return set_error(CGS_ERR_UNSUPPORTED, "edge_wide_tc: slack too small");
  const long long tiles = (long long)B * q.bands;
  if (tiles >= (1ll << 31) || (long long)B * q.H2 * q.W2 * 64 >= (1ll << 31)) return set_error(CGS_ERR_UNSUPPORTED, "batch too large; split the batch");
  q.ntiles = (int)tiles;
  q.out = p.out;
  q.ep = p.ep;
  q.debug = debug_flags();
  PFN_encodeTiledTc enc = encode_fn();
  if (!enc) return set_error(CGS_ERR_CUDA, "cuTensorMapEncodeTiled entry point not available");
  CUtensorMap tmap;
  cuuint64_t gdim[4] = {16, (cuuint64_t)q.W2, (cuuint64_t)q.H2, (cuuint64_t)B};
  cuuint64_t gstr[3] = {16 * 4, (cuuint64_t)q.W2 * 16 * 4, (cuuint64_t)q.H2 * q.W2 * 16 * 4};
  cuuint32_t box[4] = {16, (cuuint32_t)q.PW, (cuuint32_t)q.PR, 1};
  cuuint32_t estr[4] = {1, 1, 1, 1};
  CUresult r = enc(&tmap, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, const_cast<float*>(p.in), gdim, gstr, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return set_error(CGS_ERR_CUDA, "cuTensorMapEncodeTiled (edge_wide_tc) failed (%d)", (int)r);
  const size_t smem = (size_t)fixed - 2048 + (size_t)q.nstages * q.stage_bytes + 1024;
  long long grid = tiles < device_num_sms() ? tiles : device_num_sms();
  cudaError_t e = cudaSuccess, le = cudaSuccess;
  const bool aux16 = q.ep.mode == EPI_BWD && q.ep.out16;
#define CGS_WIDE_TC_CASE(PWV, EPIV)                                                                                      \
  case PWV * 8 + EPIV: {                                                                                                 \
    void (*const k32)(WideTcParams, CUtensorMap) = edge_wide_tc_kernel<PWV, EPIV>;                                       \
    static DynSmemCache smem_cache;                                                                                      \
    e = ensure_dyn_smem(k32, smem, smem_cache);                                                                          \
    if (e == cudaSuccess) le = launch_pdl(k32, dim3((unsigned)grid), dim3(WT_THREADS), smem, st, q, tmap);               \
  } break;
#define CGS_WIDE_TC_CASE16(PWV)                                                                                          \
  case PWV * 8 + EPI_BWD: {                                                                                              \
    void (*const k16)(WideTc16Params, CUtensorMap) = edge_wide_tc_kernel<PWV, EPI_BWD>;                                  \
    static DynSmemCache smem_cache;                                                                                      \
    e = ensure_dyn_smem(k16, smem, smem_cache);                                                                          \
    if (e == cudaSuccess)                                                                                                \
      le = launch_pdl(k16, dim3((unsigned)grid), dim3(WT_THREADS), smem, st, WideTc16Params{q}, tmap);                   \
  } break;
#define CGS_WIDE_TC_PW(PWV) CGS_WIDE_TC_CASE(PWV, EPI_FWD) CGS_WIDE_TC_CASE(PWV, EPI_BWD) CGS_WIDE_TC_CASE(PWV, EPI_UPDATE) CGS_WIDE_TC_CASE(PWV, EPI_RAW)
  if (aux16) {
    switch (q.PW * 8 + q.ep.mode) {
      CGS_WIDE_TC_CASE16(18)
      CGS_WIDE_TC_CASE16(34)
      CGS_WIDE_TC_CASE16(66)
      default: return set_error(CGS_ERR_UNSUPPORTED, "edge_wide_tc: row width %d", q.W2);
    }
  } else {
    switch (q.PW * 8 + q.ep.mode) {
      CGS_WIDE_TC_PW(18)
      CGS_WIDE_TC_PW(34)
      CGS_WIDE_TC_PW(66)
      default: return set_error(CGS_ERR_UNSUPPORTED, "edge_wide_tc: row width %d / epilogue %d", q.W2, q.ep.mode);
    }
  }
#undef CGS_WIDE_TC_PW
#undef CGS_WIDE_TC_CASE16
#undef CGS_WIDE_TC_CASE
  if (e != cudaSuccess) return set_error(CGS_ERR_CUDA, "cudaFuncSetAttribute(edge_wide_tc): %s", cudaGetErrorString(e));
  count_launch();
  if (le != cudaSuccess) return set_error(CGS_ERR_CUDA, "edge_wide_tc_kernel: %s", cudaGetErrorString(le));
  return check_launch("edge_wide_tc_kernel");
}

}  // namespace cgs
