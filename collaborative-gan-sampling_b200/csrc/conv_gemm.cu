// tcgen05 / TMEM implicit-GEMM kernel (TF32 or FP16 inputs, FP32 accumulate) + an FP32 SIMT twin used by the
// parity tests and as the exact-FP32 mode.  See conv_gemm.cuh for the contraction it computes.
//
// CTA = 15 warps, persistent over output tiles (128 rows x BN channels):
//   warps 0-3   epilogue: tcgen05.ld the accumulator (TMEM lane = row), transpose through padded smem so that
//               global loads/stores are 64-byte row segments, fused bias/activation/derivative/momentum update
//   warps 4-11  TMA mode (every layer with >= 32 input channels): two more epilogue groups.  Up to BN = 128 each
//               group owns whole tiles, at BN = 256 the three groups split one tile's 16-column chunks.
//               Gather mode (pixel layout, <= 4 channels): A producers, cp.async gather of 128 rows x 128 B per K
//               block into SWIZZLE_128B smem
//   warp  12    MMA issuer (one elected lane of a warp-uniform loop): 4 x tcgen05.mma.kind::tf32 (K=8) or kind::f16
//               (K=16) per K atom
//   warp  13    TMA producer for the weight tile (one 3-D box {32, BN, KB} per stage, SWIZZLE_128B)
//   warp  14    TMA producer for the A tile (one 4-D box per K atom with traversal strides, or the window map)
// Pipelines: full/empty mbarriers per smem stage (3-8 stages, 1-2 K atoms each), tmem_full/tmem_empty per
// accumulator buffer (ring of 4 x BN TMEM columns, 2 at BN = 256: tile epilogues overlap the following main loops).
// CGS_DEBUG knobs (cgs_debug_flag): CGS_DEBUG_GATHER_A forces gather mode; profiling: CGS_DEBUG_SKIP_A_GATHER,
// _SKIP_WEIGHT_TMA, _SKIP_A_TMA, _SKIP_MMA, _SKIP_EPILOGUE, _SKIP_STORES, _NO_PREFETCH, _TRACE (built with CGS_TRACE).
#include "conv_gemm.cuh"
#include "ptx.cuh"
#include "common.h"

#include <cuda.h>
#include <cstdlib>
#include <cstring>

namespace cgs {

// ---- optional event trace of CTA 0 (CGS_DEBUG_TRACE): (role, event, index, clock) records for pipeline analysis
__device__ unsigned long long g_trace[32768];
__device__ unsigned int g_trace_n;
__device__ __forceinline__ void trace(const ConvGemmParams& p, int role, int ev, unsigned idx) {
#ifdef CGS_TRACE
  // fixed slot per (role, event, index): a plain store, no atomics, so the traced thread is barely perturbed
  if ((p.debug & CGS_DEBUG_TRACE) && blockIdx.x == 0 && idx < 1024) {
    const unsigned slot = ((unsigned)(role * 4 + ev) << 10) + idx;
    g_trace[slot & 32767] = ((unsigned long long)role << 60) | ((unsigned long long)ev << 56) |
                            ((unsigned long long)(idx & 0xffffff) << 32) | (unsigned long long)(unsigned)clock64();
  }
#else
  (void)p; (void)role; (void)ev; (void)idx;      // build with CGS_NVCC_EXTRA=-DCGS_TRACE to record the trace
#endif
}

namespace {

constexpr int BM = 128;
constexpr int BK = 32;                       // floats per K block = one 128-byte swizzle row
constexpr int kEpiWarps = 4;
constexpr int kProdWarps = 8;
constexpr int kMmaWarp = kEpiWarps + kProdWarps;       // 12
constexpr int kTmaWarp = kMmaWarp + 1;                 // 13: weight tiles
constexpr int kTmaWarpA = kMmaWarp + 2;                // 14: A tiles (TMA mode)
constexpr int kThreads = (kTmaWarpA + 1) * 32;         // 480
constexpr int kRowsPerThread = BM / (kProdWarps * 4);  // 4
constexpr int A_ATOM_BYTES = BM * BK * 4;    // 16 KB: 128 rows x one 128-byte swizzle row
constexpr int EPI_CH = 16;                   // accumulator columns per TMEM load / staging pass
constexpr int EPI_PITCH = 20;                // floats per staged row (16-byte aligned; STS.128 by row is conflict-free)
constexpr int kMaxEpiWarps = kEpiWarps + kProdWarps;              // producer warps help in TMA mode
constexpr int EPI_STAGE_BYTES = kMaxEpiWarps * 32 * EPI_PITCH * 4;   // 30 KB

constexpr int K_STEPS = 4;                   // MMAs per K atom: 32 bytes each (K = 8 TF32 or K = 16 FP16)

template <int CG, bool F16>
__device__ __forceinline__ void umma(uint32_t tmem_d, uint64_t da, uint64_t db, uint32_t idesc, uint32_t accumulate) {
  if (F16) {
    if (CG == 2) umma_f16_ss_cg2(tmem_d, da, db, idesc, accumulate); else umma_f16_ss(tmem_d, da, db, idesc, accumulate);
  } else {
    if (CG == 2) umma_tf32_ss_cg2(tmem_d, da, db, idesc, accumulate); else umma_tf32_ss(tmem_d, da, db, idesc, accumulate);
  }
}
__host__ __device__ constexpr uint32_t make_idesc(bool f16, uint32_t M, uint32_t N) {
  return f16 ? make_idesc_f16(M, N) : make_idesc_tf32(M, N);
}
template <int CG>
__device__ __forceinline__ void commit(uint64_t* bar) {
  if (CG == 2) umma_commit_cg2(bar); else umma_commit(bar);
}

template <int BN, int NS = 1, int MT = 1, int CG = 1>
struct Cfg {
  // K blocks ("atoms" of 32 floats) per pipeline stage: the per-stage barrier handshakes of the single-thread TMA and
  // MMA roles cost ~400 cycles, so narrow tiles (short MMAs) take two atoms per stage to amortise them.  A class-fused
  // stage (NS > 1 accumulator slots per tile) is one A atom plus one weight atom per slot.
  // MT = 2: a CTA tile is a PAIR of adjacent M tiles that share every weight atom (one A atom per M tile, one weight
  // atom per stage): 0.75x (BN = 128) / 0.83x (BN = 64) of the L2 -> SM bytes per FLOP of one-tile stages, which is
  // what bounds these passes (profiles/round2_ncu_summary.md C4)
  // CG = 2: the CTA is one of a PAIR (cluster of two, tcgen05 cta_group::2, M = 256): each CTA loads its own M tile
  // and HALF the rows of every weight atom; the leader's MMAs read both halves.  Per CTA a stage is 16 KB of A plus
  // half the weights, so the ring is 6 stages deep where single CTAs get 4 (the load latency of ~1-2 k cycles is what
  // the 4-stage ring does not cover, profiles/round2_ncu_summary.md D2), and L2 delivers each weight byte once per pair.
  static constexpr int KB = (NS > 1 || MT > 1 || BN >= 256 || CG > 1) ? 1 : 2;
  static constexpr int B_ATOM_BYTES = BN * BK * 4 / CG;          // per CTA
  static constexpr int A_STAGE_BYTES = (MT > 1 ? MT : KB) * A_ATOM_BYTES;
  static constexpr int B_STAGE_BYTES = (NS > 1 ? NS : KB) * B_ATOM_BYTES;
  static constexpr int STAGE_BYTES = A_STAGE_BYTES + B_STAGE_BYTES;
  static constexpr int STAGES = (196608 / STAGE_BYTES) > 8 ? 8 : (196608 / STAGE_BYTES);
  // accumulator ring in TMEM: 4 buffers up to BN = 128 (512 columns), 2 for BN = 256; fused tiles take NS * BN
  // columns per buffer (two buffers)
  static constexpr int ACC_COLS = NS * MT * BN;
  static constexpr int NACC = (NS > 1 || MT > 1) ? 512 / ACC_COLS : ((BN >= 256) ? 2 : 4);
  static_assert(NS == 1 || MT == 1, "class fusion and M-tile pairs are separate modes");
  static_assert(CG == 1 || CG == 2, "clusters of one or two CTAs");
  static_assert(MT == 1 || (MT == 2 && BN <= 128), "M-tile pairs need 2 * BN TMEM columns per buffer, two buffers");
  static constexpr int TMEM_COLS = NACC * ACC_COLS;
  static_assert(NS == 1 || (ACC_COLS <= 256 && BN <= 128), "fused tiles need two TMEM buffers");
  // up to BN = 128 each epilogue warp group owns whole tiles (three tile epilogues in flight per CTA, the per-tile
  // set-up paid by 4 warps instead of 12); at BN = 256 the groups split the 16 chunks of one tile
  static constexpr bool SPLIT_TILES = (BN <= 128);
  static constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + EPI_STAGE_BYTES + 1024 /*align*/ + 256 /*barriers*/;
};

// F16: FP16 operands on kind::f16.  A 128-byte K atom holds 64 channels instead of 32, and one K = 16 MMA step covers
// the same 32 bytes as a K = 8 TF32 step: stages, ring, TMEM plan and descriptor stepping are those of the TF32 form,
// each stage simply carries twice the K.  The epilogue reads FP16 act' operands and stores FP16 where the output
// feeds another MMA (Epilogue::out16); the policy step removes the head's per-sample gradient scale (Epilogue::gexp).
// OPS: 0 = TF32 operands, FP32 outputs (the form every chain without FP16 operands runs); 1 = TF32 operands in an FP16
// chain (layer 0's forward pass: its output may be FP16); 2 = FP16 operands
template <int BN, int EPI, int NS, int MT, int CG, int OPS>
__device__ __forceinline__ void conv_gemm_tc_body(const ConvGemmParams& p, const CUtensorMap& tmap_w, const CUtensorMap& tmap_a) {
  using C = Cfg<BN, NS, MT, CG>;
  constexpr bool F16 = OPS == 2;
  constexpr int AK = F16 ? 64 : BK;            // channels per K atom
  constexpr bool FUSED = NS > 1;
  constexpr bool PAIR = MT > 1;
  constexpr bool CG2 = CG == 2;
  // CTA pair: both CTAs walk the same tile sequence (unit = two adjacent M tiles, this CTA takes tile 2 * unit + rank);
  // full / accumulator-free barriers live in the leader (rank 0), smem-slot-free and accumulator-full barriers are
  // signalled in both CTAs by the leader's multicast commits
  const uint32_t cta_rank = CG2 ? cluster_ctarank() : 0u;
  const bool leader = cta_rank == 0;
  const int tile_first = CG2 ? (int)(blockIdx.x >> 1) : (int)blockIdx.x;
  const int tile_stride = CG2 ? (int)(gridDim.x >> 1) : (int)gridDim.x;
  extern __shared__ uint8_t smem_raw[];
  // SWIZZLE_128B operands need 1024-byte aligned stage bases
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* smem_a = smem;
  uint8_t* smem_b = smem + C::STAGES * C::A_STAGE_BYTES;
  float* smem_epi = reinterpret_cast<float*>(smem + C::STAGES * C::STAGE_BYTES);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + C::STAGES * C::STAGE_BYTES + EPI_STAGE_BYTES);
  uint64_t* full_bar = bars;
  uint64_t* empty_bar = bars + C::STAGES;
  uint64_t* tmem_full_bar = bars + 2 * C::STAGES;
  uint64_t* tmem_empty_bar = bars + 2 * C::STAGES + C::NACC;
  uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(bars + 2 * C::STAGES + 2 * C::NACC);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  if (threadIdx.x == 0) {
    for (int s = 0; s < C::STAGES; ++s) {
      // TMA mode: one arrive.expect_tx from each of the two TMA warps; gather mode: weight TMA warp + the async
      // arrive of every producer thread
      mbar_init(&full_bar[s], p.a_tma ? 2 : kProdWarps * 32 + 1);
      mbar_init(&empty_bar[s], 1);
    }
    for (int a = 0; a < C::NACC; ++a) {
      mbar_init(&tmem_full_bar[a], 1);
      // one arrive per epilogue warp that reads the buffer: the 4 warps of one group, or all groups at BN = 256
      // (fused tiles: two TMEM buffers but three epilogue groups -- whole-tile ownership would let a group run two
      //  buffer uses ahead and alias the barrier parity, so the groups share every tile's chunks instead)
      // (CTA pair: the leader's barrier collects the epilogue warps of both CTAs)
      mbar_init(&tmem_empty_bar[a], CG * ((p.a_tma && (!C::SPLIT_TILES || C::NACC < 3)) ? kMaxEpiWarps : kEpiWarps));
    }
    fence_barrier_init();
  }
  if (warp == kMmaWarp) {
    if (CG2) tmem_alloc_cg2(tmem_ptr_smem, C::TMEM_COLS); else tmem_alloc(tmem_ptr_smem, C::TMEM_COLS);
  }
  if (warp == kTmaWarp && lane == 0) tma_prefetch_desc(&tmap_w);
  if (warp == kTmaWarpA && lane == 0 && p.a_tma) tma_prefetch_desc(&tmap_a);
  tcgen05_fence_before();
  __syncthreads();
  if (CG2) cluster_sync_all();                   // the partner's barriers are initialised before anything signals them
  tcgen05_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;
  // set-up done: let the next kernel of the chain start its own set-up, then wait for our predecessor's results
  pdl_launch_dependents();
  pdl_wait();

  // tile counts follow the images still in the batch (device-resident count in early-exit mode, else p.B)
  const LiveTiles lt = live_tiles(p);
  const int tiles_per_class = lt.tiles_per_class;
  const int total_tiles = lt.total;
  const unsigned long long fd_tpc = lt.fd_tiles_per_class;
  const int B_live = lt.B;
  const int m_tiles_live = ((B_live + p.BB - 1) / p.BB) * p.hy_tiles;   // M tiles that hold live images
  const int rows_per_img_tile = p.BH * p.MW;   // rows one image contributes to a tile

  if (warp >= kEpiWarps && warp < kMmaWarp && !p.a_tma) {
    // ------------------------------------------------------------------ A producers (gather mode only)
    {
    const int pw = warp - kEpiWarps;
    const int chunk = lane & 7;           // 16-byte chunk inside the 128-byte row
    const int rsub = lane >> 3;           // 0..3
    const uint32_t smem_a_u32 = smem_u32(smem_a);
    const bool pixel_mode = (p.cblocks == 0);
    uint32_t soff[kRowsPerThread];        // swizzled smem offset of (row, chunk) inside a stage
#pragma unroll
    for (int it = 0; it < kRowsPerThread; ++it) {
      const int r = pw * (4 * kRowsPerThread) + it * 4 + rsub;
      soff[it] = r * 128 + ((chunk ^ (r & 7)) << 4);
    }
    uint32_t it_global = 0;               // K blocks issued by this thread
    for (int tile = tile_first; tile < total_tiles; tile += tile_stride) {
      const int ci = tile / tiles_per_class;
      const int rem = tile - ci * tiles_per_class;
      const int m_tile = rem / p.n_tiles;
      const GemmClass& gc = p.cls[ci];
      int rbase[kRowsPerThread];
      uint32_t vmask[kRowsPerThread];     // bit t set <=> tap t of this row lies inside the image
#pragma unroll
      for (int it = 0; it < kRowsPerThread; ++it) {
        const int r = pw * (4 * kRowsPerThread) + it * 4 + rsub;
        rbase[it] = 0;
        vmask[it] = 0;
        const int bb = r / rows_per_img_tile;
        const int q = r - bb * rows_per_img_tile;
        const int hh = q / p.MW;
        const int i = q - hh * p.MW;
        const int b = (m_tile / p.hy_tiles) * p.BB + bb;
        const int j = (m_tile % p.hy_tiles) * p.BH + hh;
        if (r < p.rows_valid && b < B_live && j < p.MH) {
          const int y0 = j * p.S, x0 = i * p.S;
          rbase[it] = ((b * p.IH + y0) * p.IW + x0) * p.Cs;
          uint32_t vm = 0;                    // (taps need not form a ky x kx grid in their enumeration order)
          for (int tp = 0; tp < gc.ntaps; ++tp)
            if ((unsigned)(y0 + gc.dy[tp]) < (unsigned)p.IH && (unsigned)(x0 + gc.dx[tp]) < (unsigned)p.IW) vm |= 1u << tp;
          vmask[it] = vm;
        }
      }
      int t = 0, cb = 0;                  // block mode: current tap / channel block
      int tap_off = pixel_mode ? 0 : (gc.dy[0] * p.IW + gc.dx[0]) * p.Cs;
      for (int kb = 0; kb < gc.nkb; kb += C::KB, ++it_global) {
        const int s = it_global % C::STAGES;
        const uint32_t ph = (it_global / C::STAGES) & 1;
        mbar_wait(&empty_bar[s], ph ^ 1);
        if (pw == 0 && lane == 0) trace(p, 0, 0, it_global);
#pragma unroll
        for (int a = 0; a < C::KB; ++a) {
          if (kb + a >= gc.nkb) break;
          int off, tt;
          if (pixel_mode) {
            tt = (kb + a) * 8 + chunk;    // one tap (4 channels = 16 B) per chunk
            const bool tap_ok = tt < gc.ntaps;
            off = tap_ok ? (gc.dy[tt] * p.IW + gc.dx[tt]) * p.Cs : 0;
            if (!tap_ok) tt = 31;         // bit 31 is never set (ntaps <= 25)
          } else {
            tt = t;
            off = tap_off + (cb + gc.cb0) * BK + chunk * 4;
          }
          const uint32_t atom_base = smem_a_u32 + s * C::A_STAGE_BYTES + a * A_ATOM_BYTES;
          if (!(p.debug & CGS_DEBUG_SKIP_A_GATHER)) {
#pragma unroll
            for (int it = 0; it < kRowsPerThread; ++it) {
              const bool ok = (vmask[it] >> tt) & 1u;
              cp_async_16(atom_base + soff[it], p.in + (ok ? rbase[it] + off : 0), ok ? 16u : 0u);
            }
          }
          if (!pixel_mode && ++cb == p.cblocks) {
            cb = 0;
            ++t;
            if (t < gc.ntaps) tap_off = (gc.dy[t] * p.IW + gc.dx[t]) * p.Cs;
          }
        }
        // the copies of this thread arrive on the stage's full barrier when they land: no wait on the issue side,
        // so up to STAGES stages of gathers are in flight per CTA
        cp_async_mbar_arrive_noinc(&full_bar[s]);
        if (pw == 0 && lane == 0) trace(p, 0, 1, it_global);
      }
    }
    }  // !a_tma
  } else if (warp == kTmaWarp) {
    // ------------------------------------------------------------------ TMA producer: weight tiles
    // whole warp walks the loop (uniform control flow); one elected lane issues.  The weight matrix is viewed as
    // {32, rows, K/32} so ONE box {32, BN, KB} fetches all K atoms of a stage as consecutive atom tiles.
    const uint32_t smem_b_u32 = smem_u32(smem_b);
    if (FUSED) {
      // the whole warp walks the loop: lane 0 waits for the slot and posts the byte count, then lane q issues the box
      // of the q-th class with a tap at the shift (a single thread issuing up to four boxes per stage was the slowest
      // role of the fused tiles: 45 us of a 210 us pass)
      const bool skip = (p.debug & CGS_DEBUG_SKIP_WEIGHT_TMA) != 0;
      uint32_t stage = 0, phase = 0;
      for (int tile = tile_first; tile < total_tiles; tile += tile_stride) {
        const int ci = fast_div(tile, fd_tpc);
        const int rem = tile - ci * tiles_per_class;
        const int n_tile = rem - fast_div(rem, p.fd_n_tiles) * p.n_tiles;
        const FuseGroup& G = p.grp[ci];
        for (int si = 0; si < G.nshifts; ++si) {
          const FuseShift& sh = p.shf[G.shift0 + si];
          const int ncls = sh.ncls;
          const bool mine = lane < ncls;
          const int q = mine ? lane : 0;
          const uint32_t dst = (CG2 ? sh.pc_slot[cta_rank][q] : sh.slot[q]) * C::B_ATOM_BYTES;
          const int row = n_tile * BN + (CG2 ? sh.pc_half[cta_rank][q] * (BN / 2) : 0);
          const int katom = CG2 ? sh.pc_katom[cta_rank][q] : sh.katom0[q];
          for (int cb = 0; cb < p.cblocks; ++cb) {
            const uint32_t s = stage, ph = phase;
            if (++stage == C::STAGES) { stage = 0; phase ^= 1u; }
            if (lane == 0) {
              mbar_wait(&empty_bar[s], ph ^ 1);
              if (skip) { if (leader) mbar_arrive(&full_bar[s]); }
              else if (leader) mbar_arrive_expect_tx(&full_bar[s], (uint32_t)(ncls * CG) * C::B_ATOM_BYTES);
            }
            __syncwarp();
            if (mine && !skip) {
              if (CG2) tma_load_3d_cg2(smem_b_u32 + s * C::B_STAGE_BYTES + dst, &tmap_w, &full_bar[s], 0, row, katom + cb);
              else tma_load_3d(smem_b_u32 + s * C::B_STAGE_BYTES + dst, &tmap_w, &full_bar[s], 0, row, katom + cb);
            }
          }
        }
      }
    } else
    if (elect_one()) {                     // one thread walks the whole loop: no per-K-block election or warp sync
      uint32_t it_global = 0;
      uint32_t stage = 0, phase = 0;
      const bool skip = (p.debug & CGS_DEBUG_SKIP_WEIGHT_TMA) != 0;
      for (int tile = tile_first; tile < total_tiles; tile += tile_stride) {
        const int ci = fast_div(tile, fd_tpc);
        const int rem = tile - ci * tiles_per_class;
        const int n_tile = rem - fast_div(rem, p.fd_n_tiles) * p.n_tiles;
        const int katom0 = p.cls[ci].k0 / AK;
        const int nkb = p.cls[ci].nkb;
        for (int kb = 0; kb < nkb; kb += C::KB, ++it_global) {
          const uint32_t s = stage, ph = phase;
          if (++stage == C::STAGES) { stage = 0; phase ^= 1u; }
          mbar_wait(&empty_bar[s], ph ^ 1);
          trace(p, 1, 0, it_global);
          if (skip) {
            if (leader) mbar_arrive(&full_bar[s]);
          } else if (CG2) {                      // this CTA's half of the BN rows
            if (leader) mbar_arrive_expect_tx(&full_bar[s], 2u * C::B_STAGE_BYTES);
            tma_load_3d_cg2(smem_b_u32 + s * C::B_STAGE_BYTES, &tmap_w, &full_bar[s], 0, n_tile * BN + (int)cta_rank * (BN / 2),
                            katom0 + kb);
          } else {
            mbar_arrive_expect_tx(&full_bar[s], C::B_STAGE_BYTES);
            tma_load_3d(smem_b_u32 + s * C::B_STAGE_BYTES, &tmap_w, &full_bar[s], 0, n_tile * BN, katom0 + kb);
          }
        }
      }
    }
  } else if (warp == kTmaWarpA) {
    // ------------------------------------------------------------------ TMA producer: A tiles (TMA mode only)
    if (p.a_tma) {
      const uint32_t smem_a_u32 = smem_u32(smem_a);
      const uint32_t a_bytes = (uint32_t)p.rows_valid * 128u;
      if (elect_one()) {                   // one thread walks the whole loop
        uint32_t stage = 0, phase = 0;
        const bool skip = (p.debug & CGS_DEBUG_SKIP_A_TMA) != 0;
        const int cblocks = p.cblocks;
        for (int tile = tile_first; tile < total_tiles; tile += tile_stride) {
          const int ci = fast_div(tile, fd_tpc);
          const int rem = tile - ci * tiles_per_class;
          const int m_unit = fast_div(rem, p.fd_n_tiles);
          const int m_tile = CG2 ? 2 * m_unit + (int)cta_rank : m_unit;   // (a pair's odd tile may lie past the batch:
          const int mb = fast_div(m_tile, p.fd_hy_tiles);                 //  its box is out of range and reads zeros)
          const int b0 = mb * p.BB;
          const int y_tile = (m_tile - mb * p.hy_tiles) * p.BH * p.S;
          if (FUSED) {
            const FuseGroup& G = p.grp[ci];
            for (int si = 0; si < G.nshifts; ++si) {
              const FuseShift& sh = p.shf[G.shift0 + si];
              for (int cb = 0; cb < cblocks; ++cb) {
                const uint32_t s = stage, ph = phase;
                if (++stage == C::STAGES) { stage = 0; phase ^= 1u; }
                mbar_wait(&empty_bar[s], ph ^ 1);
                if (skip) {
                  if (leader) mbar_arrive(&full_bar[s]);
                } else if (CG2) {
                  if (leader) mbar_arrive_expect_tx(&full_bar[s], 2u * a_bytes);
                  tma_load_4d_cg2(smem_a_u32 + s * C::A_STAGE_BYTES, &tmap_a, &full_bar[s], cb * AK, sh.dx, y_tile + sh.dy, b0);
                } else {
                  mbar_arrive_expect_tx(&full_bar[s], a_bytes);
                  tma_load_4d(smem_a_u32 + s * C::A_STAGE_BYTES, &tmap_a, &full_bar[s], cb * AK, sh.dx, y_tile + sh.dy, b0);
                }
              }
            }
            continue;
          }
          const GemmClass& gc = p.cls[ci];
          const int nkb = gc.nkb;
          const int cb0 = gc.cb0;
          int t = 0, cb = 0;
          if (PAIR) {
            // m_tile above is the PAIR index: M tiles 2 * pair and 2 * pair + 1 (the last pair may be half empty)
            const int mt0 = 2 * m_tile;
            const int mbA = fast_div(mt0, p.fd_hy_tiles), mbB = fast_div(mt0 + 1, p.fd_hy_tiles);
            const int b0A = mbA * p.BB, yA = (mt0 - mbA * p.hy_tiles) * p.BH * p.S;
            const int b0B = mbB * p.BB, yB = (mt0 + 1 - mbB * p.hy_tiles) * p.BH * p.S;
            const bool second = CG2 || mt0 + 1 < m_tiles_live;   // (CTA pairs: always both, a box past the batch reads zeros)
            for (int kb = 0; kb < nkb; ++kb) {
              const uint32_t s = stage, ph = phase;
              if (++stage == C::STAGES) { stage = 0; phase ^= 1u; }
              mbar_wait(&empty_bar[s], ph ^ 1);
              if (skip) {
                if (leader) mbar_arrive(&full_bar[s]);
              } else if (CG2) {
                if (leader) mbar_arrive_expect_tx(&full_bar[s], 4u * a_bytes);
                tma_load_4d_cg2(smem_a_u32 + s * C::A_STAGE_BYTES, &tmap_a, &full_bar[s], (cb + cb0) * AK, gc.dx[t], yA + gc.dy[t], b0A);
                tma_load_4d_cg2(smem_a_u32 + s * C::A_STAGE_BYTES + A_ATOM_BYTES, &tmap_a, &full_bar[s], (cb + cb0) * AK, gc.dx[t],
                                yB + gc.dy[t], b0B);
              } else {
                mbar_arrive_expect_tx(&full_bar[s], second ? 2u * a_bytes : a_bytes);
                tma_load_4d(smem_a_u32 + s * C::A_STAGE_BYTES, &tmap_a, &full_bar[s], (cb + cb0) * AK, gc.dx[t], yA + gc.dy[t], b0A);
                if (second)
                  tma_load_4d(smem_a_u32 + s * C::A_STAGE_BYTES + A_ATOM_BYTES, &tmap_a, &full_bar[s], (cb + cb0) * AK, gc.dx[t],
                              yB + gc.dy[t], b0B);
              }
              if (++cb == cblocks) { cb = 0; ++t; }
            }
            continue;
          }
          for (int kb = 0; kb < nkb; kb += C::KB) {
            const uint32_t s = stage, ph = phase;
            if (++stage == C::STAGES) { stage = 0; phase ^= 1u; }
            const int na = (nkb - kb) < C::KB ? (nkb - kb) : C::KB;       // atoms in this stage
            mbar_wait(&empty_bar[s], ph ^ 1);
            if (skip) {
              if (leader) mbar_arrive(&full_bar[s]);
            } else if (leader) {
              mbar_arrive_expect_tx(&full_bar[s], (uint32_t)(CG * na) * a_bytes);
            }
#pragma unroll
            for (int a = 0; a < C::KB; ++a) {
              if (a >= na) break;
              // one box = BB images x BH rows x MW columns x 32 channels; out-of-image pixels read as zero
              if (!skip) {
                if (CG2)
                  tma_load_4d_cg2(smem_a_u32 + s * C::A_STAGE_BYTES + a * A_ATOM_BYTES, &tmap_a, &full_bar[s],
                                  (cb + cb0) * AK, gc.dx[t], y_tile + gc.dy[t], b0);
                else
                tma_load_4d(smem_a_u32 + s * C::A_STAGE_BYTES + a * A_ATOM_BYTES, &tmap_a, &full_bar[s],
                            (cb + cb0) * AK, gc.dx[t], y_tile + gc.dy[t], b0);
              }
              if (++cb == cblocks) {
                cb = 0;
                ++t;
              }
            }
          }
        }
      }
    }
  } else if (warp == kMmaWarp) {
    // ------------------------------------------------------------------ MMA issuer
    // whole warp walks the loop (uniform control flow); one elected lane issues the tcgen05 instructions
    constexpr uint32_t idesc = make_idesc(F16, BM * CG, BN);
    const uint64_t da0 = make_smem_desc_sw128(smem_u32(smem_a));
    const uint64_t db0 = make_smem_desc_sw128(smem_u32(smem_b));
    // The loop body is kept minimal (ring position kept incrementally, parameters hoisted, no trace code unless
    // built with CGS_TRACE): the issuing thread runs in lock-step with the tensor pipe, so every instruction here is
    // a bubble between K blocks.  Releasing a stage one K block late (commit after the next block's MMAs) was
    // measured and is slower: ring depth (3-4 stages) matters more than the issue bubble.
    if (elect_one() && leader) {               // one thread (of the pair's leader) walks the whole loop
    uint32_t it_global = 0;
    uint32_t tile_count = 0;
    uint32_t stage = 0, phase = 0;               // position in the smem ring
    const bool a_tma = p.a_tma != 0;
    const bool skip_mma = (p.debug & CGS_DEBUG_SKIP_MMA) != 0;
    for (int tile = tile_first; tile < total_tiles; tile += tile_stride, ++tile_count) {
      const int ci = fast_div(tile, fd_tpc);
      const uint32_t acc = tile_count % C::NACC;
      const uint32_t acc_ph = (tile_count / C::NACC) & 1;
      mbar_wait(&tmem_empty_bar[acc], acc_ph ^ 1);
      const uint32_t tmem_d = tmem_base + acc * C::ACC_COLS;
      if (FUSED) {
        const FuseGroup& G = p.grp[ci];
        for (int si = 0; si < G.nshifts; ++si) {
          const FuseShift& sh = p.shf[G.shift0 + si];
          // the runs of this shift, decoded once for all channel blocks (the issuing thread is the slowest role of the
          // stages with one or two classes: 64 - 256 cycles of tensor work against a loop of ~350)
          const int nrun = sh.nrun;
          uint32_t r_tm[4], r_db[4], r_idesc[4], r_acc[4];
#pragma unroll
          for (int r = 0; r < 4; ++r) {
            const uint32_t slot = sh.run_slot[r];
            r_tm[r] = slot * BN;
            r_db[r] = slot * (C::B_ATOM_BYTES >> 4);
            r_idesc[r] = make_idesc(F16, BM * CG, BN * sh.run_len[r]);
            r_acc[r] = sh.run_acc[r];
          }
          for (int cb = 0; cb < p.cblocks; ++cb, ++it_global) {
            const uint32_t s = stage;
            const bool last = (si == G.nshifts - 1) && (cb == p.cblocks - 1);
            mbar_wait(&full_bar[s], phase);
            if (++stage == C::STAGES) { stage = 0; phase ^= 1u; }
            tcgen05_fence_after();
            trace(p, 2, 0, it_global);
            const uint64_t da = da0 + (uint64_t)(s * (C::A_STAGE_BYTES >> 4));
            const uint64_t db = db0 + (uint64_t)(s * (C::B_STAGE_BYTES >> 4));
            if (!skip_mma) {
#pragma unroll
              for (int r = 0; r < 4; ++r) {
                if (r >= nrun) break;
                // one MMA of N = run_len * BN columns per k-step: adjacent class slots = adjacent TMEM columns and
                // adjacent weight atoms in the stage, the A tile is read once for all of them
                const uint32_t had = (cb > 0) ? 1u : r_acc[r];
#pragma unroll
                for (int k = 0; k < K_STEPS; ++k)
                  umma<CG, F16>(tmem_d + r_tm[r], da + 2 * k, db + r_db[r] + 2 * k, r_idesc[r], (had || k > 0) ? 1u : 0u);
              }
            }
            commit<CG>(&empty_bar[s]);
            if (last) commit<CG>(&tmem_full_bar[acc]);
            trace(p, 2, 1, it_global);
          }
        }
        continue;
      }
      const int nkb = p.cls[ci].nkb;
      for (int kb = 0; kb < nkb; kb += C::KB, ++it_global) {
        const uint32_t s = stage;
        const int na = (nkb - kb) < C::KB ? (nkb - kb) : C::KB;
        const bool last = kb + C::KB >= nkb;
        mbar_wait(&full_bar[s], phase);
        if (++stage == C::STAGES) { stage = 0; phase ^= 1u; }
        tcgen05_fence_after();
        trace(p, 2, 0, it_global);
        // cp.async (generic proxy) writes -> tensor-core (async proxy) reads
        if (!a_tma) fence_proxy_async_smem();
        // descriptor address field is in 16-byte units: + stage / atom offset, + 32 bytes per K=8 step
        const uint64_t da = da0 + (uint64_t)(s * (C::A_STAGE_BYTES >> 4));
        const uint64_t db = db0 + (uint64_t)(s * (C::B_STAGE_BYTES >> 4));
        if (!skip_mma) {
#pragma unroll
          for (int a = 0; a < C::KB; ++a) {
            if (a >= na) break;
#pragma unroll
            for (int k = 0; k < K_STEPS; ++k)
              umma<CG, F16>(tmem_d, da + a * (A_ATOM_BYTES >> 4) + 2 * k, db + a * (C::B_ATOM_BYTES >> 4) + 2 * k, idesc,
                       (kb > 0 || a > 0 || k > 0) ? 1u : 0u);
            if (PAIR) {                        // second M tile of the pair: its own A atom, the SAME weight atom
#pragma unroll
              for (int k = 0; k < K_STEPS; ++k)
                umma<CG, F16>(tmem_d + BN, da + (A_ATOM_BYTES >> 4) + 2 * k, db + 2 * k, idesc, (kb > 0 || k > 0) ? 1u : 0u);
            }
          }
        }
        commit<CG>(&empty_bar[s]);                             // smem stage reusable once these MMAs have read it
        if (last) commit<CG>(&tmem_full_bar[acc]);             // accumulator complete
        trace(p, 2, 1, it_global);
      }
    }
    }
  } else {
    // ------------------------------------------------------------------ epilogue
    // warps 0-3 always; in TMA mode the 8 idle producer warps join as two more groups.  A warp may only touch the
    // TMEM lane quarter (warp % 4).  Up to BN = 128 a group owns whole tiles (tile_count % groups), so three tile
    // epilogues overlap and a tile's set-up is paid by 4 warps; at BN = 256 the groups split one tile's chunks.
    constexpr int Q = EPI_CH / 4;                  // float4 per staged row
    constexpr int ROWS_PER_PASS = 32 / Q;          // rows covered by one warp-wide 16-byte access
    constexpr int PASSES = 32 / ROWS_PER_PASS;
    constexpr int NCH = BN / EPI_CH;
    constexpr int MAXOWN = NCH >= 2 ? 2 : 1;       // chunks pulled out of TMEM per batch (2 x 16 registers)
    const int quarter = warp & 3;
    const int group = warp >> 2;                   // 0..2
    const int ngroups = p.a_tma ? kMaxEpiWarps / 4 : 1;
    constexpr bool kSplitTiles = C::SPLIT_TILES && C::NACC >= 3;   // whole-tile ownership needs >= 3 TMEM buffers
    const int tile_groups = kSplitTiles ? ngroups : 1;       // groups that take separate tiles
    const int chunk_groups = kSplitTiles ? 1 : ngroups;      // groups that share the chunks of one tile
    float* stage = smem_epi + warp * 32 * EPI_PITCH;
    const bool dbg_skip_epi = (p.debug & CGS_DEBUG_SKIP_EPILOGUE) != 0, dbg_skip_store = (p.debug & CGS_DEBUG_SKIP_STORES) != 0;
    const bool dbg_no_prefetch = (p.debug & CGS_DEBUG_NO_PREFETCH) != 0;
    const int c4 = lane % Q;
    const int rsub = lane / Q;
    // tile-invariant part of the row -> output offset map of the PASSES rows this lane stores
    // (a tile spans either several whole images, BB > 1, or part of one image, BB == 1: one bound test per row)
    const bool multi_img = p.BB > 1;
    const int lim = multi_img ? B_live : p.MH;
    int l_off[PASSES], l_pos[PASSES];
#pragma unroll
    for (int ps = 0; ps < PASSES; ++ps) {
      const int r = quarter * 32 + ps * ROWS_PER_PASS + rsub;
      const int bb = r / rows_per_img_tile;
      const int q = r - bb * rows_per_img_tile;
      const int hh = q / p.MW;
      const int i = q - hh * p.MW;
      l_off[ps] = ((bb * p.OH + hh * p.os) * p.OW + i * p.os) * p.ON;
      l_pos[ps] = r < p.rows_valid ? (multi_img ? bb : hh) : (1 << 28);   // padding rows never pass the bound test
    }
    for (uint32_t tile_count = kSplitTiles ? group : 0;; tile_count += tile_groups) {
      const int tile = tile_first + (int)tile_count * tile_stride;
      if (tile >= total_tiles) break;
      const int ci = fast_div(tile, fd_tpc);
      const int rem = tile - ci * tiles_per_class;
      const int m_unit = fast_div(rem, p.fd_n_tiles);          // M tile, or M-tile pair
      const int n_tile = rem - m_unit * p.n_tiles;
      const uint32_t acc = tile_count % C::NACC;
      const uint32_t acc_ph = (tile_count / C::NACC) & 1;
      // a fused tile holds one accumulator per class of its group (slots): the same epilogue runs once per slot with
      // that class's output offsets; the TMEM buffer goes back to the MMA warp after the last slot has been read
      const int nslots = FUSED ? p.grp[ci].ncls : (PAIR ? ((CG2 || 2 * m_unit + 1 < m_tiles_live) ? 2 : 1) : 1);
      bool waited = false;
      for (int slot = 0; slot < nslots; ++slot) {
      const int cls_i = FUSED ? p.grp[ci].cls[slot] : ci;
      const bool last_slot = slot == nslots - 1;
      // M-tile pair: slot = which M tile of the pair; CTA pair: this CTA's tile of the unit
      const int m_tile = PAIR ? (CG2 ? 4 * m_unit + 2 * (int)cta_rank + slot : 2 * m_unit + slot)
                              : (CG2 ? 2 * m_unit + (int)cta_rank : m_unit);
      const bool tile_live = !CG2 || m_tile < m_tiles_live;    // the odd tile of the last CTA pair may not exist
      const int mb = fast_div(m_tile, p.fd_hy_tiles);
      const int b0 = mb * p.BB;
      const int j0 = (m_tile - mb * p.hy_tiles) * p.BH;
      // first chunk of this warp's group (rotated per slot so the three groups get equal shares of a fused tile)
      const int chunk_first = kSplitTiles ? 0 : ((FUSED || PAIR) ? (group + slot) % ngroups : group);
      const int t_off = ((b0 * p.OH + j0 * p.os + p.cls[cls_i].oy0) * p.OW + p.cls[cls_i].ox0) * p.ON;
      int ro[PASSES];                              // element offset of each stored row in out / aux / mom, -1 = none
#pragma unroll
      for (int ps = 0; ps < PASSES; ++ps)
        ro[ps] = (tile_live && (multi_img ? b0 : j0) + l_pos[ps] < lim) ? t_off + l_off[ps] : -1;
      // chunks of this tile that hold valid output channels (ON is a multiple of 4; the tail of the last n tile and
      // the zero columns of a narrow N are never read out of TMEM)
      const int n0 = n_tile * BN;
      const int nch = (p.ON - n0) >= BN ? NCH : (p.ON - n0 + EPI_CH - 1) / EPI_CH;
      // epilogue operands (bias / forward output / feature + momentum) of a chunk, fetched ahead of its use
      float4 x0[PASSES], x1[PASSES];
      auto prefetch = [&](int ch) {
        const int n = n0 + ch * EPI_CH + c4 * 4;
        if (ch >= nch || n >= p.ON) return;
        if (EPI == EPI_BWD) {
#pragma unroll
          for (int ps = 0; ps < PASSES; ++ps)
            if (ro[ps] >= 0)
              x0[ps] = F16 ? unpack_half4(__ldg(reinterpret_cast<const uint2*>(reinterpret_cast<const __half*>(p.ep.aux) + ro[ps] + n)))
                           : __ldg(reinterpret_cast<const float4*>(p.ep.aux + ro[ps] + n));
        } else if (EPI == EPI_UPDATE) {
#pragma unroll
          for (int ps = 0; ps < PASSES; ++ps)
            if (ro[ps] >= 0) {
              x0[ps] = *reinterpret_cast<const float4*>(p.out + ro[ps] + n);
              if (!p.ep.sgd && !p.ep.first) x1[ps] = *reinterpret_cast<const float4*>(p.ep.mom + ro[ps] + n);
            }
        } else if (EPI == EPI_FWD) {
          x0[0] = p.ep.bias ? __ldg(reinterpret_cast<const float4*>(p.ep.bias + n)) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
      };
      prefetch(chunk_first);                       // in flight while the main loop of this tile still runs
      if (!waited) {
        mbar_wait(&tmem_full_bar[acc], acc_ph);
        if (warp == 0 && lane == 0) trace(p, 3, 0, tile_count);
        tcgen05_fence_after();
        waited = true;
      }
      // FP16 chains: the gradient of this lane's TMEM row (sample b) carries the head's scale 2^gexp[b]; it is removed
      // (exactly) as the row is staged, before the policy step.  The factor waits in the staging row's padding column
      // (EPI_PITCH > EPI_CH), not in a register held across the chunk loop.
      if (F16 && (EPI == EPI_UPDATE || EPI == EPI_RAW)) {
        const int r = quarter * 32 + lane, b = b0 + (multi_img ? r / rows_per_img_tile : 0);
        stage[lane * EPI_PITCH + EPI_CH] =
            (p.ep.gexp && tile_live && r < p.rows_valid && b < B_live) ? exp2_neg(__ldg(p.ep.gexp + b)) : 1.f;
      }
      const uint32_t taddr = tmem_base + acc * C::ACC_COLS + ((FUSED || PAIR) ? slot * BN : 0) + (static_cast<uint32_t>(quarter * 32) << 16);
      bool released = false;
#pragma unroll 1
      for (int ch0 = chunk_first; ch0 < nch || !released; ch0 += chunk_groups * MAXOWN) {
        // pull a batch of this warp's chunks out of TMEM at once; after the last batch give the accumulator back
        // before touching global memory
        uint32_t v[MAXOWN][EPI_CH];
#pragma unroll
        for (int u = 0; u < MAXOWN; ++u)
          if (ch0 + u * chunk_groups < nch) tmem_ld_32x32b_x16(taddr + (ch0 + u * chunk_groups) * EPI_CH, v[u]);
        tmem_ld_wait();
        if (warp == 0 && lane == 0) trace(p, 4, 0, tile_count * 8 + ch0);
        if (ch0 + chunk_groups * MAXOWN >= nch) {
          if (last_slot) {
            tcgen05_fence_before();
            __syncwarp();
            if (lane == 0) {
              if (CG2 && !leader) mbar_arrive_cluster(&tmem_empty_bar[acc], 0); else mbar_arrive(&tmem_empty_bar[acc]);
            }
            if (warp == 0 && lane == 0) trace(p, 3, 1, tile_count);
          }
          released = true;
        }
#pragma unroll
        for (int u = 0; u < MAXOWN; ++u) {
          const int ch = ch0 + u * chunk_groups;
          if (ch >= nch) break;
          if (dbg_skip_epi) continue;                          // warp-uniform
          // lane = row: stage 32 rows x 16 columns, then re-read with lane = (row group, 16-byte column)
          const float gscale = (F16 && (EPI == EPI_UPDATE || EPI == EPI_RAW)) ? stage[lane * EPI_PITCH + EPI_CH] : 1.f;
#pragma unroll
          for (int q4 = 0; q4 < Q; ++q4)
            *reinterpret_cast<float4*>(stage + lane * EPI_PITCH + q4 * 4) =
                (F16 && (EPI == EPI_UPDATE || EPI == EPI_RAW))
                    ? make_float4(__uint_as_float(v[u][4 * q4]) * gscale, __uint_as_float(v[u][4 * q4 + 1]) * gscale,
                                  __uint_as_float(v[u][4 * q4 + 2]) * gscale, __uint_as_float(v[u][4 * q4 + 3]) * gscale)
                    : make_float4(__uint_as_float(v[u][4 * q4]), __uint_as_float(v[u][4 * q4 + 1]),
                                  __uint_as_float(v[u][4 * q4 + 2]), __uint_as_float(v[u][4 * q4 + 3]));
          __syncwarp();
          const int n = n0 + ch * EPI_CH + c4 * 4;
          const bool n_ok = n < p.ON;                // ON is a multiple of 4
          float4 a[PASSES];
#pragma unroll
          for (int ps = 0; ps < PASSES; ++ps)
            a[ps] = *reinterpret_cast<const float4*>(stage + (ps * ROWS_PER_PASS + rsub) * EPI_PITCH + c4 * 4);
          float4 o[PASSES];
#pragma unroll
          for (int ps = 0; ps < PASSES; ++ps)
            if (ro[ps] >= 0 && n_ok) o[ps] = epilogue4_t<EPI>(p.ep, ro[ps] + n, a[ps], EPI == EPI_FWD ? x0[0] : x0[ps], x1[ps]);
          if (warp == 0 && lane == 0) trace(p, 4, 1, tile_count * 8 + ch);
          if (!dbg_no_prefetch) prefetch(ch + chunk_groups);   // operands of the next chunk: overlap with these stores
#pragma unroll
          for (int ps = 0; ps < PASSES; ++ps)
            if (ro[ps] >= 0 && n_ok && !dbg_skip_store) {
              if (OPS > 0 && (EPI == EPI_FWD || EPI == EPI_BWD) && p.ep.out16)
                *reinterpret_cast<uint2*>(reinterpret_cast<__half*>(p.out) + ro[ps] + n) = pack_half4(o[ps]);
              else
                *reinterpret_cast<float4*>(p.out + ro[ps] + n) = o[ps];
            }
          if (warp == 0 && lane == 0) trace(p, 4, 2, tile_count * 8 + ch);
          __syncwarp();
          if (warp == 0 && lane == 0) trace(p, 4, 3, tile_count * 8 + ch);
        }
      }
      }  // slots
      if (warp == 0 && lane == 0) trace(p, 3, 2, tile_count);
    }
  }

  tcgen05_fence_before();
  __syncthreads();
  if (CG2) cluster_sync_all();                   // the leader's MMAs write this CTA's TMEM and barriers until its last commit
  if (warp == kMmaWarp) {
    if (CG2) tmem_dealloc_cg2(tmem_base, C::TMEM_COLS); else tmem_dealloc(tmem_base, C::TMEM_COLS);
  }
}

// One kernel name per tile shape and epilogue mode, two overloads: the passes of an FP16-operand chain take the one
// whose parameter is F16ChainParams, every other pass keeps the TF32-only code unchanged (a kernel that also held the
// FP16 body measured 59.7 k instead of 62.6 k samples/s on the MNIST-sized chain, B200).  In an FP16 chain only the
// forward pass of layer 0 runs TF32 operands (its input is the FP32 feature), and the policy step / raw gradient
// ends a data-gradient chain of strided passes, never a class-fused one: chain_instance() lists the bodies compiled.
struct F16ChainParams { ConvGemmParams p; };
__host__ __device__ constexpr bool chain_instance(int epi, int ns, bool f16) {
  return epi == EPI_FWD || (f16 && (epi == EPI_BWD || ns == 1));
}

template <int BN, int EPI, int NS, int MT, int CG>
__global__ void __launch_bounds__(kThreads, 1)
conv_gemm_tc_kernel(const __grid_constant__ ConvGemmParams p, const __grid_constant__ CUtensorMap tmap_w,
                    const __grid_constant__ CUtensorMap tmap_a) {
  conv_gemm_tc_body<BN, EPI, NS, MT, CG, 0>(p, tmap_w, tmap_a);
}
template <int BN, int EPI, int NS, int MT, int CG>
__global__ void __launch_bounds__(kThreads, 1)
conv_gemm_tc_kernel(const __grid_constant__ F16ChainParams q, const __grid_constant__ CUtensorMap tmap_w,
                    const __grid_constant__ CUtensorMap tmap_a) {
  if constexpr (EPI == EPI_FWD) {
    if (q.p.f16) conv_gemm_tc_body<BN, EPI, NS, MT, CG, 2>(q.p, tmap_w, tmap_a);
    else conv_gemm_tc_body<BN, EPI, NS, MT, CG, 1>(q.p, tmap_w, tmap_a);
  } else if constexpr (chain_instance(EPI, NS, true)) {
    conv_gemm_tc_body<BN, EPI, NS, MT, CG, 2>(q.p, tmap_w, tmap_a);
  }
}

// ---------------------------------------------------------------------------------------------
// FP32 SIMT twin: one thread per (row, 4 output channels); same parameters, same epilogue.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
conv_gemm_simt_kernel(const __grid_constant__ ConvGemmParams p, const float* __restrict__ w, int w_cols) {
  const int ngroups = p.ON / 4;
  int M_live = p.M;
  if (p.live) {                                   // early exit: rows of the images still in the batch
    const int b = *reinterpret_cast<const volatile int*>(p.live);
    const long long m = (long long)(b < 0 ? 0 : b) * p.MH * p.MW;
    if (m < M_live) M_live = (int)m;
  }
  const long long total = (long long)p.nclasses * M_live * ngroups;
  for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total;
       idx += (long long)gridDim.x * blockDim.x) {
    const int ng = (int)(idx % ngroups);
    const long long t = idx / ngroups;
    const int m = (int)(t % M_live);
    const int ci = (int)(t / M_live);
    const GemmClass& gc = p.cls[ci];
    const int per_img = p.MH * p.MW;
    const int b = m / per_img;
    const int q = m - b * per_img;
    const int j = q / p.MW;
    const int i = q - j * p.MW;
    const int cin = p.cblocks ? p.cblocks * BK : 4;
    float acc[4] = {0.f, 0.f, 0.f, 0.f};
    if (p.window) {
      for (int ky = 0; ky < gc.ntaps; ++ky) {
        const int y = j * p.S + gc.dy[ky];
        if ((unsigned)y >= (unsigned)p.IH) continue;
        const float* src = p.in + ((size_t)(b * p.IH + y) * p.in_pitch_px + (i * 2 + p.win_x0)) * 4;
        for (int q = 0; q < p.win_k * 4; ++q) {
          const float a = __ldg(src + q);
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            const int n = ng * 4 + u;
            if (n < p.N) acc[u] = fmaf(a, __ldg(w + (size_t)n * w_cols + gc.k0 + ky * 32 + q), acc[u]);
          }
        }
      }
    } else
    for (int tp = 0; tp < gc.ntaps; ++tp) {
      const int y = j * p.S + gc.dy[tp];
      const int x = i * p.S + gc.dx[tp];
      if ((unsigned)y >= (unsigned)p.IH || (unsigned)x >= (unsigned)p.IW) continue;
      const float* src = p.in + ((size_t)(b * p.IH + y) * p.IW + x) * p.Cs;
      for (int c = 0; c < cin; ++c) {
        const float a = __ldg(src + c);
        const int k = gc.k0 + tp * cin + c;             // (split-K classes are a tensor-core-path lowering only)
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const int n = ng * 4 + u;
          if (n < p.N) acc[u] = fmaf(a, __ldg(w + (size_t)n * w_cols + k), acc[u]);
        }
      }
    }
    const int row_off = ((b * p.OH + j * p.os + gc.oy0) * p.OW + (i * p.os + gc.ox0)) * p.ON;
    const int off = row_off + ng * 4;
    float4 x0, x1;
    epilogue_operands4(p.ep, p.out, off, ng * 4, x0, x1);
    *reinterpret_cast<float4*>(p.out + off) = epilogue4(p.ep, off, make_float4(acc[0], acc[1], acc[2], acc[3]), x0, x1);
  }
}

// ---------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------
typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

PFN_encodeTiled get_encode_fn() {
  static PFN_encodeTiled fn = nullptr;
  if (!fn) {
    void* ptr = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &qres) != cudaSuccess ||
        qres != cudaDriverEntryPointSuccess)
      return nullptr;
    fn = reinterpret_cast<PFN_encodeTiled>(ptr);
  }
  return fn;
}

int pick_bn(int N) {
  if (N <= 16) return 16;
  if (N <= 32) return 32;
  if (N <= 64) return 64;
  if (N <= 128) return 128;
  return 256;
}

// Row tiles of a launch (same geometry rule as launch_tc).
int count_m_tiles(const ConvGemmParams& p) {
  const int per_img = p.MH * p.MW;
  const int B = p.M / per_img;
  int BH, BB;
  if (per_img >= BM) { BB = 1; BH = BM / p.MW; } else { BH = p.MH; BB = BM / per_img; }
  return ((B + BB - 1) / BB) * ((p.MH + BH - 1) / BH);
}

// Widest BN that still gives every SM a tile; narrow problems (e.g. fc 1024x1024 at batch 1024) trade tile width
// for parallelism.  Depends on the layer shape and batch only through the tile COUNT, never on the data.
int pick_bn_for(const ConvGemmParams& p, int num_sms) {
  int bn = pick_bn(p.N);
  const int mt = count_m_tiles(p) * p.nclasses;
  while (bn > 64 && mt * ((p.N + bn - 1) / bn) < num_sms) bn >>= 1;
  return bn;
}

// Class-fusion tables of a transposed-type pass (see FuseShift): NS slots per tile; NS == 4 puts all four parity
// classes into one group, NS == 2 makes one group per output-row parity (heavier group first).
void build_fusion(ConvGemmParams& p, int NS) {
  const int ak = p.f16 ? 64 : BK;               // channels per K atom
  const int C = p.cblocks * ak;
  p.fuse = NS;
  p.ngroups = 0;
  int nshf = 0;
  int order[2] = {0, 1};
  if (NS == 2) {                                  // groups by oy0; the one with more taps first
    int taps[2] = {0, 0};
    for (int c = 0; c < p.nclasses; ++c) taps[p.cls[c].oy0 & 1] += p.cls[c].ntaps;
    if (taps[1] > taps[0]) { order[0] = 1; order[1] = 0; }
  }
  const int ngroups = NS == 2 ? 2 : 1;
  for (int gi = 0; gi < ngroups; ++gi) {
    FuseGroup& G = p.grp[p.ngroups++];
    G.ncls = 0;
    // slot order (0,0), (0,1), (1,1), (1,0): classes that share a shift sit in adjacent slots (wide MMAs)
    static const int kSlotKey[2][2] = {{0, 1}, {3, 2}};
    int cls_of_key[4] = {-1, -1, -1, -1};
    for (int c = 0; c < p.nclasses; ++c)
      if (NS != 2 || (p.cls[c].oy0 & 1) == order[gi]) cls_of_key[kSlotKey[p.cls[c].oy0 & 1][p.cls[c].ox0 & 1]] = c;
    for (int key = 0; key < 4; ++key)
      if (cls_of_key[key] >= 0) G.cls[G.ncls++] = cls_of_key[key];
    G.shift0 = nshf;
    // shifts in the canonical order of the packing (refine_conv.cu fill_transposed): the first class that has a tap at
    // a shift lists it at the position all classes agree on, so walking the taps of all classes by (users desc, dy
    // desc, dx desc) reproduces it
    struct Sh { int dy, dx, users; };
    Sh cand[kMaxShifts];
    int ncand = 0;
    for (int dy = 1; dy >= -1; --dy)
      for (int dx = 1; dx >= -1; --dx) {
        int users = 0;                              // users over ALL classes of the pass (the packing's criterion)
        for (int c = 0; c < p.nclasses; ++c)
          for (int t = 0; t < p.cls[c].ntaps; ++t)
            if (p.cls[c].dy[t] == dy && p.cls[c].dx[t] == dx) ++users;
        if (users) cand[ncand++] = Sh{dy, dx, users};
      }
    for (int a = 1; a < ncand; ++a)
      for (int b = a; b > 0 && cand[b].users > cand[b - 1].users; --b) { const Sh t = cand[b]; cand[b] = cand[b - 1]; cand[b - 1] = t; }
    unsigned touched = 0;
    for (int si = 0; si < ncand; ++si) {
      FuseShift sh;
      std::memset(&sh, 0, sizeof(sh));
      sh.dy = (signed char)cand[si].dy;
      sh.dx = (signed char)cand[si].dx;
      for (int q = 0; q < G.ncls; ++q) {
        const GemmClass& gc = p.cls[G.cls[q]];
        for (int t = 0; t < gc.ntaps; ++t)
          if (gc.dy[t] == sh.dy && gc.dx[t] == sh.dx) {
            sh.slot[sh.ncls] = (unsigned char)q;
            sh.katom0[sh.ncls] = (gc.k0 + t * C) / ak;
            ++sh.ncls;
          }
      }
      if (!sh.ncls) continue;
      // runs of adjacent slots with the same accumulate state (slots are listed in ascending order)
      for (int i = 0; i < sh.ncls;) {
        const int first = sh.slot[i];
        const unsigned acc = (touched >> first) & 1u;
        int len = 1;
        while (i + len < sh.ncls && sh.slot[i + len] == first + len && ((touched >> (first + len)) & 1u) == acc &&
               (len + 1) * p.N <= 256)
          ++len;
        sh.run_slot[sh.nrun] = (unsigned char)first;
        sh.run_len[sh.nrun] = (unsigned char)len;
        sh.run_acc[sh.nrun] = (unsigned char)acc;
        ++sh.nrun;
        i += len;
      }
      for (int i = 0; i < sh.ncls; ++i) touched |= 1u << sh.slot[i];
      for (int rank = 0; rank < 2; ++rank) {
        int n = 0, e0 = 0;
        for (int r = 0; r < sh.nrun; ++r) {
          const int L = sh.run_len[r];
          for (int j = 0; j < L; ++j, ++n) {
            const int g = rank * L + j;               // half-atom piece of the run's 2 L
            sh.pc_slot[rank][n] = (unsigned char)(sh.run_slot[r] + j);
            sh.pc_half[rank][n] = (unsigned char)(g & 1);
            sh.pc_katom[rank][n] = sh.katom0[e0 + (g >> 1)];
          }
          e0 += L;
        }
      }
      p.shf[nshf++] = sh;
    }
    G.nshifts = nshf - G.shift0;
  }
}

// Can this launch run class-fused, and with how many slots per tile?  (CGS_DEBUG_NO_FUSION switches fusion off.)
int fusion_slots(const ConvGemmParams& p, int bn) {
  if (debug_flags() & (CGS_DEBUG_NO_FUSION | CGS_DEBUG_GATHER_A)) return 0;
  if (p.nclasses != 4 || p.S != 1 || p.os != 2 || p.cblocks <= 0 || p.window || bn != p.N) return 0;
  for (int c = 0; c < 4; ++c) {
    if (p.cls[c].cb0 != 0 || p.cls[c].k0 % (p.f16 ? 64 : BK)) return 0;
    for (int t = 0; t < p.cls[c].ntaps; ++t)
      if (p.cls[c].dy[t] < -1 || p.cls[c].dy[t] > 1 || p.cls[c].dx[t] < -1 || p.cls[c].dx[t] > 1) return 0;
  }
  // a fused stage carries one weight atom per class with a tap at its shift: k = 5 averages 25 / 9 = 2.8 classes per
  // stage, k = 4 only 16 / 9 = 1.8 -- too little MMA work per pipeline hand-shake (measured slower on the MNIST nets)
  int taps = 0;
  for (int c = 0; c < 4; ++c) taps += p.cls[c].ntaps;
  if (taps < 23) return 0;      // (re-measured with wide MMAs and CTA pairs: MNIST g_dc3.fwd 43.9 us unfused, 49.7 / 54.1 fused)
  if (bn == 128) return 2;
  if (bn == 64 || bn == 32) return 4;
  return 0;
}

// Can a cluster of two CTAs of this kernel instance be resident on the current device (asked once per instance and
// device)?  On a whole B200 the answer is always yes (148 = 2 x 74 TPCs); on a partitioned or otherwise restricted
// device the launcher falls back to the single-CTA instance, which computes the same bits.
template <typename K>
bool cluster_pair_fits(K kernel, size_t smem, int threads) {
  static std::atomic<int> state[kMaxDevices];          // 0 unknown, 1 fits, -1 does not
  const int dev = current_device();
  if (dev < 0 || dev >= kMaxDevices) return true;
  int st = state[dev].load(std::memory_order_acquire);
  if (st == 0) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(2);
    cfg.blockDim = dim3(threads);
    cfg.dynamicSmemBytes = smem;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 2;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    int n = 0;
    const cudaError_t e = cudaOccupancyMaxActiveClusters(&n, kernel, &cfg);
    if (e != cudaSuccess) cudaGetLastError();
    st = (e == cudaSuccess && n >= 1) ? 1 : -1;
    state[dev].store(st, std::memory_order_release);
  }
  return st > 0;
}

template <int BN, int EPI, int NS = 1, int MT = 1, int CG = 1, bool F16 = false>
int launch_tc_epi(ConvGemmParams p, const void* w, int w_rows, int w_cols, cudaStream_t stream) {
  using C = Cfg<BN, NS, MT, CG>;
  constexpr int AK = F16 ? 64 : BK;                     // elements per 128-byte K atom
  constexpr size_t ES = F16 ? 2 : 4;                    // bytes per element
  const CUtensorMapDataType dtype = F16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32;
  const ConvGemmParams p_in = p;
  PFN_encodeTiled enc = get_encode_fn();
  if (!enc) return set_error(CGS_ERR_CUDA, "cuTensorMapEncodeTiled entry point not available");
  CUtensorMap tmap;
  // weights [rows][K] viewed as {AK (k inside an atom), rows, K/AK (atom)}: a box {AK, BN, KB} lands as KB atom tiles
  cuuint64_t gdim[3] = {(cuuint64_t)AK, (cuuint64_t)w_rows, (cuuint64_t)(w_cols / AK)};
  cuuint64_t gstride[2] = {(cuuint64_t)w_cols * ES, (cuuint64_t)AK * ES};
  cuuint32_t box[3] = {(cuuint32_t)AK, (cuuint32_t)(BN / CG), (cuuint32_t)C::KB};   // CTA pair: half an atom per box
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = enc(&tmap, dtype, 3, const_cast<void*>(w), gdim, gstride, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return set_error(CGS_ERR_CUDA, "cuTensorMapEncodeTiled failed (%d)", (int)r);
  p.debug = debug_flags();
  p.n_tiles = (p.N + BN - 1) / BN;
  // tile geometry: BB images x BH rows x MW columns (<= 128 rows) per row tile
  const int per_img = p.MH * p.MW;
  if (p.MW > BM) return set_error(CGS_ERR_UNSUPPORTED, "row width %d of the output grid exceeds the 128-row tile", p.MW);
  p.B = p.M / per_img;
  if (per_img >= BM) {
    p.BB = 1;
    p.BH = BM / p.MW;
  } else {
    p.BH = p.MH;
    p.BB = BM / per_img;
  }
  p.hy_tiles = (p.MH + p.BH - 1) / p.BH;
  p.rows_valid = p.BB * p.BH * p.MW;
  p.m_tiles = ((p.B + p.BB - 1) / p.BB) * p.hy_tiles;
  p.a_tma = (p.cblocks > 0) && !(p.debug & CGS_DEBUG_GATHER_A);
  if (F16 && (!p.a_tma || p.window)) return set_error(CGS_ERR_UNSUPPORTED, "FP16 operands need the TMA'd A operand");
  CUtensorMap tmap_a;
  std::memset(&tmap_a, 0, sizeof(tmap_a));
  if (p.window) {
    // overlapping-window view of the pitched image: dim0 = 32 floats (8 stored pixels), dim1 = output column i
    // (every 2 pixels = 32 bytes), dim2 = input row (traversal stride 2), dim3 = image
    if (p.MW > 256 || p.BH * 2 > 256) return set_error(CGS_ERR_UNSUPPORTED, "TMA box too large");
    const cuuint64_t row_bytes = (cuuint64_t)p.in_pitch_px * 16;
    cuuint64_t adim[4] = {32, (cuuint64_t)p.MW, (cuuint64_t)p.IH, (cuuint64_t)p.B};
    cuuint64_t astr[3] = {32, row_bytes, (cuuint64_t)p.IH * row_bytes};
    cuuint32_t abox[4] = {32, (cuuint32_t)p.MW, (cuuint32_t)(p.BH * 2), (cuuint32_t)p.BB};
    cuuint32_t aest[4] = {1, 1, 2, 1};
    CUresult ra = enc(&tmap_a, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, const_cast<float*>(p.in) + p.win_x0 * 4, adim, astr,
                      abox, aest, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                      CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (ra != CUDA_SUCCESS) return set_error(CGS_ERR_CUDA, "cuTensorMapEncodeTiled (window A operand) failed (%d)", (int)ra);
  } else
  if (p.a_tma) {
    // input viewed as [B][IH][IW][Cs]; traversal strides S pick every S-th pixel, so a box of
    // {32 ch, MW*S, BH*S, BB} lands as BB*BH*MW rows of 128 bytes; out-of-range coordinates read zeros
    if (p.MW * p.S > 256 || p.BH * p.S > 256) return set_error(CGS_ERR_UNSUPPORTED, "TMA box too large");
    cuuint64_t adim[4] = {(cuuint64_t)p.Cs, (cuuint64_t)p.IW, (cuuint64_t)p.IH, (cuuint64_t)p.B};
    cuuint64_t astr[3] = {(cuuint64_t)p.Cs * ES, (cuuint64_t)p.IW * p.Cs * ES, (cuuint64_t)p.IH * p.IW * p.Cs * ES};
    cuuint32_t abox[4] = {(cuuint32_t)AK, (cuuint32_t)(p.MW * p.S), (cuuint32_t)(p.BH * p.S), (cuuint32_t)p.BB};
    cuuint32_t aest[4] = {1, (cuuint32_t)p.S, (cuuint32_t)p.S, 1};
    CUresult ra = enc(&tmap_a, dtype, 4, const_cast<float*>(p.in), adim, astr, abox, aest,
                      CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                      CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (ra != CUDA_SUCCESS) return set_error(CGS_ERR_CUDA, "cuTensorMapEncodeTiled (A operand) failed (%d)", (int)ra);
  }
  const int num_sms = device_num_sms();
  void (*const k_plain)(ConvGemmParams, CUtensorMap, CUtensorMap) = conv_gemm_tc_kernel<BN, EPI, NS, MT, CG>;
  void (*const k_chain)(F16ChainParams, CUtensorMap, CUtensorMap) = conv_gemm_tc_kernel<BN, EPI, NS, MT, CG>;
  const bool chain16 = p.f16 || p.ep.out16;    // a pass of an FP16-operand chain
  if (chain16 && !chain_instance(EPI, NS, p.f16 != 0))
    return set_error(CGS_ERR_UNSUPPORTED, "no FP16-chain form of this pass (epilogue %d, %d classes per tile)", EPI, NS);
  {
    static DynSmemCache smem_cache[2];         // per kernel, per device
    cudaError_t e = chain16 ? ensure_dyn_smem(k_chain, (size_t)C::SMEM_BYTES, smem_cache[1])
                            : ensure_dyn_smem(k_plain, (size_t)C::SMEM_BYTES, smem_cache[0]);
    if (e != cudaSuccess) return set_error(CGS_ERR_CUDA, "cudaFuncSetAttribute: %s", cudaGetErrorString(e));
  }
  if (CG > 1 && !(chain16 ? cluster_pair_fits(k_chain, (size_t)C::SMEM_BYTES, kThreads)
                          : cluster_pair_fits(k_plain, (size_t)C::SMEM_BYTES, kThreads)))
    return launch_tc_epi<BN, EPI, NS, MT, 1, F16>(p_in, w, w_rows, w_cols, stream);
  if (NS > 1) build_fusion(p, NS); else p.fuse = 0;
  p.m2 = MT * CG;                             // adjacent M tiles per scheduling unit
  const int m_units = (p.m_tiles + p.m2 - 1) / p.m2;
  const long long total_ll = (long long)m_units * p.n_tiles * (NS > 1 ? p.ngroups : p.nclasses);
  if (total_ll >= (1ll << 31)) return set_error(CGS_ERR_UNSUPPORTED, "tile count exceeds 2^31");
  const int total = (int)total_ll;
  p.fd_tiles_per_class = fast_div_magic((unsigned)(m_units * p.n_tiles));
  p.fd_n_tiles = fast_div_magic((unsigned)p.n_tiles);
  p.fd_hy_tiles = fast_div_magic((unsigned)p.hy_tiles);
  // CTA pairs: one cluster of two per unit, at most one CTA per SM (148 = 2 x 74 TPCs)
  const int grid = CG > 1 ? (2 * total < (num_sms & ~1) ? 2 * total : (num_sms & ~1)) : (total < num_sms ? total : num_sms);
  cudaError_t e = chain16 ? launch_pdl_cluster(k_chain, dim3(grid), dim3(kThreads), (size_t)C::SMEM_BYTES, stream, CG,
                                                F16ChainParams{p}, tmap, tmap_a)
                          : launch_pdl_cluster(k_plain, dim3(grid), dim3(kThreads), (size_t)C::SMEM_BYTES, stream, CG, p,
                                                tmap, tmap_a);
  count_launch();
  if (e == cudaSuccess) e = cudaGetLastError();
  if (e != cudaSuccess) return set_error(CGS_ERR_CUDA, "conv_gemm_tc launch: %s", cudaGetErrorString(e));
  return CGS_OK;
}

template <bool F16, int BN, int NS = 1, int MT = 1, int CG = 1>
int launch_tc(const ConvGemmParams& p, const void* w, int w_rows, int w_cols, cudaStream_t stream) {
  switch (p.ep.mode) {                      // the epilogue mode is compiled into the kernel
    case EPI_FWD: return launch_tc_epi<BN, EPI_FWD, NS, MT, CG, F16>(p, w, w_rows, w_cols, stream);
    case EPI_BWD: return launch_tc_epi<BN, EPI_BWD, NS, MT, CG, F16>(p, w, w_rows, w_cols, stream);
    case EPI_UPDATE: return launch_tc_epi<BN, EPI_UPDATE, NS, MT, CG, F16>(p, w, w_rows, w_cols, stream);
    default: return launch_tc_epi<BN, EPI_RAW, NS, MT, CG, F16>(p, w, w_rows, w_cols, stream);
  }
}

// CTA pairs (cta_group::2) are taken for the passes whose stages are widest in bytes per MMA cycle -- class-fused tiles
// and 256-wide tiles -- when the TMA'd A operand is in use and every SM still gets a tile.  CGS_DEBUG_NO_CTA_PAIRS
// switches them off, CGS_DEBUG_FORCE_CTA_PAIRS forces them whenever legal (parity tests at small batch).
bool use_cta_pairs(const ConvGemmParams& p, long long units_total, int num_sms) {
  if (debug_flags() & (CGS_DEBUG_NO_CTA_PAIRS | CGS_DEBUG_GATHER_A)) return false;
  if (p.cblocks <= 0 || p.window) return false;
  if (debug_flags() & CGS_DEBUG_FORCE_CTA_PAIRS) return true;
  return 2 * units_total >= (num_sms & ~1);
}

int validate(const ConvGemmParams& p, int w_cols) {
  const int ak = p.f16 ? 64 : BK;
  if (p.ON % 4 != 0) return set_error(CGS_ERR_INVALID, "output channel stride %d must be a multiple of 4", p.ON);
  if (p.cblocks == 0 && p.Cs != 4) return set_error(CGS_ERR_INVALID, "pixel mode needs channel stride 4");
  if (p.window && (p.cblocks != 1 || p.in_pitch_px <= 0)) return set_error(CGS_ERR_INVALID, "bad window-mode parameters");
  if (p.nclasses < 1 || p.nclasses > kMaxClasses) return set_error(CGS_ERR_INVALID, "bad class count");
  if (w_cols % 32 != 0) return set_error(CGS_ERR_INVALID, "weight row length must be a multiple of 32 floats");
  for (int c = 0; c < p.nclasses; ++c) {
    if (p.cls[c].ntaps > kMaxTaps) return set_error(CGS_ERR_INVALID, "too many taps");
    if (p.cls[c].k0 + p.cls[c].nkb * ak > w_cols) return set_error(CGS_ERR_INVALID, "class K range exceeds weight matrix");
  }
  return CGS_OK;
}

}  // namespace

int plan_fusion(ConvGemmParams& p) {
  const int ns = fusion_slots(p, pick_bn(p.N));
  if (ns) build_fusion(p, ns);
  return ns;
}

int debug_trace_read(unsigned long long* out, int cap) {
  cudaDeviceSynchronize();
  const int n = cap < 32768 ? cap : 32768;
  cudaMemcpyFromSymbol(out, g_trace, n * sizeof(unsigned long long));
  static unsigned long long zeros[32768];
  cudaMemcpyToSymbol(g_trace, zeros, sizeof(zeros));
  return n;
}

template <bool F16>
int launch_conv_gemm_tc_t(const ConvGemmParams& p, const void* w, int w_rows, int w_cols, cudaStream_t stream) {
  if (int rc = validate(p, w_cols)) return rc;
  if (p.M <= 0) return CGS_OK;
  const int num_sms = device_num_sms();
  int bn = p.force_bn ? p.force_bn : pick_bn_for(p, num_sms);
  {
    static int force = -1;                    // developer knob: CGS_FORCE_BN=16..256 overrides the tile-width heuristic
    if (force < 0) { const char* e = getenv("CGS_FORCE_BN"); force = e ? atoi(e) : 0; }
    if (force) bn = force;
  }
  // class-fused instances of the transposed-type passes: taken when the fused tiles (4x / 2x fewer than class tiles)
  // still give every SM one; CGS_DEBUG_FORCE_FUSION forces them whenever they are legal (parity tests at small batch)
  if (!p.force_bn) {
    const int bn_full = pick_bn(p.N);
    const int ns = fusion_slots(p, bn_full);
    if (ns && ((debug_flags() & CGS_DEBUG_FORCE_FUSION) || count_m_tiles(p) * (ns == 2 ? 2 : 1) >= num_sms)) {
      const bool pairs = use_cta_pairs(p, (long long)((count_m_tiles(p) + 1) / 2) * (ns == 2 ? 2 : 1), num_sms);
      switch (ns * 1000 + bn_full) {
        case 4032: return launch_tc<F16, 32, 4>(p, w, w_rows, w_cols, stream);
        case 4064: return pairs ? launch_tc<F16, 64, 4, 1, 2>(p, w, w_rows, w_cols, stream) : launch_tc<F16, 64, 4>(p, w, w_rows, w_cols, stream);
        case 2128: return pairs ? launch_tc<F16, 128, 2, 1, 2>(p, w, w_rows, w_cols, stream) : launch_tc<F16, 128, 2>(p, w, w_rows, w_cols, stream);
        default: break;
      }
    }
  }
  // M-tile pairs sharing the weight atoms (MT = 2): 64- / 128-wide one-class tiles with a TMA'd A operand, when the
  // pairs still give every SM a tile.  Bit-identical to single tiles (each accumulator sees the same MMA sequence).
  // CGS_DEBUG_NO_MTILE_PAIRS switches them off, CGS_DEBUG_FORCE_MTILE_PAIRS forces them whenever legal.
  // (64-wide pairs on one CTA save only 17 % of the bytes and measured slower on the MNIST nets; inside CTA pairs --
  //  four M tiles per weight atom, half of it per CTA -- they save 25 % and measured 3-7 % faster: taken only there)
  if (!p.force_bn && (bn == 128 || bn == 64) && p.cblocks > 0 && !p.window && !(debug_flags() & (CGS_DEBUG_NO_MTILE_PAIRS | CGS_DEBUG_GATHER_A)) &&
      p.N > bn / 2) {
    const long long nt = (long long)((p.N + bn - 1) / bn) * p.nclasses;
    const long long tiles = (long long)count_m_tiles(p) * nt, pairs = (long long)((count_m_tiles(p) + 1) / 2) * nt;
    const long long quads = (long long)((count_m_tiles(p) + 3) / 4) * nt;
    // whole rounds over the SMs: a pair round costs two tile rounds at 0.78x / 0.85x of their bytes
    const double cost_pair = (double)((pairs + num_sms - 1) / num_sms) * 2.0 * (bn == 128 ? 0.78 : 0.85);
    const double cost_single = (double)((tiles + num_sms - 1) / num_sms);
    const bool forced = (debug_flags() & CGS_DEBUG_FORCE_MTILE_PAIRS) != 0;
    if (forced || (pairs >= num_sms && cost_pair < cost_single)) {
      // M-tile pairs inside CTA pairs: 40 KB instead of 48 KB of L2 -> SM traffic per 512 tensor cycles (BN = 128) on
      // passes that sit at the L2 throughput ceiling
      if (use_cta_pairs(p, quads, num_sms))
        return bn == 64 ? launch_tc<F16, 64, 1, 2, 2>(p, w, w_rows, w_cols, stream) : launch_tc<F16, 128, 1, 2, 2>(p, w, w_rows, w_cols, stream);
      if (bn == 128 || forced)
        return bn == 64 ? launch_tc<F16, 64, 1, 2>(p, w, w_rows, w_cols, stream) : launch_tc<F16, 128, 1, 2>(p, w, w_rows, w_cols, stream);
    }
  }
  switch (bn) {
    case 16: return launch_tc<F16, 16>(p, w, w_rows, w_cols, stream);
    case 32: return launch_tc<F16, 32>(p, w, w_rows, w_cols, stream);
    case 64: return launch_tc<F16, 64>(p, w, w_rows, w_cols, stream);
    case 128: return launch_tc<F16, 128>(p, w, w_rows, w_cols, stream);
    default:
      if (use_cta_pairs(p, (long long)((count_m_tiles(p) + 1) / 2) * ((p.N + 255) / 256) * p.nclasses, num_sms))
        return launch_tc<F16, 256, 1, 1, 2>(p, w, w_rows, w_cols, stream);
      return launch_tc<F16, 256>(p, w, w_rows, w_cols, stream);
  }
}

int launch_conv_gemm_tc(const ConvGemmParams& p, const void* w, int w_rows, int w_cols, cudaStream_t stream) {
  return p.f16 ? launch_conv_gemm_tc_t<true>(p, w, w_rows, w_cols, stream) : launch_conv_gemm_tc_t<false>(p, w, w_rows, w_cols, stream);
}

int launch_conv_gemm_simt(const ConvGemmParams& p, const float* w, int w_rows, int w_cols, cudaStream_t stream) {
  (void)w_rows;
  if (int rc = validate(p, w_cols)) return rc;
  if (p.M <= 0) return CGS_OK;
  const long long total = (long long)p.nclasses * p.M * (p.ON / 4);
  long long blocks = (total + 255) / 256;
  if (blocks > 148 * 16) blocks = 148 * 16;
  conv_gemm_simt_kernel<<<(int)blocks, 256, 0, stream>>>(p, w, w_cols); count_launch();
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return set_error(CGS_ERR_CUDA, "conv_gemm_simt launch: %s", cudaGetErrorString(e));
  return CGS_OK;
}

}  // namespace cgs
