/* libcgs -- C ABI of the B200 (sm_100a) collaborative-sampling hot path.
 *
 * This is the drop-in boundary under the reference's Python `sampling/` classes
 * (vita-epfl/collaborative-gan-sampling).  The reference has no FFI: its hot path is Python calling
 * TensorFlow-1.13 / numpy.  Each entry point below names the reference code it replaces (paths relative to the
 * reference root).  The host-side mirror of the reference classes (same module / class / method names) lives in
 * `collaborative-gan-sampling_b200/sampling/` and binds these symbols with ctypes; INTEGRATION.md shows the stub.
 *
 * Conventions
 *  - every pointer is a DEVICE pointer unless its name ends in `_host`; the caller owns all memory, including
 *    the workspace (size queried first); the library allocates nothing on the device and keeps no pointer
 *    after a call returns
 *  - all work is enqueued on the caller's stream and is asynchronous; there are no hidden synchronisations,
 *    counts are written to device integers
 *  - every call returns CGS_OK (0) or a negative cgs_status; cgs_last_error() gives the thread-local message
 *  - there is NO CPU fallback: a missing / non-sm_100 device is an error, never a silent slow path
 */
#ifndef CGS_H_
#define CGS_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct CUstream_st* cgs_stream_t; /* == cudaStream_t */

#if defined(__GNUC__)
#define CGS_API __attribute__((visibility("default")))
#else
#define CGS_API
#endif

enum cgs_status {
  CGS_OK = 0,
  CGS_ERR_INVALID = -1,     /* bad argument (maps to ValueError / AssertionError in the wrapper) */
  CGS_ERR_UNSUPPORTED = -2, /* valid in the reference, not built here (maps to NotImplementedError) */
  CGS_ERR_CUDA = -3,        /* CUDA runtime / driver error, message in cgs_last_error() */
  CGS_ERR_WORKSPACE = -4    /* workspace too small */
};

#define CGS_ABI_VERSION 1
CGS_API int cgs_version(void);
CGS_API const char* cgs_last_error(void);
/* number of CUDA kernels this library has launched in this process (bench.py's gpu_launches evidence).
 * Developer aid OUTSIDE the drop-in contract: a process-wide atomic counter, never read by any compute path. */
CGS_API long long cgs_launch_count(void);

/* ------------------------------------------------------------------------------------------------------------
 * Update policy.  Replaces sampling/policy.py:26-64 (PolicyAdaptive.apply_gradient), all three methods.
 * theta/grad/momentum/mean_square are [rows, cols] row-major FP32, loss/loss_avg are [rows].
 * `first` != 0 means the moving averages are unset (policy.py:32,40,44,48: `is not None` tests).
 * ladam: cols == 2 follows the numpy branch (policy.py:61, no upper clip); cols > 2 follows the TF branch
 * (policy.py:52-59, rescale clipped to [0, 1e4]).  In-place on theta, like the reference.
 * ---------------------------------------------------------------------------------------------------------- */
enum cgs_policy_method { CGS_POLICY_SGD = 0, CGS_POLICY_MOMENTUM = 1, CGS_POLICY_LADAM = 2 };

typedef struct cgs_policy_cfg {
  int method;        /* cgs_policy_method */
  int degree;        /* degree_  policy.py:16 (2) */
  /* doubles on purpose: the reference holds python floats and numpy rounds e.g. (1. - beta1_) to FP32 only when
   * it meets the FP32 array, so the FP32 constants must be derived from the double values to stay bit-exact */
  double step_size;  /* lambda_  policy.py:9  */
  double alpha;      /* alpha_   policy.py:10 (0.9) */
  double beta1;      /* beta1_   policy.py:13 (0.9) */
  double beta2;      /* beta2_   policy.py:14 (0.5) */
  double beta3;      /* beta3_   policy.py:15 (0.5) */
  double eps;        /* eps_     policy.py:17 (1e-8) */
} cgs_policy_cfg;

CGS_API int cgs_policy_step(const cgs_policy_cfg* cfg, float* theta, const float* grad, const float* loss,
                    float* momentum, float* mean_square, float* loss_avg, int first, int64_t rows, int64_t cols,
                    cgs_stream_t stream);

/* ------------------------------------------------------------------------------------------------------------
 * Discriminator Rejection Sampling.  Replaces sampling/rejector.py:16-38 (Rejector.sampling) and :11-14.
 * FP64 arithmetic as in the reference (rejector.py:18 astype(np.float)).
 *   sigmoids      [n] scores, dtype CGS_F32 or CGS_F64
 *   uniforms      [n] FP64 uniforms == what np.random.rand(n) returns (rejector.py:33); NULL => Philox4x32-10
 *                 counter-based stream (philox_seed, philox_offset + row), one draw per row
 *   d_tilde_m     device scalar, in: running max logit (Rejector.D_tilde_M), out: updated (rejector.py:22)
 *   shift_percent percentile shift gamma (rejector.py:27-29); negative => None (no shift)
 *   accept_out    [n] 0/1 flags;  idx_out [n] ascending row indices of accepted rows;  count_out device int
 * ---------------------------------------------------------------------------------------------------------- */
enum cgs_dtype { CGS_F32 = 0, CGS_F64 = 1 };

CGS_API size_t cgs_drs_workspace_bytes(int64_t n);
CGS_API int cgs_drs_accept(const void* sigmoids, int sig_dtype, int64_t n, const double* uniforms, uint64_t philox_seed,
                   uint64_t philox_offset, double* d_tilde_m, double epsilon, double shift_percent,
                   uint8_t* accept_out, int32_t* idx_out, int32_t* count_out, double* prob_out /* nullable [n] */,
                   void* workspace, size_t workspace_bytes, cgs_stream_t stream);
/* rejector.py:11-14: D_tilde_M = logit(clip(score_max)) */
CGS_API int cgs_drs_set_score_max(const void* score_max, int dtype, double* d_tilde_m, cgs_stream_t stream);

/* ------------------------------------------------------------------------------------------------------------
 * MH-GAN independence sampler.  Replaces sampling/idpsampler.py:17-53 (sampling + next), exactly, in parallel:
 * next-acceptance pointers -> blocked list traversal -> thinning (SURVEY.md App. A10).
 *   state (device, in/out): d_curr (value as double), d_kind (0 = None, 1 = float32-typed, 2 = float64-typed,
 *   3 = weak python float), cnt_chain (idpsampler.py:7).  alpha is evaluated in the dtype numpy would use.
 *   emit_src_out [<= n] source row of every emitted sample, count_out device int, accepted_out [n] flags.
 * ---------------------------------------------------------------------------------------------------------- */
CGS_API size_t cgs_mh_workspace_bytes(int64_t n);
CGS_API int cgs_mh_accept(const void* sigmoids, int sig_dtype, int64_t n, const double* uniforms, uint64_t philox_seed,
                  uint64_t philox_offset, double* d_curr, int32_t* d_kind, int32_t* cnt_chain, int thin_period,
                  int burn_in, uint8_t* accepted_out, int32_t* emit_src_out, int32_t* count_out, void* workspace,
                  size_t workspace_bytes, cgs_stream_t stream);

/* Order-preserving row gather: dst[r] = src[idx[r]] for r < min(*count, max_rows).  Replaces the boolean /
 * list gathers at rejector.py:34 and idpsampler.py:36,41. */
CGS_API int cgs_gather_rows(const void* src, int64_t row_bytes, const int32_t* idx, const int32_t* count,
                    int64_t max_rows, void* dst, cgs_stream_t stream);

/* ------------------------------------------------------------------------------------------------------------
 * 2-D synthetic path.  Replaces synthetic/GAN.py:28-37,108-111 (D MLP, fake_sigmoid, fake_saliency) and
 * sampling/refiner_cpu.py:19-81 (Refiner.manipulate_sample) as ONE fused kernel, weights in shared memory.
 * weights[l] is the TF dense kernel [in, out] row-major, biases[l] is [out].
 * ---------------------------------------------------------------------------------------------------------- */
#define CGS_MLP_MAX_LAYERS 8
typedef struct cgs_mlp_desc {
  int nlayers;  /* --nlayers (synthetic/main.py), 2..8 ; layer 0 is 2->nhidden, last is nhidden->1 */
  int nhidden;  /* --nhidden, a multiple of 16 from 16 to 256; at 64 every CTA holds the whole MLP, every other width
                   is held across a thread-block cluster of nhidden / 16 CTAs */
  const float* weights[CGS_MLP_MAX_LAYERS];
  const float* biases[CGS_MLP_MAX_LAYERS];
} cgs_mlp_desc;

/* sigmoid_out [n], logit_out [n] (nullable), saliency_out [n,2] (nullable) = d mean-BCE / d x, i.e. with the
 * 1/n_mean factor of synthetic/GAN.py:109-111 (n_mean = rows fed in the reference; pass the GLOBAL row count). */
CGS_API int cgs_mlp2d_score(const cgs_mlp_desc* d, const float* x, int64_t n, int64_t n_mean, float* sigmoid_out,
                    float* logit_out, float* saliency_out, cgs_stream_t stream);

typedef struct cgs_refine2d_cfg {
  int steps;                 /* rollout_steps */
  cgs_policy_cfg policy;     /* rollout_rate / rollout_method + constants */
  int64_t n_mean;            /* rows the reference's reduce_mean runs over (global batch) */
  float real_sigmoid_mean;   /* np.mean(real_sigmoid), refiner_cpu.py:23,28 (FP32 like the numpy scalar) */
} cgs_refine2d_cfg;

/* x_in [n,2] -> best_x [n,2], best_loss [n], best_step [n] (FP32, refiner_cpu.py:31-33,58-61);
 * traj_out (nullable) [n, steps+1, 3] FP32 = (x, y, loss) per step (refiner_cpu.py:37-43,64-66). */
CGS_API int cgs_refine_mlp2d(const cgs_mlp_desc* d, const cgs_refine2d_cfg* cfg, const float* x_in, int64_t n,
                     float* best_x, float* best_loss, float* best_step, float* traj_out, cgs_stream_t stream);

/* ------------------------------------------------------------------------------------------------------------
 * Image path.  Replaces sampling/collaborator.py:26-88 (Refiner.compute_forward_logits_and_grad and the K-step
 * build_refiner loop) over nsgan/GAN.py:59-101 / nsgan/ops.py:19-83 networks (conv, deconv, linear, BN folded in
 * inference mode, lrelu/relu/tanh) and the DCGAN-32/64 shapes.
 *
 * A network is a chain of layers.  Activations are NHWC FP32 with the channel stride padded to a multiple of 4.
 * Weights arrive PACKED (see collaborative-gan-sampling_b200/cgs/pack.py): one K-major matrix per direction,
 *   w_fwd [rows_fwd, kcols_fwd], w_bwd [rows_bwd, kcols_bwd], BN folded, K order = (parity class, tap, channel).
 * ---------------------------------------------------------------------------------------------------------- */
enum cgs_layer_type { CGS_LAYER_CONV = 0, CGS_LAYER_DECONV = 1, CGS_LAYER_FC = 2 };
enum cgs_act { CGS_ACT_NONE = 0, CGS_ACT_RELU = 1, CGS_ACT_LRELU = 2, CGS_ACT_TANH = 3 };

typedef struct cgs_layer_desc {
  int type;          /* cgs_layer_type */
  int k;             /* kernel size (4 or 5), stride is 2 (nsgan/ops.py:37,48) ; ignored for fc */
  int cin, cout;     /* logical channels */
  int hin, win;      /* input spatial size (fc: 1,1 and cin = flattened NHWC size) */
  int act;           /* cgs_act */
  const float* w_fwd; int rows_fwd, kcols_fwd;
  const float* w_bwd; int rows_bwd, kcols_bwd;
  const float* bias; /* folded bias, padded with zeros to the output channel stride */
  /* optional FP16 copies (__half, same layout) of w_fwd / w_bwd: with them on every GEMM layer, the DCGAN-shaped
     refinement chains run their MMAs on FP16 operands (kind::f16); null = TF32 operands */
  const void* w16_fwd;
  const void* w16_bwd;
} cgs_layer_desc;

#define CGS_MAX_LAYERS 8
typedef struct cgs_net_desc {
  int n_layers;
  cgs_layer_desc layers[CGS_MAX_LAYERS];
} cgs_net_desc;

enum cgs_refine_mode { CGS_MODE_DETERMINISTIC = 0, CGS_MODE_PROBABILISTIC = 1 };
enum cgs_math { CGS_MATH_TF32_TENSOR = 0, CGS_MATH_FP32_SIMT = 1 };

typedef struct cgs_refine_cfg {
  int steps;         /* rollout_steps (collaborator.py:10) */
  double rate;       /* rollout_rate  */
  int method;        /* CGS_POLICY_SGD | CGS_POLICY_MOMENTUM (ladam is invalid here: policy.py:51 with loss=None) */
  double alpha;      /* momentum decay 0.9 */
  int mode;          /* cgs_refine_mode */
  int clip;          /* collaborator.py:69 truthiness already resolved by the wrapper */
  float vmin, vmax;
  int math;          /* cgs_math */
  int early_exit;    /* opt-in (README.md:13): a sample whose logit reaches exit_logit keeps its best state, leaves
                        the batch and the remaining rows are compacted ON THE DEVICE (the live-row count stays in
                        device memory, grids are sized for the full batch): no host synchronisation, the launch
                        sequence is static and CUDA-graph capturable; 0 = reference behaviour (always K steps) */
  float exit_logit;
} cgs_refine_cfg;

/* largest batch one call accepts (32-bit row indexing); the wrapper refines larger batches in independent chunks */
CGS_API int64_t cgs_refine_max_batch(const cgs_net_desc* gtail, const cgs_net_desc* d);

/* bytes of workspace cgs_refine_conv needs for a batch of B */
CGS_API size_t cgs_refine_workspace_bytes(const cgs_net_desc* gtail, const cgs_net_desc* d, int64_t B);

/* feature [B, H, W, C] (C multiple of 32) is refined IN PLACE (it ends as the state after the last step);
 * outputs: best_img [B, h, w, c_stride] (the G-tail image of the best state == feature_to_data(optimal_feature),
 * collaborator.py:88), best_logit / best_step / default_logit [B] (collaborator.py:52,58-60,81-83);
 * prob_indices [B] int32 (mode probabilistic, collaborator.py:54-56) else NULL;
 * best_feature (nullable) [B,H,W,C] = optimal_feature. */
CGS_API int cgs_refine_conv(const cgs_net_desc* gtail, const cgs_net_desc* d, const cgs_refine_cfg* cfg, int64_t B,
                    float* feature, float* best_img, float* best_logit, float* best_step, float* default_logit,
                    const int32_t* prob_indices, float* best_feature, void* workspace, size_t workspace_bytes,
                    cgs_stream_t stream);

/* One forward (+ optional data-gradient) pass: collaborator.py:26-39.  logit_out [B]; grad_out (nullable)
 * [B,H,W,C] = d sum_b softplus(-logit_b) / d feature; img_out (nullable). */
CGS_API int cgs_forward_logits_and_grad(const cgs_net_desc* gtail, const cgs_net_desc* d, int math, int64_t B,
                                const float* feature, float* logit_out, float* grad_out, float* img_out,
                                void* workspace, size_t workspace_bytes, cgs_stream_t stream);

/* ------------------------------------------------------------------------------------------------------------
 * Training-mode discriminator: batch-statistic BatchNorm (nsgan/GAN.py:175 `is_training=True`, nsgan/ops.py:19-26).
 * For every D layer with a gamma: y = layer(x) + bias, mean / biased variance per channel over all B*H*W rows of
 * the batch of the call (B rows for fc), out = act(gamma * (y - mean) / sqrt(var + 1e-5) + beta); the gradient flows
 * through the statistics.  G's tail stays in inference mode, as in the reference (nsgan/GAN.py:94).  The moving
 * averages are not updated (they change no value the refinement computes) and the weights are never written.
 * ---------------------------------------------------------------------------------------------------------- */
typedef struct cgs_batchnorm_desc {
  int n_layers;                        /* == the D net's n_layers */
  const float* gamma[CGS_MAX_LAYERS];  /* [cout] per D layer; null = no batch BN after that layer */
  const float* beta[CGS_MAX_LAYERS];   /* [cout] */
} cgs_batchnorm_desc;

/* The _bn entry points are the plain ones with a batchnorm descriptor; bn == NULL is exactly the plain call.  With a
 * non-null bn, `d` carries the UNFOLDED weights of the layers that have a gamma (w * 1, bias = the layer's own).
 * CGS_ERR_UNSUPPORTED: batch BN with early exit (it would change the batch the statistics run over), on D's
 * image-edge (first) layer or on the 1-logit head.  The statistics are those of the B rows of one call: the
 * caller must not split a batch into chunks.  The chain runs on TF32 (FP32-stored) operands in this mode. */
CGS_API size_t cgs_refine_workspace_bytes_bn(const cgs_net_desc* gtail, const cgs_net_desc* d,
                                             const cgs_batchnorm_desc* bn, int64_t B);
CGS_API int cgs_refine_conv_bn(const cgs_net_desc* gtail, const cgs_net_desc* d, const cgs_batchnorm_desc* bn,
                               const cgs_refine_cfg* cfg, int64_t B, float* feature, float* best_img, float* best_logit,
                               float* best_step, float* default_logit, const int32_t* prob_indices, float* best_feature,
                               void* workspace, size_t workspace_bytes, cgs_stream_t stream);
CGS_API int cgs_forward_logits_and_grad_bn(const cgs_net_desc* gtail, const cgs_net_desc* d,
                                           const cgs_batchnorm_desc* bn, int math, int64_t B, const float* feature,
                                           float* logit_out, float* grad_out, float* img_out, void* workspace,
                                           size_t workspace_bytes, cgs_stream_t stream);

/* The batch-BN kernels alone (per-kernel tests): y, out, dz, dy are [rows, C] FP32, C a multiple of 4; every tensor
 * (gamma and beta too) 16-byte aligned, else CGS_ERR_INVALID.
 * forward: out = act(gamma * (y - mean) * rstd + beta), act a cgs_act; mean_out / rstd_out [C] nullable.
 * backward: dz = d loss / d (gamma * x^ + beta) with x^ = (y - mean) * rstd, the statistics of y recomputed ->
 *   dy = d loss / d y = rstd * (dz^ - mean(dz^) - x^ * mean(dz^ * x^)), dz^ = gamma * dz. */
CGS_API size_t cgs_batchnorm_workspace_bytes(int64_t rows, int C);
CGS_API int cgs_batchnorm_forward(int64_t rows, int C, const float* y, const float* gamma, const float* beta, int act,
                                  float* out, float* mean_out, float* rstd_out, void* workspace, size_t workspace_bytes,
                                  cgs_stream_t stream);
CGS_API int cgs_batchnorm_backward(int64_t rows, int C, const float* y, const float* gamma, const float* dz, float* dy,
                                   void* workspace, size_t workspace_bytes, cgs_stream_t stream);

/* Host-only helper (no GPU needed): K ordering of a layer's packed weight matrix.  For K index q of the forward
 * (backward != 0: data-gradient) matrix: ky[q], kx[q] = filter tap or -1 for zero padding, ch[q] = reduced channel
 * (forward: input channel; backward: output channel).  Pass NULL arrays to query the K length (multiple of 32). */
CGS_API int64_t cgs_pack_map(const cgs_layer_desc* L, int backward, int32_t* ky, int32_t* kx, int32_t* ch,
                             int64_t capacity);

/* Host-only introspection: the gathered-GEMM parameters a layer pass is lowered to, as int32s
 * [IH, IW, Cs, cblocks, MH, MW, S, M, OH, OW, ON, os, N, nclasses, window, win_k, win_x0, in_pitch_px] + per class [k0, nkb, ntaps, oy0, ox0, dy[32],
 * dx[32]] (see csrc/conv_gemm.cuh).  NULL `out` queries the length.  Lets tests replay the gather on the CPU. */
CGS_API int64_t cgs_debug_gemm_params(const cgs_layer_desc* L, int backward, int64_t B, int32_t* out,
                                      int64_t capacity);

/* Host-only introspection of the class-fused lowering of a transposed-type pass (csrc/conv_gemm.cuh FuseShift /
 * FuseGroup): returns 0 when the pass is never class-fused, else writes [slots per tile, ngroups] + per group [nshifts,
 * shift0, ncls, cls[4]] + per shift [dy, dx, ncls, nrun, slot[4], katom0[4], run_slot[4], run_len[4], run_acc[4],
 * pc_slot[2][4], pc_half[2][4], pc_katom[2][4]] (the pc_* tables are the per-CTA-rank half-atom boxes of a CTA pair).
 * NULL `out` queries the length.  Lets tests check the fused walk and the pair split on the CPU. */
CGS_API int64_t cgs_debug_fusion_plan(const cgs_layer_desc* L, int backward, int64_t B, int32_t* out, int64_t capacity);

/* Host-only introspection of a refinement chain (G tail + D without its head, bn == NULL) under `math` and the current
 * CGS_DEBUG knobs: where and in which type every tensor lives.  Writes [n, n_gtail, img_mode, f16] and then 8 int32s
 * per tensor, first act[0 .. n] (act[0] = the refined feature, act[i + 1] = output of layer i), then d loss / d act[1 .. n]
 * (exactly: the tensor data-gradient pass i - 1 reduces, i.e. the gradient w.r.t. layer i - 1's pre-activation output,
 * held in act[i]'s layout): [fp16, layout, H, W, C, values per stored pixel, stored pixels per row, elements per sample
 * (the stride from one sample to the next)].
 * fp16: 1 = __half, 0 = float.  layout: 0 = dense NHWC (channel stride = C rounded up to 4), 1 = space-to-depth
 * [H/2][W/2][2][2][4], 2 = pitched [H][W + 8][4] with pixel x at column x + 2 and zeros elsewhere.  img_mode = the
 * layout (1 or 2) of the <= 4-channel tensors; f16 = the chain's MMA operands are FP16.  NULL `out` queries the length. */
CGS_API int64_t cgs_debug_chain_layout(const cgs_net_desc* gtail, const cgs_net_desc* d, int math, int32_t* out,
                                       int64_t capacity);
/* Developer aid OUTSIDE the drop-in contract: ONE pass of the chain on the caller's tensors, launched as a refinement
 * call launches it (same kernel route, operand type, layouts and fused epilogue; cgs_debug_chain_layout gives the
 * layouts), so that each pass can be checked alone.  Tensors are batch-major with cgs_debug_chain_layout's elements
 * per sample.
 *   forward (backward == 0), 0 <= layer < n: in = act[layer], out = act[layer + 1].
 *   data-gradient, 0 < layer < n: in = d loss / d act[layer + 1], aux = act[layer] (the forward output the epilogue
 *     differentiates through), out = d loss / d act[layer].
 *   data-gradient, layer 0: in as above; step_cfg NULL: out = the raw gradient w.r.t. the feature; else out is the
 *     feature, updated in place by the fused policy step of step_cfg (method, rate, alpha, clip, vmin, vmax), with
 *     `mom` (momentum, read unless `first`, written) and `first`.  gexp (nullable, [B] int32; FP16 chains only): the
 *     input carries the per-sample factor 2^gexp[b], which the pass removes.
 *   layer == n, data-gradient: the head.  in = act[n], aux = the [B] logits (out), out = d loss / d act[n] (dpre), gexp =
 *     the [B] exponents the head writes (required when dpre is FP16).
 * The workspace is cgs_refine_workspace_bytes(gtail, d, B).  Where a refinement call runs the two image-edge passes as
 * one paired kernel (pitched image layout), this entry point runs them as the two separate kernels that
 * CGS_DEBUG_NO_EDGE_PAIR selects; the head never takes split-K partial sums here. */
CGS_API int cgs_debug_chain_pass(const cgs_net_desc* gtail, const cgs_net_desc* d, int math, int64_t B, int layer,
                                 int backward, const void* in, void* out, void* aux, int32_t* gexp,
                                 const cgs_refine_cfg* step_cfg, float* mom, int first, void* workspace,
                                 size_t workspace_bytes, cgs_stream_t stream);

/* Lowering of a pass: 0 = gather layout (K order given by cgs_pack_map), 1 = scatter layout, 2 = window layout
 * (strided passes reading a <= 4-channel image: rows = large channel, K index = ky*32 + kx*4 + small channel).  Transposed-type
 * passes with <= 4 output channels (deconv -> image forward, first-conv data-gradient) run as one GEMM over the
 * input pixels producing all k*k taps, followed by a col2im kernel with the fused epilogue; their packed matrix
 * has rows = (ky*k + kx)*4 + small_channel and K = the large channel count.  Host only. */
CGS_API int cgs_pass_layout(const cgs_layer_desc* L, int backward);

/* Single-layer entry points used by the per-layer parity tests.  x [B,hin,win,cs_in], y [B,hout,wout,cs_out];
 * workspace (cgs_layer_workspace_bytes) is only touched by scatter-lowered passes. */
CGS_API size_t cgs_layer_workspace_bytes(const cgs_layer_desc* L, int64_t B);
CGS_API int cgs_layer_forward(const cgs_layer_desc* L, int math, int64_t B, const float* x, float* y, void* workspace,
                              size_t workspace_bytes, cgs_stream_t stream);
/* dx = dgrad(dy) * act'(x_fwd) where prev_act describes the producer of x (CGS_ACT_NONE for none) */
CGS_API int cgs_layer_backward(const cgs_layer_desc* L, int math, int64_t B, const float* dy, float* dx,
                               const float* x_fwd, int prev_act, void* workspace, size_t workspace_bytes,
                               cgs_stream_t stream);

/* Developer knobs (env CGS_DEBUG at first use, or cgs_debug_set_flags): a bit set of the values below.
 * A lowering knob picks another implementation of the same pass; every one of them gives the same results
 * (bit-identical or within the stated tolerance, see tests/test_conv_gpu.py).  A profiling knob skips part of the
 * work to bound where time goes: its results are wrong by design. */
enum cgs_debug_flag {
  /* profiling */
  CGS_DEBUG_SKIP_A_GATHER = 1,            /* tcgen05 GEMM in gather mode: no A-tile copies */
  CGS_DEBUG_SKIP_WEIGHT_TMA = 2,          /* tcgen05 GEMM: no weight-tile loads */
  CGS_DEBUG_SKIP_MMA = 4,                 /* tcgen05 GEMM / edge_wide_tc: no MMA issue */
  CGS_DEBUG_SKIP_A_TMA = 8,               /* tcgen05 GEMM: no A-tile loads; edge_wide_tc: no patch loads */
  CGS_DEBUG_SKIP_EPILOGUE = 16,           /* tcgen05 GEMM: no epilogue work after the TMEM loads */
  CGS_DEBUG_TRACE = 256,                  /* CTA-0 event trace (cgs_debug_trace, cgs_debug_trace_tc) */
  CGS_DEBUG_GATHER_A = 512,               /* tcgen05 GEMM: cp.async gather of the A tiles instead of TMA boxes */
  CGS_DEBUG_SKIP_STORES = 1024,           /* tcgen05 GEMM / edge_wide_tc: no output stores */
  CGS_DEBUG_NO_PREFETCH = 2048,           /* tcgen05 GEMM: no epilogue operand prefetch; edge_wide_tc: no operand loads */
  /* lowering choices */
  CGS_DEBUG_EDGE_GENERAL = 4096,          /* image-edge passes on the general tcgen05 lowerings, not csrc/edge_*.cu */
  CGS_DEBUG_NO_FC_SPLIT = 16384,          /* no split-K on the long fc forward */
  CGS_DEBUG_PDL_ON = 32768,               /* programmatic dependent launch on everywhere (default: per refinement call) */
  CGS_DEBUG_NO_EDGE_PAIR = 65536,         /* image-edge passes as separate kernels instead of the paired kernel */
  CGS_DEBUG_NO_HEAD_PARTIALS = 131072,    /* separate split-K reduce kernel before the head */
  CGS_DEBUG_NO_FUSION = 524288,           /* no class-fused tcgen05 tiles for the transposed-type passes */
  CGS_DEBUG_FORCE_FUSION = 1048576,       /* class-fused tiles whenever legal, whatever the tile count */
  CGS_DEBUG_NO_MTILE_PAIRS = 4194304,     /* no M-tile pairs (two M tiles per CTA sharing the weight atoms) */
  CGS_DEBUG_FORCE_MTILE_PAIRS = 8388608,  /* M-tile pairs whenever legal */
  CGS_DEBUG_NO_CTA_PAIRS = 16777216,      /* no CTA pairs (clusters of two, tcgen05 cta_group::2) */
  CGS_DEBUG_FORCE_CTA_PAIRS = 33554432,   /* CTA pairs whenever legal */
  CGS_DEBUG_MLP2D_ONE_THREAD = 134217728, /* 2-D refinement with one thread per point, not the four-thread split form
                                             (nhidden == 64 only) */
  CGS_DEBUG_MLP2D_CLUSTER = 268435456,    /* 2-D score and refinement at nhidden == 64 on the cluster form that runs
                                             every other width (wins over MLP2D_ONE_THREAD) */
  CGS_DEBUG_PDL_OFF = 536870912,          /* programmatic dependent launch off everywhere (wins over PDL_ON) */
  CGS_DEBUG_TF32_OPERANDS = 1073741824    /* DCGAN refinement chain on TF32 (FP32-stored) MMA operands, not FP16 */
  /* retired, never reused: 262144, 2097152 */
};

/* Developer aid: read (and reset) the CTA-0 pipeline event trace recorded under CGS_DEBUG_TRACE. */
CGS_API int cgs_debug_trace(unsigned long long* out_host, int capacity);
/* Developer aid: CTA-0 event clocks of the last edge_wide_tc launch run under CGS_DEBUG_TRACE ([8 roles][64 tiles] int64). */
CGS_API int cgs_debug_trace_tc(long long* out_host);
/* Developer aid OUTSIDE the drop-in contract (process-wide atomic; the product never calls it -- only the parity
 * tests do, to keep alternative lowerings covered): replace the CGS_DEBUG knobs (cgs_debug_flag) at run time;
 * returns the previous value. */
CGS_API int cgs_debug_set_flags(int flags);

#ifdef __cplusplus
}
#endif
#endif /* CGS_H_ */
