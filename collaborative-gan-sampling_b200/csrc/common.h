// Shared host-side helpers: status codes, thread-local error message, CUDA error capture.
#pragma once
#include <atomic>
#include <cstdarg>
#include <cstdio>
#include <mutex>
#include <cuda_runtime.h>

#include "cgs.h"

namespace cgs {

char* error_buffer();   // thread-local, 512 bytes (api.cu)

inline int set_error(int status, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(error_buffer(), 512, fmt, ap);
  va_end(ap);
  return status;
}

inline int check_launch(const char* what) {
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return set_error(CGS_ERR_CUDA, "%s: %s", what, cudaGetErrorString(e));
  return CGS_OK;
}

// The product never runs on anything but sm_100: refuse loudly instead of falling back.
int require_sm100();

// Per-device facts and one-time kernel attributes.  cudaFuncSetAttribute and the SM count are PER DEVICE: a process
// that drives several GPUs (or several host threads) must not share one cached flag, so every cache below is indexed
// by the current device and guarded (ADVICE r1).
constexpr int kMaxDevices = 64;
int current_device();               // cudaGetDevice, -1 on error
int device_num_sms();               // multiprocessor count of the current device (cached per device, api.cu)

struct DynSmemCache {               // one per kernel instantiation (function-local static)
  std::mutex m;
  std::atomic<size_t> set[kMaxDevices];
  DynSmemCache() { for (auto& v : set) v.store(0, std::memory_order_relaxed); }
};
// Opt the kernel in to `smem` bytes of dynamic shared memory on the current device (idempotent, grows only).
template <typename K>
inline cudaError_t ensure_dyn_smem(K kernel, size_t smem, DynSmemCache& c) {
  const int dev = current_device();
  if (dev < 0 || dev >= kMaxDevices) return cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (c.set[dev].load(std::memory_order_acquire) >= smem) return cudaSuccess;
  std::lock_guard<std::mutex> lock(c.m);
  if (c.set[dev].load(std::memory_order_relaxed) >= smem) return cudaSuccess;
  cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e == cudaSuccess) c.set[dev].store(smem, std::memory_order_release);
  return e;
}

// Developer knobs (cgs_debug_flag in cgs.h): env CGS_DEBUG at first use, overridable with cgs_debug_set_flags (api.cu).
int debug_flags();

// Process-wide count of kernels launched by the library (cgs_launch_count).
void count_launch(int n = 1);

// Launch helper of the chain kernels.  With programmatic dependent launch the launch carries the programmatic stream
// serialization attribute (the kernels call pdl_wait() before they touch memory written by their predecessor, so a
// kernel's set-up -- barrier init, TMEM allocation, tensor-map prefetch -- overlaps the previous kernel's drain).
// Measured on B200 inside the replayed CUDA graph: +1.5 % on the DCGAN-64 step, +1.1 % on DCGAN-32, -0.8 % on the
// MNIST-sized nets (their kernels are 20-45 us; an early-resident successor only gets in the way), so the refinement
// loop switches it on per call from its average work per launch (refine_conv.cu).  CGS_DEBUG_PDL_ON forces it on
// everywhere, CGS_DEBUG_PDL_OFF off.
bool pdl_enabled();
struct PdlScope {            // switches programmatic dependent launch on for the launches of the calling thread
  explicit PdlScope(bool on);
  ~PdlScope();
  bool prev;
};
template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = pdl_enabled() ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}
// Same, as clusters of `cluster_x` CTAs along x (the grid must be a multiple of it).
template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl_cluster(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st,
                                      int cluster_x, Args... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[2];
  int n = 0;
  if (cluster_x > 1) {
    attr[n].id = cudaLaunchAttributeClusterDimension;
    attr[n].val.clusterDim.x = (unsigned)cluster_x;
    attr[n].val.clusterDim.y = 1;
    attr[n].val.clusterDim.z = 1;
    ++n;
  }
  if (pdl_enabled()) {
    attr[n].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[n].val.programmaticStreamSerializationAllowed = 1;
    ++n;
  }
  cfg.attrs = attr;
  cfg.numAttrs = n;
  return cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}

// cluster form of the 2-D MLP kernels, any nhidden = 16..256 divisible by 16 (mlp2d_cluster.cu); the descriptor is
// already checked, inv_n = 1 / n_mean
int mlp2d_cluster_score(const cgs_mlp_desc& d, const float* x, int64_t n, float inv_n, float* sig_out,
                        float* logit_out, float* sal_out, cudaStream_t st);
int mlp2d_cluster_refine(const cgs_mlp_desc& d, const cgs_refine2d_cfg& cfg, float inv_n, const float* x_in, int64_t n,
                         float* best_x, float* best_loss, float* best_step, float* traj, cudaStream_t st);

// shared device utilities (sampling_kernels.cu)
int compact_flags(const unsigned char* flags, long n, int* block_counts, int* idx_out, int* count_out, cudaStream_t st);
int gather_rows(const void* src, long row_bytes, const int* idx, const int* count, long max_rows, void* dst,
                cudaStream_t st);

}  // namespace cgs
