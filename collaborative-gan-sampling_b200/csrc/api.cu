// Library-level entry points: version, thread-local error string, device gate.
#include "common.h"

#include <atomic>
#include <cstdlib>

namespace cgs {

char* error_buffer() {
  static thread_local char buf[512] = {0};
  return buf;
}

static std::atomic<long long> g_launches{0};
void count_launch(int n) { g_launches.fetch_add(n, std::memory_order_relaxed); }
long long launches_total() { return g_launches.load(std::memory_order_relaxed); }

static std::atomic<int> g_debug{-1};
int debug_flags() {
  int v = g_debug.load(std::memory_order_relaxed);
  if (v < 0) {
    const char* e = getenv("CGS_DEBUG");
    v = e ? atoi(e) : 0;
    g_debug.store(v, std::memory_order_relaxed);
  }
  return v;
}
void set_debug_flags(int v) { g_debug.store(v < 0 ? 0 : v, std::memory_order_relaxed); }

static thread_local bool tl_pdl = false;
bool pdl_enabled() {
  const int f = debug_flags();
  if (f & CGS_DEBUG_PDL_OFF) return false;
  return tl_pdl || (f & CGS_DEBUG_PDL_ON) != 0;
}
PdlScope::PdlScope(bool on) : prev(tl_pdl) { tl_pdl = on; }
PdlScope::~PdlScope() { tl_pdl = prev; }

int current_device() {
  int dev = -1;
  return cudaGetDevice(&dev) == cudaSuccess ? dev : -1;
}

int device_num_sms() {
  static std::atomic<int> cache[kMaxDevices];     // zero-initialised; 0 = not queried yet
  const int dev = current_device();
  if (dev >= 0 && dev < kMaxDevices) {
    const int v = cache[dev].load(std::memory_order_relaxed);
    if (v) return v;
  }
  int n = 0;
  if (dev < 0 || cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) return 148;
  if (dev < kMaxDevices) cache[dev].store(n, std::memory_order_relaxed);
  return n;
}

int require_sm100() {
  static thread_local int cached_dev = -1;
  static thread_local int cached_ok = 0;
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return set_error(CGS_ERR_CUDA, "no CUDA device: %s (libcgs has no CPU path)", cudaGetErrorString(e));
  if (dev == cached_dev && cached_ok) return CGS_OK;
  int major = 0;
  e = cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev);
  if (e != cudaSuccess) return set_error(CGS_ERR_CUDA, "cudaDeviceGetAttribute: %s", cudaGetErrorString(e));
  if (major != 10) return set_error(CGS_ERR_CUDA, "libcgs is built for sm_100a only; device %d has compute capability %d.x", dev, major);
  cached_dev = dev;
  cached_ok = 1;
  return CGS_OK;
}

}  // namespace cgs

namespace cgs { long long launches_total(); }
extern "C" long long cgs_launch_count(void) { return cgs::launches_total(); }
extern "C" int cgs_version(void) { return CGS_ABI_VERSION; }
extern "C" const char* cgs_last_error(void) { return cgs::error_buffer(); }

namespace cgs { int debug_trace_read(unsigned long long* out, int cap); }
// Developer aid: read (and reset) the CTA-0 pipeline event trace recorded under CGS_DEBUG_TRACE.
extern "C" __attribute__((visibility("default"))) int cgs_debug_trace(unsigned long long* out_host, int capacity) {
  return cgs::debug_trace_read(out_host, capacity);
}

namespace cgs { void set_debug_flags(int v); }
// Developer aid: replace the CGS_DEBUG knobs (cgs_debug_flag) at run time; the parity tests use it to keep every
// lowering covered.  Returns the previous value.
extern "C" __attribute__((visibility("default"))) int cgs_debug_set_flags(int flags) {
  const int old = cgs::debug_flags();
  cgs::set_debug_flags(flags);
  return old;
}

namespace cgs { int debug_trace_tc(long long* out_host); }
// Developer aid: CTA-0 event clocks of the last edge_wide_tc launch run under CGS_DEBUG_TRACE ([8 roles][64 tiles]).
extern "C" CGS_API int cgs_debug_trace_tc(long long* out_host) { return cgs::debug_trace_tc(out_host); }
