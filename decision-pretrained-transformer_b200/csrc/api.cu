// Library-level entry points: version, thread-local error string, device info.
#include "common.cuh"

namespace dpt {

static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

int sm_count() {
  static thread_local int cached_dev = -1, cached = 0;
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return 148;
  if (dev != cached_dev) {
    int n = 0;
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
    cached = n;
    cached_dev = dev;
  }
  return cached;
}

int pick_envs_per_cta(int N, int slots, int min_e, int max_e, int step) {
  if (min_e < 1) min_e = 1;
  if (max_e < min_e) max_e = min_e;
  if (slots < 1) slots = 1;
  int best = -1;
  double best_eff = -1.0;
  for (int e = max_e; e >= min_e; --e) {
    if (step > 1 && e % step) continue;
    const long grid = ((long)N + e - 1) / e;
    const long waves = (grid + slots - 1) / slots;
    if (waves < 3 && e > min_e) continue;           // too coarse: keep shrinking e
    const double eff = (double)grid / (double)(waves * slots);
    if (eff > best_eff + 1e-9) best_eff = eff, best = e;
  }
  if (best < 0 && step > 1) return pick_envs_per_cta(N, slots, min_e, max_e, 1);   // no multiple of step qualifies
  return best < 0 ? min_e : best;
}

}  // namespace dpt

extern "C" int dpt_version(void) { return DPT_ABI_VERSION; }

extern "C" const char* dpt_last_error(void) { return dpt::g_err; }

extern "C" int dpt_device_info(int* sm_count, int* cc_major, int* cc_minor) {
  int dev = 0;
  DPT_CUDA(cudaGetDevice(&dev));
  int n = 0, maj = 0, min = 0;
  DPT_CUDA(cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev));
  DPT_CUDA(cudaDeviceGetAttribute(&maj, cudaDevAttrComputeCapabilityMajor, dev));
  DPT_CUDA(cudaDeviceGetAttribute(&min, cudaDevAttrComputeCapabilityMinor, dev));
  if (sm_count) *sm_count = n;
  if (cc_major) *cc_major = maj;
  if (cc_minor) *cc_minor = min;
  return DPT_OK;
}
