// Host-buffer entry points (the e2e path): the same kernels driven from HOST arrays, with the
// host<->device copies pipelined against the kernel in env chunks (double-buffered scratch).
#include <emmintrin.h>
#include <sched.h>

#include <algorithm>
#include <atomic>
#include <chrono>
#include <cstdlib>
#include <condition_variable>
#include <memory>
#include <mutex>
#include <thread>
#include <vector>

#include "common.cuh"

namespace dpt {
constexpr int HOST_CHUNK_ENVS = 8192;   // envs per pipeline chunk

struct ChunkLayout {
  size_t means, s, a, ns, r, total;  // float offsets
};
static ChunkLayout chunk_layout(int C, int H, int d) {
  auto up = [](size_t x) { return (x + 63) & ~size_t(63); };  // keep every sub-buffer 256 B aligned
  ChunkLayout L;
  size_t o = 0;
  L.means = o, o += up((size_t)C * d);
  L.s = o, o += up((size_t)C * H);
  L.a = o, o += up((size_t)C * H * d);
  L.ns = o, o += up((size_t)C * H);
  L.r = o, o += up((size_t)C * H);
  L.total = o;
  return L;
}
}  // namespace dpt

using namespace dpt;

static thread_local uint64_t t_last_d2h_bytes = 0;
extern "C" uint64_t dpt_bandit_rollin_host_last_d2h_bytes(void) { return t_last_d2h_bytes; }

extern "C" uint64_t dpt_bandit_rollin_host_scratch_bytes(int N, int H, int d) {
  if (N <= 0 || H <= 0 || d <= 0) return 0;
  const int C = N < HOST_CHUNK_ENVS ? N : HOST_CHUNK_ENVS;
  return 2 * chunk_layout(C, H, d).total * sizeof(float);
}

// ---- hybrid host pipeline --------------------------------------------------------------------
// PCIe (~56 GB/s) carries 24 B per env-step when the one-hot actions and the rewards come back as fp32, and the host
// cores are otherwise idle.  A fraction of the chunks is therefore produced in COMPACT form (arm index 1 B + reward 4 B
// per step: 5 B over PCIe) and expanded to the one-hot fp32 layout by host threads, while the other chunks keep
// coming back fully formed by DMA.  The compact arm indices are staged in the chunk's own (not yet written)
// next_states region of the caller's buffer, so no extra pinned memory is needed.  Both kinds of chunks give
// bit-identical results (the same Philox counters; tests/test_rollout_gpu.py::test_bandit_rollin_host_path).
namespace {
constexpr int HOST_PARTS = 16;  // host jobs per chunk and phase
// compact chunks queued for the host before a chunk goes by DMA; measured on a 16-core host: 1: 2.8, 2: 3.4, 3: 4.4,
// 4: 4.9, 6: 5.0 G env-steps/s
constexpr int HOST_BACKLOG = 4;

// Host-side writers use non-temporal stores: the output arrays are written once and never read here, and a normal
// store would first pull every cache line in from DRAM (read-for-ownership), doubling the memory traffic that
// already competes with the DMA engine.
void fill_ones_nt(float* lo, float* hi) {
  while (lo < hi && (reinterpret_cast<uintptr_t>(lo) & 15)) *lo++ = 1.0f;
  const __m128 one = _mm_set1_ps(1.0f);
  for (; lo + 4 <= hi; lo += 4) _mm_stream_ps(lo, one);
  while (lo < hi) *lo++ = 1.0f;
}

// one-hot rows [lo, hi) of width d from arm indices; 4 rows = d aligned 16 B vectors when lo % 4 == 0.
// d <= 5: the 4 d floats of a row quad come from a table indexed by the four arm indices (d^4 <= 625 entries x 16 d
// bytes <= 50 KB, L2-resident): ~5 instructions per row instead of ~30, so the expansion is bound by the memory system,
// not by the cores (measured: 66 -> see DESIGN.md GB/s of host stores on 16 cores).
struct OnehotLut {
  int d = 0;
  float* tab = nullptr;      // [d^4][4 d] floats, 16 B aligned
  int mul[4] = {0, 0, 0, 0};
};
static const OnehotLut* onehot_lut(int d) {
  static OnehotLut luts[6];
  static std::once_flag once[6];
  if (d < 1 || d > 5) return nullptr;
  std::call_once(once[d], [d] {
    OnehotLut& L = luts[d];
    int n = d * d * d * d;
    void* mem = nullptr;
    if (posix_memalign(&mem, 64, (size_t)n * 4 * d * sizeof(float)) != 0) return;
    float* t = reinterpret_cast<float*>(mem);
    for (int i = 0; i < n; ++i) {
      int a[4] = {i % d, (i / d) % d, (i / (d * d)) % d, i / (d * d * d)};
      for (int r = 0; r < 4; ++r)
        for (int j = 0; j < d; ++j) t[(size_t)i * 4 * d + r * d + j] = (j == a[r]) ? 1.0f : 0.0f;
    }
    L.mul[0] = 1, L.mul[1] = d, L.mul[2] = d * d, L.mul[3] = d * d * d;
    L.tab = t, L.d = d;
  });
  return luts[d].tab ? &luts[d] : nullptr;
}

void expand_onehot_nt(float* a, const uint8_t* acts, size_t lo, size_t hi, int d) {
  auto scalar = [&](size_t row) {
    float* o = a + row * d;
    const int arm = acts[row];
    for (int j = 0; j < d; ++j) o[j] = (j == arm) ? 1.0f : 0.0f;
  };
  if ((reinterpret_cast<uintptr_t>(a) & 15) || d > 64) {
    for (size_t row = lo; row < hi; ++row) scalar(row);
    return;
  }
  while (lo < hi && (lo & 3)) scalar(lo++);
  if (const OnehotLut* L = onehot_lut(d)) {
    const int m1 = L->mul[1], m2 = L->mul[2], m3 = L->mul[3];
    for (; lo + 4 <= hi; lo += 4) {
      const float* src = L->tab + (size_t)(acts[lo] + m1 * acts[lo + 1] + m2 * acts[lo + 2] + m3 * acts[lo + 3]) * 4 * d;
      float* o = a + lo * d;
      for (int v = 0; v < d; ++v) _mm_stream_ps(o + 4 * v, _mm_load_ps(src + 4 * v));
    }
  } else {
    alignas(16) float tmp[4 * 64];
    for (; lo + 4 <= hi; lo += 4) {
      for (int j = 0; j < 4 * d; ++j) tmp[j] = 0.0f;
      tmp[acts[lo]] = 1.0f, tmp[d + acts[lo + 1]] = 1.0f, tmp[2 * d + acts[lo + 2]] = 1.0f, tmp[3 * d + acts[lo + 3]] = 1.0f;
      float* o = a + lo * d;
      for (int v = 0; v < d; ++v) _mm_stream_ps(o + 4 * v, _mm_load_ps(tmp + 4 * v));
    }
  }
  while (lo < hi) scalar(lo++);
}

// ---- the reference's own dtypes (collect_data.py:23-53 returns int64 states, float64 one-hot actions / rewards) ----
void fill_ones_i64_nt(int64_t* lo, int64_t* hi) {
  while (lo < hi && (reinterpret_cast<uintptr_t>(lo) & 15)) *lo++ = 1;
  const __m128i one = _mm_set1_epi64x(1);
  for (; lo + 2 <= hi; lo += 2) _mm_stream_si128(reinterpret_cast<__m128i*>(lo), one);
  while (lo < hi) *lo++ = 1;
}
void cvt_f32_f64_nt(double* dst, const float* src, size_t lo, size_t hi) {
  while (lo < hi && ((reinterpret_cast<uintptr_t>(dst + lo) & 15) || (lo & 1))) dst[lo] = (double)src[lo], ++lo;
  for (; lo + 2 <= hi; lo += 2) _mm_stream_pd(dst + lo, _mm_cvtps_pd(_mm_castsi128_ps(_mm_loadl_epi64(reinterpret_cast<const __m128i*>(src + lo)))));
  while (lo < hi) dst[lo] = (double)src[lo], ++lo;
}
static const double* onehot_lut_f64(int d) {   // [d^4][4 d] doubles (d <= 5: <= 100 KB, L2-resident)
  static double* tabs[6] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
  static std::once_flag once[6];
  if (d < 1 || d > 5) return nullptr;
  std::call_once(once[d], [d] {
    const int n = d * d * d * d;
    void* mem = nullptr;
    if (posix_memalign(&mem, 64, (size_t)n * 4 * d * sizeof(double)) != 0) return;
    double* t = reinterpret_cast<double*>(mem);
    for (int i = 0; i < n; ++i) {
      const int a[4] = {i % d, (i / d) % d, (i / (d * d)) % d, i / (d * d * d)};
      for (int r = 0; r < 4; ++r)
        for (int j = 0; j < d; ++j) t[(size_t)i * 4 * d + r * d + j] = (j == a[r]) ? 1.0 : 0.0;
    }
    tabs[d] = t;
  });
  return tabs[d];
}
void expand_onehot_f64_nt(double* a, const uint8_t* acts, size_t lo, size_t hi, int d) {
  auto scalar = [&](size_t row) {
    double* o = a + row * d;
    const int arm = acts[row];
    for (int j = 0; j < d; ++j) o[j] = (j == arm) ? 1.0 : 0.0;
  };
  const double* tab = (reinterpret_cast<uintptr_t>(a) & 15) ? nullptr : onehot_lut_f64(d);
  if (!tab) {
    for (size_t row = lo; row < hi; ++row) scalar(row);
    return;
  }
  while (lo < hi && (lo & 3)) scalar(lo++);
  const int m1 = d, m2 = d * d, m3 = d * d * d;
  for (; lo + 4 <= hi; lo += 4) {   // 4 rows = 4 d doubles = 2 d aligned 16 B vectors
    const double* src = tab + (size_t)(acts[lo] + m1 * acts[lo + 1] + m2 * acts[lo + 2] + m3 * acts[lo + 3]) * 4 * d;
    double* o = a + lo * d;
    for (int v = 0; v < 2 * d; ++v) _mm_stream_pd(o + 2 * v, _mm_load_pd(src + 2 * v));
  }
  while (lo < hi) scalar(lo++);
}

struct HostJobs {
  int K, C, N, H, d, device;
  std::vector<char> compact;                 // per chunk
  std::vector<cudaEvent_t> d2h_done;         // per chunk, recorded on the copy stream after its D2H
  std::unique_ptr<std::atomic<int>[]> enqueued, phase1_left;
  std::atomic<int> next{0}, compact_parts_pending{0};
  std::atomic<bool> failed{false};
  float *s, *a, *ns, *r;
  bool wide = false;                         // reference dtypes: every chunk compact, expanded to int64 / float64
  int64_t *s64 = nullptr, *ns64 = nullptr;
  double *a64 = nullptr, *r64 = nullptr;

  void rows_of(int k, int part, size_t& lo, size_t& hi) const {
    const int e0 = k * C, n = std::min(C, N - e0);
    const size_t row0 = (size_t)e0 * H, nrow = (size_t)n * H;
    lo = row0 + nrow * part / HOST_PARTS, hi = row0 + nrow * (part + 1) / HOST_PARTS;
  }
  // job order: chunk k -> HOST_PARTS phase-1 jobs, then (compact chunks only) HOST_PARTS phase-2 jobs
  void run_worker() {
    cudaSetDevice(device);   // a new thread starts on device 0; the events below belong to the caller's device
    const int per_chunk = 2 * HOST_PARTS, total = K * per_chunk;
    for (;;) {
      const int j = next.fetch_add(1);
      if (j >= total) return;
      const int k = j / per_chunk, sub = j - k * per_chunk, part = sub % HOST_PARTS;
      const bool phase2 = sub >= HOST_PARTS;
      size_t lo, hi;
      rows_of(k, part, lo, hi);
      while (!enqueued[k].load(std::memory_order_acquire) && !failed.load()) std::this_thread::yield();   // kind decided
      if (failed.load()) {
        if (!phase2) phase1_left[k].fetch_sub(1);
        continue;
      }
      if (wide) {
        // staged by DMA at the start of the chunk's own output regions: arm indices (1 B per row) in next_states,
        // fp32 rewards in states; phase 1 expands actions + rewards, phase 2 overwrites the staging areas with ones
        const size_t row0 = (size_t)k * C * H;
        if (!phase2) {
          if (cudaEventSynchronize(d2h_done[k]) != cudaSuccess) {
            failed.store(true);
            phase1_left[k].fetch_sub(1);
            compact_parts_pending.fetch_sub(1);
            continue;
          }
          const uint8_t* acts = reinterpret_cast<const uint8_t*>(ns64 + row0) - row0;
          const float* rew = reinterpret_cast<const float*>(s64 + row0) - row0;
          expand_onehot_f64_nt(a64, acts, lo, hi, d);
          cvt_f32_f64_nt(r64, rew, lo, hi);
          _mm_sfence();
          phase1_left[k].fetch_sub(1, std::memory_order_release);
          compact_parts_pending.fetch_sub(1);
        } else {
          while (phase1_left[k].load(std::memory_order_acquire) > 0) std::this_thread::yield();
          fill_ones_i64_nt(s64 + lo, s64 + hi);
          fill_ones_i64_nt(ns64 + lo, ns64 + hi);
        }
        continue;
      }
      if (!compact[k]) {                      // DMA chunk: only the constant state columns are host work
        if (!phase2) {
          fill_ones_nt(s + lo, s + hi);
          fill_ones_nt(ns + lo, ns + hi);
        }
        continue;
      }
      if (!phase2) {
        if (cudaEventSynchronize(d2h_done[k]) != cudaSuccess) {
          failed.store(true);
          phase1_left[k].fetch_sub(1);
          compact_parts_pending.fetch_sub(1);
          continue;
        }
        const uint8_t* acts = reinterpret_cast<const uint8_t*>(ns + (size_t)k * C * H) - (size_t)k * C * H;  // acts[row]
        expand_onehot_nt(a, acts, lo, hi, d);
        fill_ones_nt(s + lo, s + hi);
        _mm_sfence();
        phase1_left[k].fetch_sub(1, std::memory_order_release);
        compact_parts_pending.fetch_sub(1);
      } else {                                // the staged arm indices of this chunk are consumed: overwrite them
        while (phase1_left[k].load(std::memory_order_acquire) > 0) std::this_thread::yield();
        fill_ones_nt(ns + lo, ns + hi);
      }
    }
    _mm_sfence();
  }
};
}  // namespace

// ---- host memory write peak (measurement aid for the e2e roofline) ----------------------------------------
// The host half of the e2e path is a pure write stream into the caller's arrays.  This measures what the box's
// cores can stream with non-temporal stores: `n_threads` threads (0 = every core this process may run on) each
// write their own contiguous slice of `dst` (NULL: an internal malloc'ed, first-touched buffer) of `bytes` bytes,
// three passes after one warm-up pass, best pass reported in GB/s.  Debug / bench export, not on the product path.
static int usable_cores() {
  cpu_set_t set;
  CPU_ZERO(&set);
  if (sched_getaffinity(0, sizeof(set), &set) == 0) {
    const int n = CPU_COUNT(&set);
    if (n > 0) return n;
  }
  return (int)std::max(1u, std::thread::hardware_concurrency());
}

extern "C" double dpt_host_write_peak(void* dst, uint64_t bytes, int n_threads) {
  if (bytes < (1u << 20)) bytes = 1ull << 30;
  const int T = n_threads > 0 ? n_threads : usable_cores();
  void* own = nullptr;
  if (!dst) {
    if (posix_memalign(&own, 4096, bytes) != 0) return 0.0;
    dst = own;
  }
  float* base = reinterpret_cast<float*>(dst);
  const size_t n = bytes / sizeof(float);
  double best = 0.0;
  for (int pass = 0; pass < 4; ++pass) {
    std::atomic<int> ready{0};
    std::atomic<bool> go{false};
    std::vector<std::thread> th;
    for (int t = 0; t < T; ++t)
      th.emplace_back([&, t] {
        float* lo = base + ((n * t / T) & ~size_t(15));
        float* hi = (t == T - 1) ? base + n : base + ((n * (t + 1) / T) & ~size_t(15));
        ready.fetch_add(1);
        while (!go.load(std::memory_order_acquire)) std::this_thread::yield();
        fill_ones_nt(lo, hi);
        _mm_sfence();
      });
    while (ready.load() < T) std::this_thread::yield();
    const auto t0 = std::chrono::steady_clock::now();
    go.store(true, std::memory_order_release);
    for (auto& x : th) x.join();
    const double s = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
    if (pass > 0) best = std::max(best, (double)bytes / s / 1e9);   // pass 0 first-touches the pages
  }
  free(own);
  return best;
}

// ---- persistent host worker pool ---------------------------------------------------------------------------
// The host half of the pipeline (constant columns, expansion of compact chunks) runs on worker threads that live for
// the process: created on first use, one per core of THIS rank's share of the cores the process may run on
// (sched_getaffinity, split by LOCAL_RANK / LOCAL_WORLD_SIZE under torchrun) and pinned there, so that the ranks of a
// node do not migrate onto each other's cores.
namespace {
std::vector<int> rank_cpus() {
  std::vector<int> all;
  cpu_set_t set;
  CPU_ZERO(&set);
  if (sched_getaffinity(0, sizeof(set), &set) == 0)
    for (int c = 0; c < CPU_SETSIZE; ++c)
      if (CPU_ISSET(c, &set)) all.push_back(c);
  if (all.empty())
    for (unsigned c = 0; c < std::max(1u, std::thread::hardware_concurrency()); ++c) all.push_back((int)c);
  int w = 1, r = 0;
  if (const char* e = getenv("LOCAL_WORLD_SIZE")) w = std::max(1, atoi(e));
  if (const char* e = getenv("LOCAL_RANK")) r = std::max(0, atoi(e));
  if (w > 1 && (int)all.size() >= w) {
    const size_t k = all.size() / w, lo = (size_t)(r % w) * k;
    return std::vector<int>(all.begin() + lo, all.begin() + lo + k);
  }
  return all;
}

struct HostPool {
  std::mutex m;
  std::condition_variable cv_go, cv_done;
  HostJobs* jobs = nullptr;
  uint64_t epoch = 0;
  int want = 0, active = 0;
  std::vector<std::thread> threads;
  std::vector<int> cpus;

  static HostPool& get() {
    static HostPool* p = new HostPool();   // never destroyed: the threads sleep on cv_go until the process exits
    return *p;
  }
  int capacity() {
    std::lock_guard<std::mutex> g(m);
    if (cpus.empty()) cpus = rank_cpus();
    int n = (int)cpus.size();              // the thread that drives the GPU pipeline sleeps in its waits
    if (const char* e = getenv("DPT_HOST_WORKERS")) n = atoi(e);
    return std::max(1, std::min(64, n));
  }
  void loop(int idx) {
    uint64_t seen = 0;
    for (;;) {
      HostJobs* j;
      {
        std::unique_lock<std::mutex> lk(m);
        cv_go.wait(lk, [&] { return epoch != seen && idx < want; });
        seen = epoch;
        j = jobs;
      }
      j->run_worker();
      {
        std::lock_guard<std::mutex> g(m);
        if (--active == 0) cv_done.notify_all();
      }
    }
  }
  void start(HostJobs* j, int n) {
    std::lock_guard<std::mutex> g(m);
    while ((int)threads.size() < n) {
      const int idx = (int)threads.size();
      threads.emplace_back([this, idx] { loop(idx); });
      if (cpus.size() > 1) {   // worker idx -> core idx of the rank's share
        cpu_set_t one;
        CPU_ZERO(&one);
        CPU_SET(cpus[(size_t)idx % cpus.size()], &one);
        pthread_setaffinity_np(threads.back().native_handle(), sizeof(one), &one);
      }
      threads.back().detach();
    }
    jobs = j, want = n, active = n, ++epoch;
    cv_go.notify_all();
  }
  void wait() {
    std::unique_lock<std::mutex> lk(m);
    cv_done.wait(lk, [&] { return active == 0; });
  }
};
}  // namespace

static int rollin_host_impl(const float* means_host, float var, uint64_t seed, uint64_t env_id0, int N, int H, int d,
                            float* ctx_states_host, float* ctx_actions_host, float* ctx_next_states_host,
                            float* ctx_rewards_host, int64_t* s64, double* a64, int64_t* ns64, double* r64, void* scratch,
                            uint64_t scratch_bytes, void* stream) {
  const bool wide = a64 != nullptr;
  DPT_CHECK_ARG(N >= 0 && H >= 0 && d >= 1, "dpt_bandit_rollin_host: bad sizes N=%d H=%d d=%d", N, H, d);
  if (N == 0 || H == 0) return DPT_OK;
  DPT_CHECK_ARG(means_host && (wide ? (s64 && ns64 && r64) : (ctx_states_host && ctx_actions_host && ctx_next_states_host && ctx_rewards_host)),
                "dpt_bandit_rollin_host: null host pointer");
  DPT_CHECK_ARG(!wide || d <= 255, "dpt_bandit_rollin_host_f64: d=%d > 255", d);
  DPT_CHECK_ARG(scratch && scratch_bytes >= dpt_bandit_rollin_host_scratch_bytes(N, H, d),
                "dpt_bandit_rollin_host: scratch too small (%llu < %llu bytes)", (unsigned long long)scratch_bytes,
                (unsigned long long)dpt_bandit_rollin_host_scratch_bytes(N, H, d));
  const int C = N < HOST_CHUNK_ENVS ? N : HOST_CHUNK_ENVS;
  const ChunkLayout L = chunk_layout(C, H, d);
  cudaStream_t cs = (cudaStream_t)stream;
  struct Res {   // the pipeline's own stream and events: released on every return path
    cudaStream_t copy = nullptr;   // D2H stream, so chunk k's copies overlap chunk k+1's kernel
    cudaEvent_t done[2] = {nullptr, nullptr}, freed[2] = {nullptr, nullptr};
    std::vector<cudaEvent_t> d2h;
    ~Res() {
      for (int i = 0; i < 2; ++i) {
        if (done[i]) cudaEventDestroy(done[i]);
        if (freed[i]) cudaEventDestroy(freed[i]);
      }
      for (auto& ev : d2h)
        if (ev) cudaEventDestroy(ev);
      if (copy) cudaStreamDestroy(copy);
    }
  } res;
  DPT_CUDA(cudaStreamCreateWithFlags(&res.copy, cudaStreamNonBlocking));
  for (int i = 0; i < 2; ++i) {
    DPT_CUDA(cudaEventCreateWithFlags(&res.done[i], cudaEventDisableTiming));
    // (blocking sync: the thread that drives the pipeline sleeps in its pacing waits instead of spinning on a core
    //  the workers can use -- 4 cores per rank at 8 GPUs)
    DPT_CUDA(cudaEventCreateWithFlags(&res.freed[i], cudaEventDisableTiming | cudaEventBlockingSync));
  }
  cudaStream_t copy = res.copy;
  cudaEvent_t* done = res.done;
  cudaEvent_t* freed = res.freed;
  // The bandit state is the constant [1] (envs/bandit_env.py:38): context_states / context_next_states never cross
  // PCIe, host threads write them (and expand the compact chunks) while the GPU pipeline runs.
  HostJobs jobs;
  jobs.K = (N + C - 1) / C, jobs.C = C, jobs.N = N, jobs.H = H, jobs.d = d;
  DPT_CUDA(cudaGetDevice(&jobs.device));
  jobs.s = ctx_states_host, jobs.a = ctx_actions_host, jobs.ns = ctx_next_states_host, jobs.r = ctx_rewards_host;
  jobs.wide = wide, jobs.s64 = s64, jobs.a64 = a64, jobs.ns64 = ns64, jobs.r64 = r64;
  jobs.compact.assign(jobs.K, 0);
  jobs.enqueued.reset(new std::atomic<int>[jobs.K]);
  jobs.phase1_left.reset(new std::atomic<int>[jobs.K]);
  const bool balance = !wide && jobs.K >= 4 && d <= 255;   // wide: every chunk compact; few chunks or d > 255: every chunk by DMA
  for (int kk = 0; kk < jobs.K; ++kk) {
    jobs.enqueued[kk].store(0);
    jobs.phase1_left[kk].store(HOST_PARTS);
  }
  res.d2h.assign(jobs.K, nullptr);
  for (int kk = 0; kk < jobs.K; ++kk) DPT_CUDA(cudaEventCreateWithFlags(&res.d2h[kk], cudaEventDisableTiming));
  jobs.d2h_done = res.d2h;
  const size_t total_rows = (size_t)N * H;
  HostPool& pool = HostPool::get();
  const int n_workers = (int)std::min<size_t>((size_t)pool.capacity(), std::max<size_t>(1, total_rows >> 18));
  pool.start(&jobs, n_workers);
  int rc = DPT_OK;
  int k = 0;
  uint64_t d2h_bytes = 0;
  for (int e0 = 0; e0 < N && rc == DPT_OK; e0 += C, ++k) {
    const int n = (N - e0) < C ? (N - e0) : C;
    const int b = k & 1;
    float* buf = reinterpret_cast<float*>(scratch) + (size_t)b * L.total;
    cudaError_t ce = cudaSuccess;
    auto ck = [&](cudaError_t e) {
      if (ce == cudaSuccess) ce = e;
    };
    if (k >= 2) ck(cudaEventSynchronize(freed[b]));    // buffer b's previous D2H has drained (host-side pacing)
    // kind of this chunk: compact when the host workers would otherwise run out of expansion work
    // balance: the host cores expand compact chunks (5 B per step over PCIe) as fast as they can -- with the table-driven
    // expansion that alone reaches the host's measured store bandwidth on a 16-core box -- and a chunk goes by DMA
    // (24 B per step over PCIe, 8 B per step of host work) only while more than HOST_BACKLOG compact chunks are queued
    // for the host, i.e. when the cores, not PCIe, are what the pipeline waits for (few cores per rank at 8 GPUs)
    jobs.compact[k] = wide || (balance && jobs.compact_parts_pending.load() < HOST_BACKLOG * HOST_PARTS);
    if (jobs.compact[k]) jobs.compact_parts_pending.fetch_add(HOST_PARTS);
    ck(cudaMemcpyAsync(buf + L.means, means_host + (size_t)e0 * d, sizeof(float) * n * d, cudaMemcpyHostToDevice, cs));
    const size_t row = (size_t)e0 * H, nrow = (size_t)n * H;
    if (jobs.compact[k]) {
      uint8_t* acts_dev = reinterpret_cast<uint8_t*>(buf + L.a);
      rc = bandit_rollin_compact(buf + L.means, var, seed, env_id0 + (uint64_t)e0, n, H, d, acts_dev, buf + L.r, cs);
      if (rc != DPT_OK) break;
      ck(cudaEventRecord(done[b], cs));
      ck(cudaStreamWaitEvent(copy, done[b], 0));
      if (wide) {   // staged arm indices / fp32 rewards at the start of the chunk's next_states / states regions
        ck(cudaMemcpyAsync(ns64 + row, acts_dev, nrow, cudaMemcpyDeviceToHost, copy));
        ck(cudaMemcpyAsync(s64 + row, buf + L.r, sizeof(float) * nrow, cudaMemcpyDeviceToHost, copy));
      } else {
        ck(cudaMemcpyAsync(ctx_next_states_host + row, acts_dev, nrow, cudaMemcpyDeviceToHost, copy));   // staged arm indices
        ck(cudaMemcpyAsync(ctx_rewards_host + row, buf + L.r, sizeof(float) * nrow, cudaMemcpyDeviceToHost, copy));
      }
    } else {
      rc = dpt_bandit_rollin(buf + L.means, var, DPT_REWARD_GAUSSIAN, seed, env_id0 + (uint64_t)e0, n, H, d, buf + L.s, buf + L.a,
                             buf + L.ns, buf + L.r, nullptr, nullptr, nullptr, cs);
      if (rc != DPT_OK) break;
      ck(cudaEventRecord(done[b], cs));
      ck(cudaStreamWaitEvent(copy, done[b], 0));
      ck(cudaMemcpyAsync(ctx_actions_host + row * d, buf + L.a, sizeof(float) * nrow * d, cudaMemcpyDeviceToHost, copy));
      ck(cudaMemcpyAsync(ctx_rewards_host + row, buf + L.r, sizeof(float) * nrow, cudaMemcpyDeviceToHost, copy));
    }
    d2h_bytes += jobs.compact[k] ? nrow * 5 : nrow * 4 * (uint64_t)(d + 1);
    ck(cudaEventRecord(freed[b], copy));
    ck(cudaEventRecord(jobs.d2h_done[k], copy));
    if (ce != cudaSuccess) {   // a failed enqueue: stop here, release the workers (they see `failed`), report below
      set_error("dpt_bandit_rollin_host: %s while enqueueing chunk %d", cudaGetErrorString(ce), k);
      rc = DPT_ERR_CUDA;
      break;
    }
    jobs.enqueued[k].store(1, std::memory_order_release);
  }
  if (rc != DPT_OK) jobs.failed.store(true);
  t_last_d2h_bytes = d2h_bytes;
  pool.wait();
  cudaError_t e1 = cudaStreamSynchronize(copy);
  cudaError_t e2 = cudaStreamSynchronize(cs);
  if (jobs.failed.load() && rc == DPT_OK) {
    set_error("dpt_bandit_rollin_host: a host worker failed while waiting for its chunk");
    return DPT_ERR_CUDA;
  }
  if (rc != DPT_OK) return rc;
  if (e1 != cudaSuccess || e2 != cudaSuccess) {
    set_error("dpt_bandit_rollin_host: %s", cudaGetErrorString(e1 != cudaSuccess ? e1 : e2));
    return DPT_ERR_CUDA;
  }
  return DPT_OK;
}

extern "C" int dpt_bandit_rollin_host(const float* means_host, float var, uint64_t seed, uint64_t env_id0, int N,
                                      int H, int d, float* ctx_states_host, float* ctx_actions_host,
                                      float* ctx_next_states_host, float* ctx_rewards_host, void* scratch,
                                      uint64_t scratch_bytes, void* stream) {
  return rollin_host_impl(means_host, var, seed, env_id0, N, H, d, ctx_states_host, ctx_actions_host, ctx_next_states_host,
                          ctx_rewards_host, nullptr, nullptr, nullptr, nullptr, scratch, scratch_bytes, stream);
}

extern "C" int dpt_bandit_rollin_host_f64(const float* means_host, float var, uint64_t seed, uint64_t env_id0, int N, int H, int d,
                                          int64_t* ctx_states_host, double* ctx_actions_host, int64_t* ctx_next_states_host,
                                          double* ctx_rewards_host, void* scratch, uint64_t scratch_bytes, void* stream) {
  DPT_CHECK_ARG(ctx_actions_host, "dpt_bandit_rollin_host_f64: null host pointer");
  return rollin_host_impl(means_host, var, seed, env_id0, N, H, d, nullptr, nullptr, nullptr, nullptr, ctx_states_host,
                          ctx_actions_host, ctx_next_states_host, ctx_rewards_host, scratch, scratch_bytes, stream);
}
