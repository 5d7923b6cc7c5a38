// Ordered multi-source sum: dst[i] = ((src[0][i] + src[1][i]) + ...) + src[M-1][i], always in source order.
//
// The data-parallel interactive trainer (dist.train_interactive_sharded) keeps one gradient slot per micro-batch, each on
// the GPU that computed it.  Every rank sums ALL slots with this kernel, reading the other ranks' slots through their
// peer mappings (CUDA IPC, NVLink) with ordinary loads.  Because the order of the additions is fixed by the slot index
// and not by the rank layout, every rank computes the same bits whatever the number of GPUs.  Ordering against the
// writers is the caller's job (stream synchronise + barrier before the call, a second barrier before a slot is rewritten).
#include <algorithm>

#include "common.cuh"

namespace dpt {

constexpr int OS_CHUNK = 128;      // source pointers per launch (1 KB of kernel parameters)
constexpr int OS_THREADS = 256;

struct OrderedSumParams {
  const float* src[OS_CHUNK];
  int m;          // sources in this launch
  int first;      // 1: the first launch (the sum starts at src[0]); 0: continue from dst
  uint64_t n;     // floats
  float* dst;
};

// VEC: every pointer is 16 B aligned, so each thread adds float4s; the n % 4 tail is added by the first threads.
template <bool VEC>
__global__ void __launch_bounds__(OS_THREADS) ordered_sum_kernel(const OrderedSumParams p) {
  const uint64_t tid = (uint64_t)blockIdx.x * OS_THREADS + threadIdx.x, stride = (uint64_t)gridDim.x * OS_THREADS;
  uint64_t done = 0;
  if constexpr (VEC) {
    const uint64_t n4 = p.n >> 2;
    for (uint64_t i = tid; i < n4; i += stride) {
      float4 acc = p.first ? reinterpret_cast<const float4*>(p.src[0])[i] : reinterpret_cast<const float4*>(p.dst)[i];
      for (int s = p.first; s < p.m; ++s) {
        const float4 v = reinterpret_cast<const float4*>(p.src[s])[i];
        acc.x += v.x, acc.y += v.y, acc.z += v.z, acc.w += v.w;
      }
      reinterpret_cast<float4*>(p.dst)[i] = acc;
    }
    done = n4 << 2;
  }
  for (uint64_t i = done + tid; i < p.n; i += stride) {
    float acc = p.first ? p.src[0][i] : p.dst[i];
    for (int s = p.first; s < p.m; ++s) acc += p.src[s][i];
    p.dst[i] = acc;
  }
}

}  // namespace dpt

using namespace dpt;

extern "C" int dpt_ordered_sum_f32(const float* const* src, int M, int64_t n, float* dst, void* stream) {
  DPT_CHECK_ARG(M >= 0 && n >= 0, "dpt_ordered_sum_f32: M=%d n=%lld must be >= 0", M, (long long)n);
  if (M == 0 || n == 0) return DPT_OK;
  DPT_CHECK_ARG(src && dst, "dpt_ordered_sum_f32: null %s", src ? "dst" : "src array");
  bool vec = aligned16(dst);
  for (int s = 0; s < M; ++s) {
    DPT_CHECK_ARG(src[s], "dpt_ordered_sum_f32: src[%d] is null", s);
    DPT_CHECK_ARG(src[s] != dst, "dpt_ordered_sum_f32: src[%d] aliases dst", s);
    vec = vec && aligned16(src[s]);
  }
  const long blocks = std::min<long>(((long)((n + 3) / 4) + OS_THREADS - 1) / OS_THREADS, (long)sm_count() * 8);
  for (int s0 = 0; s0 < M; s0 += OS_CHUNK) {
    OrderedSumParams p{};
    p.m = std::min(OS_CHUNK, M - s0), p.first = s0 == 0, p.n = (uint64_t)n, p.dst = dst;
    for (int s = 0; s < p.m; ++s) p.src[s] = src[s0 + s];
    if (vec)
      ordered_sum_kernel<true><<<(int)blocks, OS_THREADS, 0, (cudaStream_t)stream>>>(p);
    else
      ordered_sum_kernel<false><<<(int)blocks, OS_THREADS, 0, (cudaStream_t)stream>>>(p);
    DPT_LAUNCH_CHECK();
  }
  return DPT_OK;
}
