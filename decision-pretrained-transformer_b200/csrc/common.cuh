// Shared host/device helpers for libdpt_b200.so (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdarg.h>

#include "../../include/dpt_b200.h"

#if defined(__CUDA_ARCH__) && (__CUDA_ARCH__ < 1000)
#error "libdpt_b200 is written for sm_100a (B200) only"
#endif

namespace dpt {

void set_error(const char* fmt, ...);
int sm_count();
// bandit_rollin.cu: compact form of the rollin launch (arm index + reward per step), used by the host pipeline
int bandit_rollin_compact(const float* means, float var, uint64_t seed, uint64_t env_id0, int N, int H, int d, uint8_t* acts_u8,
                          float* ctx_rewards, void* stream);
// Envs per CTA such that the grid (ceil(N / e) CTAs, `slots` resident at a time) ends close to a whole number
// of waves: among e in [min_e, max_e] with at least 3 waves, the one with the fullest last wave (ties: larger e).
// step > 1: only multiples of step are candidates; when none of them qualifies, the rule above without step.
int pick_envs_per_cta(int N, int slots, int min_e, int max_e, int step = 1);

#define DPT_CHECK_ARG(cond, ...)                \
  do {                                          \
    if (!(cond)) {                              \
      dpt::set_error(__VA_ARGS__);              \
      return DPT_ERR_INVALID_ARG;               \
    }                                           \
  } while (0)

#define DPT_CUDA(call)                                                                  \
  do {                                                                                  \
    cudaError_t _e = (call);                                                            \
    if (_e != cudaSuccess) {                                                            \
      dpt::set_error("%s failed: %s (%s:%d)", #call, cudaGetErrorString(_e), __FILE__, __LINE__); \
      return DPT_ERR_CUDA;                                                              \
    }                                                                                   \
  } while (0)

#define DPT_LAUNCH_CHECK()                                                              \
  do {                                                                                  \
    cudaError_t _e = cudaGetLastError();                                                \
    if (_e != cudaSuccess) {                                                            \
      dpt::set_error("kernel launch failed: %s (%s:%d)", cudaGetErrorString(_e), __FILE__, __LINE__); \
      return DPT_ERR_CUDA;                                                              \
    }                                                                                   \
  } while (0)

static inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

#ifdef __CUDACC__
// Streaming (write-once) stores: keep them out of L1, they are never re-read by this kernel.
__device__ __forceinline__ void st_stream(float4* p, float4 v) {
  asm volatile("st.global.L1::no_allocate.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z),
               "f"(v.w)
               : "memory");
}
// predicated forms (one instruction, no branch around the store)
__device__ __forceinline__ void st_stream_if(bool pred, float4* p, float4 v) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %5, 0;\n\t@p st.global.L1::no_allocate.v4.f32 [%0], {%1, %2, %3, %4};\n\t}"
      ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w), "r"((int)pred)
      : "memory");
}
__device__ __forceinline__ void st_stream_if(bool pred, float2* p, float2 v) {
  asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %3, 0;\n\t@p st.global.L1::no_allocate.v2.f32 [%0], {%1, %2};\n\t}" ::"l"(p),
               "f"(v.x), "f"(v.y), "r"((int)pred)
               : "memory");
}
__device__ __forceinline__ void st_stream(float2* p, float2 v) {
  asm volatile("st.global.L1::no_allocate.v2.f32 [%0], {%1, %2};" ::"l"(p), "f"(v.x), "f"(v.y) : "memory");
}
__device__ __forceinline__ void st_stream(float* p, float v) {
  asm volatile("st.global.L1::no_allocate.f32 [%0], %1;" ::"l"(p), "f"(v) : "memory");
}

// Fill base[begin, end) (float indices) with `v`, cooperatively by `nthreads` threads: scalar head
// up to the first 16 B-aligned address, float4 body, scalar tail.  Works for any alignment of base.
__device__ __forceinline__ void fill_range(float* base, size_t begin, size_t end, float v, int tid, int nthreads) {
  const size_t mis = (reinterpret_cast<uintptr_t>(base + begin) >> 2) & 3;   // floats past a 16 B boundary
  size_t b4 = begin + ((4 - mis) & 3);
  if (b4 > end) b4 = end;
  const size_t e4 = b4 + ((end - b4) & ~size_t(3));
  if (tid < (int)(b4 - begin)) st_stream(base + begin + tid, v);
  if (tid < (int)(end - e4)) st_stream(base + e4 + tid, v);
  const float4 v4 = make_float4(v, v, v, v);
  float4* p = reinterpret_cast<float4*>(base + b4);
  const size_t n4 = (e4 - b4) >> 2;
  for (size_t i = tid; i < n4; i += nthreads) st_stream(p + i, v4);
}

// One-hot rows from bit strings.  s_nib[t] holds the 4-bit pattern t as four 0 / 1 floats; threads 0 .. 15 fill it.
__device__ __forceinline__ void onehot_nib_init(float4* s_nib, int t) {
  if (t < 16) s_nib[t] = make_float4((t & 1) ? 1.f : 0.f, (t & 2) ? 1.f : 0.f, (t & 4) ? 1.f : 0.f, (t & 8) ? 1.f : 0.f);
}

// The one-hot rows of a warp task of 32 step quads (lane = quad), D floats per step.  Lane l passes its quad's 4D-bit string `bq`
// (bit u * D + j: step u took arm j), so a quad's rows are exactly D float4 and float4 g of the task is nibble g % D of quad
// g / D's string: D stores per lane, each one shuffle, one shift and one table lookup, 512 B per warp and store.  Float4s at
// g >= nvalid (past the end of the row) are not stored.  per_it(it) runs after store `it`: independent work to interleave.
template <int D, typename F>
__device__ __forceinline__ void onehot_quad_store(float4* abase, uint64_t bq, int lane, int nvalid, const float4* s_nib, F&& per_it) {
  const uint32_t blo = (uint32_t)bq, bhi = (uint32_t)(bq >> 32);
#pragma unroll
  for (int it = 0; it < D; ++it) {
    const int g = it * 32 + lane;
    const int src = g / D, f = g - src * D;
    uint32_t w = __shfl_sync(0xffffffffu, blo, src);
    if (4 * D > 32) {
      const uint32_t wh = __shfl_sync(0xffffffffu, bhi, src);
      w = (uint32_t)((((uint64_t)wh << 32) | w) >> (4 * f));
    } else {
      w >>= 4 * f;
    }
    st_stream_if(g < nvalid, abase + g, s_nib[w & 15u]);
    per_it(it);
  }
}
#endif

}  // namespace dpt
