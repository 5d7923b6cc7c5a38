// fp32 CUDA-core building blocks of the dense GPT-2 kernels (gpt2_dense_fp32.cu forward, gpt2_train.cu backward):
// one thread owns one token row and keeps its 32-wide vectors in registers.
#pragma once
#include "gpt2_model.cuh"

namespace dpt {

__device__ __forceinline__ float2 ffma2_(float2 a, float2 b, float2 c) {
  float2 d;
  asm("fma.rn.f32x2 %0, %1, %2, %3;"
      : "=l"(reinterpret_cast<unsigned long long&>(d))
      : "l"(reinterpret_cast<unsigned long long&>(a)), "l"(reinterpret_cast<unsigned long long&>(b)),
        "l"(reinterpret_cast<unsigned long long&>(c)));
  return d;
}

// acc[0..31] += sum_i xs[i] * W[i][col0 .. col0+31],  W in shared memory with row stride `ld` floats
template <int IN>
__device__ __forceinline__ void row_matvec32(const float* xs, const float* W, int ld, int col0, float2* acc) {
#pragma unroll 4
  for (int i = 0; i < IN; ++i) {
    const float2 xx = make_float2(xs[i], xs[i]);
    const float4* row = reinterpret_cast<const float4*>(W + i * ld + col0);
#pragma unroll
    for (int o = 0; o < 8; ++o) {
      const float4 w = row[o];
      acc[2 * o] = ffma2_(xx, make_float2(w.x, w.y), acc[2 * o]);
      acc[2 * o + 1] = ffma2_(xx, make_float2(w.z, w.w), acc[2 * o + 1]);
    }
  }
}

template <bool STATS = false>
__device__ __forceinline__ void ln_row_f(const float* x, const float* w, const float* b, float* y, float* stats = nullptr) {
  float mean = 0.f;
#pragma unroll
  for (int c = 0; c < G_E; ++c) mean += x[c];
  mean *= (1.0f / G_E);
  float var = 0.f;
#pragma unroll
  for (int c = 0; c < G_E; ++c) var = fmaf(x[c] - mean, x[c] - mean, var);
  const float rs = 1.0f / sqrtf(var * (1.0f / G_E) + 1e-5f);
  if (STATS) stats[0] = mean, stats[1] = rs;
#pragma unroll
  for (int c = 0; c < G_E; ++c) y[c] = (x[c] - mean) * rs * __ldg(w + c) + __ldg(b + c);
}

__device__ __forceinline__ float gelu_new_f(float x) {
  return 0.5f * x * (1.0f + tanhf(0.7978845608028654f * (x + 0.044715f * x * x * x)));
}

__device__ __forceinline__ void store32_(float* dst, const float* v) {
  float4* d4 = reinterpret_cast<float4*>(dst);
#pragma unroll
  for (int o = 0; o < 8; ++o) d4[o] = make_float4(v[4 * o], v[4 * o + 1], v[4 * o + 2], v[4 * o + 3]);
}

__device__ __forceinline__ void load32_(float* v, const float* src) {
  const float4* s4 = reinterpret_cast<const float4*>(src);
#pragma unroll
  for (int o = 0; o < 8; ++o) {
    const float4 t = s4[o];
    v[4 * o] = t.x, v[4 * o + 1] = t.y, v[4 * o + 2] = t.z, v[4 * o + 3] = t.w;
  }
}

}  // namespace dpt
