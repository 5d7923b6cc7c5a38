// Philox4x32-10 counter-based RNG (Salmon et al., SC'11) and the draw transforms of the DPT
// rollout kernels.  The integer layer is restated bit-for-bit in oracle/philox.py.
//
// Counter = (index, env_lo, env_hi, stream), key = (seed_lo, seed_hi): every draw is addressed by
// the GLOBAL env id, a per-stream index (step / block) and a stream tag, never by thread id, so
// results are independent of launch geometry and of the sharding over GPUs.  This replaces the
// reference's order-dependent global np.random / torch.randn streams (SURVEY.md §5).
#pragma once
#include <stdint.h>

namespace dpt {

enum : uint32_t {
  STREAM_TASK = 0,            // bandit means / theta
  STREAM_ROLLIN_SETUP = 1,    // rollin_bandit: cov, rand_index, dirichlet
  STREAM_ROLLIN_STEP = 2,     // rollin_bandit: per step-pair (categorical uniforms, reward normals)
  STREAM_DARKROOM_STEP = 3,   // rollin_mdp uniform: one word per step
  STREAM_DARKROOM_QUERY = 4,  // query state per sample
  STREAM_ENV_REWARD = 5,      // env.step reward noise (index = step pair)
  STREAM_CTRL = 6,            // controller draws
  STREAM_OFFLINE = 7,         // offline evaluation: Thompson sample=False draws (index = (slot * n_draws + draw) * ceil(d/4) + block)
};

struct Key {
  uint32_t k0, k1;
};

// The key schedule written out: round r uses (k0 + r * 0x9E3779B9, k1 + r * 0xBB67AE85).  Computed on the host into a kernel
// parameter, the round keys sit in the constant bank and each round's XOR takes them as an operand instead of recomputing the
// schedule in the kernel's loop.
struct RoundKeys {
  uint32_t k0[10], k1[10];
};
__host__ __device__ inline RoundKeys round_keys(Key key) {
  RoundKeys rk;
  for (int r = 0; r < 10; ++r) rk.k0[r] = key.k0 + (uint32_t)r * 0x9E3779B9u, rk.k1[r] = key.k1 + (uint32_t)r * 0xBB67AE85u;
  return rk;
}

__device__ __forceinline__ void philox_round(uint32_t& c0, uint32_t& c1, uint32_t& c2, uint32_t& c3, uint32_t k0, uint32_t k1) {
  const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
  const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
  c0 = hi1 ^ c1 ^ k0;
  c1 = lo1;
  c2 = hi0 ^ c3 ^ k1;
  c3 = lo0;
}

__device__ __forceinline__ uint4 philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, Key key) {
  uint32_t k0 = key.k0, k1 = key.k1;
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    philox_round(c0, c1, c2, c3, k0, k1);
    k0 += 0x9E3779B9u;
    k1 += 0xBB67AE85u;
  }
  return make_uint4(c0, c1, c2, c3);
}

__device__ __forceinline__ uint4 philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, const RoundKeys& rk) {
#pragma unroll
  for (int r = 0; r < 10; ++r) philox_round(c0, c1, c2, c3, rk.k0[r], rk.k1[r]);
  return make_uint4(c0, c1, c2, c3);
}

__device__ __forceinline__ uint4 philox_words(Key key, uint64_t env, uint32_t index, uint32_t stream) {
  return philox4x32_10(index, (uint32_t)env, (uint32_t)(env >> 32), stream, key);
}
__device__ __forceinline__ uint4 philox_words(const RoundKeys& rk, uint64_t env, uint32_t index, uint32_t stream) {
  return philox4x32_10(index, (uint32_t)env, (uint32_t)(env >> 32), stream, rk);
}

__device__ __forceinline__ uint32_t word_of(uint4 w, int i) {
  return i == 0 ? w.x : i == 1 ? w.y : i == 2 ? w.z : w.w;
}

// bounded integer in [0, n): (w * n) >> 32
__device__ __forceinline__ uint32_t bounded(uint32_t w, uint32_t n) { return __umulhi(w, n); }

// uniform in [0,1) with 24 bits -- exact in fp32 and fp64
__device__ __forceinline__ float u24(uint32_t w) { return (float)(w >> 8) * 5.9604644775390625e-08f; }

// uniform in (0,1]
__device__ __forceinline__ float u32_open0(uint32_t w) {
  return fmaf((float)w, 2.3283064365386963e-10f, 1.1641532182693481e-10f);
}

// Box-Muller: two words -> two standard normals (fast intrinsics; the oracle consumes the
// dumped values, so only the distribution matters here -- checked statistically in tests).
__device__ __forceinline__ float fast_lg2(float x) {
  float y;
  asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float fast_sqrt(float x) {
  float y;
  asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ void box_muller(uint32_t a, uint32_t b, float& z0, float& z1) {
  // u in [2^-33, 1]: no denormals, -2 ln u = -2 ln2 * lg2 u >= 0
  float r = fast_sqrt(-1.3862943611198906f * fast_lg2(u32_open0(a)));
  float s, c;
  __sincosf((float)b * 1.4629180792671596e-09f /* 2*pi*2^-32 */, &s, &c);
  z0 = r * c;
  z1 = r * s;
}

}  // namespace dpt
