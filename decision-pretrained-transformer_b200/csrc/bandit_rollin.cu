// Fused bandit rollout kernel: rollin_bandit (reference collect_data.py:23-53) + BanditEnv.transit
// (envs/bandit_env.py:56-64) for N envs x H steps in one launch.
//
// Layout of work ("one warp per env batch"): a CTA owns `envs_per_cta` consecutive envs.
//   1. setup, one thread per env: behaviour policy of rollin_bandit -- cov ~ U{0,.1,..,1},
//      probs ~ Dirichlet(1_d), rand_index ~ U{0..d-1}, probs = (1-cov) probs + cov e_idx -- then the
//      normalised cdf of np.random.choice(p=) computed with the SAME float64 operation sequence
//      as numpy (no FMA contraction), turned into integer thresholds so the per-step categorical
//      draw is (d-1) integer compares and bit-exact against the oracle;
//   2. meanwhile the other warps stream the constant context_states / context_next_states (== 1);
//   3. step loop: each warp takes 128-step ranges of one env; a lane owns a step quad and makes
//      two Philox4x32-10 calls for it (one per step pair: 2 categorical uniforms + 1 Box-Muller
//      pair each, round keys from the constant bank).  Rewards go out as one float4 per lane
//      (512 B per warp store); the quad's one-hot rows (4d floats = d float4) are re-tiled across
//      the warp by shuffling the quads' 4d-bit strings, one 16-entry table lookup per float4
//      (onehot_quad_store, shared with the online loop's context expansion).
// HBM traffic is write-only: 4*(2+d+1) B per env-step (32 B for d=5), inputs are < 0.1 B/step.
#include <string.h>

#include <type_traits>
#include <unordered_map>

#include "common.cuh"
#include "philox.cuh"

namespace dpt {

constexpr int RB_THREADS = 256;
constexpr int RB_WARPS = RB_THREADS / 32;
constexpr int RB_MAX_ENVS = 32;
constexpr int RB_MAX_D = 32;

enum { MODE_PHILOX = 0, MODE_PHILOX_DUMP = 1, MODE_INJECT = 2 };

struct RollinParams {
  const float* means;
  float var;
  int rtype;  // DPT_REWARD_*
  Key key;
  RoundKeys rk;  // key schedule of `key` (fast path: round keys from the constant bank)
  uint64_t env_id0;
  int N, H, d, envs_per_cta;
  float *ctx_s, *ctx_a, *ctx_ns, *ctx_r;
  uint8_t* acts_u8;  // compact form (host pipeline): arm index per step [N,H] instead of the one-hot / state tensors
  double* stats;  // nullable: += (sum r, sum r^2, #pulls of the optimal arm) over all env-steps
  // fused all-gather over NVLink peer memory (nullable): when the LAST CTA of the launch has seen every
  // CTA's contribution, it stores this rank's three totals into slot `peer_slot` of every rank's gather
  // buffer (peer pointers are CUDA-IPC mappings; plain system-scope stores, no collective launch)
  dpt_bandit_inject_t in;
  dpt_bandit_dump_t out;
};

__constant__ double c_cov_grid[11] = {0.0, .1, .2, .3, .4, .5, .6, .7, .8, .9, 1.0};  // collect_data.py:30

template <int MODE>
struct Thr {
  using type = uint32_t;
};
template <>
struct Thr<MODE_INJECT> {
  using type = double;
};

// Per-env behaviour policy -> thresholds of the categorical draw (thread-local, runs once per env).
template <int MODE, int DMAX>
__device__ __forceinline__ void rollin_setup_env(const RollinParams& p, int env, int D, float* s_means,
                                                 typename Thr<MODE>::type* s_thr) {
  const uint64_t gid = p.env_id0 + (uint64_t)env;
  for (int j = 0; j < D; ++j) s_means[j] = p.means[(size_t)env * D + j];
  if (MODE == MODE_INJECT && p.in.actions != nullptr) return;  // action stream injected
  int cov_idx, ridx;
  double probs[DMAX];
  if (MODE == MODE_INJECT) {
    cov_idx = p.in.cov_idx[env];
    ridx = p.in.rand_idx[env];
#pragma unroll
    for (int j = 0; j < DMAX; ++j)
      if (j < D) probs[j] = p.in.dir_probs[(size_t)env * D + j];
  } else {
    const uint4 w = philox_words(p.key, gid, 0, STREAM_ROLLIN_SETUP);
    cov_idx = (int)bounded(w.x, 11);
    ridx = (int)bounded(w.y, (uint32_t)D);
    double sum = 0.0;
#pragma unroll
    for (int b = 0; b < (DMAX + 3) / 4; ++b) {
      if (4 * b < D) {
        const uint4 g = philox_words(p.key, gid, 1 + b, STREAM_ROLLIN_SETUP);
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const int j = 4 * b + i;
          if (j < DMAX && j < D) {  // Gamma(1) = -log U; Dirichlet(1_d) = normalised gammas
            probs[j] = (double)(-__logf(u32_open0(word_of(g, i))));
            sum += probs[j];
          }
        }
      }
    }
#pragma unroll
    for (int j = 0; j < DMAX; ++j)
      if (j < D) probs[j] = probs[j] / sum;
    if (MODE == MODE_PHILOX_DUMP) {
      if (p.out.cov_idx) p.out.cov_idx[env] = cov_idx;
      if (p.out.rand_idx) p.out.rand_idx[env] = ridx;
      if (p.out.dir_probs)
        for (int j = 0; j < D; ++j) p.out.dir_probs[(size_t)env * D + j] = probs[j];
    }
  }
  // probs = (1 - cov) * probs + cov * onehot(rand_index)   (collect_data.py:36), then
  // cdf = cumsum(probs); cdf /= cdf[-1]                    (numpy RandomState.choice)
  const double cov = c_cov_grid[cov_idx];
  const double omc = __dsub_rn(1.0, cov);
  double acc = 0.0;
#pragma unroll
  for (int j = 0; j < DMAX; ++j) {
    if (j < D) {
      const double pm = __dadd_rn(__dmul_rn(omc, probs[j]), __dmul_rn(cov, j == ridx ? 1.0 : 0.0));
      acc = (j == 0) ? pm : __dadd_rn(acc, pm);
      probs[j] = acc;
    }
  }
#pragma unroll
  for (int j = 0; j < DMAX - 1; ++j) {
    if (j < D - 1) {
      const double c = __ddiv_rn(probs[j], acc);
      if (MODE == MODE_INJECT) {
        s_thr[j] = c;
      } else {  // u = k * 2^-31 exactly, so  cdf_j <= u  <=>  ceil(cdf_j * 2^31) <= k
        s_thr[j] = (typename Thr<MODE>::type)ceil(c * 2147483648.0);
      }
    }
  }
}

// CTA-level reduction of the return statistics: warp shuffles, then one double atomic per CTA and
// statistic (the only cross-env operation of the whole path; shards on other GPUs add theirs via
// the NCCL gather on the host side).
__device__ __forceinline__ void reduce_stats(const RollinParams& p, float sr, float sr2, float nopt) {
  double* stats = p.stats;
  __shared__ float s_part[3][RB_WARPS];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    sr += __shfl_xor_sync(0xffffffffu, sr, o);
    sr2 += __shfl_xor_sync(0xffffffffu, sr2, o);
    nopt += __shfl_xor_sync(0xffffffffu, nopt, o);
  }
  if (lane == 0) s_part[0][warp] = sr, s_part[1][warp] = sr2, s_part[2][warp] = nopt;
  __syncthreads();
  if (threadIdx.x < 3) {
    double acc = 0.0;
    for (int w = 0; w < RB_WARPS; ++w) acc += (double)s_part[threadIdx.x][w];
    atomicAdd(stats + threadIdx.x, acc);   // fire-and-forget: the kernel boundary orders it before any reader
  }
}

// Multi-GPU form: a one-warp kernel behind the rollin launch stores the rank's three totals into slot `rank` of every
// rank's gather buffer over NVLink (plain system-visible stores through the CUDA-IPC mappings, one thread per (peer,
// statistic): all n_peers * 3 stores are in flight together; the kernel boundary makes them visible, readers order
// themselves with stream sync + barrier).  Round 1 did this inside the rollin kernel ("last CTA" pattern) with
// `st.global.release.sys` issued one after the other: every release store waited for the previous one to become
// visible system-wide, ~1.5 us per peer -- the whole 1 -> 8 GPU efficiency loss (launch 0.3105 ms with the statistics
// off, 0.3206 / 0.3241 / 0.3296 ms at 2 / 4 / 8 GPUs, linear in the number of peers; profiles/r02_scale_n8_*.json).
struct PeerPublish {
  double* dst[DPT_MAX_PEERS];
  int n;
};
__global__ void peer_publish_kernel(const double* __restrict__ stats, const PeerPublish pp) {
  const int r = threadIdx.x / 3, t = threadIdx.x - 3 * r;
  if (r < pp.n) asm volatile("st.global.relaxed.sys.f64 [%0], %1;" ::"l"(pp.dst[r] + t), "d"(stats[t]) : "memory");
}

// packed fp32 pair arithmetic (sm_100: FADD2 / FFMA2, one issue slot for two lanes of work)
__device__ __forceinline__ float2 add2(float2 a, float2 b) {
  float2 r;
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(reinterpret_cast<uint64_t&>(r)) : "l"(reinterpret_cast<uint64_t&>(a)), "l"(reinterpret_cast<uint64_t&>(b)));
  return r;
}
__device__ __forceinline__ float2 fma2(float2 a, float2 b, float2 c) {
  float2 r;
  asm("fma.rn.f32x2 %0, %1, %2, %3;"
      : "=l"(reinterpret_cast<uint64_t&>(r))
      : "l"(reinterpret_cast<uint64_t&>(a)), "l"(reinterpret_cast<uint64_t&>(b)), "l"(reinterpret_cast<uint64_t&>(c)));
  return r;
}

__device__ __forceinline__ int argmax_first(const float* m, int D) {
  int best = 0;
  for (int j = 1; j < D; ++j)
    if (m[j] > m[best]) best = j;
  return best;
}

// ---------------------------------------------------------------------------------------------
// Fast path: compile-time d (2d <= 32), H % 4 == 0, 16 B-aligned outputs.
// A warp task is one env x 128 steps; lane l owns the step quad 4l .. 4l + 3 (never partial: H % 4 == 0, only the last range
// of an env is ragged, predicated per quad).  Per lane and task: two Philox calls (step pairs 2l, 2l + 1 of the range: the
// same counters as the generic path), one float4 of rewards (512 B per warp store) and D float4 of one-hot rows from the
// quad's 4D-bit string (onehot_quad_store).
// ---------------------------------------------------------------------------------------------
// Resident CTAs per SM the fast kernel is compiled for: 5 up to d = 5 (48 registers; left to itself ptxas takes 50-64 and the SM
// holds 4 CTAs: 0.320 against 0.292 ms at 125k x 500, d = 5); d = 6 .. 10: 4 (<= 64 registers); d = 16: 2 (<= 128; at 3 the
// Philox instantiations spill).  No instantiation spills.
template <int D>
constexpr int rb_min_blocks() { return D <= 5 ? 5 : D <= 10 ? 4 : 2; }
template <int D, int MODE, int RT>   // RT: DPT_REWARD_* (compile-time: the kernel sits at the issue / HBM balance point)
__global__ void __launch_bounds__(RB_THREADS, rb_min_blocks<D>()) bandit_rollin_fast(const RollinParams p) {
  using thr_t = typename Thr<MODE>::type;
  using qbits_t = typename std::conditional<(4 * D > 32), uint64_t, uint32_t>::type;   // a quad's one-hot bit string
  __shared__ float4 s_nib[16];
  __shared__ float s_means[RB_MAX_ENVS][D];
  __shared__ thr_t s_thr[RB_MAX_ENVS][D];
  __shared__ qbits_t s_optmask[RB_MAX_ENVS];   // one-hot bits of the optimal arm in all four steps of a quad
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int env0 = blockIdx.x * p.envs_per_cta;
  const int ne = min(p.envs_per_cta, p.N - env0);
  const int H = p.H;

  if (warp == 0) {
    onehot_nib_init(s_nib, lane);
    if (lane < ne) {
      rollin_setup_env<MODE, D>(p, env0 + lane, D, s_means[lane], s_thr[lane]);
      const qbits_t o = (qbits_t)1 << argmax_first(s_means[lane], D);
      s_optmask[lane] = o | (o << D) | (o << (2 * D)) | (o << (3 * D));
    }
  } else {  // bandit state is the constant [1] (envs/bandit_env.py:38): dx = 1
    const size_t b = (size_t)env0 * H, e = (size_t)(env0 + ne) * H;
    fill_range(p.ctx_s, b, e, 1.0f, tid - 32, RB_THREADS - 32);
    fill_range(p.ctx_ns, b, e, 1.0f, tid - 32, RB_THREADS - 32);
  }
  __syncthreads();

  const int chunks = (H + 127) >> 7;
  const bool inj_actions = (MODE == MODE_INJECT) && p.in.actions != nullptr;
  float2 st_r = make_float2(0.f, 0.f), st_r2 = make_float2(0.f, 0.f);   // per pair component, packed f32x2 updates
  int st_opt = 0;
  // (env, range) of this warp's task: task index t = warp + i * RB_WARPS = e * chunks + c, advanced by the
  // constant (de, dc) = divmod(RB_WARPS, chunks) with one predicated carry -- no division, no data-dependent loop
  const int de = RB_WARPS / chunks, dc = RB_WARPS - de * chunks;
  int e = warp / chunks, c = warp - e * chunks;
  for (; e < ne; e += de, c += dc) {
    if (c >= chunks) {
      c -= chunks, ++e;
      if (e >= ne) break;
    }
    const int env = env0 + e;
    const int h0 = c * 128 + 4 * lane;
    const bool valid = h0 < H;
    const size_t row = (size_t)env * H + h0;
    int a[4] = {0, 0, 0, 0};
    float z[4] = {0.f, 0.f, 0.f, 0.f};
    if (MODE != MODE_INJECT) {
      const uint64_t gid = p.env_id0 + (uint64_t)env;
      const uint4 w0 = philox_words(p.rk, gid, (uint32_t)(h0 >> 1), STREAM_ROLLIN_STEP);
      const uint4 w1 = philox_words(p.rk, gid, (uint32_t)(h0 >> 1) + 1u, STREAM_ROLLIN_STEP);
      const uint32_t k[4] = {w0.x >> 1, w0.y >> 1, w1.x >> 1, w1.y >> 1};
      // a = #{j : k >= t_j}.  k < 2^31 and t_j <= 2^31, so k - t_j fits in 32 bits and its sign bit is (k < t_j): one
      // subtract and one shift-add per compare
#pragma unroll
      for (int j = 0; j < D - 1; ++j) {
        const uint32_t t = s_thr[e][j];
#pragma unroll
        for (int u = 0; u < 4; ++u) a[u] -= (int)((k[u] - t) >> 31);
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) a[u] += D - 1;
      if (RT == DPT_REWARD_GAUSSIAN) {
        box_muller(w0.z, w0.w, z[0], z[1]);
        box_muller(w1.z, w1.w, z[2], z[3]);
      } else {
        z[0] = u24(w0.z), z[1] = u24(w0.w), z[2] = u24(w1.z), z[3] = u24(w1.w);
      }
      if (MODE == MODE_PHILOX_DUMP && valid) {
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          if (p.out.u) p.out.u[row + u] = (double)k[u] * 4.656612873077392578125e-10;
          if (p.out.z) p.out.z[row + u] = z[u];
          if (p.out.actions) p.out.actions[row + u] = a[u];
        }
      }
    } else if (valid) {
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        if (inj_actions) {
          a[u] = p.in.actions[row + u];
        } else {  // searchsorted(cdf, u, side='right') = #{j : cdf_j <= u}
          const double uu = p.in.u[row + u];
#pragma unroll
          for (int j = 0; j < D - 1; ++j) a[u] += (s_thr[e][j] <= uu);
        }
        z[u] = p.in.z[row + u];
      }
    }
    // r = means[a] + var * z   (envs/bandit_env.py:59); else Bernoulli(mean): envs/bandit_env.py:61
    float r[4];
    qbits_t bq = 0;
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const float m = s_means[e][a[u]];
      r[u] = RT == DPT_REWARD_GAUSSIAN ? fmaf(p.var, z[u], m) : (z[u] < m ? 1.f : 0.f);
      bq |= ((qbits_t)1 << a[u]) << (u * D);
    }
    st_stream_if(valid, reinterpret_cast<float4*>(p.ctx_r + row), make_float4(r[0], r[1], r[2], r[3]));
    if (p.stats && valid) {
      const float2 r01 = make_float2(r[0], r[1]), r23 = make_float2(r[2], r[3]);
      st_r = add2(add2(st_r, r01), r23);
      st_r2 = fma2(r23, r23, fma2(r01, r01, st_r2));
      st_opt += 4 * D > 32 ? __popcll((uint64_t)(bq & s_optmask[e])) : __popc((uint32_t)(bq & s_optmask[e]));
    }
    const int nq = min(32, (H - c * 128) >> 2);
    onehot_quad_store<D>(reinterpret_cast<float4*>(p.ctx_a + ((size_t)env * H + (size_t)c * 128) * D), bq, lane, nq * D, s_nib,
                         [](int) {});
  }
  if (p.stats) reduce_stats(p, st_r.x + st_r.y, st_r2.x + st_r2.y, (float)st_opt);
}

// ---------------------------------------------------------------------------------------------
// Generic path: runtime d <= 32, any H, any alignment.  One lane per step; the SAME Philox
// counters as the fast path (pair index = h / 2, component by parity), so both paths draw
// identical noise.  All stores are coalesced 4 B scalars.
// ---------------------------------------------------------------------------------------------
template <int MODE>
__global__ void __launch_bounds__(RB_THREADS) bandit_rollin_generic(const RollinParams p) {
  using thr_t = typename Thr<MODE>::type;
  __shared__ float s_means[RB_MAX_ENVS][RB_MAX_D];
  __shared__ thr_t s_thr[RB_MAX_ENVS][RB_MAX_D];
  __shared__ int s_opt[RB_MAX_ENVS];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int env0 = blockIdx.x * p.envs_per_cta;
  const int ne = min(p.envs_per_cta, p.N - env0);
  const int H = p.H, D = p.d;

  if (tid < ne) {
    rollin_setup_env<MODE, RB_MAX_D>(p, env0 + tid, D, s_means[tid], s_thr[tid]);
    s_opt[tid] = argmax_first(s_means[tid], D);
  }
  if (!p.acts_u8) {
    for (size_t i = (size_t)env0 * H + tid; i < (size_t)(env0 + ne) * H; i += RB_THREADS) {
      st_stream(p.ctx_s + i, 1.0f);
      st_stream(p.ctx_ns + i, 1.0f);
    }
  }
  __syncthreads();

  const int chunks = (H + 31) >> 5;
  const bool inj_actions = (MODE == MODE_INJECT) && p.in.actions != nullptr;
  float st_r = 0.f, st_r2 = 0.f, st_opt = 0.f;
  for (int task = warp; task < ne * chunks; task += RB_WARPS) {
    const int e = task / chunks, c = task - e * chunks;
    const int env = env0 + e;
    const int h = c * 32 + lane;
    const size_t row = (size_t)env * H + h;
    int a = 0;
    float z = 0.f;
    if (MODE != MODE_INJECT) {
      const uint4 w = philox_words(p.key, p.env_id0 + (uint64_t)env, (uint32_t)(h >> 1), STREAM_ROLLIN_STEP);
      const uint32_t k = ((h & 1) ? w.y : w.x) >> 1;
      for (int j = 0; j < D - 1; ++j) a += (k >= s_thr[e][j]);
      if (p.rtype == DPT_REWARD_GAUSSIAN) {
        float z0, z1;
        box_muller(w.z, w.w, z0, z1);
        z = (h & 1) ? z1 : z0;
      } else {
        z = u24((h & 1) ? w.w : w.z);
      }
      if (MODE == MODE_PHILOX_DUMP && h < H) {
        if (p.out.u) p.out.u[row] = (double)k * 4.656612873077392578125e-10;
        if (p.out.z) p.out.z[row] = z;
        if (p.out.actions) p.out.actions[row] = a;
      }
    } else if (h < H) {
      if (inj_actions) {
        a = p.in.actions[row];
      } else {
        const double u = p.in.u[row];
        for (int j = 0; j < D - 1; ++j) a += (s_thr[e][j] <= u);
      }
      z = p.in.z[row];
    }
    if (h < H) {
      const float ma = s_means[e][a];
      const float r = p.rtype == DPT_REWARD_GAUSSIAN ? fmaf(p.var, z, ma) : (z < ma ? 1.f : 0.f);
      st_stream(p.ctx_r + row, r);
      if (p.stats) st_r += r, st_r2 = fmaf(r, r, st_r2), st_opt += (float)(a == s_opt[e]);
    }
    if (p.acts_u8) {   // compact: 1 B per step, expanded on the host
      if (h < H) p.acts_u8[row] = (uint8_t)a;
      continue;
    }
    const int nvalid = min(32, H - c * 32) * D;
    float* abase = p.ctx_a + ((size_t)env * H + (size_t)c * 32) * D;
    for (int it = 0; it < D; ++it) {
      const int i = it * 32 + lane;
      const int s = i / D;
      const int as = __shfl_sync(0xffffffffu, a, s & 31);
      if (i < nvalid) st_stream(abase + i, (i - s * D) == as ? 1.f : 0.f);
    }
  }
  if (p.stats) reduce_stats(p, st_r, st_r2, st_opt);
}

// resident CTAs per SM of a kernel (occupancy API), cached per kernel POINTER: every instantiation has the same
// function type, so a function-local static inside a generic lambda would be shared by all of them
template <typename K>
static int resident_ctas(K kern) {
  static thread_local std::unordered_map<const void*, int> cache;
  const void* key = reinterpret_cast<const void*>(kern);
  auto it = cache.find(key);
  if (it != cache.end()) return it->second;
  int n = 0;
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, kern, RB_THREADS, 0) != cudaSuccess || n < 1) n = 4;
  cache[key] = n;
  return n;
}

template <int MODE>
static void launch_mode(RollinParams p, bool fast, cudaStream_t st) {
  // envs per CTA: up to 32, few enough that the grid covers the machine >= 3 times, and chosen so that the
  // last wave is nearly full (the kernel's real occupancy decides what a wave is)
  auto go = [&](auto kern, int step, int min_e) {
    const int slots = sm_count() * resident_ctas(kern);
    p.envs_per_cta = pick_envs_per_cta(p.N, slots, min_e, RB_MAX_ENVS, step);
    if (min_e > 1 && (p.N + p.envs_per_cta - 1) / p.envs_per_cta < 3 * slots)   // small N: spread the envs over the machine
      p.envs_per_cta = pick_envs_per_cta(p.N, slots, 1, RB_MAX_ENVS);
    const int grid = (p.N + p.envs_per_cta - 1) / p.envs_per_cta;
    kern<<<grid, RB_THREADS, 0, st>>>(p);
  };
  if (fast) {
    // envs per CTA a multiple of `step`: the CTA's (env, 128-step range) tasks then split evenly over its warps (125k x 500:
    // 0.307 -> 0.292 ms); and at least 4 tasks per warp, or the per-CTA setup is paid for too little work (100k x 200, d = 10:
    // the fullest last wave alone picks 4 envs per CTA, one task per warp, 0.242 ms against 0.173 for the 64-step kernel)
    const int chunks = (p.H + 127) >> 7;
    int step = 1;
    while ((step * chunks) % RB_WARPS) ++step;
    const int min_e = (4 * RB_WARPS / chunks + step - 1) / step * step;
    switch (p.d) {
#define DPT_CASE(DD)                                                   \
  case DD:                                                             \
    if (p.rtype == DPT_REWARD_GAUSSIAN)                                \
      go(bandit_rollin_fast<DD, MODE, DPT_REWARD_GAUSSIAN>, step, min_e);  \
    else                                                               \
      go(bandit_rollin_fast<DD, MODE, DPT_REWARD_BERNOULLI>, step, min_e); \
    return;
      DPT_CASE(2)
      DPT_CASE(3)
      DPT_CASE(4)
      DPT_CASE(5)
      DPT_CASE(6)
      DPT_CASE(8)
      DPT_CASE(10)
      DPT_CASE(16)
#undef DPT_CASE
      default:
        break;
    }
  }
  go(bandit_rollin_generic<MODE>, 1, 1);
}

}  // namespace dpt

using namespace dpt;

static int bandit_rollin_impl(const float* means, float var, int reward_type, uint64_t seed, uint64_t env_id0, int N, int H, int d,
                              float* ctx_states, float* ctx_actions, float* ctx_next_states, float* ctx_rewards,
                              double* return_stats, const dpt_bandit_inject_t* inject, const dpt_bandit_dump_t* dump,
                              double* const* peer_dst, int n_peers, unsigned int* done_counter, void* stream,
                              uint8_t* acts_u8 = nullptr) {
  DPT_CHECK_ARG(N >= 0 && H >= 0, "dpt_bandit_rollin: N=%d H=%d must be >= 0", N, H);
  DPT_CHECK_ARG(reward_type == DPT_REWARD_GAUSSIAN || reward_type == DPT_REWARD_BERNOULLI,
                "dpt_bandit_rollin: unknown reward_type %d (0 uniform/gaussian, 1 bernoulli)", reward_type);
  DPT_CHECK_ARG(d >= 1 && d <= RB_MAX_D, "dpt_bandit_rollin: d=%d outside [1,%d]", d, RB_MAX_D);
  if (N == 0 || H == 0) return DPT_OK;
  DPT_CHECK_ARG(means && ctx_rewards && (acts_u8 || (ctx_states && ctx_actions && ctx_next_states)),
                "dpt_bandit_rollin: null means/context pointer");
  RollinParams p{};
  p.acts_u8 = acts_u8;
  p.means = means;
  p.var = var;
  p.rtype = reward_type;
  p.key = Key{(uint32_t)seed, (uint32_t)(seed >> 32)};
  p.rk = round_keys(p.key);
  p.env_id0 = env_id0;
  p.N = N, p.H = H, p.d = d;
  p.ctx_s = ctx_states, p.ctx_a = ctx_actions, p.ctx_ns = ctx_next_states, p.ctx_r = ctx_rewards;
  p.stats = return_stats;
  if (n_peers > 0)
    DPT_CHECK_ARG(n_peers <= DPT_MAX_PEERS && peer_dst && return_stats,
                  "dpt_bandit_rollin_p2p: needs return_stats and 1..%d peer pointers", DPT_MAX_PEERS);
  int mode = MODE_PHILOX;
  if (inject) {
    DPT_CHECK_ARG(!dump, "dpt_bandit_rollin: inject and dump are mutually exclusive");
    DPT_CHECK_ARG(inject->z, "dpt_bandit_rollin: inject->z is required");
    DPT_CHECK_ARG(inject->actions || (inject->cov_idx && inject->dir_probs && inject->rand_idx && inject->u),
                  "dpt_bandit_rollin: inject needs actions or (cov_idx, dir_probs, rand_idx, u)");
    p.in = *inject;
    mode = MODE_INJECT;
  } else if (dump) {
    p.out = *dump;
    mode = MODE_PHILOX_DUMP;
  }
  const bool fast = !acts_u8 && (H % 4 == 0) && 2 * d <= 32 && aligned16(ctx_states) && aligned16(ctx_actions) &&
                    aligned16(ctx_next_states) && aligned16(ctx_rewards);
  cudaStream_t st = (cudaStream_t)stream;
  if (mode == MODE_PHILOX)
    launch_mode<MODE_PHILOX>(p, fast, st);
  else if (mode == MODE_PHILOX_DUMP)
    launch_mode<MODE_PHILOX_DUMP>(p, fast, st);
  else
    launch_mode<MODE_INJECT>(p, fast, st);
  DPT_LAUNCH_CHECK();
  if (n_peers > 0) {
    PeerPublish pp{};
    for (int r = 0; r < n_peers; ++r) pp.dst[r] = peer_dst[r];
    pp.n = n_peers;
    peer_publish_kernel<<<1, 3 * DPT_MAX_PEERS <= 32 ? 32 : 3 * DPT_MAX_PEERS, 0, st>>>(return_stats, pp);
    DPT_LAUNCH_CHECK();
  }
  (void)done_counter;   // kept in the ABI (round 1's in-kernel protocol used it); unused
  return DPT_OK;
}

extern "C" int dpt_bandit_rollin(const float* means, float var, int reward_type, uint64_t seed, uint64_t env_id0, int N, int H, int d,
                                 float* ctx_states, float* ctx_actions, float* ctx_next_states, float* ctx_rewards,
                                 double* return_stats, const dpt_bandit_inject_t* inject,
                                 const dpt_bandit_dump_t* dump, void* stream) {
  return bandit_rollin_impl(means, var, reward_type, seed, env_id0, N, H, d, ctx_states, ctx_actions, ctx_next_states,
                            ctx_rewards, return_stats, inject, dump, nullptr, 0, nullptr, stream);
}

// compact form for the host pipeline (host_paths.cu): same draws, outputs = arm index (1 B) + reward (4 B) per step
namespace dpt {
int bandit_rollin_compact(const float* means, float var, uint64_t seed, uint64_t env_id0, int N, int H, int d, uint8_t* acts_u8,
                          float* ctx_rewards, void* stream) {
  return bandit_rollin_impl(means, var, DPT_REWARD_GAUSSIAN, seed, env_id0, N, H, d, nullptr, nullptr, nullptr, ctx_rewards,
                            nullptr, nullptr, nullptr, nullptr, 0, nullptr, stream, acts_u8);
}
}  // namespace dpt

extern "C" int dpt_bandit_rollin_p2p(const float* means, float var, uint64_t seed, uint64_t env_id0, int N, int H, int d,
                                     float* ctx_states, float* ctx_actions, float* ctx_next_states, float* ctx_rewards,
                                     double* return_stats, double* const* peer_dst, int n_peers,
                                     unsigned int* done_counter, void* stream) {
  DPT_CHECK_ARG(N > 0 && H > 0, "dpt_bandit_rollin_p2p: empty shard (N=%d, H=%d) cannot signal its peers", N, H);
  return bandit_rollin_impl(means, var, DPT_REWARD_GAUSSIAN, seed, env_id0, N, H, d, ctx_states, ctx_actions,
                            ctx_next_states, ctx_rewards, return_stats, nullptr, nullptr, peer_dst, n_peers, done_counter,
                            stream);
}

// ---- peer-memory plumbing: buffers that other ranks' kernels can store into over NVLink ----
extern "C" int dpt_peer_buffer_create(uint64_t bytes, void** dev_ptr, unsigned char handle[64]) {
  DPT_CHECK_ARG(bytes > 0 && dev_ptr && handle, "dpt_peer_buffer_create: bad arguments");
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "cudaIpcMemHandle_t is 64 bytes");
  void* ptr = nullptr;
  DPT_CUDA(cudaMalloc(&ptr, bytes));
  DPT_CUDA(cudaMemset(ptr, 0, bytes));
  cudaIpcMemHandle_t h;
  DPT_CUDA(cudaIpcGetMemHandle(&h, ptr));
  memcpy(handle, &h, 64);
  *dev_ptr = ptr;
  return DPT_OK;
}
extern "C" int dpt_peer_buffer_open(const unsigned char handle[64], void** dev_ptr) {
  DPT_CHECK_ARG(handle && dev_ptr, "dpt_peer_buffer_open: bad arguments");
  cudaIpcMemHandle_t h;
  memcpy(&h, handle, 64);
  DPT_CUDA(cudaIpcOpenMemHandle(dev_ptr, h, cudaIpcMemLazyEnablePeerAccess));
  return DPT_OK;
}
extern "C" int dpt_peer_buffer_close(void* dev_ptr) {
  if (dev_ptr) DPT_CUDA(cudaIpcCloseMemHandle(dev_ptr));
  return DPT_OK;
}
extern "C" int dpt_peer_buffer_destroy(void* dev_ptr) {
  if (dev_ptr) DPT_CUDA(cudaFree(dev_ptr));
  return DPT_OK;
}
extern "C" int dpt_peer_buffer_zero(void* dev_ptr, uint64_t bytes, void* stream) {
  DPT_CHECK_ARG(dev_ptr, "dpt_peer_buffer_zero: null pointer");
  DPT_CUDA(cudaMemsetAsync(dev_ptr, 0, bytes, (cudaStream_t)stream));
  return DPT_OK;
}
extern "C" int dpt_peer_buffer_read(const void* dev_ptr, void* host_dst, uint64_t bytes, void* stream) {
  DPT_CHECK_ARG(dev_ptr && host_dst, "dpt_peer_buffer_read: null pointer");
  DPT_CUDA(cudaMemcpyAsync(host_dst, dev_ptr, bytes, cudaMemcpyDeviceToHost, (cudaStream_t)stream));
  DPT_CUDA(cudaStreamSynchronize((cudaStream_t)stream));
  return DPT_OK;
}
