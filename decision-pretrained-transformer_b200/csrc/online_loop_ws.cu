// Fast fused online evaluation loop for the classical bandit controllers (d <= 10).
//
// Same contract as online_loop.cu's general kernel (reference evals/eval_bandit.py:56-103 + envs/bandit_env.py:56-64,
// :98-149 + ctrls/ctrl_bandit.py act_numpy_vec / set_batch_numpy_vec), re-cut around what ncu showed of that kernel
// (39-52 % issue utilisation, 21 warps per SM at 100k envs, 145-540 instructions per warp-step of which the
// controller proper is a minority).  One warp owns 32 envs (lane = env) for all H steps:
//   per step   pick arm -> reward -> O(1) statistics update -> stage the arm (as a byte and as a bit of the step quad's
//       one-hot bit string) and the reward in shared memory, store cum_means[h, env] (coalesced across the warp).
//       The per-arm (sum, count) live in shared memory (only the pulled arm is touched), the cached decision
//       statistics in registers: 80 registers per thread, 24 warps resident per SM, so that 100k envs
//       (21.1 warps per SM) are ONE wave.  Everything that depends on a count only (1/n, the UCB bonus, Thompson's
//       1/(var + n prior_var) and posterior std) comes from a [2][H+1] float64 table, so a step has no float64
//       division or square root.  float64 like the reference: the arm is the reference's arm.
//       Reward noise: one Philox block + two Box-Muller pairs per step quad, off the controller's dependency chain.
//   per tile (WT steps)   the warp drains its own staging tile: rewards and one-hot rows leave as contiguous 16 B stores --
//       a float4 of an env's one-hot run is one nibble of the quad's bit string, i.e. one shared load + one 16-entry
//       table lookup -- in batches of four independent load / lookup / store chains.
//   The per-step regret sums [H,4] are NOT accumulated here: regret_pass_kernel (below) streams cum_means [H,N]
//   once afterwards.
// This single fused kernel is what Thompson / LinUCB use at large batches; Opt / EmpMean / UCB and small batches run the split
// pipeline in the second half of this file (controller kernel + context-expansion kernel), see launch_online_ws / dpt_online_loop.
// Measured dead end kept in DESIGN.md: the warp-specialised form of this kernel (3 controller warps + 1 flush / noise
// warp per CTA, tiles handed over through mbarriers) -- the single helper warp runs ~50-230 dependent instructions
// per step for its three controllers and becomes the bottleneck (controllers stalled 12 % of their time on the
// "tile drained" barrier); letting every warp drain its own tile has no hand-over and the same instruction count.
// HBM traffic per env-step: 4 (2 + d + 1) B of context rows + 4 B of cum_means (36 B at d = 5).
#include <stdlib.h>

#include "online_loop.cuh"

namespace dpt {

// steps per staging tile (multiple of 4): 32 at d <= 5, 16 at d <= 10 (shared memory per warp: 32 warps must stay resident)
template <int DMAX>
constexpr int ws_wt() { return DMAX <= 5 ? 32 : 16; }
constexpr int WS_NCONS = 4; // warps per CTA

template <int DMAX>
struct alignas(16) WsTile {
  static constexpr int WT = ws_wt<DMAX>(), WQ = WT / 4;   // steps / float4 slots per env and tile
  static constexpr int BWQ = (4 * DMAX + 31) / 32;   // words of one-hot bits per step quad (4 DMAX bits)
  static constexpr int BROW = (WQ * BWQ) | 1;        // odd row lengths: lane = env accesses are bank-conflict free
  float4 rew[32][WQ];        // rewards; float4 slot q of env e lives in column q ^ swz(e) (conflict-free 16 B accesses)
  uint32_t acts[32][WQ | 1]; // pulled arm per step, one byte each
  uint32_t bits[32][BROW];   // one-hot rows of each step quad as a bit string (DMAX bits per step): nibble f of quad q is
                             // float4 q DMAX + f of the env's run of T d floats
};

struct WsNoTile {};

// SPLIT: the controller kernel of the split pipeline (below) stages nothing -- it emits the pulled arms as one coalesced
// 4-byte word per env and step quad and leaves the context rows to online_expand_kernel
template <int DMAX, bool STATS, bool SPLIT>
struct alignas(16) WsCons {
  std::conditional_t<SPLIT, WsNoTile, WsTile<DMAX>> tile;
  float means[32][DMAX];
  double sum[STATS ? DMAX : 1][32];   // reward sum per arm   (only the pulled arm is touched in a step)
  int cnt[STATS ? DMAX : 1][32];      // pull count per arm
};

// a quarter warp (8 envs) x one float4 slot must hit 8 distinct 16 B bank groups: rows are WQ groups long
template <int WQ>
__device__ __forceinline__ int swz_t(int e) { return WQ >= 8 ? (e & 7) : ((e / (8 / (WQ >= 8 ? 8 : WQ))) & (WQ - 1)); }

// a / n for a count n >= 1 with rc = RN(1 / n) from the table: two FMA corrections give the correctly rounded
// quotient (Markstein), i.e. the reference's b / max(1, counts) bit for bit -- checked by dpt_selftest_div
__device__ __forceinline__ double div_by_count(double a, int n, double rc) {
  const double nd = (double)n;
  double q = a * rc;
  q = fma(fma(-nd, q, a), rc, q);
  q = fma(fma(-nd, q, a), rc, q);
  return q;
}

// LinUCB (lin_d = 2): per-arm row of constants in shared memory -- x0, x1, x0^2, 2 x0 x1, x1^2, pad
constexpr int LIN_AW = 6;
__device__ __forceinline__ void lin_arm_row(double* row, double x0, double x1) {
  row[0] = x0, row[1] = x1, row[2] = x0 * x0, row[3] = 2.0 * (x0 * x1), row[4] = x1 * x1, row[5] = 0.0;
}

// sqrt of a positive, normal float64 to ~1 ulp without the IEEE routine's special-case branches: hardware reciprocal square
// root seed (20 bits) + two coupled Newton steps (Goldschmidt); 0 -> 0
__device__ __forceinline__ double sqrt_nr(double q) {
  double y;
  asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(q));
  double g = q * y, h = 0.5 * y;
  double r = fma(-h, g, 0.5);
  g = fma(g, r, g), h = fma(h, r, h);
  r = fma(-h, g, 0.5);
  g = fma(g, r, g);
  return q > 0.0 ? g : 0.0;
}

__device__ __forceinline__ void lin_arm_load(uint32_t sa, double* A) {   // the row's first five entries
  asm("ld.shared.v2.f64 {%0, %1}, [%2];" : "=d"(A[0]), "=d"(A[1]) : "r"(sa));
  asm("ld.shared.v2.f64 {%0, %1}, [%2+16];" : "=d"(A[2]), "=d"(A[3]) : "r"(sa));
  asm("ld.shared.f64 %0, [%1+32];" : "=d"(A[4]) : "r"(sa));
}

// First-maximum argmax (np.argmax) of v[LO..HI) as a balanced tournament: the right half wins only when strictly greater, so ties
// go to the lower index exactly as in the sequential scan, but the dependent compare / select chain is log2(n) deep instead of n
// (the controller kernels run 5 warps per scheduler; a step's latency chain matters as much as its instruction count)
template <int LO, int HI>
__device__ __forceinline__ void argmax_tree(const double* v, double& best, int& idx) {
  if constexpr (HI - LO == 1) {
    best = v[LO], idx = LO;
  } else {
    constexpr int MID = LO + (HI - LO + 1) / 2;
    double bl, br;
    int il, ir;
    argmax_tree<LO, MID>(v, bl, il);
    argmax_tree<MID, HI>(v, br, ir);
    const bool right = br > bl;
    best = right ? br : bl, idx = right ? ir : il;
  }
}

// the env step's reward in float64, as the reference forms it; shared by the controller (statistics) and the expander (context rows)
__device__ __forceinline__ double reward_f64(float ma, float z, double var, int rtype) {
  return rtype == DPT_REWARD_GAUSSIAN ? (double)ma + (0.0 + var * (double)z)   // envs/bandit_env.py:59
                                      : (z < ma ? 1.0 : 0.0);                  // :61 Bernoulli(mean)
}

// what the controller kernel of the split pipeline needs besides OnlineParams
struct SplitArgs {
  uint32_t* arms4;       // [ceil(H/4)][N]: byte u of word (q, env) = arm pulled at step 4 q + u; NULL = context not materialised
  double* creg;          // [ceil(H/128) + 1][N]: cumulative regret of the env before step 128 k (float64), last row: max(means);
                         // NULL = the expander does not accumulate the regret sums
  bool fill;             // the controller warps also write the constant state columns (H % 4 == 0, 16 B-aligned arrays)
};

// per-lane state of the split controller besides the controller's own (quad() takes it by reference)
struct SplitLane {
  uint32_t* arms4;     // this env's word of the current step quad
  double* creg_out;    // this env's carry slot of the current 128-step range
  double sum_ma, mmax; // sum of the pulled arms' means so far; max(means)
  float4* fill_p;      // next float4 of the constant-column fill (context_states; context_next_states = + fill_off bytes)
  ptrdiff_t fill_off;
  int fill_n;          // step quads in which this lane still has a float4 to write
};

template <int DMAX, int KIND, bool IO, bool SPLIT = false>
struct WsKernel {
  static constexpr bool STATS = (KIND == K_EMP || KIND == K_UCB || KIND == K_THOMPSON);
  using Cons = WsCons<DMAX, STATS, SPLIT>;
  using Tile = WsTile<DMAX>;
  static constexpr int BWQ = Tile::BWQ, WT = Tile::WT, WQ = Tile::WQ;
  static __device__ __forceinline__ int swz(int e) { return swz_t<WQ>(e); }
  // Thompson's control normals are drawn for ZSPAN steps at a time: a whole step quad at d <= 5 (20 normals = exactly 5 Philox
  // blocks; per step pair it was 3 blocks for 10 normals, one sixth of the words unused), a step pair at d <= 10 (5 blocks, 40
  // live floats per quad would not fit the registers).  Block index on STREAM_CTRL: (step / ZSPAN) * NBZ + block.
  static constexpr int ZSPAN = DMAX <= 5 ? 4 : 2;
  static constexpr int NBZ = (ZSPAN * DMAX + 3) / 4;

  // ------------------------------------------------------------------------------- drain one staging tile
  static __device__ __forceinline__ void flush(const OnlineParams& p, const Tile& tl, const float4* s_nib, int env0, int nl, int h0, int T,
                                               bool bits_ok, bool vec_r, int lane) {
    const int H = p.H, d = p.d;
    // rewards: T * 4 B per env and tile
    if (vec_r) {
#pragma unroll
      for (int it = 0; it < WQ; ++it) {
        const int e = it * (32 / WQ) + lane / WQ, q = lane % WQ;
        if (e < nl && 4 * q < T)
          st_stream(reinterpret_cast<float4*>(p.ctx_r + (size_t)(env0 + e) * H + h0) + q, tl.rew[e][q ^ swz(e)]);
      }
    } else {
      for (int i = lane; i < nl * WT; i += 32) {
        const int e = i / WT, t = i % WT;
        if (t < T) {
          const float4 r4 = tl.rew[e][(t >> 2) ^ swz(e)];
          const int u = t & 3;
          st_stream(p.ctx_r + (size_t)(env0 + e) * H + h0 + t, u == 0 ? r4.x : u == 1 ? r4.y : u == 2 ? r4.z : r4.w);
        }
      }
    }
    // one-hot rows
    if (bits_ok) {   // d == DMAX and T % 4 == 0: float4 g of an env's run of T*d floats is nibble g % DMAX of step quad g / DMAX
      // lane = (env of a group of 4, 8 consecutive float4): every store covers whole 128 B lines of 4 envs
      const int nbn = (T >> 2) * DMAX;                 // float4 per env in this tile
      const int gl = lane & 7;
      const size_t estride = ((size_t)H * DMAX) >> 2;
      float4* dst0 = reinterpret_cast<float4*>(p.ctx_a + ((size_t)env0 * H + h0) * DMAX) + gl;
      constexpr int NK = (WQ * DMAX + 7) / 8;          // iterations over g = 8 k + gl
#pragma unroll 2
      for (int e = lane >> 3; e < nl; e += 4) {
        const uint32_t* brow = tl.bits[e];
        float4* dst = dst0 + (size_t)e * estride;
        uint32_t nib[NK];
#pragma unroll
        for (int k = 0; k < NK; ++k) {
          const int g = min(8 * k + gl, WQ * DMAX - 1);
          const int q = g / DMAX, f = g - q * DMAX;
          nib[k] = (brow[q * BWQ + (f >> 3)] >> (4 * (f & 7))) & 15u;
        }
#pragma unroll
        for (int k = 0; k < NK; ++k) st_stream_if(8 * k + gl < nbn, dst + 8 * k, s_nib[nib[k]]);
      }
    } else {
      const int per = T * d;
      for (int e = 0; e < nl; ++e)
        for (int el = lane; el < per; el += 32) {
          const int t = (d == 1) ? el : (int)__umulhi((uint32_t)el, p.magic_d);
          const int a = (tl.acts[e][t >> 2] >> (8 * (t & 3))) & 255;
          st_stream(p.ctx_a + ((size_t)(env0 + e) * H + h0) * d + el, (a == el - t * d) ? 1.f : 0.f);
        }
    }
  }

  // ------------------------------------------------------------------------------- controller warp
  struct State {
    double st0[STATS ? DMAX : 1];              // EMP: mean; UCB: mean + bonus; THOMPSON: posterior mean
    double st1[KIND == K_THOMPSON ? DMAX : 1]; // THOMPSON: posterior std
    double s00, s01, s11, b0, b1;              // LinUCB (lin_d = 2): Sigma = I + sum x x^T, b = sum x r
    uint32_t untried;
  };

  // one step quad (4 steps; FULL: all four exist).  Returns nothing; stages rewards / arms / one-hot bits of the quad.
  template <bool FULL>
  static __device__ __forceinline__ void quad(const OnlineParams& p, Cons& cs, State& S, const double* s_arms,
                                              const double* __restrict__ tab0, const double* __restrict__ tab1, int h, int nsteps, int q,
                                              int opt, int env, bool live, uint64_t gid, float*& cmp, double sigma2tc0, bool stage, int lane,
                                              SplitLane& sl) {
    const int N = p.N, H = p.H, d = p.d;
    // reward noise of the quad: one Philox block + two Box-Muller pairs, off the controller's dependency chain
    float zz[4];
    if (IO && p.in.reward_z) {
#pragma unroll
      for (int t = 0; t < 4; ++t) zz[t] = (live && h + t < H) ? p.in.reward_z[(size_t)(h + t) * N + env] : 0.f;
    } else {
      reward_noise4(p.key, gid, (uint32_t)(h >> 2), p.rtype, zz);   // h is a multiple of 4 (tiles and quads are)
    }
    if (IO && p.out.reward_z && live) {
#pragma unroll
      for (int t = 0; t < 4; ++t)
        if (h + t < H) p.out.reward_z[(size_t)(h + t) * N + env] = zz[t];
    }
    float rr[4] = {0.f, 0.f, 0.f, 0.f};
    uint32_t aw = 0u;
    uint64_t bq = 0ull;
    if (sl.creg_out && (h & 127) == 0) {   // regret carry (expander / regret pass): cumulative regret before every 128th step
      if (live) *sl.creg_out = fma((double)h, sl.mmax, -sl.sum_ma);   // = sum over h' < h of (max(means) - means[arm_h'])
      sl.creg_out += N;
    }
    if (SPLIT && FULL && sl.fill_n > 0) {
      // constant states (bandit dx = 1, envs/bandit_env.py:38): the warp's 32 envs are one contiguous run of 32 H floats per array,
      // written 128 floats per step quad and array -- HBM-only work spread over the controller's (latency-bound) lifetime
      const float4 one4 = make_float4(1.f, 1.f, 1.f, 1.f);
      if (q < sl.fill_n) {
        st_stream(sl.fill_p, one4);
        st_stream(reinterpret_cast<float4*>(reinterpret_cast<char*>(sl.fill_p) + sl.fill_off), one4);
      }
      sl.fill_p += 32;
    }
    float zc[KIND == K_THOMPSON ? ZSPAN * DMAX : 1];              // control normals of the current ZSPAN steps
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      if (!FULL && u >= nsteps) break;
      const int hh = h + u;
      // ------------------------------------------------ controller: pick an arm ------------
      int a = 0;
      if (KIND == K_OPT) {
        a = opt;                                                        // ctrl_bandit.py:35-37
      } else if (KIND == K_EMP || KIND == K_UCB) {
        double best;               // padding arms j >= d carry -inf and are never picked
        argmax_tree<0, DMAX>(S.st0, best, a);                           // np.argmax: first maximum  :106 | :369-370
        if ((KIND == K_UCB || p.p0 != 0.0) && S.untried) a = __ffs(S.untried) - 1;   // np.argmin(counts) when min == 0  :110-113 | :373-375
      } else if (KIND == K_THOMPSON) {
        if ((u % ZSPAN) == 0) {           // control normals of steps hh .. hh + ZSPAN - 1: NBZ Philox blocks
          if (IO && p.in.ctrl_z) {
#pragma unroll
            for (int s2 = 0; s2 < ZSPAN; ++s2)
#pragma unroll
              for (int j = 0; j < DMAX; ++j)
                zc[s2 * DMAX + j] = (live && j < d && hh + s2 < H) ? p.in.ctrl_z[((size_t)(hh + s2) * N + env) * d + j] : 0.f;
          } else {
#pragma unroll
            for (int bk = 0; bk < NBZ; ++bk) {
              float z4n[4];
              normals4(philox_words(p.key, gid, (uint32_t)((hh / ZSPAN) * NBZ + bk), STREAM_CTRL), z4n);
#pragma unroll
              for (int k = 0; k < 4; ++k)
                if (4 * bk + k < ZSPAN * DMAX) zc[4 * bk + k] = z4n[k];
            }
          }
        }
        if constexpr (DMAX <= 5) {
          double vs[DMAX], best;
#pragma unroll
          for (int j = 0; j < DMAX; ++j) {
            const float zj = zc[(u % ZSPAN) * DMAX + j];
            if (IO && p.out.ctrl_z && live && j < d) p.out.ctrl_z[((size_t)hh * N + env) * d + j] = zj;
            vs[j] = fma(S.st1[j], (double)zj, S.st0[j]);                // np.random.normal(means, sqrt(variances)) :234
          }                                                             // (padding arms: mean -inf, std 0)
          argmax_tree<0, DMAX>(vs, best, a);
        } else {   // d = 10: 10 live samples do not fit beside the 40 cached statistics (tournament: 0.50 -> 0.70 ms, spills)
          double best = -INFINITY;
#pragma unroll
          for (int j = 0; j < DMAX; ++j) {
            const float zj = zc[(u % ZSPAN) * DMAX + j];
            if (IO && p.out.ctrl_z && live && j < d) p.out.ctrl_z[((size_t)hh * N + env) * d + j] = zj;
            const double v = fma(S.st1[j], (double)zj, S.st0[j]);
            if (v > best) best = v, a = j;
          }
        }
      } else if (KIND == K_LINUCB2) {
        if (hh == 0) {                                                  // :496-500 uniform random first arm
          if (IO && p.in.first_arm)
            a = live ? p.in.first_arm[env] : 0;
          else
            a = (int)bounded(philox_words(p.key, gid, 0u, STREAM_CTRL).x, (uint32_t)d);
          if (IO && p.out.first_arm && live) p.out.first_arm[env] = a;
        } else {   // lin_d == 2: closed-form inverse, everything in registers
          const double idet = 1.0 / (S.s00 * S.s11 - S.s01 * S.s01);
          const double i00 = S.s11 * idet, i01 = -S.s01 * idet, i11 = S.s00 * idet;
          const double t0 = i00 * S.b0 + i01 * S.b1, t1 = i01 * S.b0 + i11 * S.b1;   // theta = cov_inv @ A^T r  :513
          // per arm (s_arms row: x0, x1, x0^2, 2 x0 x1, x1^2): arm @ cov_inv @ arm = i00 x0^2 + i01 (2 x0 x1) + i11 x1^2 -- 3 float64
          // operations on the arm's constant products instead of 6 on (x0, x1); like the reference's LAPACK inverse / BLAS
          // products this is float64-accurate, not bit-identical, arithmetic: the argmax is what is pinned (goldens)
          double best = -INFINITY;
          const uint32_t arms_sa = (uint32_t)__cvta_generic_to_shared(s_arms);   // (one conversion; per-access generic addressing cost 3 uniform instructions per load)
#pragma unroll
          for (int j = 0; j < DMAX; ++j) {
            if (j < d) {
              double A[LIN_AW];
              lin_arm_load(arms_sa + 8 * LIN_AW * j, A);
              const double qf = fma(i00, A[2], fma(i01, A[3], i11 * A[4]));
              const double v = fma(p.p0, sqrt_nr(qf), fma(t0, A[0], t1 * A[1]));       // :519
              if (v > best) best = v, a = j;                                           // strict >: first maximum :520
            }
          }
        }
      }
      // ------------------------------------------------ env step ---------------------------
      const float z = zz[u];
      const float ma = cs.means[lane][a];
      const double r = reward_f64(ma, z, p.var, p.rtype);
      // ------------------------------------------------ controller statistics --------------
      if (STATS) {
        const double sa = cs.sum[a][lane] + r;
        const int ca = cs.cnt[a][lane] + 1;
        cs.sum[a][lane] = sa, cs.cnt[a][lane] = ca;
        S.untried &= ~(1u << a);
        double n0, n1 = 0.0;
        if (KIND == K_THOMPSON) {   // update_posterior_all :196-203, over the common denominator var + n*prior_var
          n0 = fma(p.p2, sa, sigma2tc0) * __ldg(tab0 + ca);   // = w*prior_mean + (1-w)*sum/n,  w = var/(var + n*prior_var)
          n1 = __ldg(tab1 + ca);                              // = sqrt(1 / (1/prior_var + n/var))
        } else {
          n0 = div_by_count(sa, ca, __ldg(tab0 + ca));        // b / max(1, counts)
          if (KIND == K_UCB) n0 += __ldg(tab1 + ca);          // + const / max(1, sqrt(counts)) :366
        }
#pragma unroll
        for (int j = 0; j < DMAX; ++j) {
          if (j == a) {
            S.st0[j] = n0;
            if (KIND == K_THOMPSON) S.st1[j] = n1;
          }
        }
      } else if (KIND == K_LINUCB2) {
        const double* A = s_arms + LIN_AW * a;
        S.b0 += A[0] * r, S.b1 += A[1] * r;
        S.s00 += A[2], S.s01 += 0.5 * A[3], S.s11 += A[4];   // (0.5 * (2 x0 x1) is exact)
      }
      // ------------------------------------------------ outputs ----------------------------
      if (live) st_stream(cmp, ma);                                     // get_arm_value :151-153 -> cum_means[hh, env]
      cmp += N;
      if (sl.creg_out) sl.sum_ma += (double)ma;
      rr[u] = (float)r;
      aw |= (uint32_t)a << (8 * u);
      bq |= (uint64_t)(1u << a) << (u * DMAX);                          // one-hot row of step u at bit u * DMAX of the quad's string
    }
    if constexpr (SPLIT) {
      if (sl.arms4) {
        if (live) *sl.arms4 = aw;   // 128 B per warp and step quad
        sl.arms4 += N;
      }
    } else if (stage) {
      Tile& tl = cs.tile;
      tl.rew[lane][q ^ swz(lane)] = make_float4(rr[0], rr[1], rr[2], rr[3]);
      tl.acts[lane][q] = aw;
      tl.bits[lane][q * BWQ] = (uint32_t)bq;
      if (BWQ > 1) tl.bits[lane][q * BWQ + 1] = (uint32_t)(bq >> 32);
    }
  }

  static __device__ __forceinline__ void controller(const OnlineParams& p, Cons& cs, const double* s_arms, const float4* s_nib,
                                                    const double* __restrict__ tab0, const double* __restrict__ tab1, int env, bool live, int lane) {
    const int N = p.N, H = p.H, d = p.d;
    const bool stage = p.ctx_a != nullptr;     // context materialised: tiles go through the flush warp
    const uint64_t gid = p.env_id0 + (uint64_t)env;
    float mmax = -INFINITY;
    int opt = 0;
#pragma unroll
    for (int j = 0; j < DMAX; ++j) {
      const float mj = (live && j < d) ? p.means[(size_t)env * d + j] : -INFINITY;
      if (mj > mmax) mmax = mj, opt = j;
      cs.means[lane][j] = mj;
      if (STATS) cs.sum[j][lane] = 0.0, cs.cnt[j][lane] = 0;
    }
    __syncwarp();
    State S;
#pragma unroll
    for (int j = 0; j < DMAX; ++j) {   // before the first pull: EMP mean 0, UCB 0 + bonus(0) = const, THOMPSON the prior;
      const bool real = j < d;         // padding arms (j >= d) can never win an argmax
      if (KIND == K_EMP) S.st0[j] = real ? 0.0 : -INFINITY;
      if (KIND == K_UCB) S.st0[j] = real ? 0.0 + p.p0 : -INFINITY;
      if (KIND == K_THOMPSON) S.st0[j] = real ? p.p1 : -INFINITY, S.st1[j] = real ? sqrt(p.p2) : 0.0;
    }
    S.untried = (d >= 32) ? 0xffffffffu : ((1u << d) - 1u);
    S.s00 = 1.0, S.s01 = 0.0, S.s11 = 1.0, S.b0 = 0.0, S.b1 = 0.0;
    const double sigma2tc0 = p.p0 * p.p0 * p.p1;                  // Thompson: std^2 (ctrls/ctrl_bandit.py:126) * prior_mean
    float* cmp = p.cum_means + env;       // (never NULL here: online_ws_supported)
    const int env0 = env - lane, nl = min(32, N - env0);
    const bool bits_ok = p.vec && d == DMAX && (H % 4 == 0);
    const bool vec_r = (H % 4 == 0) && (reinterpret_cast<uintptr_t>(p.ctx_r) & 15) == 0;
    if (stage) {   // constant states (bandit dx = 1): this warp's envs are one contiguous run
      fill_range(p.ctx_s, (size_t)env0 * H, (size_t)(env0 + nl) * H, 1.0f, lane, 32);
      fill_range(p.ctx_ns, (size_t)env0 * H, (size_t)(env0 + nl) * H, 1.0f, lane, 32);
    }
    Tile& tl = cs.tile;
    SplitLane sl{};   // (the fused kernel uses the regret carries only)
    if (p.creg_carry) sl.creg_out = p.creg_carry + env, sl.mmax = (double)mmax;
    for (int h0 = 0, T; h0 < H; h0 += T) {
      T = min(WT, H - h0);
      const int nq = T >> 2;
#pragma unroll 1
      for (int q = 0; q < nq; ++q)
        quad<true>(p, cs, S, s_arms, tab0, tab1, h0 + 4 * q, 4, q, opt, env, live, gid, cmp, sigma2tc0, stage, lane, sl);
      if (T & 3) quad<false>(p, cs, S, s_arms, tab0, tab1, h0 + 4 * nq, T & 3, nq, opt, env, live, gid, cmp, sigma2tc0, stage, lane, sl);
      if (stage) {
        __syncwarp();
        flush(p, tl, s_nib, env0, nl, h0, T, bits_ok, vec_r, lane);
        __syncwarp();
      }
    }
  }

  // ------------------------------------------------------------------------------- controller warp, split pipeline
  static __device__ __forceinline__ void controller_split(const OnlineParams& p, const SplitArgs& sa, Cons& cs, const double* s_arms,
                                                          const double* __restrict__ tab0, const double* __restrict__ tab1, int env, bool live,
                                                          int lane) {
    const int H = p.H, d = p.d;
    const uint64_t gid = p.env_id0 + (uint64_t)env;
    const double sigma2tc0 = p.p0 * p.p0 * p.p1;
    float mmax = -INFINITY;
    int opt = 0;
    State S;
#pragma unroll
    for (int j = 0; j < DMAX; ++j) {
      const bool real = j < d;         // padding arms (j >= d) carry -inf and can never win an argmax
      const float mj = (live && real) ? p.means[(size_t)env * d + j] : -INFINITY;
      if (mj > mmax) mmax = mj, opt = j;
      cs.means[lane][j] = mj;
      if (STATS) cs.sum[j][lane] = 0.0, cs.cnt[j][lane] = 0;
      if (KIND == K_EMP) S.st0[j] = real ? 0.0 : -INFINITY;
      if (KIND == K_UCB) S.st0[j] = real ? 0.0 + p.p0 : -INFINITY;
      if (KIND == K_THOMPSON) S.st0[j] = real ? p.p1 : -INFINITY, S.st1[j] = real ? sqrt(p.p2) : 0.0;
    }
    S.untried = (1u << d) - 1u;
    S.s00 = 1.0, S.s01 = 0.0, S.s11 = 1.0, S.b0 = 0.0, S.b1 = 0.0;
    __syncwarp();
    float* cmp = p.cum_means + env;
    SplitLane sl{};
    sl.arms4 = sa.arms4 ? sa.arms4 + env : nullptr, sl.creg_out = sa.creg ? sa.creg + env : nullptr, sl.mmax = (double)mmax;
    if (sa.creg && live) sa.creg[(size_t)((H + 127) >> 7) * p.N + env] = (double)mmax;   // row ceil(H / 128): max(means), for the expander
    if (sa.fill) {   // this lane's float4 of every 128-float piece of the warp's run of min(32, N - env0) * H floats
      const int env0 = env - lane;
      const long long run = (long long)min(32, p.N - env0) * H - 4 * lane;
      sl.fill_n = run > 0 ? (int)((run + 127) >> 7) : 0;
      sl.fill_p = reinterpret_cast<float4*>(p.ctx_s + (size_t)env0 * H) + lane;
      sl.fill_off = reinterpret_cast<char*>(p.ctx_ns) - reinterpret_cast<char*>(p.ctx_s);
    }
    const int nq = H >> 2, rem = H & 3;
#pragma unroll 1
    for (int q = 0; q < nq; ++q) quad<true>(p, cs, S, s_arms, tab0, tab1, 4 * q, 4, q, opt, env, live, gid, cmp, sigma2tc0, false, lane, sl);
    if (rem) quad<false>(p, cs, S, s_arms, tab0, tab1, 4 * nq, rem, nq, opt, env, live, gid, cmp, sigma2tc0, false, lane, sl);
  }
};

// resident CTAs per SM the kernels are compiled for: 6 (80 registers, no spills; 100k envs = 5.3 CTAs per SM are still ONE wave),
// Thompson at d = 10 keeps 40 float64 statistics in registers and gets 4 (128 registers)
template <int DMAX, int KIND>
constexpr int ws_min_blocks() { return (DMAX > 5 && KIND == K_THOMPSON) ? 4 : 6; }

template <int DMAX, int KIND, bool IO>
__global__ void __launch_bounds__(WS_NCONS * 32, ws_min_blocks<DMAX, KIND>()) online_loop_ws_kernel(const OnlineParams p, const double* __restrict__ tab) {
  using K = WsKernel<DMAX, KIND, IO>;
  using Cons = typename K::Cons;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  __shared__ float4 s_nib[16];   // 4-bit pattern -> four 0/1 floats (one-hot flush)
  Cons* cons = reinterpret_cast<Cons*>(smem_raw);
  double* s_arms = reinterpret_cast<double*>(smem_raw + sizeof(Cons) * WS_NCONS);   // [d][LIN_AW] (LinUCB)
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  onehot_nib_init(s_nib, tid);
  if (KIND == K_LINUCB2)
    for (int j = tid; j < p.d; j += blockDim.x) lin_arm_row(s_arms + LIN_AW * j, p.arms[2 * j], p.arms[2 * j + 1]);
  __syncthreads();
  const int env = (blockIdx.x * WS_NCONS + warp) * 32 + lane;
  if (env - lane < p.N)            // warp-uniform
    K::controller(p, cons[warp], s_arms, s_nib, tab, tab + (p.H + 1), env, env < p.N, lane);
}

// =============================================================================================
// Split pipeline (round 2, second half): controller kernel -> context expansion (+ regret sums)
// =============================================================================================
// The fused kernel above is bound by its context stores: every 32 steps an env's rows leave as 640 B + 128 B pieces scattered over
// 100k rows, drained by the same warps whose controller chains are the critical path (store-stream elimination in DESIGN.md section 4:
// 0.10 ms of controller against 0.46 ms of stores at 100k x 500).  Here the sequential part does only what is sequential:
//   online_ctrl_kernel     lane = env, all H steps: arm, reward (for its statistics), cum_means[h, env], ONE coalesced 4-byte word
//                          of arms per env and step quad into a scratch [H/4][N] (1 B per env-step), the constant state columns in
//                          512 B pieces per step quad (the warp's 32 envs are one contiguous run per array) and, every 128 steps,
//                          the env's cumulative regret (float64 carries for the expander / the regret pass);
//   online_expand_kernel   fully parallel over (env, step quad), behind the controller kernel on the same stream: re-derives the
//                          rewards from the same Philox block and the same float64 expression, writes rewards and one-hot rows as
//                          contiguous 128-step runs (16 B per lane, 512 B per warp and instruction) and accumulates the [H,3] regret
//                          sums in thread-local float64 registers;
//   ones_fill_kernel       the constant state columns when the shapes are not 16 B-friendly (otherwise the controller writes them);
//   regret_pass_kernel     the regret sums from cum_means when the context is not materialised (and after the fused kernel).
// Everything runs on the caller's stream.  Measured and dropped (DESIGN.md section 4, dead ends): controller chunks in time running
// beside expansion chunks on internal streams -- co-running kernels are issue-bound together, 128-step pieces lose DRAM locality.
// resident CTAs per SM the controller kernel is compiled for: 6 (80 registers, no spills; 100k envs = 5.3 CTAs per SM are still one
// wave), Thompson at d = 10 (40 float64 statistics in registers) 4
template <int DMAX, int KIND>
constexpr int ctrl_min_blocks() { return (DMAX > 5 && KIND == K_THOMPSON) ? 4 : 6; }
template <int DMAX, int KIND, bool IO>
__global__ void __launch_bounds__(WS_NCONS * 32, ctrl_min_blocks<DMAX, KIND>()) online_ctrl_kernel(const OnlineParams p, const double* __restrict__ tab,
                                                                                                   const SplitArgs sa) {
  using K = WsKernel<DMAX, KIND, IO, true>;
  using Cons = typename K::Cons;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  Cons* cons = reinterpret_cast<Cons*>(smem_raw);
  double* s_arms = reinterpret_cast<double*>(smem_raw + sizeof(Cons) * WS_NCONS);   // [d][LIN_AW] (LinUCB)
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (KIND == K_LINUCB2) {
    for (int j = tid; j < p.d; j += blockDim.x) lin_arm_row(s_arms + LIN_AW * j, p.arms[2 * j], p.arms[2 * j + 1]);
    __syncthreads();
  }
  const int env = (blockIdx.x * WS_NCONS + warp) * 32 + lane;
  if (env - lane < p.N)            // warp-uniform
    K::controller_split(p, sa, cons[warp], s_arms, tab, tab + (p.H + 1), env, env < p.N, lane);
}

constexpr int EX_WARPS = 4;
constexpr int EX_Q = 32;      // step quads per warp task (lane = quad): 128 steps
constexpr int EX_TASKS = 32;  // envs per warp: the 32 arms words a lane gathers are one 128 B line
// resident CTAs per SM the fast expander is compiled for: the 12 float64 accumulators of REG need 80 registers (96 at d = 10)
template <int D, bool REG>
constexpr int ex_min_blocks() { return REG ? (D > 5 ? 5 : 6) : 8; }

// Fast expander: compile-time d, H % 4 == 0, 16 B-aligned context rows.  A warp task is one env x 32 step quads (lane = quad); a
// warp walks up to 32 consecutive envs at a fixed 128-step range.  Its arms words arrive as coalesced [quad][env] rows (one line
// each) and are transposed through a per-warp shared-memory tile -- a lane-per-quad gather costs 32 LSU wavefronts per task (ncu:
// LSU data pipe at 59 %).  Rewards are re-derived from the same Philox block and float64 expression as in the controller (letting
// the controller store them in place, 16 B per lane at a row stride, cost it 258 -> 402 us).  The env's means sit in lanes
// 0 .. d - 1 and are picked with a shuffle by the arm.  One-hot rows: the task's 32 D float4 are re-tiled across the warp by
// shuffling the quads' bit strings; a float4 is one nibble = one 16-entry table lookup.  Warp slots are enumerated range-fastest,
// so CTAs in flight together cover whole rows of consecutive envs and DRAM sees one compact write window (env-block-fastest
// order: 4.2 TB/s, this order: 5.5 TB/s).
// REG: the per-step regret sums [H,3] (evals/eval_bandit.py:169-178: sum over envs of reg = max(means) - means[arm], reg^2 and the
// squared cumulative regret) are accumulated here instead of by a pass over cum_means: a lane owns the same 4 steps for all of its
// warp's envs, so the sums over envs are thread-local float64 accumulators; the cumulative regret of a step is the carry the
// controller left for this 128-step range + a warp scan over the quads + the prefix inside the quad.
template <int D, bool INJ, bool REG>
__global__ void __launch_bounds__(EX_WARPS * 32, ex_min_blocks<D, REG>()) online_expand_kernel(const OnlineParams p, const uint32_t* __restrict__ arms4,
                                                                                               const double* __restrict__ creg_in, int nqt, int ngy) {
  __shared__ float4 s_nib[16];   // 4-bit pattern -> four 0/1 floats
  __shared__ uint32_t s_arm[EX_WARPS][EX_Q][33];   // per warp: arms words [quad][env], read back by lane = quad (conflict-free)
  onehot_nib_init(s_nib, threadIdx.x);
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int N = p.N, H = p.H;
  // warp slot W = (env block of 32, 128-step range), range fastest: the warps of a CTA write the ranges of the SAME envs' rows at
  // the same time, env after env -- one contiguous burst per row, like a sequential stream
  const int W = blockIdx.x * EX_WARPS + warp;
  const int bx = W / ngy, by = W - bx * ngy;
  const int env0 = bx * EX_TASKS, ne = min(EX_TASKS, N - env0);
  const int q0 = by * EX_Q, nq = min(EX_Q, nqt - q0);
  if (ne <= 0) return;
  const int q = q0 + lane;
  const bool qv = lane < nq;
  // the warp's arms words: 32 coalesced row loads (one 128 B line each; a lane-per-quad gather would cost 32 LSU wavefronts per
  // task -- ncu showed the LSU data pipe at 59 %), transposed through shared memory
#pragma unroll 8
  for (int k = 0; k < nq; ++k) s_arm[warp][k][lane] = lane < ne ? __ldcs(arms4 + (size_t)(q0 + k) * N + env0 + lane) : 0u;
  __syncwarp();
  const float* msrc = p.means + (size_t)env0 * D + (lane < D ? lane : 0);
  const double* csrc = creg_in + (size_t)by * N + env0;      // (REG only) range `by` starts at step 128 by
  float m_n = __ldg(msrc);
  const double* xsrc = creg_in + (size_t)ngy * N + env0;     // (REG only) row ngy: max(means) of the env
  double c_n = REG ? __ldg(csrc) : 0.0, x_n = REG ? __ldg(xsrc) : 0.0;
  double s1[4] = {0.0, 0.0, 0.0, 0.0}, s2[4] = {0.0, 0.0, 0.0, 0.0}, c2[4] = {0.0, 0.0, 0.0, 0.0};
  for (int e = 0; e < ne; ++e) {
    const int env = env0 + e;
    const uint32_t aw = qv ? s_arm[warp][lane][e] : 0u;
    const float m = m_n;
    const double carry = c_n, mmax = x_n;
    if (e + 1 < ne) {
      m_n = __ldg(msrc + (e + 1) * D);
      if (REG) c_n = __ldg(csrc + e + 1), x_n = __ldg(xsrc + e + 1);
    }
    float zz[4];
    if (INJ) {
#pragma unroll
      for (int t = 0; t < 4; ++t) zz[t] = qv ? p.in.reward_z[(size_t)(4 * q + t) * N + env] : 0.f;
    } else {
      reward_noise4(p.key, p.env_id0 + (uint64_t)env, (uint32_t)q, p.rtype, zz);
    }
    float rr[4], ma[4];
    uint64_t bq = 0ull;
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int a = qv ? (aw >> (8 * u)) & 255 : 0;
      ma[u] = __shfl_sync(0xffffffffu, m, a);
      rr[u] = (float)reward_f64(ma[u], zz[u], p.var, p.rtype);
      bq |= (uint64_t)(1u << a) << (u * D);
    }
    const size_t row = (size_t)env * H + 4 * (size_t)q0;   // first step of this task
    st_stream_if(qv, reinterpret_cast<float4*>(p.ctx_r + row) + lane, make_float4(rr[0], rr[1], rr[2], rr[3]));
    // regret of the quad's steps and their prefix; the inclusive scan of the quad totals over the lanes (5 dependent shuffle
    // rounds) is interleaved with the one-hot stores below, which do not depend on it
    double reg[4], sc = 0.0;
    if (REG) {
#pragma unroll
      for (int u = 0; u < 4; ++u) reg[u] = qv ? mmax - (double)ma[u] : 0.0;
      sc = ((reg[0] + reg[1]) + reg[2]) + reg[3];
    }
    auto scan_round = [&](int o) {
      const double v = __shfl_up_sync(0xffffffffu, sc, o);
      if (lane >= o) sc += v;
    };
    // one-hot rows: the task's 32 quads are 32 D float4
    onehot_quad_store<D>(reinterpret_cast<float4*>(p.ctx_a + row * D), bq, lane, nq * D, s_nib, [&](int it) {
      if (REG && it < 5) scan_round(1 << it);
    });
    if (REG) {
#pragma unroll
      for (int it = D; it < 5; ++it) scan_round(1 << it);
      double cr = carry + (sc - (((reg[0] + reg[1]) + reg[2]) + reg[3]));   // cumulative regret before this quad
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        cr += reg[u];                                                       // (lanes past the range: reg = 0, sums land nowhere)
        s1[u] += reg[u], s2[u] = fma(reg[u], reg[u], s2[u]), c2[u] = fma(cr, cr, c2[u]);
      }
    }
  }
  if (REG && qv) {
    double* acc = p.regret + 3 * ((size_t)(bx & (p.regret_reps - 1)) * H + 4 * (size_t)q);
#pragma unroll
    for (int u = 0; u < 4; ++u) atomicAdd(acc + 3 * u, s1[u]), atomicAdd(acc + 3 * u + 1, s2[u]), atomicAdd(acc + 3 * u + 2, c2[u]);
  }
}

// Generic expander: any d <= 10, any H, any alignment; lane = step quad, scalar stores (odd shapes only)
__global__ void __launch_bounds__(EX_WARPS * 32) online_expand_generic_kernel(const OnlineParams p, const uint32_t* __restrict__ arms4, int q_lo,
                                                                              int q_hi) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int N = p.N, H = p.H, d = p.d;
  const int env = blockIdx.x * EX_WARPS + warp;
  if (env >= N) return;
  const bool inj = p.in.reward_z != nullptr;
  for (int q = q_lo + lane; q < q_hi; q += 32) {
    const uint32_t aw = arms4[(size_t)q * N + env];
    float zz[4];
    if (inj) {
#pragma unroll
      for (int t = 0; t < 4; ++t) zz[t] = (4 * q + t < H) ? p.in.reward_z[(size_t)(4 * q + t) * N + env] : 0.f;
    } else {
      reward_noise4(p.key, p.env_id0 + (uint64_t)env, (uint32_t)q, p.rtype, zz);
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int h = 4 * q + u;
      if (h >= H) break;
      const int a = (aw >> (8 * u)) & 255;
      const size_t row = (size_t)env * H + h;
      st_stream(p.ctx_r + row, (float)reward_f64(p.means[(size_t)env * d + a], zz[u], p.var, p.rtype));
      for (int j = 0; j < d; ++j) st_stream(p.ctx_a + row * d + j, j == a ? 1.f : 0.f);
    }
  }
}

// constant states (bandit dx = 1, envs/bandit_env.py:38): context_states = context_next_states = 1
__global__ void __launch_bounds__(256) ones_fill_kernel(float* __restrict__ a, float* __restrict__ b, size_t n) {
  const size_t per = ((n + gridDim.x - 1) / gridDim.x + 3) & ~size_t(3);
  const size_t lo = min(n, per * blockIdx.x), hi = min(n, lo + per);
  fill_range(a, lo, hi, 1.0f, threadIdx.x, 256);
  fill_range(b, lo, hi, 1.0f, threadIdx.x, 256);
}

// ---------------------------------------------------------------------------------------------
// Regret statistics (evals/eval_bandit.py:169-178) from cum_means [H,N]: sums over envs, per step, of the regret
// reg = max(means) - cum_means, reg^2, the cumulative regret and its square.  One warp per 32 envs: lane = env for
// the loads (128 B per step row) and the float64 prefix over steps, lane = step for the sums over the 32 envs
// (32 x 32 tile through shared memory), then one atomic per (step, statistic) and warp into replicated accumulators.
// ---------------------------------------------------------------------------------------------
constexpr int RP_WARPS = 4;
constexpr int RP_T = 16;      // steps per tile: 32 envs x 16 steps (6.5 KB of shared memory per warp, so 100k envs are one wave)
__global__ void __launch_bounds__(RP_WARPS * 32, 6) regret_pass_kernel(const float* __restrict__ cum_means, const float* __restrict__ means, int N,
                                                                       int H, int d, double* __restrict__ reps, int n_reps,
                                                                       const double* __restrict__ creg_in) {
  // blockIdx.y = a 128-step range; its starting cumulative regret per env is what the loop kernel left in creg_in [range][N].
  // (Measured, 100k x 500: one warp per 32 envs over all H 0.09 ms; ranges -- 4x the warps -- the same; 4 env blocks per warp
  // with the sums meeting in shared memory -- 4x fewer atomics -- 0.11 ms: neither parallelism nor the atomics bound it.)
  const int h_lo = 128 * (int)blockIdx.y, h_hi = min(H, h_lo + 128);
  __shared__ float s_cm[RP_WARPS][32][RP_T + 1];
  __shared__ double s_cr[RP_WARPS][32][RP_T + 1];
  __shared__ float s_mx[RP_WARPS][32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int gw = blockIdx.x * RP_WARPS + warp, env0 = gw * 32;
  if (env0 >= N) return;
  const int env = env0 + lane, nl = min(32, N - env0);
  const bool live = env < N;
  float mmax = -INFINITY;
  if (live)
    for (int j = 0; j < d; ++j) mmax = fmaxf(mmax, means[(size_t)env * d + j]);
  s_mx[warp][lane] = mmax;
  double creg = live ? creg_in[(size_t)blockIdx.y * N + env] : 0.0;
  double* acc = reps + 3 * (size_t)(gw & (n_reps - 1)) * H;    // [n_reps][H][3]: sum reg, sum reg^2, sum creg^2
  const int t = lane & (RP_T - 1), half = lane >> 4;           // sums over envs: lane = (half of the envs, step)
  const float* src = cum_means + env;
  float cm[RP_T], nx[RP_T];
#pragma unroll
  for (int k = 0; k < RP_T; ++k) nx[k] = (live && h_lo + k < h_hi) ? __ldcs(src + (size_t)(h_lo + k) * N) : 0.f;
  for (int h0 = h_lo; h0 < h_hi; h0 += RP_T) {
    const int T = min(RP_T, h_hi - h0);
#pragma unroll
    for (int k = 0; k < RP_T; ++k) cm[k] = nx[k];
#pragma unroll
    for (int k = 0; k < RP_T; ++k)   // next tile's loads are in flight while this one is reduced
      nx[k] = (live && h0 + RP_T + k < h_hi) ? __ldcs(src + (size_t)(h0 + RP_T + k) * N) : 0.f;
#pragma unroll
    for (int k = 0; k < RP_T; ++k) {
      if (k < T) creg += (double)mmax - (double)cm[k];   // (the prefix must not see the padding of a partial tile)
      s_cm[warp][lane][k] = cm[k];
      s_cr[warp][lane][k] = creg;
    }
    __syncwarp();
    double s1 = 0.0, s2 = 0.0, c2 = 0.0;
#pragma unroll 4
    for (int e = half; e < nl; e += 2) {
      const double reg = (double)s_mx[warp][e] - (double)s_cm[warp][e][t];
      const double cr = s_cr[warp][e][t];
      s1 += reg, s2 = fma(reg, reg, s2), c2 = fma(cr, cr, c2);
    }
    s1 += __shfl_xor_sync(0xffffffffu, s1, 16), s2 += __shfl_xor_sync(0xffffffffu, s2, 16), c2 += __shfl_xor_sync(0xffffffffu, c2, 16);
    if (lane < T) {
      double* dst = acc + 3 * (size_t)(h0 + lane);
      atomicAdd(dst, s1), atomicAdd(dst + 1, s2), atomicAdd(dst + 2, c2);
    }
    __syncwarp();
  }
}

// regret[h] += (S1, S2, C1, C2)[h]: S1, S2, C2 folded over the replicas in a fixed order; the sum over envs of the cumulative
// regret is linear in the per-step sums, C1[h] = sum_{h' <= h} S1[h'], so it is a prefix over steps (one block, carry per chunk)
__global__ void __launch_bounds__(1024) regret_finish_kernel(const double* __restrict__ reps, int n_reps, int H, double* __restrict__ regret) {
  __shared__ double s_warp[32];
  __shared__ double s_carry;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (threadIdx.x == 0) s_carry = 0.0;
  __syncthreads();
  for (int h0 = 0; h0 < H; h0 += 1024) {
    const int h = h0 + threadIdx.x;
    double s1 = 0.0, s2 = 0.0, c2 = 0.0;
    if (h < H) {
#pragma unroll 16
      for (int r = 0; r < n_reps; ++r) {   // fixed order; independent loads
        const double* src = reps + 3 * ((size_t)r * H + h);
        s1 += src[0], s2 += src[1], c2 += src[2];
      }
    }
    double sc = s1;                         // inclusive scan of s1 over the 1024 steps of this chunk
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const double v = __shfl_up_sync(0xffffffffu, sc, o);
      if (lane >= o) sc += v;
    }
    if (lane == 31) s_warp[warp] = sc;
    __syncthreads();
    if (warp == 0) {
      double w = s_warp[lane];
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const double v = __shfl_up_sync(0xffffffffu, w, o);
        if (lane >= o) w += v;
      }
      s_warp[lane] = w;
    }
    __syncthreads();
    const double c1 = s_carry + (warp ? s_warp[warp - 1] : 0.0) + sc;
    if (h < H) {
      double* dst = regret + 4 * (size_t)h;
      dst[0] += s1, dst[1] += s2, dst[2] += c1, dst[3] += c2;
    }
    __syncthreads();
    if (threadIdx.x == 1023) s_carry = c1;
    __syncthreads();
  }
}

// count-indexed float64 terms, n = 0..H.  EMP / UCB: tab0 = 1 / max(1, n), tab1 = const / max(1, sqrt(n));
// THOMPSON: tab0 = 1 / (var + n prior_var), tab1 = sqrt(var prior_var tab0)  -- the expressions of online_loop.cu
__global__ void online_ws_table_kernel(int kind, double p0, double p2, int H, double* __restrict__ tab) {
  const int n = blockIdx.x * blockDim.x + threadIdx.x;
  if (n > H) return;
  double t0, t1;
  if (kind == K_THOMPSON) {
    const double sigma2 = p0 * p0;
    t0 = 1.0 / (sigma2 + (double)n * p2);
    t1 = sqrt(sigma2 * p2 * t0);
  } else {
    t0 = 1.0 / fmax(1.0, (double)n);
    t1 = p0 / fmax(1.0, sqrt((double)n));
  }
  tab[n] = t0, tab[(H + 1) + n] = t1;
}

// selftest: div_by_count(a, n, RN(1/n)) == a / n bit for bit
__global__ void selftest_div_kernel(const double* __restrict__ a, const int* __restrict__ n, int count, int* __restrict__ mismatches) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= count) return;
  const double want = a[i] / (double)n[i];
  const double got = div_by_count(a[i], n[i], 1.0 / (double)n[i]);
  if (__double_as_longlong(want) != __double_as_longlong(got)) atomicAdd(mismatches, 1);
}

bool online_ws_supported(int kind, const OnlineParams& p) {
  if (p.d > 10) return false;
  if (!p.cum_means) return false;               // cum_means is the kernel's primary output (and what the regret pass reads)
  if (kind == K_LINUCB && p.lin_d != 2) return false;
  return true;
}

template <int DMAX, int KIND>
static cudaError_t launch_ws(const OnlineParams& p, double* tab, cudaStream_t st) {
  const bool io = p.in.reward_z || p.in.ctrl_z || p.in.first_arm || p.out.reward_z || p.out.ctrl_z || p.out.first_arm;
  auto kern = io ? online_loop_ws_kernel<DMAX, KIND, true> : online_loop_ws_kernel<DMAX, KIND, false>;
  using Cons = typename WsKernel<DMAX, KIND, false>::Cons;
  const size_t smem = sizeof(Cons) * WS_NCONS + (KIND == K_LINUCB2 ? sizeof(double) * LIN_AW * p.d : 0);
  if (smem > 48 * 1024) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
  }
  if (KIND == K_EMP || KIND == K_UCB || KIND == K_THOMPSON)
    online_ws_table_kernel<<<(p.H + 1 + 255) / 256, 256, 0, st>>>(KIND, p.p0, p.p2, p.H, tab);
  const int warps_total = (p.N + 31) / 32;
  kern<<<(warps_total + WS_NCONS - 1) / WS_NCONS, WS_NCONS * 32, smem, st>>>(p, tab);
  return cudaGetLastError();
}

template <int DMAX>
static cudaError_t launch_ws_kind(int kind, const OnlineParams& p, double* tab, cudaStream_t st) {
  switch (kind) {
    case K_OPT: return launch_ws<DMAX, K_OPT>(p, tab, st);
    case K_EMP: return launch_ws<DMAX, K_EMP>(p, tab, st);
    case K_UCB: return launch_ws<DMAX, K_UCB>(p, tab, st);
    case K_THOMPSON: return launch_ws<DMAX, K_THOMPSON>(p, tab, st);
    default: return launch_ws<DMAX, K_LINUCB2>(p, tab, st);
  }
}

// ------------------------------------------------------------------------------------------- split pipeline, host side
namespace {
int fill_grid(size_t n, int per_sm) {
  const size_t want = (n + 16383) / 16384, cap = (size_t)sm_count() * per_sm;
  const size_t g = want < cap ? want : cap;
  return g ? (int)g : 1;
}

}  // namespace

#define SPLIT_TRY(call)                  \
  do {                                   \
    cudaError_t _e = (call);             \
    if (_e != cudaSuccess) return _e;    \
  } while (0)

static bool expand_is_fast(const OnlineParams& p) {
  return p.vec && p.H % 4 == 0 && aligned16(p.ctx_r) && (p.d == 10 || (p.d >= 2 && p.d <= 5));
}

template <int D>
static void launch_expand_fast(const OnlineParams& p, const uint32_t* arms4, const double* creg, cudaStream_t st) {
  const int nqt = p.H / 4, ngy = (nqt + EX_Q - 1) / EX_Q;
  const unsigned slots = (unsigned)((p.N + EX_TASKS - 1) / EX_TASKS) * ngy, grid = (slots + EX_WARPS - 1) / EX_WARPS;
  const bool inj = p.in.reward_z != nullptr, reg = creg != nullptr;
  auto kern = inj ? (reg ? online_expand_kernel<D, true, true> : online_expand_kernel<D, true, false>)
                  : (reg ? online_expand_kernel<D, false, true> : online_expand_kernel<D, false, false>);
  kern<<<grid, EX_WARPS * 32, 0, st>>>(p, arms4, creg, nqt, ngy);
}

static void launch_expand(const OnlineParams& p, const uint32_t* arms4, const double* creg, cudaStream_t st) {
  if (expand_is_fast(p)) {
    switch (p.d) {
      case 2: return launch_expand_fast<2>(p, arms4, creg, st);
      case 3: return launch_expand_fast<3>(p, arms4, creg, st);
      case 4: return launch_expand_fast<4>(p, arms4, creg, st);
      case 5: return launch_expand_fast<5>(p, arms4, creg, st);
      default: return launch_expand_fast<10>(p, arms4, creg, st);
    }
  }
  online_expand_generic_kernel<<<(p.N + EX_WARPS - 1) / EX_WARPS, EX_WARPS * 32, 0, st>>>(p, arms4, 0, (p.H + 3) / 4);
}

// One pass, all on the caller's stream: count tables -> controller (+ constant-column fill) -> expansion (+ regret sums) ->
// regret_finish.
template <int DMAX, int KIND>
static cudaError_t launch_split(const OnlineParams& p, double* tab, double* regret_out, cudaStream_t st) {
  const bool io = p.in.reward_z || p.in.ctrl_z || p.in.first_arm || p.out.reward_z || p.out.ctrl_z || p.out.first_arm;
  auto kern = io ? online_ctrl_kernel<DMAX, KIND, true> : online_ctrl_kernel<DMAX, KIND, false>;
  using Cons = typename WsKernel<DMAX, KIND, false, true>::Cons;
  const size_t smem = sizeof(Cons) * WS_NCONS + (KIND == K_LINUCB2 ? sizeof(double) * LIN_AW * p.d : 0);
  const int N = p.N, H = p.H;
  const bool mat = p.ctx_a != nullptr;
  const bool reg_fused = mat && regret_out && expand_is_fast(p);   // regret sums in the expander; otherwise a pass over cum_means
  const int HQ = (H + 3) / 4, HC = (H + 127) / 128;
  const size_t b_arms = mat ? (((size_t)HQ * N * 4 + 255) & ~size_t(255)) : 0;
  const size_t b_creg = regret_out ? (size_t)(HC + 1) * N * 8 : 0;   // regret carries: for the expander, else for the regret pass
  unsigned char* scratch = nullptr;
  if (b_arms + b_creg) {
    keep_pool_memory();
    SPLIT_TRY(cudaMallocAsync(reinterpret_cast<void**>(&scratch), b_arms + b_creg, st));
  }
  SplitArgs sa{};
  sa.arms4 = mat ? reinterpret_cast<uint32_t*>(scratch) : nullptr;
  sa.creg = regret_out ? reinterpret_cast<double*>(scratch + b_arms) : nullptr;
  if (KIND == K_EMP || KIND == K_UCB || KIND == K_THOMPSON)
    online_ws_table_kernel<<<(H + 1 + 255) / 256, 256, 0, st>>>(KIND, p.p0, p.p2, H, tab);
  const int warps_total = (N + 31) / 32;
  const int ctrl_grid = (warps_total + WS_NCONS - 1) / WS_NCONS;
  sa.fill = mat && H % 4 == 0 && aligned16(p.ctx_s) && aligned16(p.ctx_ns);
  kern<<<ctrl_grid, WS_NCONS * 32, smem, st>>>(p, tab, sa);
  if (mat && !sa.fill) ones_fill_kernel<<<fill_grid((size_t)N * H, 8), 256, 0, st>>>(p.ctx_s, p.ctx_ns, (size_t)N * H);
  if (mat) launch_expand(p, sa.arms4, reg_fused ? sa.creg : nullptr, st);
  if (regret_out) {
    if (!reg_fused)
      regret_pass_kernel<<<dim3((warps_total + RP_WARPS - 1) / RP_WARPS, HC), RP_WARPS * 32, 0, st>>>(p.cum_means, p.means, N, H, p.d, p.regret,
                                                                                                    p.regret_reps, sa.creg);
    regret_finish_kernel<<<1, 1024, 0, st>>>(p.regret, p.regret_reps, H, regret_out);
  }
  const cudaError_t err = cudaGetLastError();
  if (scratch) SPLIT_TRY(cudaFreeAsync(scratch, st));
  return err;
}

template <int DMAX>
static cudaError_t launch_split_kind(int kind, const OnlineParams& p, double* tab, double* regret_out, cudaStream_t st) {
  switch (kind) {
    case K_OPT: return launch_split<DMAX, K_OPT>(p, tab, regret_out, st);
    case K_EMP: return launch_split<DMAX, K_EMP>(p, tab, regret_out, st);
    case K_UCB: return launch_split<DMAX, K_UCB>(p, tab, regret_out, st);
    case K_THOMPSON: return launch_split<DMAX, K_THOMPSON>(p, tab, regret_out, st);
    default: return launch_split<DMAX, K_LINUCB2>(p, tab, regret_out, st);
  }
}

// the split pipeline; fused = true: the single fused kernel of this file's first half (dpt_online_loop picks one by controller
// kind and batch size)
cudaError_t launch_online_ws(int kind, const OnlineParams& p, double* tab, double* regret_out, cudaStream_t st, bool fused) {
  if (!online_ws_supported(kind, p)) return cudaErrorNotSupported;
  if (!fused) return p.d <= 5 ? launch_split_kind<5>(kind, p, tab, regret_out, st) : launch_split_kind<10>(kind, p, tab, regret_out, st);
  OnlineParams q = p;
  const int HC = (p.H + 127) / 128;
  if (regret_out) {   // regret carries [HC][N] for the ranged regret pass
    keep_pool_memory();
    SPLIT_TRY(cudaMallocAsync(reinterpret_cast<void**>(&q.creg_carry), (size_t)HC * p.N * sizeof(double), st));
  }
  cudaError_t e = p.d <= 5 ? launch_ws_kind<5>(kind, q, tab, st) : launch_ws_kind<10>(kind, q, tab, st);
  if (e == cudaSuccess && regret_out) {   // [H,4] regret sums from cum_means: p.regret = zeroed [regret_reps][H][3] scratch
    const int ctas = ((p.N + 31) / 32 + RP_WARPS - 1) / RP_WARPS;   // one atomic set per warp (32 envs) and 16-step tile
    regret_pass_kernel<<<dim3(ctas, HC), RP_WARPS * 32, 0, st>>>(p.cum_means, p.means, p.N, p.H, p.d, p.regret, p.regret_reps, q.creg_carry);
    regret_finish_kernel<<<1, 1024, 0, st>>>(p.regret, p.regret_reps, p.H, regret_out);
    e = cudaGetLastError();
  }
  if (q.creg_carry) SPLIT_TRY(cudaFreeAsync(q.creg_carry, st));
  return e;
}

}  // namespace dpt

using namespace dpt;

extern "C" int dpt_selftest_div(const double* a, const int* n, int count, int* mismatches, void* stream) {
  DPT_CHECK_ARG(a && n && mismatches && count >= 0, "dpt_selftest_div: bad arguments");
  if (count == 0) return DPT_OK;
  selftest_div_kernel<<<(count + 255) / 256, 256, 0, (cudaStream_t)stream>>>(a, n, count, mismatches);
  DPT_LAUNCH_CHECK();
  return DPT_OK;
}
