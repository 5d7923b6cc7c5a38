// Fused online evaluation loop for the classical bandit controllers, and the stand-alone
// per-arm statistics kernel.
//
//   dpt_online_loop : deploy_online_vec (reference evals/eval_bandit.py:56-103) + BanditEnvVec.deploy /
//                     step / transit (envs/bandit_env.py:98-149, :56-64) + the controller's
//                     set_batch_numpy_vec / act_numpy_vec (ctrls/ctrl_bandit.py) for all H steps in ONE
//                     launch.  The reference recounts every arm from the whole context at every step
//                     (O(N d h) Python per step, O(H^2) per trajectory); here one thread owns one env and
//                     keeps the per-arm (count, reward sum) in registers, so a step is O(d).
//                     All controller statistics are float64 like the reference, so the chosen arm is the
//                     reference's arm unless two arms tie to ~1e-16.
//   dpt_arm_stats   : the same statistics from an arbitrary pre-filled context (offline evaluation /
//                     set_batch on a given context), one warp per env with warp-shuffle reductions.
//
// HBM traffic of the loop: 4*(2+d+1) B of context rows + 4 B of cum_means per env-step (36 B for d=5).
// A thread's own rows are strided by H*d*4 B, so rows are staged per warp in shared memory (1 B per
// action, 4 B per reward, 32 envs x 32 steps) and flushed as contiguous, 16 B-aligned float4 runs
// (32 steps * d * 4 B per env).
#include <atomic>

#include "online_loop.cuh"

namespace dpt {

// dynamic shared memory: [nwarps] WarpTile | [nwarps*32][DMAX] float means | (8 B-aligned) [d][lin_d] double arms
__host__ __device__ inline size_t ol_arms_offset(int nwarps, int dmax) {
  return (sizeof(WarpTile) * nwarps + sizeof(float) * 32 * nwarps * dmax + 7) & ~size_t(7);
}

// IO: the launch injects or dumps noise (parity runs); the production instantiation carries none of those branches
template <int DMAX, int KIND, bool IO>
__global__ void __launch_bounds__(OL_THREADS) online_loop_kernel(const OnlineParams p) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  __shared__ float4 s_nib[16];   // 4-bit pattern -> four 0/1 floats (one-hot flush)
  const int nthreads = blockDim.x, nwarps = nthreads >> 5;   // 1 or 2 warps per CTA (host picks the wave fit)
  WarpTile* tiles = reinterpret_cast<WarpTile*>(smem_raw);
  float* s_means_all = reinterpret_cast<float*>(smem_raw + sizeof(WarpTile) * nwarps);   // [nthreads][DMAX]
  double* s_arms = reinterpret_cast<double*>(smem_raw + ol_arms_offset(nwarps, DMAX));   // [d][lin_d]
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  WarpTile& tile = tiles[warp];
  float(*s_means)[DMAX] = reinterpret_cast<float(*)[DMAX]>(s_means_all) + warp * 32;
  const int env0w = (blockIdx.x * nwarps + warp) * 32;  // first env of this warp
  onehot_nib_init(s_nib, tid);
  const int env = env0w + lane;
  const bool live = env < p.N;
  const int N = p.N, H = p.H, d = p.d;
  const uint64_t gid = p.env_id0 + (uint64_t)env;
  const bool materialise = p.ctx_a != nullptr;

  if (KIND == K_LINUCB || KIND == K_LINUCB2) {
    for (int i = tid; i < d * p.lin_d; i += nthreads) s_arms[i] = p.arms[i];
  }
  float m[DMAX];
  float mmax = -INFINITY;
  int opt = 0;
#pragma unroll
  for (int j = 0; j < DMAX; ++j) {
    m[j] = (live && j < d) ? p.means[(size_t)env * d + j] : -INFINITY;
    if (m[j] > mmax) mmax = m[j], opt = j;
    s_means[lane][j] = m[j];
  }
  __syncthreads();


  // constant states (bandit dx = 1): this warp's envs are one contiguous run
  if (p.ctx_s) {
    const int nl = min(32, N - env0w);
    if (nl > 0) {
      fill_range(p.ctx_s, (size_t)env0w * H, (size_t)(env0w + nl) * H, 1.0f, lane, 32);
      fill_range(p.ctx_ns, (size_t)env0w * H, (size_t)(env0w + nl) * H, 1.0f, lane, 32);
    }
  }

  ArmState<DMAX> st;
#pragma unroll
  for (int j = 0; j < DMAX; ++j) {
    st.sum[j] = 0.0, st.cnt[j] = 0;
    st.aux0[j] = (KIND == K_THOMPSON) ? p.p1 : 0.0;                  // prior mean | empirical mean 0
    st.aux1[j] = (KIND == K_THOMPSON) ? sqrt(p.p2) : p.p0;           // prior std  | UCB bonus const/max(1,0)
  }
  // LinUCB: S = I + sum x x^T, bvec = sum x r  (ctrls/ctrl_bandit.py:510-513)
  double S[KIND == K_LINUCB ? OL_MAX_LD * OL_MAX_LD : 1], bv[KIND == K_LINUCB ? OL_MAX_LD : 1];
  double s00 = 1.0, s01 = 0.0, s11 = 1.0, b0 = 0.0, b1 = 0.0;   // K_LINUCB2: Sigma = I + sum x x^T (symmetric), b = sum x r
  if (KIND == K_LINUCB) {
    for (int i = 0; i < p.lin_d; ++i) {
      bv[i] = 0.0;
      for (int j = 0; j < p.lin_d; ++j) S[i * p.lin_d + j] = (i == j) ? 1.0 : 0.0;
    }
  }
  const double sigma2 = p.p0 * p.p0;  // Thompson: std^2 (ctrls/ctrl_bandit.py:126)
  double creg = 0.0;  // this env's cumulative regret (evals/eval_bandit.py:176)
  const int nb_ctrl = (d + 3) >> 2;

  // Thompson: the d control normals of the step about to run; those of step h + 1 are generated while the
  // float64 posterior arithmetic of step h is in flight (they do not depend on the controller state)
  float zc[KIND == K_THOMPSON ? DMAX : 1];
  auto gen_ctrl = [&](int h, float* out) {
    if (IO && p.in.ctrl_z) {
#pragma unroll
      for (int j = 0; j < DMAX; ++j) out[j] = (live && j < d) ? p.in.ctrl_z[((size_t)h * N + env) * d + j] : 0.f;
    } else {
#pragma unroll
      for (int j0 = 0; j0 < DMAX; j0 += 4) {
        if (j0 < d) {
          float zz[4];
          normals4(philox_words(p.key, gid, (uint32_t)(h * nb_ctrl + (j0 >> 2)), STREAM_CTRL), zz);
#pragma unroll
          for (int c = 0; c < 4; ++c)
            if (j0 + c < DMAX) out[j0 + c] = zz[c];
        }
      }
    }
  };
  if (KIND == K_THOMPSON) gen_ctrl(0, zc);

  for (int h0 = 0; h0 < H; h0 += OL_T) {
    const int T = min(OL_T, H - h0);
    // ---- phase A: reward noise of the whole tile (independent Philox / Box-Muller chains, 4 in flight) ----
    if (IO && p.in.reward_z) {
      for (int t = 0; t < T; ++t) tile.rew[lane][(t + lane) & (OL_T - 1)] = live ? p.in.reward_z[(size_t)(h0 + t) * N + env] : 0.f;
    } else {
#pragma unroll 2
      for (int t = 0; t < T; t += 4) {   // one Philox block per 4 steps: (x, y) -> steps 4k, 4k+1; (z, w) -> 4k+2, 4k+3
        float z4[4];
        reward_noise4(p.key, gid, (uint32_t)((h0 + t) >> 2), p.rtype, z4);
#pragma unroll
        for (int k = 0; k < 4; ++k) tile.rew[lane][(t + k + lane) & (OL_T - 1)] = z4[k];
      }
    }
    // ---- phase B: the sequential controller / env steps ----
    for (int t = 0; t < T; ++t) {
      const int h = h0 + t;
      int a = 0;
      // ------------------------------------------------ controller: pick an arm ------------
      if (KIND == K_OPT) {
        a = opt;                                                        // :35-37
      } else if (KIND == K_EMP || KIND == K_UCB) {
        double best = -INFINITY;
        int first_untried = -1;
#pragma unroll
        for (int j = 0; j < DMAX; ++j) {
          if (j < d) {
            const double v = (KIND == K_UCB) ? st.aux0[j] + st.aux1[j] : st.aux0[j];   // :106 | :369-370
            if (v > best) best = v, a = j;                              // np.argmax: first maximum
            if (st.cnt[j] == 0 && first_untried < 0) first_untried = j; // np.argmin(counts) when min == 0
          }
        }
        if ((KIND == K_UCB || p.p0 != 0.0) && first_untried >= 0) a = first_untried;   // :110-113 | :373-375
      } else if (KIND == K_THOMPSON) {
        float zn[DMAX];
        if (h + 1 < H) gen_ctrl(h + 1, zn);
        double best = -INFINITY;
#pragma unroll
        for (int j = 0; j < DMAX; ++j) {
          if (j < d) {
            const float zj = zc[j];
            if (IO && p.out.ctrl_z && live) p.out.ctrl_z[((size_t)h * N + env) * d + j] = zj;
            const double v = st.aux0[j] + st.aux1[j] * (double)zj;      // np.random.normal(means, sqrt(variances)) :234
            if (v > best) best = v, a = j;
          }
        }
#pragma unroll
        for (int j = 0; j < DMAX; ++j) zc[j] = zn[j];
      } else if (KIND == K_LINUCB2 && h > 0) {   // lin_d == 2: closed-form inverse, everything in registers
        const double idet = 1.0 / (s00 * s11 - s01 * s01);
        const double i00 = s11 * idet, i01 = -s01 * idet, i11 = s00 * idet;
        const double t0 = i00 * b0 + i01 * b1, t1 = i01 * b0 + i11 * b1;          // theta = cov_inv @ A^T r  :513
        double best = -INFINITY;
        for (int j = 0; j < d; ++j) {
          const double x0 = s_arms[2 * j], x1 = s_arms[2 * j + 1];
          const double q = x0 * (i00 * x0 + i01 * x1) + x1 * (i01 * x0 + i11 * x1);
          const double v = (t0 * x0 + t1 * x1) + p.p0 * sqrt(q);                  // :519
          if (v > best) best = v, a = j;                                           // strict >: first maximum :520
        }
      } else {  // LinUCB
        if (h == 0) {                                                   // :496-500 uniform random first arm
          if (IO && p.in.first_arm)
            a = live ? p.in.first_arm[env] : 0;
          else
            a = (int)bounded(philox_words(p.key, gid, 0u, STREAM_CTRL).x, (uint32_t)d);
          if (IO && p.out.first_arm && live) p.out.first_arm[env] = a;
        } else if (KIND == K_LINUCB) {
          const int ld = p.lin_d;
          double Si[OL_MAX_LD * OL_MAX_LD], theta[OL_MAX_LD];
          if (ld == 2) {
            const double det = S[0] * S[3] - S[1] * S[2];
            Si[0] = S[3] / det, Si[1] = -S[1] / det, Si[2] = -S[2] / det, Si[3] = S[0] / det;
          } else {
            inv_small<OL_MAX_LD>(S, Si, ld);
          }
          for (int i = 0; i < ld; ++i) {
            double acc = 0.0;
            for (int j = 0; j < ld; ++j) acc += Si[i * ld + j] * bv[j];
            theta[i] = acc;                                             // cov_inv @ A^T r  :513
          }
          double best = -INFINITY;
          for (int j = 0; j < d; ++j) {
            const double* x = s_arms + j * ld;
            double mean = 0.0, q = 0.0;
            for (int i = 0; i < ld; ++i) {
              mean += theta[i] * x[i];
              double row = 0.0;
              for (int k = 0; k < ld; ++k) row += Si[i * ld + k] * x[k];
              q += x[i] * row;
            }
            const double v = mean + p.p0 * sqrt(q);                     // :519
            if (v > best) best = v, a = j;                              // strict >: first maximum :520
          }
        }
      }
      // ------------------------------------------------ env step ---------------------------
      const float z = tile.rew[lane][(t + lane) & (OL_T - 1)];
      if (IO && p.out.reward_z && live) p.out.reward_z[(size_t)h * N + env] = z;
      const float ma = s_means[lane][a];
      const double r = p.rtype == DPT_REWARD_GAUSSIAN ? (double)ma + (0.0 + p.var * (double)z)   // envs/bandit_env.py:59
                                                      : (z < ma ? 1.0 : 0.0);                    // :61 Bernoulli(mean)
      // ------------------------------------------------ controller statistics --------------
      if (KIND == K_EMP || KIND == K_UCB || KIND == K_THOMPSON) {
        // gather the pulled arm's (sum, count) with selects, update once, scatter back with selects:
        // no divergence although the lanes of a warp pull different arms
        double sa = 0.0;
        int ca = 0;
#pragma unroll
        for (int j = 0; j < DMAX; ++j)
          if (j == a) sa = st.sum[j], ca = st.cnt[j];
        sa += r;
        ca += 1;
        const double n = (double)ca;
        double n0, n1 = 0.0;
        if (KIND == K_THOMPSON) {   // update_posterior_all :196-203, over the common denominator var + n*prior_var
          const double inv = 1.0 / (sigma2 + n * p.p2);
          n0 = (sigma2 * p.p1 + p.p2 * sa) * inv;          // = w*prior_mean + (1-w)*sum/n,  w = var/(var + n*prior_var)
          n1 = sqrt(sigma2 * p.p2 * inv);                  // = sqrt(1 / (1/prior_var + n/var))
        } else {
          n0 = sa / n;                                      // b / max(1, counts)
          if (KIND == K_UCB) n1 = p.p0 / fmax(1.0, sqrt(n));  // const / max(1, sqrt(counts)) :366
        }
#pragma unroll
        for (int j = 0; j < DMAX; ++j) {
          const bool hit = (j == a);
          st.sum[j] = hit ? sa : st.sum[j];
          st.cnt[j] = hit ? ca : st.cnt[j];
          st.aux0[j] = hit ? n0 : st.aux0[j];
          if (KIND != K_EMP) st.aux1[j] = hit ? n1 : st.aux1[j];
        }
      } else if (KIND == K_LINUCB2) {
        const double x0 = s_arms[2 * a], x1 = s_arms[2 * a + 1];
        b0 += x0 * r, b1 += x1 * r;
        s00 += x0 * x0, s01 += x0 * x1, s11 += x1 * x1;
      } else if (KIND == K_LINUCB) {
        const int ld = p.lin_d;
        const double* x = s_arms + a * ld;
        for (int i = 0; i < ld; ++i) {
          bv[i] += x[i] * r;
          for (int j = 0; j < ld; ++j) S[i * ld + j] += x[i] * x[j];
        }
      }
      // ------------------------------------------------ outputs ----------------------------
      if (live && p.cum_means) st_stream(p.cum_means + (size_t)h * N + env, ma);   // get_arm_value :151-153
      tile.acts[lane][t] = (unsigned char)a;
      tile.rew[lane][(t + lane) & (OL_T - 1)] = (float)r;
      creg += (double)mmax - (double)ma;
      tile.creg[lane][(t + lane) & (OL_T - 1)] = (float)creg;
    }
    __syncwarp();
    // ------------------------------------------------ flush 32 envs x T steps ----------------
    const int nl = min(32, N - env0w);
    if (nl > 0 && p.regret) {     // per-step sums over this warp's envs (evals/eval_bandit.py:169-178); lane = step
      double s1 = 0.0, s2 = 0.0, c1 = 0.0, c2 = 0.0;
      for (int e = 0; e < nl; ++e) {   // warp-uniform trip count: the shuffle below needs all lanes
        const int ae = lane < T ? tile.acts[e][lane] : 0;
        const double reg = (double)__shfl_sync(0xffffffffu, mmax, e) - (double)s_means[e][ae];
        const double cr = (double)tile.creg[e][(lane + e) & (OL_T - 1)];
        s1 += reg, s2 += reg * reg, c1 += cr, c2 += cr * cr;
      }
      double* dst = p.regret + 4 * ((size_t)((blockIdx.x * nwarps + warp) & (p.regret_reps - 1)) * H + (size_t)(h0 + lane));
      if (lane < T) atomicAdd(dst, s1), atomicAdd(dst + 1, s2), atomicAdd(dst + 2, c1), atomicAdd(dst + 3, c2);
    }
    if (nl > 0 && materialise) {
      if (lane < T) {
        size_t idx = (size_t)env0w * H + h0 + lane;
        for (int e = 0; e < nl; ++e, idx += H) {
          st_stream(p.ctx_r + idx, tile.rew[e][(lane + e) & (OL_T - 1)]);
        }
      }
      if (p.vec) {
        // float4 q of an env's run covers flat elements 4q..4q+3 = bits [r0, r0+4) of the one-hot bit string of
        // steps t0, t0+1 (d >= 4) or t0..t0+3 (d < 4); (t0, r0) depend on the lane only, the 4-bit pattern
        // indexes a 16-entry float4 table: 2 byte loads + 5 integer ops + 1 table load per 16 B store
        using mask_t = typename std::conditional<(DMAX <= 16), uint32_t, uint64_t>::type;
        const int nq = (T * d) >> 2;   // float4 per env in this flush
        const int nsteps = (d >= 4) ? 2 : 4;
        const size_t estride = ((size_t)H * d) >> 2;
        float4* dst0 = reinterpret_cast<float4*>(p.ctx_a + ((size_t)env0w * H + h0) * d);
        for (int q = lane; q < nq; q += 32) {
          const int t0 = (d == 1) ? 4 * q : (int)__umulhi((uint32_t)(4 * q), p.magic_d);
          const int r0 = 4 * q - t0 * d;
          const int t1 = min(t0 + 1, T - 1), t2 = min(t0 + 2, T - 1), t3 = min(t0 + 3, T - 1);   // never read a step this tile did not write
          float4* dst = dst0 + q;
          for (int e = 0; e < nl; ++e, dst += estride) {
            mask_t M = ((mask_t)1 << tile.acts[e][t0]) | ((mask_t)1 << (d + tile.acts[e][t1]));
            if (nsteps == 4) M |= ((mask_t)1 << (2 * d + tile.acts[e][t2])) | ((mask_t)1 << (3 * d + tile.acts[e][t3]));
            st_stream(dst, s_nib[(uint32_t)(M >> r0) & 15u]);
          }
        }
      } else {
        const int per = T * d;
        for (int e = 0; e < nl; ++e)
          for (int el = lane; el < per; el += 32) {
            const int t = (d == 1) ? el : (int)__umulhi((uint32_t)el, p.magic_d);
            st_stream(p.ctx_a + ((size_t)(env0w + e) * H + h0) * d + el, (tile.acts[e][t] == el - t * d) ? 1.f : 0.f);
          }
      }
    }
    __syncwarp();
  }
}

// ---------------------------------------------------------------------------------------------
// dpt_arm_stats: one warp per env, lanes stride over the context steps, per-arm partials in
// registers, warp-shuffle reductions.
// ---------------------------------------------------------------------------------------------
template <int DMAX>
__global__ void __launch_bounds__(256) arm_stats_kernel(const float* __restrict__ ctx_a, const float* __restrict__ ctx_r,
                                                        int N, int h, int Hs, int d, double* __restrict__ sums,
                                                        int32_t* __restrict__ counts) {
  const int lane = threadIdx.x & 31;
  const int env = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (env >= N) return;
  double s[DMAX];
  int c[DMAX];
#pragma unroll
  for (int j = 0; j < DMAX; ++j) s[j] = 0.0, c[j] = 0;
  for (int t = lane; t < h; t += 32) {
    const float* row = ctx_a + ((size_t)env * Hs + t) * d;
    int a = 0;
    float bv = row[0];
    for (int j = 1; j < d; ++j) {
      const float v = row[j];
      if (v > bv) bv = v, a = j;       // np.argmax(actions, axis=-1)
    }
    const double r = (double)ctx_r[(size_t)env * Hs + t];
#pragma unroll
    for (int j = 0; j < DMAX; ++j)
      if (j == a) s[j] += r, c[j] += 1;
  }
#pragma unroll
  for (int j = 0; j < DMAX; ++j) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      s[j] += __shfl_xor_sync(0xffffffffu, s[j], o);
      c[j] += __shfl_xor_sync(0xffffffffu, c[j], o);
    }
    if (lane == 0 && j < d) sums[(size_t)env * d + j] = s[j], counts[(size_t)env * d + j] = c[j];
  }
}

// The scratch (regret replicas; split pipeline: the arms words, 1 B per env-step) comes from the device's default
// stream-ordered pool; let the pool keep up to 256 MB across synchronisations so that repeated calls do not go back to the driver.
void keep_pool_memory() {
  static thread_local int done_dev = -1;
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev == done_dev) return;
  cudaMemPool_t pool;
  if (cudaDeviceGetDefaultMemPool(&pool, dev) == cudaSuccess) {
    uint64_t cur = 0, want = 256ull << 20;
    if (cudaMemPoolGetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &cur) == cudaSuccess && cur < want)
      cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &want);
  }
  cudaGetLastError();
  done_dev = dev;
}

// regret[i] += sum over replicas (fixed order: the result does not depend on which replica a warp used)
__global__ void __launch_bounds__(256) regret_reduce_kernel(const double* __restrict__ reps, int n_reps, int n, double* __restrict__ regret) {
  const int i = blockIdx.x * 256 + threadIdx.x;
  if (i >= n) return;
  double acc = 0.0;
#pragma unroll 8
  for (int r = 0; r < n_reps; ++r) acc += reps[(size_t)r * n + i];   // (fixed order; independent loads, 8 in flight)
  regret[i] += acc;
}

template <int DMAX, int KIND>
static cudaError_t launch_online(const OnlineParams& p, cudaStream_t st) {
  const bool io = p.in.reward_z || p.in.ctrl_z || p.in.first_arm || p.out.reward_z || p.out.ctrl_z || p.out.first_arm;
  auto kern = io ? online_loop_kernel<DMAX, KIND, true> : online_loop_kernel<DMAX, KIND, false>;
  const size_t arms = sizeof(double) * ((KIND == K_LINUCB || KIND == K_LINUCB2) ? p.d * p.lin_d : 0);
  // One thread per env and H sequential steps: a partly filled last wave costs a whole wave.  Pick 2 or 1
  // warps per CTA so that the grid needs the fewest waves (ties: the larger CTA).
  const int warps_total = (p.N + 31) / 32;
  int best_nw = OL_WARPS;
  long best_waves = -1;
  for (int nw = OL_WARPS; nw >= 1; nw >>= 1) {
    const size_t smem = ol_arms_offset(nw, DMAX) + arms;
    if (smem > 48 * 1024 && cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) {
      cudaGetLastError();
      continue;
    }
    int per_sm = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, nw * 32, smem) != cudaSuccess || per_sm < 1) {
      cudaGetLastError();
      continue;
    }
    const long grid = (warps_total + nw - 1) / nw, cap = (long)per_sm * sm_count();
    const long waves = (grid + cap - 1) / cap;
    if (best_waves < 0 || waves < best_waves) best_waves = waves, best_nw = nw;
  }
  if (best_waves < 0) return cudaErrorInvalidConfiguration;
  const size_t smem = ol_arms_offset(best_nw, DMAX) + arms;
  if (smem > 48 * 1024) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
  }
  kern<<<(warps_total + best_nw - 1) / best_nw, best_nw * 32, smem, st>>>(p);
  return cudaGetLastError();
}

template <int DMAX>
static cudaError_t launch_online_kind(int kind, const OnlineParams& p, cudaStream_t st) {
  switch (kind) {
    case K_OPT: return launch_online<DMAX, K_OPT>(p, st);
    case K_EMP: return launch_online<DMAX, K_EMP>(p, st);
    case K_UCB: return launch_online<DMAX, K_UCB>(p, st);
    case K_THOMPSON: return launch_online<DMAX, K_THOMPSON>(p, st);
    default:
      return p.lin_d == 2 ? launch_online<DMAX, K_LINUCB2>(p, st) : launch_online<DMAX, K_LINUCB>(p, st);
  }
}

}  // namespace dpt

using namespace dpt;

static std::atomic<int> g_online_impl{-1};
extern "C" int dpt_debug_online_impl(int impl) { return g_online_impl.exchange(impl < -1 || impl > 3 ? -1 : impl); }

extern "C" int dpt_online_loop(int ctrl_kind, double p0, double p1, double p2, const float* means, const double* arms,
                               int lin_d, double var, int reward_type, uint64_t seed, uint64_t env_id0, int N, int H, int d,
                               float* ctx_states, float* ctx_actions, float* ctx_next_states, float* ctx_rewards,
                               float* cum_means, double* regret_sums, const dpt_online_inject_t* inject,
                               const dpt_online_dump_t* dump, void* stream) {
  DPT_CHECK_ARG(ctrl_kind >= K_OPT && ctrl_kind <= K_LINUCB, "dpt_online_loop: unknown controller kind %d", ctrl_kind);
  DPT_CHECK_ARG(N >= 0 && H >= 0, "dpt_online_loop: N=%d H=%d must be >= 0", N, H);
  DPT_CHECK_ARG(reward_type == DPT_REWARD_GAUSSIAN || reward_type == DPT_REWARD_BERNOULLI,
                "dpt_online_loop: unknown reward_type %d (0 uniform/gaussian, 1 bernoulli)", reward_type);
  DPT_CHECK_ARG(d >= 1 && d <= 32, "dpt_online_loop: d=%d outside [1,32]", d);
  if (N == 0 || H == 0) return DPT_OK;
  DPT_CHECK_ARG(means, "dpt_online_loop: null means");
  const bool any = ctx_states || ctx_actions || ctx_next_states || ctx_rewards;
  DPT_CHECK_ARG(!any || (ctx_states && ctx_actions && ctx_next_states && ctx_rewards),
                "dpt_online_loop: context pointers must be all NULL or all non-NULL");
  if (ctrl_kind == K_LINUCB) {
    DPT_CHECK_ARG(arms && lin_d >= 1 && lin_d <= OL_MAX_LD, "dpt_online_loop: LinUCB needs arms and 1 <= lin_d <= %d",
                  OL_MAX_LD);
  }
  if (ctrl_kind == K_THOMPSON) DPT_CHECK_ARG(p0 > 0.0 && p2 > 0.0, "dpt_online_loop: Thompson needs std > 0 and prior_var > 0");
  OnlineParams p{};
  p.p0 = p0, p.p1 = p1, p.p2 = p2, p.var = var;
  p.means = means, p.arms = arms, p.lin_d = lin_d;
  p.key = Key{(uint32_t)seed, (uint32_t)(seed >> 32)};
  p.env_id0 = env_id0;
  p.N = N, p.H = H, p.d = d;
  p.rtype = reward_type;
  p.magic_d = (uint32_t)((0x100000000ull + (uint64_t)d - 1) / (uint64_t)d);
  p.ctx_s = ctx_states, p.ctx_a = ctx_actions, p.ctx_ns = ctx_next_states, p.ctx_r = ctx_rewards;
  p.cum_means = cum_means, p.regret = regret_sums;
  if (inject) p.in = *inject;
  if (dump) p.out = *dump;
  p.vec = any && ((size_t)H * d) % 4 == 0 && (OL_T * d) % 4 == 0 && aligned16(ctx_actions);
  cudaError_t e;
  cudaStream_t st = (cudaStream_t)stream;
  // Every warp adds its 32 envs' partial sums to the same [H,4] block, tile by tile and nearly in lockstep:
  // spread them over replicated accumulators (stream-ordered scratch, <= 4 MB) and fold the replicas afterwards.
  // Automatic choice (dpt_debug_online_impl -1 / 0): online_loop_ws.cu where it applies (d <= 10, lin_d == 2): the split pipeline
  // (controller kernel, then context expansion) for Opt / EmpMean / UCB and for small batches, the single fused kernel for Thompson /
  // LinUCB at large batches (their controller chains are long enough to hide the fused kernel's scattered stores: 100k x 200,
  // d = 10: 0.50 / 0.65 ms fused against 0.56 / 0.71 ms split); 2 = always fused, 3 = always split, 1 = always the general kernel
  const int impl = g_online_impl.load(std::memory_order_relaxed);
  const bool ws = impl != 1 && online_ws_supported(ctrl_kind, p);
  double* reps = nullptr;
  unsigned char* scratch = nullptr;
  p.regret_reps = 1;
  int r = 1;
  if (ws) {
    if (regret_sums) r = N > 32 * 64 ? 16 : 1;      // regret_pass_kernel: one atomic set per warp (32 envs) and 16-step tile
  } else if (regret_sums && N > 32 * 8) {
    r = 64;
    while (r > 1 && (size_t)r * H * 32 > (4u << 20)) r >>= 1;
  }
  const size_t reps_bytes = (ws ? (regret_sums != nullptr) : r > 1) ? (size_t)r * H * 32 : 0;
  const size_t tab_bytes = ws ? 2 * (size_t)(H + 1) * sizeof(double) : 0;
  if (reps_bytes + tab_bytes) {
    keep_pool_memory();
    e = cudaMallocAsync(reinterpret_cast<void**>(&scratch), reps_bytes + tab_bytes, st);
    if (e == cudaSuccess && reps_bytes) e = cudaMemsetAsync(scratch, 0, reps_bytes, st);
    if (e != cudaSuccess) {
      set_error("dpt_online_loop: scratch: %s", cudaGetErrorString(e));
      return DPT_ERR_CUDA;
    }
    if (reps_bytes) reps = reinterpret_cast<double*>(scratch), p.regret = reps, p.regret_reps = r;
  }
  if (ws)
    e = launch_online_ws(ctrl_kind, p, reinterpret_cast<double*>(scratch + reps_bytes), regret_sums, st,
                         impl == 2 || (impl != 3 && (ctrl_kind == K_THOMPSON || ctrl_kind == K_LINUCB) && N > 32768));
  else if (d <= 5)
    e = launch_online_kind<5>(ctrl_kind, p, st);
  else if (d <= 10)
    e = launch_online_kind<10>(ctrl_kind, p, st);
  else if (d <= 16)
    e = launch_online_kind<16>(ctrl_kind, p, st);
  else
    e = launch_online_kind<32>(ctrl_kind, p, st);
  if (!ws && reps && e == cudaSuccess) {
    regret_reduce_kernel<<<(H * 4 + 255) / 256, 256, 0, st>>>(reps, p.regret_reps, H * 4, regret_sums);
    e = cudaGetLastError();
  }
  if (scratch) cudaFreeAsync(scratch, st);
  if (e != cudaSuccess) {
    set_error("dpt_online_loop launch failed: %s", cudaGetErrorString(e));
    return DPT_ERR_CUDA;
  }
  return DPT_OK;
}

extern "C" int dpt_arm_stats(const float* ctx_actions, const float* ctx_rewards, int N, int h, int H_stride, int d,
                             double* sums, int32_t* counts, void* stream) {
  DPT_CHECK_ARG(N >= 0 && h >= 0 && H_stride >= h, "dpt_arm_stats: N=%d h=%d H_stride=%d", N, h, H_stride);
  DPT_CHECK_ARG(d >= 1 && d <= 32, "dpt_arm_stats: d=%d outside [1,32]", d);
  if (N == 0) return DPT_OK;
  DPT_CHECK_ARG(sums && counts && (h == 0 || (ctx_actions && ctx_rewards)), "dpt_arm_stats: null pointer");
  const int grid = (N + 7) / 8;
  cudaStream_t st = (cudaStream_t)stream;
  if (d <= 5)
    arm_stats_kernel<5><<<grid, 256, 0, st>>>(ctx_actions, ctx_rewards, N, h, H_stride, d, sums, counts);
  else if (d <= 10)
    arm_stats_kernel<10><<<grid, 256, 0, st>>>(ctx_actions, ctx_rewards, N, h, H_stride, d, sums, counts);
  else if (d <= 16)
    arm_stats_kernel<16><<<grid, 256, 0, st>>>(ctx_actions, ctx_rewards, N, h, H_stride, d, sums, counts);
  else
    arm_stats_kernel<32><<<grid, 256, 0, st>>>(ctx_actions, ctx_rewards, N, h, H_stride, d, sums, counts);
  DPT_LAUNCH_CHECK();
  return DPT_OK;
}
