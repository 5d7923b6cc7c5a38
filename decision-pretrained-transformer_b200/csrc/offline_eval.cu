// Offline bandit evaluation for every dataset size in one pass over the context.
//
//   dpt_offline_eval : evals/eval_bandit.py:214-335 (offline / offline_graph) and evals/eval_linear_bandit.py:202-330 for a
//                      whole list of horizons.  Each controller sees the first h context rows of an env and plays one
//                      noise-free pull (BanditEnvVec.deploy_eval, envs/bandit_env.py:115-123: the reward is means[a]).
//
// The per-arm statistics of a prefix are cumulative, so one warp per env streams its context once, 32 steps at a time,
// and stops at every horizon of the (host-sorted) list to evaluate the controllers on the statistics so far:
//   - lane j < d owns arm j's (reward sum, pull count), in float64 like the reference;
//   - a run of steps is folded in either step by step (shuffle of the step's arm and reward) or, for long runs and few
//     arms, with one ballot/popc and one warp sum per arm;
//   - EmpMean / LCB / LinReg / the learner's argmax are warp-uniform and cheap; Thompson (sample=False) spreads its
//     n_draws posterior draws over the lanes and counts the winners with ballots.
// The sums over envs go to a per-CTA shared accumulator and leave with one set of double atomics per CTA.
#include <algorithm>
#include <vector>

#include "common.cuh"
#include "online_loop.cuh"
#include "philox.cuh"

namespace dpt {

constexpr int OE_WARPS = 8;
constexpr int OE_THREADS = OE_WARPS * 32;
constexpr int OE_MAX_LD = 8;
constexpr int OE_C = DPT_OFFLINE_NSLOTS;

struct OffWarp {  // per-warp scratch: the statistics every lane needs at a checkpoint
  double mu[32], sd[32], b[32];
  double aug[OE_MAX_LD][2 * OE_MAX_LD];  // [Sigma | I] -> [I | Sigma^-1]
  double rhs[OE_MAX_LD], theta[OE_MAX_LD];
  int n[32];
};

struct OffParams {
  const float* means;
  const float* ctx_a;
  const float* ctx_r;
  const int2* sched;  // [K] (horizon, slot) sorted by horizon
  int N, d, Hs, K, Hmax;
  int mask;
  double lcb_c, std2, prior_mean, prior_var, lin_c;
  int n_draws, nb;  // nb: Philox blocks per draw = ceil(d / 4)
  const double* arms;
  int lin_d;
  const float* logits;
  int logits_T;
  RoundKeys rk;
  uint64_t env_id0;
  const double* inject_z;
  double* dump_z;
  double* sums;     // [K][C][2]
  double* rewards;  // [K][C][N] or NULL
  bool smem_acc;    // accumulate sums in shared memory (else global atomics per env)
};

// first maximum: larger value wins, ties go to the lower index (np.argmax)
__device__ __forceinline__ int warp_argmax(double v, int idx) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const double ov = __shfl_xor_sync(0xffffffffu, v, o);
    const int oi = __shfl_xor_sync(0xffffffffu, idx, o);
    if (ov > v || (ov == v && oi < idx)) v = ov, idx = oi;
  }
  return idx;
}

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

__global__ void __launch_bounds__(OE_THREADS, 3) offline_eval_kernel(const OffParams p) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  OffWarp* wsall = reinterpret_cast<OffWarp*>(smem_raw);
  double* s_arms = reinterpret_cast<double*>(smem_raw + sizeof(OffWarp) * OE_WARPS);
  double* s_acc = s_arms + 32 * OE_MAX_LD;   // [K][C][2], when p.smem_acc
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  OffWarp& ws = wsall[warp];
  const int N = p.N, d = p.d, K = p.K;
  const bool use_emp = p.mask & (1 << DPT_OFFLINE_EMP), use_lcb = p.mask & (1 << DPT_OFFLINE_LCB);
  const bool use_thmp = p.mask & (1 << DPT_OFFLINE_THMP), use_lin = p.mask & (1 << DPT_OFFLINE_LINREG);
  const bool use_lnr = p.mask & (1 << DPT_OFFLINE_LNR);
  const bool need_ctx = use_emp || use_lcb || use_thmp || use_lin;
  const int ld = p.lin_d;

  if (use_lin)
    for (int i = tid; i < d * ld; i += OE_THREADS) s_arms[i] = p.arms[i];
  if (p.smem_acc)
    for (int i = tid; i < K * OE_C * 2; i += OE_THREADS) s_acc[i] = 0.0;
  __syncthreads();

  for (int env = blockIdx.x * OE_WARPS + warp; env < N; env += gridDim.x * OE_WARPS) {
    const uint64_t gid = p.env_id0 + (uint64_t)env;
    const float m = lane < d ? p.means[(size_t)env * d + lane] : -INFINITY;
    const int a_opt = warp_argmax((double)m, lane);
    const double mmax = (double)__shfl_sync(0xffffffffu, m, a_opt);
    double bsum = 0.0;  // lane j < d: arm j's reward sum and pull count so far
    int cnt = 0;
    int ci = 0;
    int hc = K > 0 ? p.sched[0].x : 0;
    int a_emp = 0, a_lcb = 0, a_lin = 0, a_lnr = 0;

    for (int t0 = 0; t0 < p.Hmax; t0 += 32) {
      const int n_in = min(32, p.Hmax - t0);
      int a = -1;
      float r = 0.f;
      if (need_ctx && lane < n_in) {
        const size_t row = (size_t)env * p.Hs + t0 + lane;
        const float* x = p.ctx_a + row * d;
        float bv = x[0];
        a = 0;
        for (int j = 1; j < d; ++j) {
          const float v = x[j];
          if (v > bv) bv = v, a = j;  // np.argmax(actions, axis=-1)
        }
        r = p.ctx_r[row];
      }
      int s0 = 0;
      while (s0 < n_in) {
        const bool stop = ci < K && hc <= t0 + n_in;  // a checkpoint ends inside this chunk
        const int s1 = stop ? hc - t0 : n_in;
        // ---- fold steps [s0, s1) into the per-arm statistics ----
        if (need_ctx && s1 > s0) {
          if (s1 - s0 > 2 * d) {
            const bool in = lane >= s0 && lane < s1;
            for (int j = 0; j < d; ++j) {
              const bool hit = in && a == j;
              const unsigned bal = __ballot_sync(0xffffffffu, hit);
              const double sj = warp_sum(hit ? (double)r : 0.0);
              if (lane == j) bsum += sj, cnt += __popc(bal);
            }
          } else {
            for (int s = s0; s < s1; ++s) {
              const int as = __shfl_sync(0xffffffffu, a, s);
              const float rs = __shfl_sync(0xffffffffu, r, s);
              if (lane == as) bsum += (double)rs, cnt += 1;
            }
          }
        }
        s0 = s1;
        if (!stop) continue;
        // ---- checkpoint: every slot whose horizon is hc ----
        const int h = hc;
        const double n = (double)cnt;
        if (lane < d) ws.b[lane] = bsum, ws.n[lane] = cnt;
        if (use_emp || use_lcb) {
          const double mean = bsum / fmax(1.0, n);                                    // b / max(1, counts)
          if (use_emp) a_emp = warp_argmax(lane < d ? mean : -INFINITY, lane);
          if (use_lcb) {
            const double v = mean - p.lcb_c / fmax(1.0, sqrt(n));                     // ctrl_bandit.py:255-314
            a_lcb = warp_argmax(lane < d ? v : -INFINITY, lane);
          }
        }
        if (use_thmp && lane < d) {  // ThompsonSamplingPolicy._posterior, operation for operation (no FMA contraction)
          const double am = cnt > 0 ? bsum / fmax(n, 1.0) : 0.0;
          const double pw = p.std2 / __dadd_rn(p.std2, __dmul_rn(n, p.prior_var));
          const double nm = __dadd_rn(__dmul_rn(pw, p.prior_mean), __dmul_rn(1.0 - pw, am));
          const double nv = 1.0 / __dadd_rn(1.0 / p.prior_var, n / p.std2);
          ws.mu[lane] = cnt > 0 ? nm : p.prior_mean;
          ws.sd[lane] = sqrt(cnt > 0 ? nv : p.prior_var);
        }
        __syncwarp();
        if (use_lin && ld == 2) {  // closed-form 2x2 inverse; Sigma and sum_a b_a x_a as warp sums over the arm lanes
          const double x0 = lane < d ? s_arms[2 * lane] : 0.0, x1 = lane < d ? s_arms[2 * lane + 1] : 0.0;
          const double s00 = 1.0 + warp_sum(n * (x0 * x0)), s01 = warp_sum(n * (x0 * x1)), s11 = 1.0 + warp_sum(n * (x1 * x1));
          const double r0 = warp_sum(bsum * x0), r1 = warp_sum(bsum * x1);
          const double idet = 1.0 / (s00 * s11 - s01 * s01);
          const double i00 = s11 * idet, i01 = -s01 * idet, i11 = s00 * idet;
          const double t0 = i00 * r0 + i01 * r1, t1 = i01 * r0 + i11 * r1;
          const double q = x0 * (i00 * x0 + i01 * x1) + x1 * (i01 * x0 + i11 * x1);
          a_lin = warp_argmax(lane < d ? (t0 * x0 + t1 * x1) + p.lin_c * sqrt(q) : -INFINITY, lane);
        } else if (use_lin) {  // theta = (I + sum_a n_a x_a x_a^T)^-1 sum_a b_a x_a;  value theta.x + c sqrt(x^T Sigma^-1 x)
          for (int e = lane; e < ld * ld + ld; e += 32) {
            double acc = 0.0;
            if (e < ld * ld) {
              const int i = e / ld, k = e - i * ld;
              acc = i == k ? 1.0 : 0.0;
              for (int j = 0; j < d; ++j) acc += (double)ws.n[j] * (s_arms[j * ld + i] * s_arms[j * ld + k]);
              ws.aug[i][k] = acc;
              ws.aug[i][ld + k] = i == k ? 1.0 : 0.0;
            } else {
              const int i = e - ld * ld;
              for (int j = 0; j < d; ++j) acc += ws.b[j] * s_arms[j * ld + i];
              ws.rhs[i] = acc;
            }
          }
          // Gauss-Jordan with partial pivoting, one lane per column of [Sigma | I]
          for (int c = 0; c < ld; ++c) {
            __syncwarp();
            int piv = c;
            double pv = fabs(ws.aug[c][c]);
            for (int rr = c + 1; rr < ld; ++rr)
              if (fabs(ws.aug[rr][c]) > pv) pv = fabs(ws.aug[rr][c]), piv = rr;
            __syncwarp();
            if (piv != c && lane < 2 * ld) {
              const double tmp = ws.aug[c][lane];
              ws.aug[c][lane] = ws.aug[piv][lane];
              ws.aug[piv][lane] = tmp;
            }
            __syncwarp();
            const double inv = 1.0 / ws.aug[c][c];
            double f[OE_MAX_LD];
#pragma unroll
            for (int rr = 0; rr < OE_MAX_LD; ++rr) f[rr] = rr < ld ? ws.aug[rr][c] : 0.0;
            __syncwarp();
            if (lane < 2 * ld) {
              const double pc = ws.aug[c][lane] * inv;
              ws.aug[c][lane] = pc;
#pragma unroll
              for (int rr = 0; rr < OE_MAX_LD; ++rr)
                if (rr < ld && rr != c) ws.aug[rr][lane] -= f[rr] * pc;
            }
          }
          __syncwarp();
          if (lane < ld) {
            double acc = 0.0;
            for (int k = 0; k < ld; ++k) acc += ws.aug[lane][ld + k] * ws.rhs[k];
            ws.theta[lane] = acc;
          }
          __syncwarp();
          double v = -INFINITY;
          if (lane < d) {
            const double* x = s_arms + lane * ld;
            double mean = 0.0, q = 0.0;
            for (int i = 0; i < ld; ++i) {
              mean += ws.theta[i] * x[i];
              double row = 0.0;
              for (int k = 0; k < ld; ++k) row += ws.aug[i][ld + k] * x[k];
              q += x[i] * row;
            }
            v = mean + p.lin_c * sqrt(q);
          }
          a_lin = warp_argmax(v, lane);
        }
        if (use_lnr) {  // row h-1 of the test=False forward = the test=True forward on context[:, :h]
          const float lg = lane < d ? p.logits[((size_t)env * p.logits_T + (h - 1)) * d + lane] : -INFINITY;
          a_lnr = warp_argmax((double)lg, lane);
        }
        while (ci < K && p.sched[ci].x == h) {
          const int k = p.sched[ci].y;
          int a_thmp = 0;
          if (use_thmp) {  // sample=False: n_draws posterior draws, per-arm win counts, the arm with most wins
            int wins = 0;
            for (int base = 0; base < p.n_draws; base += 32) {
              const int draw = base + lane;
              int w = -1;
              if (draw < p.n_draws) {
                double best = -INFINITY;
                const size_t zoff = (((size_t)k * p.n_draws + draw) * N + env) * d;
                for (int b = 0; b < p.nb; ++b) {
                  float z4[4];
                  if (!p.inject_z)
                    normals4(philox_words(p.rk, gid, (uint32_t)(((size_t)k * p.n_draws + draw) * p.nb + b), STREAM_OFFLINE), z4);
#pragma unroll
                  for (int c = 0; c < 4; ++c) {
                    const int j = 4 * b + c;
                    if (j < d) {
                      const double z = p.inject_z ? p.inject_z[zoff + j] : (double)z4[c];
                      if (p.dump_z) p.dump_z[zoff + j] = z;
                      const double v = __dadd_rn(ws.mu[j], __dmul_rn(ws.sd[j], z));   // np.random.normal(means, sqrt(var))
                      if (v > best) best = v, w = j;
                    }
                  }
                }
              }
              for (int j = 0; j < d; ++j) {
                const unsigned bal = __ballot_sync(0xffffffffu, w == j);
                if (lane == j) wins += __popc(bal);
              }
            }
            a_thmp = warp_argmax(lane < d ? (double)wins : -INFINITY, lane);
          }
          if (lane < OE_C && (p.mask >> lane) & 1) {
            const int a_c = lane == DPT_OFFLINE_OPT ? a_opt : lane == DPT_OFFLINE_EMP ? a_emp : lane == DPT_OFFLINE_LCB ? a_lcb
                          : lane == DPT_OFFLINE_THMP ? a_thmp : lane == DPT_OFFLINE_LINREG ? a_lin : a_lnr;
            const double rew = (double)p.means[(size_t)env * d + a_c];
            const double reg = mmax - rew;
            if (p.rewards) p.rewards[((size_t)k * OE_C + lane) * N + env] = rew;
            double* dst = (p.smem_acc ? s_acc : p.sums) + ((size_t)k * OE_C + lane) * 2;
            atomicAdd(dst, reg);
            atomicAdd(dst + 1, reg * reg);
          }
          ++ci;
        }
        __syncwarp();
        hc = ci < K ? p.sched[ci].x : 0;
      }
    }
  }
  if (p.smem_acc) {
    __syncthreads();
    for (int i = tid; i < K * OE_C * 2; i += OE_THREADS)
      if ((p.mask >> ((i >> 1) % OE_C)) & 1) atomicAdd(p.sums + i, s_acc[i]);
  }
}

}  // namespace dpt

using namespace dpt;

extern "C" int dpt_offline_eval(const dpt_offline_params_t* prm, const float* means, const float* ctx_actions,
                                const float* ctx_rewards, double* sums, double* rewards, void* stream) {
  DPT_CHECK_ARG(prm, "dpt_offline_eval: null params");
  const dpt_offline_params_t& q = *prm;
  DPT_CHECK_ARG(q.d >= 1 && q.d <= 32, "dpt_offline_eval: d=%d outside [1,32]", q.d);
  DPT_CHECK_ARG(q.N >= 0 && q.K >= 0, "dpt_offline_eval: N=%d K=%d must be >= 0", q.N, q.K);
  DPT_CHECK_ARG(q.H_stride >= 1, "dpt_offline_eval: H_stride=%d must be >= 1", q.H_stride);
  DPT_CHECK_ARG(q.ctrl_mask > 0 && q.ctrl_mask < (1 << OE_C), "dpt_offline_eval: ctrl_mask=0x%x selects no known slot",
                q.ctrl_mask);
  DPT_CHECK_ARG(q.K == 0 || q.horizons_host, "dpt_offline_eval: null horizons_host");
  int hmax = 0;
  for (int i = 0; i < q.K; ++i) {
    const int h = q.horizons_host[i];
    DPT_CHECK_ARG(h >= 1 && h <= q.H_stride, "dpt_offline_eval: horizon %d (entry %d) outside [1, H_stride=%d]", h, i, q.H_stride);
    hmax = std::max(hmax, h);
  }
  const bool thmp = q.ctrl_mask & (1 << DPT_OFFLINE_THMP), lin = q.ctrl_mask & (1 << DPT_OFFLINE_LINREG);
  const bool lnr = q.ctrl_mask & (1 << DPT_OFFLINE_LNR);
  if (lin) DPT_CHECK_ARG(q.lin_d >= 1 && q.lin_d <= OE_MAX_LD, "dpt_offline_eval: lin_d=%d outside [1,%d]", q.lin_d, OE_MAX_LD);
  if (thmp) {
    DPT_CHECK_ARG(q.n_draws >= 1, "dpt_offline_eval: n_draws=%d must be >= 1", q.n_draws);
    DPT_CHECK_ARG(q.thmp_std > 0.0 && q.thmp_prior_var > 0.0, "dpt_offline_eval: Thompson needs std > 0 and prior_var > 0");
    const uint64_t nb = (uint64_t)(q.d + 3) / 4;
    DPT_CHECK_ARG((uint64_t)q.K * (uint64_t)q.n_draws * nb <= 0xFFFFFFFFull,
                  "dpt_offline_eval: K * n_draws * ceil(d/4) exceeds the 32-bit Philox index");
  }
  if (lnr) DPT_CHECK_ARG(q.logits_T >= hmax, "dpt_offline_eval: logits_T=%d < largest horizon %d", q.logits_T, hmax);
  if (q.N == 0 || q.K == 0) return DPT_OK;
  DPT_CHECK_ARG(means && sums, "dpt_offline_eval: null means / sums");
  DPT_CHECK_ARG(!(thmp || lin || (q.ctrl_mask & ((1 << DPT_OFFLINE_EMP) | (1 << DPT_OFFLINE_LCB)))) || (ctx_actions && ctx_rewards),
                "dpt_offline_eval: null ctx_actions / ctx_rewards");
  DPT_CHECK_ARG(!lin || q.arms, "dpt_offline_eval: LinReg needs arms");
  DPT_CHECK_ARG(!lnr || q.learner_logits, "dpt_offline_eval: null learner_logits");

  // the horizons in ascending order (ties: slot order), as (horizon, slot) pairs
  std::vector<int2> sched(q.K);
  for (int i = 0; i < q.K; ++i) sched[i] = make_int2(q.horizons_host[i], i);
  std::stable_sort(sched.begin(), sched.end(), [](const int2& a, const int2& b) { return a.x < b.x; });

  OffParams p{};
  p.means = means, p.ctx_a = ctx_actions, p.ctx_r = ctx_rewards;
  p.N = q.N, p.d = q.d, p.Hs = q.H_stride, p.K = q.K, p.Hmax = hmax;
  p.mask = q.ctrl_mask;
  p.lcb_c = q.lcb_const, p.std2 = q.thmp_std * q.thmp_std, p.prior_mean = q.thmp_prior_mean, p.prior_var = q.thmp_prior_var;
  p.lin_c = q.linreg_const;
  p.n_draws = q.n_draws, p.nb = (q.d + 3) / 4;
  p.arms = q.arms, p.lin_d = lin ? q.lin_d : 0;
  p.logits = q.learner_logits, p.logits_T = q.logits_T;
  p.rk = round_keys(Key{(uint32_t)q.seed, (uint32_t)(q.seed >> 32)});
  p.env_id0 = q.env_id0;
  p.inject_z = q.inject_z, p.dump_z = q.dump_z;
  p.sums = sums, p.rewards = rewards;

  cudaStream_t st = (cudaStream_t)stream;
  const size_t base = sizeof(OffWarp) * OE_WARPS + sizeof(double) * 32 * OE_MAX_LD;
  const size_t acc = sizeof(double) * (size_t)q.K * OE_C * 2;
  p.smem_acc = acc <= 96 * 1024;   // larger horizon lists accumulate straight into `sums`
  const size_t smem = base + (p.smem_acc ? acc : 0);
  if (smem > 48 * 1024) DPT_CUDA(cudaFuncSetAttribute(offline_eval_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  int per_sm = 0;
  DPT_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, offline_eval_kernel, OE_THREADS, smem));
  const long want = ((long)q.N + OE_WARPS - 1) / OE_WARPS, cap = (long)std::max(per_sm, 1) * sm_count();
  const int grid = (int)std::min(want, cap);

  keep_pool_memory();
  int2* d_sched = nullptr;
  cudaError_t e = cudaMallocAsync(reinterpret_cast<void**>(&d_sched), sizeof(int2) * q.K, st);
  if (e == cudaSuccess) e = cudaMemcpyAsync(d_sched, sched.data(), sizeof(int2) * q.K, cudaMemcpyHostToDevice, st);
  if (e == cudaSuccess) {
    p.sched = d_sched;
    offline_eval_kernel<<<grid, OE_THREADS, smem, st>>>(p);
    e = cudaGetLastError();
  }
  if (d_sched) cudaFreeAsync(d_sched, st);
  if (e != cudaSuccess) {
    set_error("dpt_offline_eval: %s", cudaGetErrorString(e));
    return DPT_ERR_CUDA;
  }
  return DPT_OK;
}
