/*
 * dpt_b200.h -- C ABI of the B200-native DPT rollout hot path (libdpt_b200.so).
 *
 * The reference (titanium-47/decision-pretrained-transformer) is 100 % Python and has no
 * FFI layer; the drop-in boundary is its duck-typed Python API (SURVEY.md §8b).  This header
 * is the thin C ABI the Python mirror classes call through ctypes.  Every entry point cites
 * the reference interface it replaces (file:line relative to the reference root).
 *
 * Conventions
 *   - all pointers are DEVICE pointers unless the name ends in _host; buffers are owned by
 *     the caller (PyTorch); the library never allocates except opaque model handles;
 *   - `stream` is a cudaStream_t passed as void*; all work is enqueued asynchronously on it,
 *     there are no hidden synchronisations;
 *   - return value: 0 = ok, <0 = error (DPT_ERR_*); dpt_last_error() gives a thread-local
 *     message; nothing throws or aborts;
 *   - context tensors use the reference consumer's fp32 layout (dataset.py:54-61,
 *     utils.py:193-197): [N,H,dx], [N,H,du], [N,H,dx], [N,H,1] row-major;
 *   - randomness: Philox4x32-10, key = seed, counter = (index, env_lo, env_hi, stream) with the
 *     GLOBAL env id (env_id0 + i), so results do not depend on launch geometry or on how the
 *     env range is sharded over GPUs.  Every randomised entry point has an `inject` argument
 *     (consume caller-provided noise instead -- used for parity against the reference) and a
 *     `dump` argument (write out the noise that was used).
 */
#ifndef DPT_B200_H
#define DPT_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DPT_OK 0
#define DPT_ERR_INVALID_ARG (-1)
#define DPT_ERR_CUDA (-2)
#define DPT_ERR_UNSUPPORTED (-3)

#define DPT_ABI_VERSION 9

/* reward_type of the bandit entry points (envs/bandit_env.py:56-63, envs/gpu_bandit_env.py:53-63):
 * 0 'uniform'  : r = means[a] + var * z, z ~ N(0,1);
 * 1 'bernoulli': r = (u < means[a]) ? 1 : 0, u ~ U[0,1) (24 bits); injected / dumped `z` arrays then hold u. */
#define DPT_REWARD_GAUSSIAN 0
#define DPT_REWARD_BERNOULLI 1
#define DPT_MAX_PEERS 16

int dpt_version(void);
const char* dpt_last_error(void);
/* sm count / compute capability of the current device (fails loudly if there is none). */
int dpt_device_info(int* sm_count, int* cc_major, int* cc_minor);

/* ---------------------------------------------------------------- E1: task draw ------------
 * envs/bandit_env.py:10-18 (sample) + :29-34 (BanditEnv.__init__ argmax / one-hot) and
 * envs/gpu_bandit_env.py:18-28.  means ~ U[0,1)^d (24-bit, fp32-exact).
 * opt_a_index [N] int32 and opt_a [N,d] fp32 one-hot may be NULL. */
int dpt_bandit_sample_means(uint64_t seed, uint64_t env_id0, int N, int d, float* means,
                            int32_t* opt_a_index, float* opt_a, void* stream);
/* argmax / one-hot for caller-provided means (BanditEnv.__init__, LinearBanditEnv.__init__ :162-165). */
int dpt_bandit_opt_action(const float* means, int N, int d, int32_t* opt_a_index, float* opt_a, void* stream);

/* ---------------------------------------------------------------- R1: rollin_bandit --------
 * collect_data.py:23-53 fused with envs/bandit_env.py:56-64 (transit) for N envs x H steps.
 * inject: either `actions` (int32 [N,H]) or all of (cov_idx [N], dir_probs f64 [N,d],
 * rand_idx [N], u f64 [N,H]); `z` fp32 [N,H] always.  dump: any subset, NULL = skip.
 * return_stats: NULL or f64 [3], += (sum of rewards, sum of squared rewards, number of pulls of
 * the optimal arm) over all N*H env-steps (caller zeroes it; atomics, so shards may share it) --
 * the small per-shard statistic that is gathered over NCCL in the multi-GPU collection. */
typedef struct {
  const int32_t* cov_idx;
  const double* dir_probs;
  const int32_t* rand_idx;
  const double* u;
  const int32_t* actions;
  const float* z;
} dpt_bandit_inject_t;

typedef struct {
  int32_t* cov_idx;
  double* dir_probs;
  int32_t* rand_idx;
  double* u;
  int32_t* actions;
  float* z;
} dpt_bandit_dump_t;

int dpt_bandit_rollin(const float* means, float var, int reward_type, uint64_t seed, uint64_t env_id0, int N, int H, int d,
                      float* ctx_states, float* ctx_actions, float* ctx_next_states, float* ctx_rewards,
                      double* return_stats, const dpt_bandit_inject_t* inject, const dpt_bandit_dump_t* dump,
                      void* stream);

/* Multi-GPU form: the same launch, plus an all-gather of the three return statistics over NVLink peer memory without a
 * collective: a one-warp kernel enqueued behind the rollin launch stores return_stats[0..2] to peer_dst[r][0..2] for
 * r < n_peers with system-scope stores (peer_dst: HOST array of device pointers, normally slot `rank` of every rank's
 * gather buffer, opened with dpt_peer_buffer_open; one of them may be this rank's own buffer).  return_stats must be zero
 * before the launch (it holds this launch's totals only).  done_counter: unused (round 1's in-kernel protocol), may be
 * NULL.  No host synchronisation; readers must order themselves after all ranks' launches (stream sync + barrier). */
int dpt_bandit_rollin_p2p(const float* means, float var, uint64_t seed, uint64_t env_id0, int N, int H, int d,
                          float* ctx_states, float* ctx_actions, float* ctx_next_states, float* ctx_rewards,
                          double* return_stats, double* const* peer_dst, int n_peers, unsigned int* done_counter,
                          void* stream);
/* Buffers other ranks' kernels may write: cudaMalloc + CUDA IPC handle (64 bytes) / open in a peer process. */
int dpt_peer_buffer_create(uint64_t bytes, void** dev_ptr, unsigned char handle[64]);
int dpt_peer_buffer_open(const unsigned char handle[64], void** dev_ptr);
int dpt_peer_buffer_close(void* dev_ptr);
int dpt_peer_buffer_destroy(void* dev_ptr);
int dpt_peer_buffer_read(const void* dev_ptr, void* host_dst, uint64_t bytes, void* stream);  /* D2H + stream sync */
int dpt_peer_buffer_zero(void* dev_ptr, uint64_t bytes, void* stream);  /* cudaMemsetAsync through a (peer) mapping:
                                                                         * what a rank with an empty env shard publishes */
/* Protocol notes for dpt_bandit_rollin_p2p / the peer buffers (reference: none -- the reference is single-process):
 *  - a slot may be re-used only after every rank has read it: order readers with stream-sync + barrier BEFORE the
 *    read and a second barrier AFTER it (dist.collect_bandit_sharded does both). */

/* Host-buffer form of the same call (the e2e path): means_host [N,d] in, the four context
 * arrays out, all HOST pointers (pinned for full speed).  Uses `scratch` (device, at least
 * dpt_bandit_rollin_host_scratch_bytes(...) bytes) for double-buffered chunks so the D2H copies
 * overlap the kernel; the constant state columns (bandit state == [1]) are written by host threads
 * instead of crossing PCIe, and a self-balancing share of the chunks comes back as arm index + reward (5 B per step)
 * and is expanded to the one-hot fp32 layout by the same host threads.  Results are
 * identical whichever way a chunk travels.  Synchronises `stream` before returning. */
uint64_t dpt_bandit_rollin_host_scratch_bytes(int N, int H, int d);
int dpt_bandit_rollin_host(const float* means_host, float var, uint64_t seed, uint64_t env_id0, int N, int H, int d,
                           float* ctx_states_host, float* ctx_actions_host, float* ctx_next_states_host,
                           float* ctx_rewards_host, void* scratch, uint64_t scratch_bytes, void* stream);
/* The same collection in the reference's OWN host dtypes (collect_data.py:23-53: states / next_states int64, one-hot
 * actions and rewards float64; [N,H,1], [N,H,d], [N,H,1], [N,H] row-major) -- what collect_data.generate_bandit_histories
 * hands to its callers.  Only 5 B per env-step cross PCIe (arm index + fp32 reward, staged inside the output arrays);
 * the host cores expand them (64 B per env-step of stores).  The arrays may be pageable. */
int dpt_bandit_rollin_host_f64(const float* means_host, float var, uint64_t seed, uint64_t env_id0, int N, int H, int d,
                               int64_t* ctx_states_host, double* ctx_actions_host, int64_t* ctx_next_states_host,
                               double* ctx_rewards_host, void* scratch, uint64_t scratch_bytes, void* stream);
/* Bytes that crossed PCIe device->host in this thread's last dpt_bandit_rollin_host call (the pipeline returns a
 * self-balancing share of the chunks as arm index + reward, 5 B per step, and expands them on the host cores). */
uint64_t dpt_bandit_rollin_host_last_d2h_bytes(void);
/* Measurement aid for the e2e roofline (no reference counterpart): GB/s that `n_threads` host threads (0 = every
 * core this process may run on) reach with non-temporal stores into `dst` (NULL: an internal buffer) of `bytes`
 * bytes, best of three passes after a first-touch pass.  The host half of dpt_bandit_rollin_host is such a stream. */
double dpt_host_write_peak(void* dst, uint64_t bytes, int n_threads);

/* ---------------------------------------------------------------- R3/R4: rollin_mdp --------
 * collect_data.py:83-111 (rollin_mdp) fused with envs/darkroom_env.py:37-55 (transit), :69-82
 * (opt_action), :96-111 (permuted variant) and collect_data.py:200-201 (query state + optimal
 * action, n_samples per env).  goals int32 [N,2]; perm_index int32 [N] or NULL;
 * mode 0 = 'uniform', 1 = 'expert'. */
typedef struct {
  const int32_t* states;   /* [N,H,2]  (uniform mode) */
  const int32_t* actions;  /* [N,H]    (uniform mode) */
  const int32_t* query;    /* [N,S,2] */
} dpt_darkroom_inject_t;

typedef struct {
  int32_t* states;
  int32_t* actions;
  int32_t* query;
} dpt_darkroom_dump_t;

int dpt_darkroom_rollin(const int32_t* goals, const int32_t* perm_index, int dim, int mode, uint64_t seed,
                        uint64_t env_id0, int N, int H, int n_samples, float* ctx_states, float* ctx_actions,
                        float* ctx_next_states, float* ctx_rewards, float* query_states, float* optimal_actions,
                        const dpt_darkroom_inject_t* inject, const dpt_darkroom_dump_t* dump, void* stream);

/* One batched transition: DarkroomEnvVec.step (envs/darkroom_env.py:126-133 -> :57-64 -> :37-55).
 * states int32 [N,2], actions fp32 one-hot [N,5] -> next_states int32 [N,2], rewards int32 [N]. */
int dpt_darkroom_step(const int32_t* states, const float* actions, const int32_t* goals, const int32_t* perm_index,
                      int dim, int N, int32_t* next_states, int32_t* rewards, void* stream);
/* Batched DarkroomEnv.opt_action (envs/darkroom_env.py:69-82, :105-111): fp32 one-hot [N,5]. */
int dpt_darkroom_opt_action(const int32_t* states, const int32_t* goals, const int32_t* perm_index, int N,
                            float* actions, void* stream);

/* Policy rollout of one darkroom episode from a per-env logits table (SURVEY.md §8(f) row 1:
 * DarkroomEnvVec.deploy_eval + DarkroomTransformerController.act, envs/darkroom_env.py:151-175,
 * ctrls/ctrl_darkroom.py:35-66).  Within an episode the context is fixed, so the controller's logits
 * depend only on the query state: logits [N, dim*dim, 5] holds them for every state (index x*dim+y).
 * Each env starts at (0,0) and runs `horizon` steps: softmax (float64) + categorical draw (sample != 0;
 * uniforms from Philox or inject_u f64 [horizon,N]) or argmax, then the grid transition.  Outputs are the
 * episode's fp32 context rows [N,horizon,.] and returns [N] (sum of rewards, nullable). */
int dpt_darkroom_policy_rollout(const float* logits, const int32_t* goals, const int32_t* perm_index, int dim,
                                int horizon, int sample, uint64_t seed, uint64_t env_id0, int64_t episode, int N,
                                float* states, float* actions, float* next_states, float* rewards, float* returns,
                                const double* inject_u, double* dump_u, void* stream);

/* ---------------------------------------------------------------- E5: GPUBanditEnv.step ----
 * envs/gpu_bandit_env.py:53-63 (transit) in one launch: a = argmax(actions), r = means[a] +
 * var * z (type 0, 'uniform') or Bernoulli(means[a]) (type 1).  `step` is the env's step
 * counter (part of the Philox counter).  inject_noise: fp32 [N] standard normals (type 0) or
 * uniforms in [0,1) (type 1); dump_noise likewise. */
int dpt_gpu_bandit_step(const float* means, const float* actions, float var, int type, uint64_t seed,
                        uint64_t env_id0, int64_t step, int N, int d, float* reward, const float* inject_noise,
                        float* dump_noise, void* stream);

/* ---------------------------------------------------------------- K2-K4 stats --------------
 * Per-(env, arm) reward sums and pull counts of an arbitrary context prefix
 * (ctrls/ctrl_bandit.py:95-104, :165-177, :355-364): ctx_actions fp32 [N,Hs,d] (row stride Hs
 * steps, first h used), ctx_rewards fp32 [N,Hs,1] -> sums f64 [N,d], counts int32 [N,d]. */
int dpt_arm_stats(const float* ctx_actions, const float* ctx_rewards, int N, int h, int H_stride, int d,
                  double* sums, int32_t* counts, void* stream);
/* Selftest of the online loop's count division (no reference counterpart): counts how many of the `count` pairs
 * (a[i], n[i] >= 1) give a / n != the table-reciprocal + two-FMA-correction quotient the fused loop uses in place of
 * the reference's `b / np.maximum(1, counts)` (ctrls/ctrl_bandit.py:105).  Must be 0. */
int dpt_selftest_div(const double* a, const int32_t* n, int count, int32_t* mismatches, void* stream);
/* Which implementation dpt_online_loop uses for shapes the fast kernels cover (d <= 10; LinUCB: lin_d == 2), for A/B
 * measurements and for the parity test that runs every implementation on the same inputs (no reference counterpart):
 * 0 = automatic (split pipeline -- controller kernel, then context expansion -- or the single fused kernel, by
 * controller kind and batch size), 1 = general kernel, 2 = fused kernel, 3 = split pipeline; -1 = automatic as well
 * (the setting a fresh process starts with).  Returns the previous setting. */
int dpt_debug_online_impl(int impl);

/* ---------------------------------------------------------------- L1: deploy_online_vec ----
 * evals/eval_bandit.py:56-103 fused with BanditEnvVec.deploy/step (envs/bandit_env.py:98-149) and
 * the controller's set_batch_numpy_vec/act_numpy_vec: all H steps in one call and no host synchronisation.  d <= 10 (LinUCB:
 * lin_d == 2) runs either as ONE fused kernel or as a controller kernel followed by a context-expansion kernel (chosen by
 * controller kind and batch size; results are bit-identical), other shapes as one general kernel; every launch goes to `stream`
 * (graph-capturable); scratch (1 B per env-step of arm indices, a few [N] / [H] float64 arrays) is stream-ordered
 * (cudaMallocAsync / cudaFreeAsync on `stream`).
 * ctrl kinds and the reference classes they replace (ctrls/ctrl_bandit.py):
 *   0 OptPolicy :22-38 | 1 EmpMeanPolicy :57-118 (p0 = online flag) | 2 UCBPolicy :318-380 (p0 = const)
 *   3 ThompsonSamplingPolicy sample=True :122-251 (p0 = std, p1 = prior_mean, p2 = prior_var)
 *   4 LinUCBPolicy :447-528 (p0 = const; arms f64 [d,lin_d])
 * Outputs: ctx_* (any may be NULL = not materialised), cum_means fp32 [H,N] (expected reward of
 * the chosen arm, envs/bandit_env.py:151-153), regret_sums f64 [H,4] += over envs of (reg, reg^2,
 * cumreg, cumreg^2) with reg = max(means) - cum_means and cumreg its running sum over steps
 * (evals/eval_bandit.py:169-178: enough for the per-step and cumulative regret mean / sem; NULL =
 * skip; zeroed by the caller; accumulated with atomics; the [H,4] block is what crosses NVLink). */
typedef struct {
  const float* reward_z;     /* [H,N] standard normals, env order per step (eval loop order) */
  const float* ctrl_z;       /* Thompson: [H,N,d] standard normals */
  const int32_t* first_arm;  /* LinUCB: [N] arm pulled at h = 0 */
} dpt_online_inject_t;

typedef struct {
  float* reward_z;
  float* ctrl_z;
  int32_t* first_arm;
} dpt_online_dump_t;

int dpt_online_loop(int ctrl_kind, double p0, double p1, double p2, const float* means, const double* arms,
                    int lin_d, double var, int reward_type, uint64_t seed, uint64_t env_id0, int N, int H, int d,
                    float* ctx_states,
                    float* ctx_actions, float* ctx_next_states, float* ctx_rewards, float* cum_means,
                    double* regret_sums, const dpt_online_inject_t* inject, const dpt_online_dump_t* dump,
                    void* stream);

/* ---------------------------------------------------------------- L2: offline evaluation ----
 * evals/eval_bandit.py:214-335 (offline / offline_graph) and evals/eval_linear_bandit.py:202-330 for a whole horizon list
 * in ONE launch: for every env and every entry k of horizons_host, each selected controller sees the first h = horizons[k]
 * context rows and plays one noise-free pull (BanditEnvVec.deploy_eval, envs/bandit_env.py:115-123: reward = means[a]).
 * The context is read once (one warp per env, horizons visited in ascending order).
 * Slots (bit c of ctrl_mask selects slot c; the output layout always has DPT_OFFLINE_NSLOTS slots):
 *   0 opt    OptPolicy: the first best arm
 *   1 emp    EmpMeanPolicy(online=False): argmax b / max(1, n)
 *   2 lcb    PessMeanPolicy (ctrls/ctrl_bandit.py:255-314): argmax b/max(1,n) - lcb_const/max(1, sqrt(n))
 *   3 thmp   ThompsonSamplingPolicy(sample=False) :122-251: posterior from (thmp_std, prior_mean, prior_var), n_draws
 *            float64 draws mu + sqrt(v) z, argmax of each, the arm that won most often
 *   4 linreg LinUCBPolicy(const = linreg_const) :447-528: arms f64 [d, lin_d], theta = (I + sum_a n_a x_a x_a^T)^-1 sum_a b_a x_a,
 *            value theta.x + c sqrt(x^T Sigma^-1 x)
 *   5 lnr    BanditTransformerController(sample=False): argmax of row h-1 of learner_logits [N, logits_T, d] fp32, the
 *            test=False forward over the full context (row h-1 attends to the same tokens as the test=True forward on
 *            context[:, :h])
 * Every argmax takes the first maximum.  Inputs: means [N,d] fp32, ctx_actions [N,H_stride,d] fp32 one-hot (the arm of a
 * step is the first max of its row), ctx_rewards [N,H_stride] fp32; horizons_host is a HOST array [K], each in [1, H_stride],
 * any order, duplicates allowed.  Outputs: sums f64 [K, NSLOTS, 2] += over envs of (max mean - reward, its square) for the
 * selected slots (zeroed by the caller, accumulated with atomics, so shards may share it; other slots are not written);
 * rewards f64 [K, NSLOTS, N] (NULL = skip; only selected slots are written).  Thompson normals: Philox, key = seed,
 * counter ((k * n_draws + draw) * ceil(d/4) + block, global env id, STREAM 7), 4 normals per block; inject_z / dump_z f64
 * [K, n_draws, N, d] (the reference's np.random.normal order per horizon; local env index).  The (horizon, slot) schedule
 * is copied to stream-ordered device scratch from pageable host memory, so the call is not graph-capturable. */
#define DPT_OFFLINE_OPT 0
#define DPT_OFFLINE_EMP 1
#define DPT_OFFLINE_LCB 2
#define DPT_OFFLINE_THMP 3
#define DPT_OFFLINE_LINREG 4
#define DPT_OFFLINE_LNR 5
#define DPT_OFFLINE_NSLOTS 6

typedef struct {
  int N, d, H_stride, K;
  const int32_t* horizons_host;  /* [K] */
  int ctrl_mask;
  double lcb_const;
  double thmp_std, thmp_prior_mean, thmp_prior_var;
  int n_draws;
  const double* arms;            /* [d, lin_d] */
  int lin_d;
  double linreg_const;
  const float* learner_logits;   /* [N, logits_T, d] */
  int logits_T;
  uint64_t seed, env_id0;
  const double* inject_z;        /* [K, n_draws, N, d] or NULL */
  double* dump_z;                /* [K, n_draws, N, d] or NULL */
} dpt_offline_params_t;

int dpt_offline_eval(const dpt_offline_params_t* params, const float* means, const float* ctx_actions,
                     const float* ctx_rewards, double* sums, double* rewards, void* stream);

/* ---------------------------------------------------------------- M1: Transformer ----------
 * models/net.py:9-60 (GPT2Model trunk with n_head = 1, embed_transition, pred_actions).
 * Weights are fp32 device pointers in the reference state_dict layout; they are repacked once
 * into the handle. */
typedef struct {
  int horizon, state_dim, action_dim, n_layer, n_embd, n_positions;
  const float* wpe;                 /* [n_positions, E] */
  const float* embed_w;             /* embed_transition.weight [E, 2dx+du+1] */
  const float* embed_b;             /* [E] */
  const float* pred_w;              /* pred_actions.weight [du, E] */
  const float* pred_b;              /* [du] */
  const float* lnf_w;
  const float* lnf_b;
  /* per layer arrays of n_layer pointers (HOST arrays of DEVICE pointers) */
  const float* const* ln1_w;
  const float* const* ln1_b;
  const float* const* attn_w;       /* c_attn.weight [E, 3E] */
  const float* const* attn_b;       /* [3E] */
  const float* const* proj_w;       /* attn.c_proj.weight [E, E] */
  const float* const* proj_b;
  const float* const* ln2_w;
  const float* const* ln2_b;
  const float* const* fc_w;         /* mlp.c_fc.weight [E, 4E] */
  const float* const* fc_b;
  const float* const* fc2_w;        /* mlp.c_proj.weight [4E, E] */
  const float* const* fc2_b;
} dpt_gpt2_weights_t;

typedef struct dpt_gpt2 dpt_gpt2_t;

int dpt_gpt2_create(const dpt_gpt2_weights_t* w, dpt_gpt2_t** out, void* stream);
int dpt_gpt2_destroy(dpt_gpt2_t* m);

/* Transformer.forward(x) (models/net.py:41-60): query_states [B,dx], context_* [B,T,.] fp32,
 * context row stride `T_stride` steps (so views context[:, :h] of a [B,H,.] buffer can be passed
 * without a copy, as evals/eval_bandit.py:71-76 does).  test != 0 -> out [B,du] (last position);
 * test == 0 -> out [B,T,du] (positions 1..T).  precision: 0 = fp32 everywhere (1e-5 logit bar);
 * 1 = bf16 (2e-2 bar): sequences of <= 512 tokens run the dense tcgen05 kernels (bf16 operands, fp32
 * accumulation in tensor memory; one 128-token tile, or 2..4 tiles attended flash-style).  With precision 0
 * sequences of <= 512 tokens run the dense fp32 CUDA-core kernel (neither needs a workspace); longer ones
 * the token-sequential kernel with an fp32 / bf16 K/V cache in `workspace`.
 * ctx_share >= 1: consecutive groups of ctx_share sequences share ONE context row (sequence b reads
 * context row b / ctx_share; query_states and out stay per sequence) -- used to evaluate every
 * possible query state of an env against its context in one launch (darkroom policy table).
 * workspace: device scratch of dpt_gpt2_forward_workspace_bytes(m, B, T, precision) bytes (per-sequence K/V). */
uint64_t dpt_gpt2_forward_workspace_bytes(const dpt_gpt2_t* m, int B, int T, int precision);
int dpt_gpt2_forward(dpt_gpt2_t* m, const float* query_states, const float* ctx_states, const float* ctx_actions,
                     const float* ctx_next_states, const float* ctx_rewards, int B, int T, int T_stride, int ctx_share,
                     int test, int precision, float* out, void* workspace, uint64_t workspace_bytes, void* stream);

/* Training (train.py:252-331 with Transformer.forward, models/net.py:41-60): fp32, sequences of <= 512 tokens, the
 * parameter tensors read in place through dpt_gpt2_weights_t (no handle, no repack, no host synchronisation).
 * dpt_gpt2_train_forward computes the same logits as dpt_gpt2_forward(precision = 0), bit for bit, and saves the
 * activations the backward needs in `workspace` (dpt_gpt2_train_workspace_bytes(w, B, T) bytes, 16 B aligned, the same
 * buffer for both calls).  dpt_gpt2_train_backward takes dout, the gradient of the logits ([B,du] if test, else
 * [B,T,du]), and OVERWRITES every gradient of `grads` (transformer.wte is not an input and has none): weight gradients
 * are sums over all B*(T+1) rows reduced in a fixed order (two identical calls give bit-identical gradients); wpe's
 * gradient has n_positions rows, zero past row T.  The context inputs get no gradient.  B = 0 is a no-op.  n_embd != 32,
 * n_layer > 8 and T + 1 > 512 return DPT_ERR_UNSUPPORTED. */
typedef struct {
  float* wpe;
  float* embed_w;
  float* embed_b;
  float* pred_w;
  float* pred_b;
  float* lnf_w;
  float* lnf_b;
  /* per layer arrays of n_layer pointers (HOST arrays of DEVICE pointers), as in dpt_gpt2_weights_t */
  float* const* ln1_w;
  float* const* ln1_b;
  float* const* attn_w;
  float* const* attn_b;
  float* const* proj_w;
  float* const* proj_b;
  float* const* ln2_w;
  float* const* ln2_b;
  float* const* fc_w;
  float* const* fc_b;
  float* const* fc2_w;
  float* const* fc2_b;
} dpt_gpt2_grads_t;

uint64_t dpt_gpt2_train_workspace_bytes(const dpt_gpt2_weights_t* w, int B, int T);
int dpt_gpt2_train_forward(const dpt_gpt2_weights_t* w, const float* query_states, const float* ctx_states,
                           const float* ctx_actions, const float* ctx_next_states, const float* ctx_rewards, int B, int T,
                           int T_stride, int test, float* out, void* workspace, uint64_t workspace_bytes, void* stream);
int dpt_gpt2_train_backward(const dpt_gpt2_weights_t* w, const float* dout, int B, int T, int test,
                            const dpt_gpt2_grads_t* grads, void* workspace, uint64_t workspace_bytes, void* stream);

/* Population training: n_models same-shape models (members share n_layer, state_dim, action_dim and n_positions) trained
 * in the same launches, each exactly as dpt_gpt2_train_forward / dpt_gpt2_train_backward would train it alone: member i's
 * logits and gradients are bit-identical to the one-model calls on its own weights, inputs and dout (same row chunking,
 * same fixed-order sums).  w and grads are arrays of n_models structs; query_states, ctx_*, out and dout are HOST arrays
 * of n_models DEVICE pointers, with the shapes of the one-model calls; B, T, T_stride and test are shared.  The workspace
 * holds one member region after another: dpt_gpt2_train_population_workspace_bytes(w, n_models, B, T) =
 * n_models * dpt_gpt2_train_workspace_bytes(w, B, T) bytes, 16 B aligned, the same buffer for both calls.  The per-member
 * tables travel in the kernel parameters: no host synchronisation, no upload, capturable in a CUDA graph.
 * 1 <= n_models <= DPT_GPT2_POPULATION_MAX per call; n_models = 0 or B = 0 is a no-op.  n_models < 0 or above the limit,
 * null pointers and a member of another shape (the message names the member and the field) return DPT_ERR_INVALID_ARG;
 * n_embd != 32, n_layer > 8 and T + 1 > 512 return DPT_ERR_UNSUPPORTED. */
#define DPT_GPT2_POPULATION_MAX 32
uint64_t dpt_gpt2_train_population_workspace_bytes(const dpt_gpt2_weights_t* w, int n_models, int B, int T);
int dpt_gpt2_train_population_forward(const dpt_gpt2_weights_t* w, int n_models, const float* const* query_states,
                                      const float* const* ctx_states, const float* const* ctx_actions,
                                      const float* const* ctx_next_states, const float* const* ctx_rewards, int B, int T,
                                      int T_stride, int test, float* const* out, void* workspace, uint64_t workspace_bytes,
                                      void* stream);
int dpt_gpt2_train_population_backward(const dpt_gpt2_weights_t* w, int n_models, const float* const* dout, int B, int T,
                                       int test, const dpt_gpt2_grads_t* grads, void* workspace, uint64_t workspace_bytes,
                                       void* stream);

/* Mixed-precision training: the population calls above with a `precision` argument.  precision = 0 runs exactly the
 * fp32 kernels of the calls without _ex (same results, bit for bit).  precision = 1 is bf16 training: bf16 operands at the
 * tensor-core inputs, fp32 accumulation, fp32 LayerNorm, softmax statistics, residual stream and gradient sums.
 * - forward: the tcgen05 dense forward of dpt_gpt2_forward(precision = 1) on the parameter tensors; member i's logits are
 *   bit-identical to dpt_gpt2_forward(precision = 1) on a handle of the same weights.
 * - backward: the attention backward on mma.sync tensor-core products (bf16 in, fp32 out), split over ceil((T+1)/64)
 *   CTAs per sequence; the projection, MLP and LayerNorm backward and every weight-gradient sum in fp32.  Two identical
 *   calls give bit-identical gradients, and member i's equal the one-member call's.
 * Workspace at precision 1: dpt_gpt2_train_population_workspace_bytes_ex(w, n_models, B, T, 1) bytes, 16 B aligned, the
 * same buffer for the forward and the backward.  It is larger than at precision 0: each member region also holds the bf16
 * weight images the forward packs from the parameters (40 KB per layer) and the attention-output gradients of one layer
 * (144 B per row); the two precisions' workspaces are not interchangeable.
 * B = 0 (and n_models = 0) only validates: the same argument checks run, nothing is launched.  precision outside {0, 1},
 * n_embd != 32, n_layer > 8 and T + 1 > 512 return DPT_ERR_UNSUPPORTED with a message; the other errors are those of the
 * calls without _ex.  workspace_bytes_ex returns 0 for arguments it cannot size (as the call without _ex does). */
uint64_t dpt_gpt2_train_population_workspace_bytes_ex(const dpt_gpt2_weights_t* w, int n_models, int B, int T, int precision);
int dpt_gpt2_train_population_forward_ex(const dpt_gpt2_weights_t* w, int n_models, const float* const* query_states,
                                         const float* const* ctx_states, const float* const* ctx_actions,
                                         const float* const* ctx_next_states, const float* const* ctx_rewards, int B, int T,
                                         int T_stride, int test, int precision, float* const* out, void* workspace,
                                         uint64_t workspace_bytes, void* stream);
int dpt_gpt2_train_population_backward_ex(const dpt_gpt2_weights_t* w, int n_models, const float* const* dout, int B, int T,
                                          int test, int precision, const dpt_gpt2_grads_t* grads, void* workspace,
                                          uint64_t workspace_bytes, void* stream);

/* Ordered multi-source sum (the gradient exchange of the data-parallel interactive trainer, train_interactive.py:97-139;
 * the reference is single-GPU): dst[i] = (((src[0][i] + src[1][i]) + ...) + src[M-1][i]) for i < n, fp32, added in
 * source order whatever the launch geometry, so every rank that sums the same M slots gets the same bits.  src is a HOST
 * array of M device pointers; each may be local or a peer mapping opened with dpt_peer_buffer_open (read with ordinary
 * loads).  No source may alias dst.  M = 0 or n = 0 is a no-op; negative M or n and null pointers return
 * DPT_ERR_INVALID_ARG.  The caller orders the call after every writer of the sources (stream sync + barrier). */
int dpt_ordered_sum_f32(const float* const* src, int M, int64_t n, float* dst, void* stream);

/* Fused bandit online loop with the transformer controller: evals/eval_bandit.py:56-103 +
 * ctrls/ctrl_bandit.py:383-444 (BanditTransformerController, sample != 0 -> softmax + categorical
 * draw, else argmax) + env step, with a per-env KV cache (valid because the bandit query token is
 * constant, SURVEY.md §3.3).  kv_cache: device scratch of dpt_gpt2_online_kv_bytes(...) bytes.
 * inject: reward_z [H,N] fp32, ctrl_u f64 [H,N] (uniforms of the categorical draw). */
typedef struct {
  const float* reward_z;
  const double* ctrl_u;
} dpt_gpt2_online_inject_t;

typedef struct {
  float* reward_z;
  double* ctrl_u;
  float* logits;   /* [H,N,du] logits the controller saw at each step */
} dpt_gpt2_online_dump_t;

uint64_t dpt_gpt2_online_kv_bytes(const dpt_gpt2_t* m, int N, int H, int precision);
int dpt_gpt2_online_loop(dpt_gpt2_t* m, const float* means, double var, int reward_type, int sample, uint64_t seed,
                         uint64_t env_id0,
                         int N, int H, int precision, void* kv_cache, uint64_t kv_bytes, float* ctx_states,
                         float* ctx_actions, float* ctx_next_states, float* ctx_rewards, float* cum_means,
                         double* regret_sums, const dpt_gpt2_online_inject_t* inject,
                         const dpt_gpt2_online_dump_t* dump, void* stream);

/* Population evaluation: the online loop of n_models same-shape models (members share n_layer and action_dim, have
 * state_dim == 1 and n_positions >= H) in one launch, on the same tasks and the same noise: member i's outputs are bit for
 * bit those of dpt_gpt2_online_loop(models[i], ...) with the same means, var, reward_type, sample, seed, env_id0, N, H,
 * precision and inject, whichever kernel variant the population's total of n_models * N env-warps selects (regret sums
 * are float64 atomics: equal up to their order of addition).  models, ctx_*, cum_means, regret_sums: HOST arrays of
 * n_models pointers (device pointers with the shapes of the one-model call); a whole array may be NULL, an entry may be
 * NULL where the one-model call allows it, and a member's four context pointers are all NULL or all set.  dump: n_models
 * structs or NULL.  inject is shared by every member.  kv_cache holds n_models regions of
 * dpt_gpt2_online_kv_bytes(models[0], N, H, precision) bytes, one after another.  The per-member tables travel in the
 * kernel parameters: no host synchronisation, no upload, capturable in a CUDA graph.
 * 1 <= n_models <= DPT_GPT2_ONLINE_POPULATION_MAX per call; n_models = 0, N = 0 or H = 0 is a no-op.  n_models outside
 * [0, max], null pointers, a K/V buffer that is too small and a member of another shape (the message names the member and
 * the field) return DPT_ERR_INVALID_ARG. */
#define DPT_GPT2_ONLINE_POPULATION_MAX 16
int dpt_gpt2_online_loop_population(dpt_gpt2_t* const* models, int n_models, const float* means, double var, int reward_type,
                                    int sample, uint64_t seed, uint64_t env_id0, int N, int H, int precision, void* kv_cache,
                                    uint64_t kv_bytes, float* const* ctx_states, float* const* ctx_actions,
                                    float* const* ctx_next_states, float* const* ctx_rewards, float* const* cum_means,
                                    double* const* regret_sums, const dpt_gpt2_online_inject_t* inject,
                                    const dpt_gpt2_online_dump_t* dump, void* stream);

/* One decode step for callers that drive their own loop (the rollout half of train_interactive.py:97-132 /
 * train_explorer_exploiter.py:110-166, where the arm that is pulled is chosen outside): append the token of position
 * `pos` (tokens [N, 2*dx+du+1] = [state | action | next_state | reward]; position 0 is the query token
 * [query_state, 0, ...], models/net.py:45-53) to every sequence's K/V cache and write the logits at that position
 * (= Transformer.forward(...)[:, -1] over the pos transitions appended so far) to logits [N, du].  Positions must be
 * appended in order 0, 1, 2, ...; kv_cache as for dpt_gpt2_online_loop: dpt_gpt2_online_kv_bytes(m, N, T_max, precision). */
int dpt_gpt2_decode_step(dpt_gpt2_t* m, const float* tokens, int N, int pos, int T_max, int precision, void* kv_cache,
                         uint64_t kv_bytes, float* logits, void* stream);

/* ---------------------------------------------------------------- (f)4: explorer / exploiter rollout ----
 * The no-grad half of an episode of train_explorer_exploiter.py:110-166 in ONE launch (fp32, K/V-cached, one cache per
 * model): per step t both models score the context so far; the explorer's sampled arm is RECORDED in the context
 * (:131-136, :155) while the env is stepped with a uniformly random arm (:137-152); advantages[n, t-1] =
 * CE(exploiter logits_t, optimal arm) - CE(exploiter logits_{t-1}, optimal arm) (:158-164).  As published the reference
 * raises IndexError at t = 0 (its test=False models return preds[:, 1:, :] of an empty context); here, as in
 * GPUBanditEnv.rollout_explorer_exploiter's step-by-step form, position 0 is the query token.  Outputs: ctx_* fp32
 * [N,K,.], advantages fp32 [N,K-1].  Draws are Philox (global env id, step); inject / dump: ctrl_u f64 [K,N] (the
 * explorer's categorical uniforms), random_arm int32 [K,N], reward_z fp32 [K,N]; dump only: both models' logits [K,N,du].
 * kv_explorer / kv_exploiter: two distinct scratch buffers of >= max over the models of
 * dpt_gpt2_online_kv_bytes(model, N, K, 0) bytes each. */
typedef struct {
  const double* ctrl_u;
  const int32_t* random_arm;
  const float* reward_z;
} dpt_explore_inject_t;

typedef struct {
  double* ctrl_u;
  int32_t* random_arm;
  float* reward_z;
  float* logits_explorer;
  float* logits_exploiter;
} dpt_explore_dump_t;

int dpt_gpt2_explore_exploit_rollout(dpt_gpt2_t* explorer, dpt_gpt2_t* exploiter, const float* means, double var, int reward_type,
                                     uint64_t seed, uint64_t env_id0, int N, int K, void* kv_explorer, void* kv_exploiter,
                                     uint64_t kv_bytes_each, float* ctx_states, float* ctx_actions, float* ctx_next_states,
                                     float* ctx_rewards, float* advantages, const dpt_explore_inject_t* inject,
                                     const dpt_explore_dump_t* dump, void* stream);

/* ---------------------------------------------------------------- bring-up / regression ----
 * D[128,N] = A[128,K] * B[N,K]^T through tcgen05.mma (bf16 operands, fp32 accumulate in tensor memory):
 * the self-test of the UMMA helpers (descriptors, 128 B swizzle, TMEM loads) used by the dense forward. */
int dpt_debug_umma_gemm(const float* A, const float* B, float* D, int N, int K, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* DPT_B200_H */
