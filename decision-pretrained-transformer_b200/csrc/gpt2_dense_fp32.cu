// Dense Transformer.forward(x) in fp32 on the CUDA cores (precision = 0, sequences of <= 512 tokens).
//
// Same decomposition as the tensor-core kernel (gpt2_dense.cu) -- one CTA per sequence, thread t owns token
// row t, residual stream in fp32 registers -- but every contraction is fp32 FFMA2 (fma.rn.f32x2) so the
// result meets the 1e-5 logit bar against the reference.  The layer's weights (48 KB fp32) and the
// sequence's K and V (2 x 16 KB) live in shared memory; a thread's matvec reads weight rows as broadcast
// LDS.128 (all threads of a warp read the same address) and keeps 32 outputs in registers.  Attention is a
// per-row online softmax over the keys <= t (K/V rows broadcast from shared memory).  Compared with the
// token-sequential kernel there is no K/V traffic to HBM and all tokens of a sequence advance in parallel.
//
// SAVE = true is the forward of training (gpt2_train_forward_kernel, called from gpt2_train.cu): the same rows
// (dense_fp32_rows) on the parameter tensors as they are (embed_transition.weight [E, din], pred_actions.weight [du, E]
// instead of the handle's transposed copies), and every row also stores what the backward needs (TrainSave, layout
// TA_* / TF_* in gpt2_model.cuh).  Its logits are bit-identical to SAVE = false.  A training launch covers a population
// of same-shape models: CTA (b, member = blockIdx.y), each member with its own parameters, inputs, logits and save area.
#include "common.cuh"
#include "gpt2_model.cuh"
#include "gpt2_fp32.cuh"

namespace dpt {

// shared memory (floats); the CTA has THREADS = 128 / 256 / 512 threads = token rows
constexpr int DF_WQKV = 0;                     // [32][96]
constexpr int DF_WPROJ = DF_WQKV + 32 * 96;    // [32][32]
constexpr int DF_WFC = DF_WPROJ + 32 * 32;     // [32][128]
constexpr int DF_WFC2 = DF_WFC + 32 * 128;     // [128][32]
constexpr int DF_K = DF_WFC2 + 128 * 32;       // [THREADS][32], then V [THREADS][32]
constexpr int df_floats(int threads) { return DF_K + 2 * threads * 32; }   // 80 KB / 112 KB / 176 KB

// The rows of sequence b.  W is Gpt2Dev (SAVE = false: the handle's transposed embed / pred copies) or TrainW
// (SAVE = true: the parameter tensors); sh gives L, dx, du, din; p the inputs, the output and B, T, Ts, test, share.
// tid = threadIdx.x and b are read by the kernel, which knows the range of threadIdx.x from its launch bounds.
template <int DF_THREADS, bool SAVE, class W, class Sh, class P>
__device__ __forceinline__ void dense_fp32_rows(const int tid, const int b, const W& m, const Sh& sh, const P& p, const TrainSave& sv) {
  constexpr int DF_V = DF_K + DF_THREADS * 32;
  extern __shared__ __align__(16) float sm[];
  const int S = p.T + 1;
  const bool valid = tid < S;
  const int dx = sh.dx, du = sh.du, din = sh.din;

  float x[G_E];
  {
    float tok[32];
#pragma unroll
    for (int i = 0; i < 32; ++i) tok[i] = 0.f;
    if (valid) {
      if (tid == 0) {
        for (int i = 0; i < dx; ++i) tok[i] = p.query[(size_t)b * dx + i];
      } else {
        const size_t row = (size_t)(b / p.share) * p.Ts + (tid - 1);
        for (int i = 0; i < dx; ++i) tok[i] = p.cs[row * dx + i];
        for (int i = 0; i < du; ++i) tok[dx + i] = p.ca[row * du + i];
        for (int i = 0; i < dx; ++i) tok[dx + du + i] = p.cns[row * dx + i];
        tok[2 * dx + du] = p.cr[row];
      }
    }
    if (SAVE && valid) store32_(sv.fin + ((size_t)b * S + tid) * TF_STRIDE + TF_TOK, tok);
#pragma unroll
    for (int c = 0; c < G_E; ++c) x[c] = valid ? __ldg(m.embed_b + c) + __ldg(m.wpe + (size_t)tid * G_E + c) : 0.f;
    for (int i = 0; i < din; ++i) {
      const float tv = tok[i];
#pragma unroll
      for (int c = 0; c < G_E; ++c) {
        const float* e;
        if constexpr (SAVE) e = m.embed_w + c * din + i;
        else e = m.embed_wT + i * G_E + c;
        x[c] = fmaf(tv, __ldg(e), x[c]);
      }
    }
  }

  for (int l = 0; l < sh.L; ++l) {
    const auto& w = m.layer[l];
    float* const rec = SAVE && valid ? sv.act + (((size_t)l * p.B + b) * S + tid) * TA_STRIDE : nullptr;   // SAVE: this row's record
    __syncthreads();   // previous layer's readers of the weights / K / V are done
    {
      auto cp = [&](const float* src, int off, int n) {
        const float4* s4 = reinterpret_cast<const float4*>(src);
        float4* d4 = reinterpret_cast<float4*>(sm + off);
        for (int i = tid; i < n / 4; i += DF_THREADS) d4[i] = __ldg(s4 + i);
      };
      cp(w.attn_w, DF_WQKV, 32 * 96);
      cp(w.proj_w, DF_WPROJ, 32 * 32);
      cp(w.fc_w, DF_WFC, 32 * 128);
      cp(w.fc2_w, DF_WFC2, 128 * 32);
    }
    __syncthreads();
    float y[G_E];
    float2 acc[16];
    // ---- LN1, then k and v rows -> shared memory, q stays in registers ----
    if (SAVE) {
      if (valid) store32_(rec + TA_XIN, x);
      float st[2];
      ln_row_f<true>(x, w.ln1_w, w.ln1_b, y, st);
      if (valid) rec[TA_MU1] = st[0], rec[TA_RS1] = st[1];
    } else {
      ln_row_f(x, w.ln1_w, w.ln1_b, y);
    }
#pragma unroll
    for (int part = 1; part <= 2; ++part) {      // 1: k, 2: v
#pragma unroll
      for (int o = 0; o < 16; ++o) acc[o] = make_float2(__ldg(w.attn_b + part * 32 + 2 * o), __ldg(w.attn_b + part * 32 + 2 * o + 1));
      row_matvec32<G_E>(y, sm + DF_WQKV, 96, part * 32, acc);
      float4* dst = reinterpret_cast<float4*>(sm + (part == 1 ? DF_K : DF_V) + tid * G_E);
#pragma unroll
      for (int o = 0; o < 8; ++o) dst[o] = make_float4(acc[2 * o].x, acc[2 * o].y, acc[2 * o + 1].x, acc[2 * o + 1].y);
      if (SAVE && valid) {
        float4* g4 = reinterpret_cast<float4*>(rec + (part == 1 ? TA_K : TA_V));
#pragma unroll
        for (int o = 0; o < 8; ++o) g4[o] = make_float4(acc[2 * o].x, acc[2 * o].y, acc[2 * o + 1].x, acc[2 * o + 1].y);
      }
    }
    float q[G_E];
#pragma unroll
    for (int o = 0; o < 16; ++o) acc[o] = make_float2(__ldg(w.attn_b + 2 * o), __ldg(w.attn_b + 2 * o + 1));
    row_matvec32<G_E>(y, sm + DF_WQKV, 96, 0, acc);
#pragma unroll
    for (int o = 0; o < 16; ++o) q[2 * o] = acc[o].x * 0.17677669529663687f, q[2 * o + 1] = acc[o].y * 0.17677669529663687f;
    if (SAVE && valid) store32_(rec + TA_Q, q);
    __syncthreads();
    // ---- causal attention of row tid: online softmax over keys 0..tid ----
    {
      float mx = -INFINITY, lsum = 0.f;
#pragma unroll
      for (int o = 0; o < 16; ++o) acc[o] = make_float2(0.f, 0.f);
      const int jmax = __shfl_sync(0xffffffffu, tid, 31);   // last row of this warp: warp-uniform trip count
      for (int j = 0; j <= jmax; ++j) {
        const float4* kr = reinterpret_cast<const float4*>(sm + DF_K + j * G_E);
        float2 d0 = make_float2(0.f, 0.f), d1 = make_float2(0.f, 0.f);
#pragma unroll
        for (int o = 0; o < 8; ++o) {
          const float4 kk = kr[o];
          d0 = ffma2_(make_float2(q[4 * o], q[4 * o + 1]), make_float2(kk.x, kk.y), d0);
          d1 = ffma2_(make_float2(q[4 * o + 2], q[4 * o + 3]), make_float2(kk.z, kk.w), d1);
        }
        const float s = (d0.x + d0.y) + (d1.x + d1.y);
        if (j <= tid) {
          if (s > mx) {   // rescale only when the running maximum moves
            const float sc = expf(mx - s);
            lsum *= sc;
#pragma unroll
            for (int o = 0; o < 16; ++o) acc[o].x *= sc, acc[o].y *= sc;
            mx = s;
          }
          const float pr = expf(s - mx);
          lsum += pr;
          const float2 pp = make_float2(pr, pr);
          const float4* vr = reinterpret_cast<const float4*>(sm + DF_V + j * G_E);
#pragma unroll
          for (int o = 0; o < 8; ++o) {
            const float4 vv = vr[o];
            acc[2 * o] = ffma2_(pp, make_float2(vv.x, vv.y), acc[2 * o]);
            acc[2 * o + 1] = ffma2_(pp, make_float2(vv.z, vv.w), acc[2 * o + 1]);
          }
        }
      }
      const float inv = 1.0f / lsum;
#pragma unroll
      for (int o = 0; o < 16; ++o) y[2 * o] = acc[o].x * inv, y[2 * o + 1] = acc[o].y * inv;
      if (SAVE && valid) store32_(rec + TA_O, y), rec[TA_LSE] = mx + logf(lsum);
    }
    // ---- x += o Wproj + b ----
#pragma unroll
    for (int o = 0; o < 16; ++o) acc[o] = make_float2(__ldg(w.proj_b + 2 * o), __ldg(w.proj_b + 2 * o + 1));
    row_matvec32<G_E>(y, sm + DF_WPROJ, 32, 0, acc);
#pragma unroll
    for (int o = 0; o < 16; ++o) x[2 * o] += acc[o].x, x[2 * o + 1] += acc[o].y;
    // ---- MLP: 4 slices of 32 hidden units, each consumed by fc2 as soon as it is activated ----
    if (SAVE) {
      if (valid) store32_(rec + TA_XMID, x);
      float st[2];
      ln_row_f<true>(x, w.ln2_w, w.ln2_b, y, st);
      if (valid) rec[TA_MU2] = st[0], rec[TA_RS2] = st[1];
    } else {
      ln_row_f(x, w.ln2_w, w.ln2_b, y);
    }
    float2 out2[16];
#pragma unroll
    for (int o = 0; o < 16; ++o) out2[o] = make_float2(__ldg(w.fc2_b + 2 * o), __ldg(w.fc2_b + 2 * o + 1));
#pragma unroll 1
    for (int part = 0; part < 4; ++part) {
#pragma unroll
      for (int o = 0; o < 16; ++o) acc[o] = make_float2(__ldg(w.fc_b + part * 32 + 2 * o), __ldg(w.fc_b + part * 32 + 2 * o + 1));
      row_matvec32<G_E>(y, sm + DF_WFC, 128, part * 32, acc);
      if (SAVE && valid) {
        float4* h4 = reinterpret_cast<float4*>(rec + TA_H + part * 32);
#pragma unroll
        for (int o = 0; o < 8; ++o) h4[o] = make_float4(acc[2 * o].x, acc[2 * o].y, acc[2 * o + 1].x, acc[2 * o + 1].y);
      }
      float g[G_E];
#pragma unroll
      for (int o = 0; o < 16; ++o) g[2 * o] = gelu_new_f(acc[o].x), g[2 * o + 1] = gelu_new_f(acc[o].y);
      row_matvec32<G_E>(g, sm + DF_WFC2 + part * 32 * G_E, 32, 0, out2);
    }
#pragma unroll
    for (int o = 0; o < 16; ++o) x[2 * o] += out2[o].x, x[2 * o + 1] += out2[o].y;
  }

  if (SAVE && valid) {   // final residual and ln_f statistics of every row (rows without logits get gradient 0 there)
    float* f = sv.fin + ((size_t)b * S + tid) * TF_STRIDE;
    store32_(f + TF_X, x);
    float y[G_E], st[2];
    ln_row_f<true>(x, m.lnf_w, m.lnf_b, y, st);
    f[TF_MU] = st[0], f[TF_RS] = st[1];
  }
  if (p.test ? (tid == p.T) : (tid >= 1 && tid <= p.T)) {
    float y[G_E];
    ln_row_f(x, m.lnf_w, m.lnf_b, y);
    float* o = p.test ? p.out + (size_t)b * du : p.out + ((size_t)b * p.T + (tid - 1)) * du;
    for (int j = 0; j < du; ++j) {
      float lg = __ldg(m.pred_b + j);
#pragma unroll
      for (int c = 0; c < G_E; ++c) {
        const float* e;
        if constexpr (SAVE) e = m.pred_w + j * G_E + c;
        else e = m.pred_wT + c * du + j;
        lg = fmaf(y[c], __ldg(e), lg);
      }
      o[j] = lg;
    }
  }
}

// inference (dpt_gpt2_forward, precision 0): one CTA per sequence
template <int DF_THREADS, bool SAVE = false>
__global__ void __launch_bounds__(DF_THREADS) gpt2_dense_fp32_kernel(const DenseParams p, const TrainSave sv = TrainSave{}) {
  static_assert(!SAVE, "the forward of training is gpt2_train_forward_kernel");
  dense_fp32_rows<DF_THREADS, false>(threadIdx.x, blockIdx.x, p.m, p.m, p, sv);
}

// the forward of training: CTA (b, member), member = blockIdx.y reads its own parameters, inputs, logits and save area
template <int DF_THREADS, int NM>
__global__ void __launch_bounds__(DF_THREADS) gpt2_train_forward_kernel(const __grid_constant__ TrainFwdParams<NM> p) {
  const TrainFwdMember& mb = p.mem[NM == 1 ? 0 : blockIdx.y];
  struct {
    const float *query, *cs, *ca, *cns, *cr;
    float* out;
    int B, T, Ts, test, share;
  } io{mb.query, mb.cs, mb.ca, mb.cns, mb.cr, mb.out, p.B, p.T, p.Ts, p.test, 1};
  dense_fp32_rows<DF_THREADS, true>(threadIdx.x, blockIdx.x, mb.w, p, io, mb.sv);
}

template <int THREADS>
static cudaError_t launch_df(const DenseParams& p, cudaStream_t st) {
  const int smem = df_floats(THREADS) * (int)sizeof(float);
  cudaError_t e = cudaFuncSetAttribute(gpt2_dense_fp32_kernel<THREADS>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
  if (e != cudaSuccess) return e;
  gpt2_dense_fp32_kernel<THREADS><<<p.B, THREADS, smem, st>>>(p);
  return cudaGetLastError();
}

int gpt2_dense_fp32_launch(const DenseParams& p, cudaStream_t st) {
  const int S = p.T + 1;
  cudaError_t e = S <= 128 ? launch_df<128>(p, st) : S <= 256 ? launch_df<256>(p, st) : launch_df<512>(p, st);
  if (e != cudaSuccess) {
    set_error("gpt2_dense_fp32 launch failed: %s", cudaGetErrorString(e));
    return DPT_ERR_CUDA;
  }
  return DPT_OK;
}

template <int THREADS, int NM>
static cudaError_t launch_train_fwd(const TrainFwdParams<NM>& p, int n, cudaStream_t st) {
  const int smem = df_floats(THREADS) * (int)sizeof(float);
  cudaError_t e = cudaFuncSetAttribute(gpt2_train_forward_kernel<THREADS, NM>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
  if (e != cudaSuccess) return e;
  gpt2_train_forward_kernel<THREADS, NM><<<dim3(p.B, n), THREADS, smem, st>>>(p);
  return cudaGetLastError();
}

template <int NM>
int gpt2_train_forward_launch(const TrainFwdParams<NM>& p, int n, cudaStream_t st) {
  const int S = p.T + 1;
  cudaError_t e = S <= 128 ? launch_train_fwd<128>(p, n, st) : S <= 256 ? launch_train_fwd<256>(p, n, st)
                                                                         : launch_train_fwd<512>(p, n, st);
  if (e != cudaSuccess) {
    set_error("gpt2_train_forward launch failed: %s", cudaGetErrorString(e));
    return DPT_ERR_CUDA;
  }
  return DPT_OK;
}
template int gpt2_train_forward_launch<1>(const TrainFwdParams<1>&, int, cudaStream_t);
template int gpt2_train_forward_launch<TRAIN_POP_MAX>(const TrainFwdParams<TRAIN_POP_MAX>&, int, cudaStream_t);

}  // namespace dpt
