// Training of the GPT-2 (models/net.py:9-60) in fp32 on the CUDA cores, sequences of <= 512 tokens.
//
//   dpt_gpt2_train_forward : the dense fp32 forward (gpt2_dense_fp32.cu, SAVE = true) on the parameter tensors as
//                            they are -- no handle, no repack -- which also stores each row's activations (TA_* / TF_*).
//   dpt_gpt2_train_backward: three launches on the caller's stream.
//     1. gpt2_train_backward_kernel: one CTA per sequence, thread t = token row t (as the forward), layers in reverse.
//        It computes every row's data gradients and writes, per layer and row, the operand pairs of the weight
//        gradients (GR_* / GF_*).  Causal attention is flash-attention-2 style from the saved log-sum-exp:
//        D_i = dO_i . O_i, a query-side pass for dQ (K, V in shared memory) and key-side passes for dV and dK
//        (Q, dO, lse, D in shared memory).
//     2. weight_grad_partial_kernel: every weight gradient is a sum over the B*S rows of an outer product
//        A_r^T G_r (or of A_r * G_r for LayerNorm weights; biases: of G_r).  The rows are cut into NC fixed chunks;
//        CTA (tile, chunk) writes its 32 x 32 tile's chunk sum to slot `chunk` of the partial buffer.
//     3. weight_grad_reduce_kernel sums the NC slots in chunk order into the gradient tensors; wpe_grad_kernel sums
//        the position gradients over the batch in sequence order (rows past T are zero).
//   Every sum has a fixed order, so two identical calls give bit-identical gradients.
//
// Population training (dpt_gpt2_train_population_*): n same-shape models in the same launches.  Every kernel takes its
// member from the grid (forward / backward: blockIdx.y, partial sums and reduction: blockIdx.z, wpe: blockIdx.y); member i
// uses workspace region i (train_layout(...).total floats each) and its own pointer table in the kernel parameters.  The
// chunking depends on B and T only, so each member runs exactly the arithmetic of the one-model call; the one-model entry
// points are the n = 1 case (kernels instantiated with a member capacity NM of 1, so their parameter blocks stay small).
//
// bf16 training (precision = 1, the *_ex entry points): bf16 operands at the tensor-core inputs, fp32 accumulation,
// LayerNorm, softmax statistics, residual stream, loss, master weights and gradient sums.
//   forward : the weight images of every member and layer are packed from the parameters (pack_train_wimg_kernel), then
//             the tcgen05 dense forward (gpt2_dense.cu, SAVE = true) runs and saves the same fp32 records as the fp32
//             forward of training; its logits are bit-identical to dpt_gpt2_forward(precision = 1).
//   backward: 2 L + 1 launches, then the same weight-gradient reduction as fp32.
//     gpt2_train_rows_bf16_kernel (phase l = L-1 .. -1, one thread per row of all B*S rows): the ln_1 backward of layer
//       l + 1 (from its dq, dk, dv) or, at l = L-1, pred_actions and ln_f; then the MLP / ln_2 backward of layer l and
//       dO = d(attn output), D = rowsum(dO * O), kept in the DOS scratch.  It writes the GR_* / GF_* operands as fp32.
//     gpt2_train_attn_bf16_kernel (layer l): flash-attention-2 backward on mma.sync.m16n8k16 (bf16 in, fp32 out).  CTA
//       (sequence, tile t of 64 rows) computes dq of query tile t over key tiles 0..t and dk, dv of key tile t over query
//       tiles t..nt-1, so a sequence runs on nt = ceil(S / 64) CTAs, each with nt + 1 tile steps, and no sum crosses CTAs.
//   Every sum has a fixed order and no atomics, so two identical calls give bit-identical gradients.
#include <algorithm>

#include <cuda_bf16.h>

#include "common.cuh"
#include "gpt2_model.cuh"
#include "gpt2_fp32.cuh"

namespace dpt {

// per layer and row: what the weight-gradient reduction reads, [L][B][S][GR_STRIDE]
constexpr int GR_DX = 0;       // gradient of the layer's output residual [32]   (G of mlp.c_proj + bias)
constexpr int GR_G = 32;       // gelu_new(h) [128]                                (A of mlp.c_proj)
constexpr int GR_DH = 160;     // gradient of h [128]                              (G of mlp.c_fc + bias)
constexpr int GR_Y2 = 288;     // ln_2 output [32]                                 (A of mlp.c_fc)
constexpr int GR_XH2 = 320;    // ln_2 normalised input [32]                       (A of ln_2.weight)
constexpr int GR_DY2 = 352;    // gradient of the ln_2 output [32]                 (G of ln_2)
constexpr int GR_DXM = 384;    // gradient of the post-attention residual [32]     (G of attn.c_proj + bias)
constexpr int GR_DQKV = 416;   // gradient of q, k, v (unscaled q) [96]            (G of attn.c_attn + bias)
constexpr int GR_Y1 = 512;     // ln_1 output [32]                                 (A of attn.c_attn)
constexpr int GR_XH1 = 544;    // [32]                                             (A of ln_1.weight)
constexpr int GR_DY1 = 576;    // [32]                                             (G of ln_1)
constexpr int GR_STRIDE = 608;
// per row, once: [B][S][GF_STRIDE]
constexpr int GF_DLOG = 0;     // gradient of the logits, zero-padded to 32        (G of pred_actions + bias)
constexpr int GF_YF = 32;      // ln_f output                                      (A of pred_actions)
constexpr int GF_XHF = 64;     // ln_f normalised input                            (A of ln_f.weight)
constexpr int GF_DYF = 96;     // gradient of the ln_f output                      (G of ln_f)
constexpr int GF_DX0 = 128;    // gradient of the embedded token (G of embed_transition + bias, and of wpe)
constexpr int GF_STRIDE = 160;

// backward shared memory (floats): transposed layer weights, then two [THREADS][32] row arrays and [THREADS][2]
constexpr int DB_WQKVT = 0;                      // [96][32]  = attn_w^T
constexpr int DB_WPROJT = DB_WQKVT + 96 * 32;    // [32][32]  = proj_w^T
constexpr int DB_WFCT = DB_WPROJT + 32 * 32;     // [128][32] = fc_w^T
constexpr int DB_WFC2T = DB_WFCT + 128 * 32;     // [32][128] = fc2_w^T
constexpr int DB_X1 = DB_WFC2T + 32 * 128;
constexpr int db_floats(int threads) { return DB_X1 + 2 * threads * 32 + 2 * threads; }   // 84 KB / 120 KB / 184 KB

constexpr float ATT_SCALE = 0.17677669529663687f;   // 1 / sqrt(32)

struct BackMember {   // one member of the population: its parameter tensors, dout and workspace region
  TrainW w;
  const float* dout;
  const float *act, *fin;
  float *grec, *gfin;
};
template <int NM>
struct BackParams {
  int L, du, B, T, test;
  BackMember mem[NM];
};

// dx += d LayerNorm(x)/dx applied to dy, from the normalised input xh, rstd rs and the LN weight w
__device__ __forceinline__ void ln_back_(const float* xh, float rs, const float* dy, const float* w, float* dx) {
  float m1 = 0.f, m2 = 0.f;
#pragma unroll
  for (int c = 0; c < G_E; ++c) {
    const float d = dy[c] * __ldg(w + c);
    m1 += d;
    m2 = fmaf(d, xh[c], m2);
  }
  m1 *= (1.0f / G_E), m2 *= (1.0f / G_E);
#pragma unroll
  for (int c = 0; c < G_E; ++c) dx[c] += rs * (dy[c] * __ldg(w + c) - m1 - xh[c] * m2);
}

__device__ __forceinline__ void acc_to_(const float2* acc, float* v) {
#pragma unroll
  for (int o = 0; o < 16; ++o) v[2 * o] = acc[o].x, v[2 * o + 1] = acc[o].y;
}

__device__ __forceinline__ float dot32_(const float* a, const float* b_sm) {
  const float4* b4 = reinterpret_cast<const float4*>(b_sm);
  float2 d0 = make_float2(0.f, 0.f), d1 = make_float2(0.f, 0.f);
#pragma unroll
  for (int o = 0; o < 8; ++o) {
    const float4 bb = b4[o];
    d0 = ffma2_(make_float2(a[4 * o], a[4 * o + 1]), make_float2(bb.x, bb.y), d0);
    d1 = ffma2_(make_float2(a[4 * o + 2], a[4 * o + 3]), make_float2(bb.z, bb.w), d1);
  }
  return (d0.x + d0.y) + (d1.x + d1.y);
}

// acc[0..31] += s * v_sm[0..31]
__device__ __forceinline__ void axpy32_(float s, const float* v_sm, float2* acc) {
  const float2 ss = make_float2(s, s);
  const float4* v4 = reinterpret_cast<const float4*>(v_sm);
#pragma unroll
  for (int o = 0; o < 8; ++o) {
    const float4 vv = v4[o];
    acc[2 * o] = ffma2_(ss, make_float2(vv.x, vv.y), acc[2 * o]);
    acc[2 * o + 1] = ffma2_(ss, make_float2(vv.z, vv.w), acc[2 * o + 1]);
  }
}

// CTA (b, member = blockIdx.y)
template <int THREADS, int NM>
__global__ void __launch_bounds__(THREADS) gpt2_train_backward_kernel(const __grid_constant__ BackParams<NM> p) {
  extern __shared__ __align__(16) float sm[];
  float* const X1 = sm + DB_X1;
  float* const X2 = sm + DB_X1 + THREADS * 32;
  float* const SV = sm + DB_X1 + 2 * THREADS * 32;
  const BackMember& mb = p.mem[NM == 1 ? 0 : blockIdx.y];
  const TrainW& m = mb.w;
  const int tid = threadIdx.x, b = blockIdx.x;
  const int S = p.T + 1, du = p.du;
  const bool valid = tid < S;
  const int row = valid ? tid : S - 1;   // rows past the sequence load a valid row and store nothing
  const size_t r = (size_t)b * S + row;
  const size_t NR = (size_t)p.B * S;

  float dx[G_E];
  // ---- pred_actions and ln_f ----
  {
    const float* f = mb.fin + r * TF_STRIDE;
    float xh[G_E], dl[G_E], dy[G_E];
    load32_(xh, f + TF_X);
    const float mu = f[TF_MU], rs = f[TF_RS];
#pragma unroll
    for (int c = 0; c < G_E; ++c) xh[c] = (xh[c] - mu) * rs, dl[c] = 0.f, dy[c] = 0.f;
    const bool has_out = p.test ? row == p.T : row >= 1;
    if (has_out) {
      const float* d = p.test ? mb.dout + (size_t)b * du : mb.dout + ((size_t)b * p.T + (row - 1)) * du;
      for (int j = 0; j < du; ++j) {
        const float g = d[j];
        dl[j] = g;
#pragma unroll
        for (int c = 0; c < G_E; ++c) dy[c] = fmaf(g, __ldg(m.pred_w + j * G_E + c), dy[c]);
      }
    }
#pragma unroll
    for (int c = 0; c < G_E; ++c) dx[c] = 0.f;
    ln_back_(xh, rs, dy, m.lnf_w, dx);
    if (valid) {
      float* g = mb.gfin + r * GF_STRIDE;
      store32_(g + GF_DLOG, dl), store32_(g + GF_XHF, xh), store32_(g + GF_DYF, dy);
#pragma unroll
      for (int c = 0; c < G_E; ++c) dl[c] = fmaf(xh[c], __ldg(m.lnf_w + c), __ldg(m.lnf_b + c));
      store32_(g + GF_YF, dl);
    }
  }

  for (int l = p.L - 1; l >= 0; --l) {
    const TrainLayerW& lw = m.layer[l];
    __syncthreads();   // the previous layer's readers of the weights and row arrays are done
    for (int i = tid; i < 32 * 96; i += THREADS) sm[DB_WQKVT + (i % 96) * 32 + i / 96] = __ldg(lw.attn_w + i);
    for (int i = tid; i < 32 * 32; i += THREADS) sm[DB_WPROJT + (i % 32) * 32 + i / 32] = __ldg(lw.proj_w + i);
    for (int i = tid; i < 32 * 128; i += THREADS) sm[DB_WFCT + (i % 128) * 32 + i / 128] = __ldg(lw.fc_w + i);
    for (int i = tid; i < 128 * 32; i += THREADS) sm[DB_WFC2T + (i % 32) * 128 + i / 32] = __ldg(lw.fc2_w + i);
    const float* a = mb.act + ((size_t)l * NR + r) * TA_STRIDE;
    float* g = mb.grec + ((size_t)l * NR + r) * GR_STRIDE;
    if (valid) store32_(g + GR_DX, dx);
    __syncthreads();
    float2 acc[16];
    // ---- MLP: x_out = x_mid + fc2(gelu_new(fc(ln_2(x_mid)))) ----
    float dxm[G_E];   // becomes the gradient of x_mid
    {
      float xh[G_E], dy[G_E];
      load32_(xh, a + TA_XMID);
      const float mu = a[TA_MU2], rs = a[TA_RS2];
#pragma unroll
      for (int c = 0; c < G_E; ++c) xh[c] = (xh[c] - mu) * rs;
      if (valid) {
        float y[G_E];
#pragma unroll
        for (int c = 0; c < G_E; ++c) y[c] = fmaf(xh[c], __ldg(lw.ln2_w + c), __ldg(lw.ln2_b + c));
        store32_(g + GR_Y2, y), store32_(g + GR_XH2, xh);
      }
      float2 dy2[16];
#pragma unroll
      for (int o = 0; o < 16; ++o) dy2[o] = make_float2(0.f, 0.f);
#pragma unroll 1
      for (int part = 0; part < 4; ++part) {
#pragma unroll
        for (int o = 0; o < 16; ++o) acc[o] = make_float2(0.f, 0.f);
        row_matvec32<G_E>(dx, sm + DB_WFC2T, 128, part * 32, acc);   // d gelu(h)
        float h[G_E], dh[G_E];
        load32_(h, a + TA_H + part * 32);
        acc_to_(acc, dh);
#pragma unroll
        for (int c = 0; c < G_E; ++c) {
          const float x = h[c], x2 = x * x;
          const float t = tanhf(0.7978845608028654f * (x + 0.044715f * x2 * x));
          h[c] = 0.5f * x * (1.0f + t);
          const float dg = 0.5f * (1.0f + t) + 0.5f * x * (1.0f - t * t) * 0.7978845608028654f * (1.0f + 3.0f * 0.044715f * x2);
          dh[c] *= dg;
        }
        if (valid) store32_(g + GR_G + part * 32, h), store32_(g + GR_DH + part * 32, dh);
        row_matvec32<G_E>(dh, sm + DB_WFCT + part * 32 * 32, 32, 0, dy2);
      }
      acc_to_(dy2, dy);
      if (valid) store32_(g + GR_DY2, dy);
#pragma unroll
      for (int c = 0; c < G_E; ++c) dxm[c] = dx[c];
      ln_back_(xh, rs, dy, lw.ln2_w, dxm);
    }
    if (valid) store32_(g + GR_DXM, dxm);
    // ---- attention: x_mid = x_in + proj(softmax(q k^T) v) ----
    float dO[G_E];
#pragma unroll
    for (int o = 0; o < 16; ++o) acc[o] = make_float2(0.f, 0.f);
    row_matvec32<G_E>(dxm, sm + DB_WPROJT, 32, 0, acc);
    acc_to_(acc, dO);
    float Dm;
    {
      float o_[G_E];
      load32_(o_, a + TA_O);
      Dm = 0.f;
#pragma unroll
      for (int c = 0; c < G_E; ++c) Dm = fmaf(dO[c], o_[c], Dm);
    }
    const float lse = a[TA_LSE];
    {   // K, V rows -> shared memory
      float t[G_E];
      load32_(t, a + TA_K);
      store32_(X1 + tid * G_E, t);
      load32_(t, a + TA_V);
      store32_(X2 + tid * G_E, t);
    }
    __syncthreads();
    const int jmax = __shfl_sync(0xffffffffu, tid, 31);   // last row of this warp: warp-uniform trip counts
    const int jmin = tid & ~31;                           // first row of this warp
    float dqk[G_E];   // dq (unscaled), later dk
    {
      float q[G_E];
      load32_(q, a + TA_Q);
#pragma unroll
      for (int o = 0; o < 16; ++o) acc[o] = make_float2(0.f, 0.f);
      for (int j = 0; j <= jmax; ++j) {
        const float s = dot32_(q, X1 + j * G_E);
        if (j <= tid) {
          const float pr = expf(s - lse);
          const float ds = pr * (dot32_(dO, X2 + j * G_E) - Dm);
          axpy32_(ds, X1 + j * G_E, acc);
        }
      }
#pragma unroll
      for (int o = 0; o < 16; ++o) dqk[2 * o] = acc[o].x * ATT_SCALE, dqk[2 * o + 1] = acc[o].y * ATT_SCALE;
    }
    if (valid) store32_(g + GR_DQKV, dqk);
    float dy1[G_E];
#pragma unroll
    for (int o = 0; o < 16; ++o) acc[o] = make_float2(0.f, 0.f);
    row_matvec32<G_E>(dqk, sm + DB_WQKVT, 32, 0, acc);
    __syncthreads();   // K, V readers done
    {   // Q, dO, lse, D -> shared memory
      float t[G_E];
      load32_(t, a + TA_Q);
      store32_(X1 + tid * G_E, t);
      store32_(X2 + tid * G_E, dO);
      SV[2 * tid] = lse, SV[2 * tid + 1] = Dm;
    }
    __syncthreads();
    {
      float k[G_E];
      load32_(k, a + TA_K);
      // dv_j = sum_{i >= j} P_ij dO_i
      float2 dv[16];
#pragma unroll
      for (int o = 0; o < 16; ++o) dv[o] = make_float2(0.f, 0.f);
      for (int i = jmin; i < S; ++i) {
        const float s = dot32_(k, X1 + i * G_E);
        if (i >= tid) axpy32_(expf(s - SV[2 * i]), X2 + i * G_E, dv);
      }
      acc_to_(dv, dO);   // dO is not needed any more: it holds dv
      if (valid) store32_(g + GR_DQKV + 64, dO);
      row_matvec32<G_E>(dO, sm + DB_WQKVT + 64 * 32, 32, 0, acc);
      // dk_j = sum_{i >= j} P_ij (dO_i . v_j - D_i) q_i
      float v[G_E];
      load32_(v, a + TA_V);
      float2 dk[16];
#pragma unroll
      for (int o = 0; o < 16; ++o) dk[o] = make_float2(0.f, 0.f);
      for (int i = jmin; i < S; ++i) {
        const float s = dot32_(k, X1 + i * G_E);
        if (i >= tid) {
          const float ds = expf(s - SV[2 * i]) * (dot32_(v, X2 + i * G_E) - SV[2 * i + 1]);
          axpy32_(ds, X1 + i * G_E, dk);
        }
      }
      acc_to_(dk, dqk);
      if (valid) store32_(g + GR_DQKV + 32, dqk);
      row_matvec32<G_E>(dqk, sm + DB_WQKVT + 32 * 32, 32, 0, acc);
    }
    acc_to_(acc, dy1);
    // ---- ln_1 ----
    {
      float xh[G_E];
      load32_(xh, a + TA_XIN);
      const float mu = a[TA_MU1], rs = a[TA_RS1];
#pragma unroll
      for (int c = 0; c < G_E; ++c) xh[c] = (xh[c] - mu) * rs;
      if (valid) {
        float y[G_E];
#pragma unroll
        for (int c = 0; c < G_E; ++c) y[c] = fmaf(xh[c], __ldg(lw.ln1_w + c), __ldg(lw.ln1_b + c));
        store32_(g + GR_Y1, y), store32_(g + GR_XH1, xh), store32_(g + GR_DY1, dy1);
      }
#pragma unroll
      for (int c = 0; c < G_E; ++c) dx[c] = dxm[c];
      ln_back_(xh, rs, dy1, lw.ln1_w, dx);
    }
  }
  if (valid) store32_(mb.gfin + r * GF_STRIDE + GF_DX0, dx);
}

// ---- weight gradients: fixed-chunk partial sums, then a fixed-order reduction ----
struct RJob {
  const float *A, *G;   // row r of the operands at A + r * sa, G + r * sg
  int sa, sg, nin, nout;
  int diag;             // 0: W[i][o] = sum_r A[r][i] G[r][o]; 1: W[c] = sum_r A[r][c] G[r][c] (nin = nout = 32)
  int trans;            // W is stored [nout][nin] (nn.Linear) instead of [nin][nout] (Conv1D)
  int woff, boff;       // flat offsets of the weight and of the bias (sum_r G[r][o]) in a partial slot
};
struct RTile {
  short job, i0, o0;
};
constexpr int R_MAX_JOBS = 6 * G_MAX_L + 3;
constexpr int R_MAX_TILES = 14 * G_MAX_L + 3;
struct RParams {   // the operands of member 0; member z's are at the same offsets in its workspace region (+ z * mstride)
  RJob job[R_MAX_JOBS];
  RTile tile[R_MAX_TILES];
  int NR, CH, P;
  size_t mstride;
  float* part;   // [NC][P]
};
struct RSeg {
  int off, n;
};
constexpr int R_MAX_SEGS = 2 * R_MAX_JOBS;
template <int NM>
struct RSegs {
  RSeg seg[R_MAX_SEGS];
  int NC, P;
  size_t mstride;
  const float* part;
  float* dst[NM][R_MAX_SEGS];   // per member: the gradient tensor of each segment
};
template <int NM>
struct WpeParams {
  const float* gfin;
  size_t mstride;
  int B, S, n_pos;
  float* dwpe[NM];
};
static_assert(sizeof(TrainFwdParams<TRAIN_POP_MAX>) <= 32764 && sizeof(BackParams<TRAIN_POP_MAX>) <= 32764 &&
                  sizeof(RSegs<TRAIN_POP_MAX>) <= 32764 && sizeof(RParams) <= 32764,
              "the per-member tables of TRAIN_POP_MAX members must fit the kernel parameter limit");

// CTA (tile, chunk, member)
__global__ void __launch_bounds__(256) weight_grad_partial_kernel(const RParams p) {
  __shared__ __align__(16) float As[32][32];
  __shared__ __align__(16) float Gs[32][32];
  __shared__ float red[2][8][32];
  const RTile t = p.tile[blockIdx.x];
  const RJob& j = p.job[t.job];
  const int tid = threadIdx.x, chunk = blockIdx.y;
  const size_t moff = (size_t)blockIdx.z * p.mstride;
  const float* const A = j.A + moff;
  const float* const G = j.G + moff;
  const int r0 = chunk * p.CH, r1 = min(p.NR, r0 + p.CH);
  const int lr = tid >> 3, l4 = (tid & 7) * 4;   // loader: row, 4 columns
  const int i = tid >> 3, o4 = (tid & 7) * 4;    // outer product: input i, outputs o4..o4+3
  const int dc = tid & 31, dg = tid >> 5;        // diagonal: column, row group
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f), bacc = acc;
  float dacc = 0.f, dbacc = 0.f;
  for (int rb = r0; rb < r1; rb += 32) {
    const int rr = rb + lr;
    float4 av = make_float4(0.f, 0.f, 0.f, 0.f), gv = av;
    if (rr < r1) {
      av = *reinterpret_cast<const float4*>(A + (size_t)rr * j.sa + t.i0 + l4);
      gv = *reinterpret_cast<const float4*>(G + (size_t)rr * j.sg + t.o0 + l4);
    }
    __syncthreads();
    *reinterpret_cast<float4*>(&As[lr][l4]) = av;
    *reinterpret_cast<float4*>(&Gs[lr][l4]) = gv;
    __syncthreads();
    if (!j.diag) {
#pragma unroll 8
      for (int k = 0; k < 32; ++k) {
        const float a = As[k][i];
        const float4 gg = *reinterpret_cast<const float4*>(&Gs[k][o4]);
        acc.x = fmaf(a, gg.x, acc.x), acc.y = fmaf(a, gg.y, acc.y), acc.z = fmaf(a, gg.z, acc.z), acc.w = fmaf(a, gg.w, acc.w);
        bacc.x += gg.x, bacc.y += gg.y, bacc.z += gg.z, bacc.w += gg.w;
      }
    } else {
#pragma unroll
      for (int k = dg; k < 32; k += 8) dacc = fmaf(As[k][dc], Gs[k][dc], dacc), dbacc += Gs[k][dc];
    }
  }
  float* part = p.part + moff + (size_t)chunk * p.P;
  if (!j.diag) {
    const float v[4] = {acc.x, acc.y, acc.z, acc.w}, bv[4] = {bacc.x, bacc.y, bacc.z, bacc.w};
    const int gi = t.i0 + i;
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const int go = t.o0 + o4 + e;
      if (gi < j.nin && go < j.nout) part[j.woff + (j.trans ? go * j.nin + gi : gi * j.nout + go)] = v[e];
      if (i == 0 && t.i0 == 0 && go < j.nout) part[j.boff + go] = bv[e];
    }
  } else {
    red[0][dg][dc] = dacc, red[1][dg][dc] = dbacc;
    __syncthreads();
    if (tid < 32) {
      float s = 0.f, sb = 0.f;
#pragma unroll
      for (int k = 0; k < 8; ++k) s += red[0][k][tid], sb += red[1][k][tid];
      part[j.woff + tid] = s, part[j.boff + tid] = sb;
    }
  }
}

// CTA (x, segment, member)
template <int NM>
__global__ void __launch_bounds__(256) weight_grad_reduce_kernel(const __grid_constant__ RSegs<NM> s) {
  const RSeg& g = s.seg[blockIdx.y];
  const int mz = NM == 1 ? 0 : blockIdx.z;
  const int e = blockIdx.x * 256 + threadIdx.x;
  if (e >= g.n) return;
  const float* src = s.part + (size_t)mz * s.mstride + g.off + e;
  float acc = 0.f;
  for (int c = 0; c < s.NC; ++c) acc += src[(size_t)c * s.P];
  s.dst[mz][blockIdx.y][e] = acc;
}

// CTA (x, member)
template <int NM>
__global__ void wpe_grad_kernel(const __grid_constant__ WpeParams<NM> p) {
  const int mz = NM == 1 ? 0 : blockIdx.y;
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= p.n_pos * G_E) return;
  const int t = e / G_E, c = e % G_E;
  const float* gfin = p.gfin + (size_t)mz * p.mstride;
  float acc = 0.f;
  if (t < p.S)
    for (int b = 0; b < p.B; ++b) acc += gfin[((size_t)b * p.S + t) * GF_STRIDE + GF_DX0 + c];
  p.dwpe[mz][e] = acc;
}

// ---- bf16 backward (precision 1) ----
constexpr int DOS_STRIDE = 36;   // per row: dO [32] (gradient of the attention output), D = dO . O, pad
// rows kernel shared memory (floats): the transposed weights of the backward kernel, attn_w^T of layer l + 1 first
constexpr int RB_FLOATS = DB_X1;   // 48 KB

template <int NM>
struct Rows16Params {
  BackParams<NM> b;
  float* dos[NM];
  int l;   // phase: layer l's MLP (l >= 0) after layer l + 1's ln_1 (l + 1 < L)
};

// CTA (block of 128 rows, member = blockIdx.y): thread = row r of the B*S rows
template <int NM>
__global__ void __launch_bounds__(128) gpt2_train_rows_bf16_kernel(const __grid_constant__ Rows16Params<NM> p) {
  extern __shared__ __align__(16) float sm[];
  const BackMember& mb = p.b.mem[NM == 1 ? 0 : blockIdx.y];
  const TrainW& m = mb.w;
  const int tid = threadIdx.x, l = p.l, L = p.b.L, du = p.b.du;
  const int S = p.b.T + 1;
  const size_t NR = (size_t)p.b.B * S;
  if (l + 1 < L) {
    const TrainLayerW& u = m.layer[l + 1];
    for (int i = tid; i < 32 * 96; i += 128) sm[DB_WQKVT + (i % 96) * 32 + i / 96] = __ldg(u.attn_w + i);
  }
  if (l >= 0) {
    const TrainLayerW& lw = m.layer[l];
    for (int i = tid; i < 32 * 32; i += 128) sm[DB_WPROJT + (i % 32) * 32 + i / 32] = __ldg(lw.proj_w + i);
    for (int i = tid; i < 32 * 128; i += 128) sm[DB_WFCT + (i % 128) * 32 + i / 128] = __ldg(lw.fc_w + i);
    for (int i = tid; i < 128 * 32; i += 128) sm[DB_WFC2T + (i % 32) * 128 + i / 32] = __ldg(lw.fc2_w + i);
  }
  __syncthreads();
  const size_t r = (size_t)blockIdx.x * 128 + tid;
  if (r >= NR) return;
  const int row = (int)(r % S), b = (int)(r / S);
  float dx[G_E];
  float2 acc[16];
  if (l + 1 == L) {   // ---- pred_actions and ln_f ----
    const float* f = mb.fin + r * TF_STRIDE;
    float xh[G_E], dl[G_E], dy[G_E];
    load32_(xh, f + TF_X);
    const float mu = f[TF_MU], rs = f[TF_RS];
#pragma unroll
    for (int c = 0; c < G_E; ++c) xh[c] = (xh[c] - mu) * rs, dl[c] = 0.f, dy[c] = 0.f;
    const bool has_out = p.b.test ? row == p.b.T : row >= 1;
    if (has_out) {
      const float* d = p.b.test ? mb.dout + (size_t)b * du : mb.dout + ((size_t)b * p.b.T + (row - 1)) * du;
      for (int j = 0; j < du; ++j) {
        const float g = d[j];
        dl[j] = g;
#pragma unroll
        for (int c = 0; c < G_E; ++c) dy[c] = fmaf(g, __ldg(m.pred_w + j * G_E + c), dy[c]);
      }
    }
#pragma unroll
    for (int c = 0; c < G_E; ++c) dx[c] = 0.f;
    ln_back_(xh, rs, dy, m.lnf_w, dx);
    float* g = mb.gfin + r * GF_STRIDE;
    store32_(g + GF_DLOG, dl), store32_(g + GF_XHF, xh), store32_(g + GF_DYF, dy);
#pragma unroll
    for (int c = 0; c < G_E; ++c) dl[c] = fmaf(xh[c], __ldg(m.lnf_w + c), __ldg(m.lnf_b + c));
    store32_(g + GF_YF, dl);
  } else {            // ---- ln_1 of layer l + 1: dy1 = dq Wq^T + dk Wk^T + dv Wv^T ----
    const TrainLayerW& u = m.layer[l + 1];
    const float* a = mb.act + ((size_t)(l + 1) * NR + r) * TA_STRIDE;
    float* g = mb.grec + ((size_t)(l + 1) * NR + r) * GR_STRIDE;
    float t[G_E], dy1[G_E], xh[G_E];
#pragma unroll
    for (int o = 0; o < 16; ++o) acc[o] = make_float2(0.f, 0.f);
#pragma unroll 1
    for (int part = 0; part < 3; ++part) {
      load32_(t, g + GR_DQKV + part * 32);
      row_matvec32<G_E>(t, sm + DB_WQKVT + part * 32 * 32, 32, 0, acc);
    }
    acc_to_(acc, dy1);
    load32_(xh, a + TA_XIN);
    const float mu = a[TA_MU1], rs = a[TA_RS1];
#pragma unroll
    for (int c = 0; c < G_E; ++c) xh[c] = (xh[c] - mu) * rs, t[c] = fmaf(xh[c], __ldg(u.ln1_w + c), __ldg(u.ln1_b + c));
    store32_(g + GR_Y1, t), store32_(g + GR_XH1, xh), store32_(g + GR_DY1, dy1);
    load32_(dx, g + GR_DXM);
    ln_back_(xh, rs, dy1, u.ln1_w, dx);
  }
  if (l < 0) {
    store32_(mb.gfin + r * GF_STRIDE + GF_DX0, dx);
    return;
  }
  // ---- MLP of layer l: x_out = x_mid + fc2(gelu_new(fc(ln_2(x_mid)))) ----
  const TrainLayerW& lw = m.layer[l];
  const float* a = mb.act + ((size_t)l * NR + r) * TA_STRIDE;
  float* g = mb.grec + ((size_t)l * NR + r) * GR_STRIDE;
  store32_(g + GR_DX, dx);
  float dxm[G_E];
  {
    float xh[G_E], dy[G_E];
    load32_(xh, a + TA_XMID);
    const float mu = a[TA_MU2], rs = a[TA_RS2];
#pragma unroll
    for (int c = 0; c < G_E; ++c) xh[c] = (xh[c] - mu) * rs;
    {
      float y[G_E];
#pragma unroll
      for (int c = 0; c < G_E; ++c) y[c] = fmaf(xh[c], __ldg(lw.ln2_w + c), __ldg(lw.ln2_b + c));
      store32_(g + GR_Y2, y), store32_(g + GR_XH2, xh);
    }
    float2 dy2[16];
#pragma unroll
    for (int o = 0; o < 16; ++o) dy2[o] = make_float2(0.f, 0.f);
#pragma unroll 1
    for (int part = 0; part < 4; ++part) {
#pragma unroll
      for (int o = 0; o < 16; ++o) acc[o] = make_float2(0.f, 0.f);
      row_matvec32<G_E>(dx, sm + DB_WFC2T, 128, part * 32, acc);   // d gelu(h)
      float h[G_E], dh[G_E];
      load32_(h, a + TA_H + part * 32);
      acc_to_(acc, dh);
#pragma unroll
      for (int c = 0; c < G_E; ++c) {
        const float x = h[c], x2 = x * x;
        const float t = tanhf(0.7978845608028654f * (x + 0.044715f * x2 * x));
        h[c] = 0.5f * x * (1.0f + t);
        const float dg = 0.5f * (1.0f + t) + 0.5f * x * (1.0f - t * t) * 0.7978845608028654f * (1.0f + 3.0f * 0.044715f * x2);
        dh[c] *= dg;
      }
      store32_(g + GR_G + part * 32, h), store32_(g + GR_DH + part * 32, dh);
      row_matvec32<G_E>(dh, sm + DB_WFCT + part * 32 * 32, 32, 0, dy2);
    }
    acc_to_(dy2, dy);
    store32_(g + GR_DY2, dy);
#pragma unroll
    for (int c = 0; c < G_E; ++c) dxm[c] = dx[c];
    ln_back_(xh, rs, dy, lw.ln2_w, dxm);
  }
  store32_(g + GR_DXM, dxm);
  // ---- attention output: dO = dxm Wproj^T, D = dO . O ----
  float dO[G_E], o_[G_E];
#pragma unroll
  for (int o = 0; o < 16; ++o) acc[o] = make_float2(0.f, 0.f);
  row_matvec32<G_E>(dxm, sm + DB_WPROJT, 32, 0, acc);
  acc_to_(acc, dO);
  load32_(o_, a + TA_O);
  float D = 0.f;
#pragma unroll
  for (int c = 0; c < G_E; ++c) D = fmaf(dO[c], o_[c], D);
  float* d = p.dos[NM == 1 ? 0 : blockIdx.y] + r * DOS_STRIDE;
  store32_(d, dO);
  d[32] = D;
}

constexpr int AT_ROWS = 64;        // rows of a tile: 4 warps x 16 (one mma.m16n8k16 row block each)
constexpr int AT_LD = 40;          // bf16 row stride of the [row][32] tiles (80 B: conflict-free fragment reads)
constexpr int AT_LDT = 72;         // bf16 row stride of the transposed [32][row] tiles (144 B)

template <int NM>
struct Attn16Params {
  int B, S, nt, l;
  size_t NR;
  const float* act[NM];
  float* grec[NM];
  const float* dos[NM];
};

__device__ __forceinline__ void mma_bf16_16816(float* d, const uint32_t* a, uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ uint32_t bf2_(float lo, float hi) {
  __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&v);
}
__device__ __forceinline__ uint32_t w32_(const __nv_bfloat16* p) { return *reinterpret_cast<const uint32_t*>(p); }

struct AttnSmem {
  __nv_bfloat16 ra[AT_ROWS][AT_LD];    // K (dq pass) or Q (dk/dv pass), [row][head]
  __nv_bfloat16 rb[AT_ROWS][AT_LD];    // V or dO
  __nv_bfloat16 ta[G_E][AT_LDT];       // K^T or Q^T, [head][row]
  __nv_bfloat16 tb[G_E][AT_LDT];       // dO^T
  float lse[AT_ROWS], dd[AT_ROWS];
};

// rows [row0, row0 + 64) of sequence b -> tiles (bf16; rows >= S are zero, with lse = D = 0): ra/rb from the act record
// fields fa/fb, or rb from dO (fb < 0); transposed copies when asked
__device__ __forceinline__ void load_tile_(AttnSmem& s, const float* act, const float* dos, size_t base, int row0, int S,
                                           int fa, int fb, bool trans_a, bool trans_b, bool stats) {
  const int tid = threadIdx.x, rr = tid >> 1, h0 = (tid & 1) * 16, row = row0 + rr;
  float va[16], vb[16];
  float lse = 0.f, dd = 0.f;
  if (row < S) {
    const float* a = act + (base + row) * TA_STRIDE;
    const float* d = dos + (base + row) * DOS_STRIDE;
    const float4* pa = reinterpret_cast<const float4*>(a + fa + h0);
    const float4* pb = reinterpret_cast<const float4*>(fb < 0 ? d + h0 : a + fb + h0);
#pragma unroll
    for (int o = 0; o < 4; ++o) {
      const float4 x = pa[o], y = pb[o];
      va[4 * o] = x.x, va[4 * o + 1] = x.y, va[4 * o + 2] = x.z, va[4 * o + 3] = x.w;
      vb[4 * o] = y.x, vb[4 * o + 1] = y.y, vb[4 * o + 2] = y.z, vb[4 * o + 3] = y.w;
    }
    if (stats) lse = a[TA_LSE], dd = d[32];
  } else {
#pragma unroll
    for (int c = 0; c < 16; ++c) va[c] = 0.f, vb[c] = 0.f;
  }
#pragma unroll
  for (int c = 0; c < 16; c += 2) {
    *reinterpret_cast<uint32_t*>(&s.ra[rr][h0 + c]) = bf2_(va[c], va[c + 1]);
    *reinterpret_cast<uint32_t*>(&s.rb[rr][h0 + c]) = bf2_(vb[c], vb[c + 1]);
  }
  if (trans_a) {
#pragma unroll
    for (int c = 0; c < 16; ++c) s.ta[h0 + c][rr] = __float2bfloat16_rn(va[c]);
  }
  if (trans_b) {
#pragma unroll
    for (int c = 0; c < 16; ++c) s.tb[h0 + c][rr] = __float2bfloat16_rn(vb[c]);
  }
  if (stats && h0 == 0) s.lse[rr] = lse, s.dd[rr] = dd;
}

// A fragments (16 rows from r0, head k-steps 0 and 1) of a [row][head] tile
__device__ __forceinline__ void a_frags_(const __nv_bfloat16 (*t)[AT_LD], int r0, uint32_t (*f)[4]) {
  const int lane = threadIdx.x & 31, g = lane >> 2, c = lane & 3;
#pragma unroll
  for (int ks = 0; ks < 2; ++ks) {
    f[ks][0] = w32_(&t[r0 + g][ks * 16 + 2 * c]);
    f[ks][1] = w32_(&t[r0 + g + 8][ks * 16 + 2 * c]);
    f[ks][2] = w32_(&t[r0 + g][ks * 16 + 2 * c + 8]);
    f[ks][3] = w32_(&t[r0 + g + 8][ks * 16 + 2 * c + 8]);
  }
}

// acc[2][4] (16 x 16) = A (16 x 32, fragments a) times the rows n0..n0+15 of a [row][head] tile, transposed
__device__ __forceinline__ void mma_rows_(const uint32_t (*a)[4], const __nv_bfloat16 (*t)[AT_LD], int n0, float (*acc)[4]) {
  const int lane = threadIdx.x & 31, g = lane >> 2, c = lane & 3;
#pragma unroll
  for (int nt = 0; nt < 2; ++nt) {
#pragma unroll
    for (int e = 0; e < 4; ++e) acc[nt][e] = 0.f;
#pragma unroll
    for (int ks = 0; ks < 2; ++ks)
      mma_bf16_16816(acc[nt], a[ks], w32_(&t[n0 + nt * 8 + g][ks * 16 + 2 * c]), w32_(&t[n0 + nt * 8 + g][ks * 16 + 2 * c + 8]));
  }
}

// out[4][4] (16 x 32) += A (16 x 16 over rows k0..k0+15) times a [head][row] tile
__device__ __forceinline__ void mma_cols_(const uint32_t* a, const __nv_bfloat16 (*t)[AT_LDT], int k0, float (*out)[4]) {
  const int lane = threadIdx.x & 31, g = lane >> 2, c = lane & 3;
#pragma unroll
  for (int hn = 0; hn < 4; ++hn)
    mma_bf16_16816(out[hn], a, w32_(&t[hn * 8 + g][k0 + 2 * c]), w32_(&t[hn * 8 + g][k0 + 2 * c + 8]));
}

// out[4][4] (rows r0 + g, r0 + g + 8; head columns 8 hn + 2c, +1) * scale -> dst + row * GR_STRIDE, rows < S
__device__ __forceinline__ void store_rows_(float* dst, int r0, int S, const float (*out)[4], float scale) {
  const int lane = threadIdx.x & 31, g = lane >> 2, c = lane & 3;
#pragma unroll
  for (int h = 0; h < 2; ++h) {
    const int row = r0 + g + 8 * h;
    if (row >= S) continue;
#pragma unroll
    for (int hn = 0; hn < 4; ++hn)
      *reinterpret_cast<float2*>(dst + (size_t)row * GR_STRIDE + hn * 8 + 2 * c) =
          make_float2(out[hn][2 * h] * scale, out[hn][2 * h + 1] * scale);
  }
}

// CTA (sequence b * nt + tile t, member = blockIdx.y), 4 warps; warp w owns rows 16 w .. 16 w + 15 of the tile
template <int NM>
__global__ void __launch_bounds__(128) gpt2_train_attn_bf16_kernel(const __grid_constant__ Attn16Params<NM> p) {
  __shared__ __align__(16) AttnSmem s;
  const int z = NM == 1 ? 0 : blockIdx.y;
  const int b = blockIdx.x / p.nt, t = blockIdx.x % p.nt, S = p.S;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, c = lane & 3;
  const float* act = p.act[z] + (size_t)p.l * p.NR * TA_STRIDE;
  float* grec = p.grec[z] + ((size_t)p.l * p.NR + (size_t)b * S) * GR_STRIDE;
  const float* dos = p.dos[z];
  const size_t base = (size_t)b * S;
  const int r0 = 16 * warp;
  uint32_t fa[2][4], fb[2][4];
  float out0[4][4], out1[4][4];

  // ---- dq of query tile t: dS = P o (dO V^T - D), dq = dS K / sqrt(32) over key tiles 0..t ----
  load_tile_(s, act, dos, base, t * AT_ROWS, S, TA_Q, -1, false, false, true);
  __syncthreads();
  a_frags_(s.ra, r0, fa);   // q
  a_frags_(s.rb, r0, fb);   // dO
  const int q0 = t * AT_ROWS + r0;
  const float lse0 = s.lse[r0 + g], lse1 = s.lse[r0 + g + 8], d0 = s.dd[r0 + g], d1 = s.dd[r0 + g + 8];
#pragma unroll
  for (int hn = 0; hn < 4; ++hn)
#pragma unroll
    for (int e = 0; e < 4; ++e) out0[hn][e] = 0.f;
  for (int j = 0; j <= t; ++j) {
    __syncthreads();
    load_tile_(s, act, dos, base, j * AT_ROWS, S, TA_K, TA_V, true, false, false);
    __syncthreads();
#pragma unroll 1
    for (int kc = 0; kc < AT_ROWS; kc += 16) {
      const int k0 = j * AT_ROWS + kc;
      if (k0 > q0 + 15) break;   // every key of the chunk is after every query of the warp
      float sc[2][4], dp[2][4];
      mma_rows_(fa, s.ra, kc, sc);
      mma_rows_(fb, s.rb, kc, dp);
      uint32_t ds[4];
#pragma unroll
      for (int nt = 0; nt < 2; ++nt) {
        float v[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const int q = q0 + g + (e >> 1) * 8, k = k0 + nt * 8 + 2 * c + (e & 1);
          const float pr = (k <= q && q < S) ? __expf(sc[nt][e] - (e >> 1 ? lse1 : lse0)) : 0.f;
          v[e] = pr * (dp[nt][e] - (e >> 1 ? d1 : d0));
        }
        ds[2 * nt] = bf2_(v[0], v[1]), ds[2 * nt + 1] = bf2_(v[2], v[3]);
      }
      mma_cols_(ds, s.ta, kc, out0);
    }
  }
  store_rows_(grec + GR_DQKV, q0, S, out0, ATT_SCALE);

  // ---- dk, dv of key tile t: dv = P^T dO, dk = dS^T q over query tiles t..nt-1 ----
  __syncthreads();
  load_tile_(s, act, dos, base, t * AT_ROWS, S, TA_K, TA_V, false, false, false);
  __syncthreads();
  a_frags_(s.ra, r0, fa);   // k
  a_frags_(s.rb, r0, fb);   // v
  const int k0 = t * AT_ROWS + r0;
#pragma unroll
  for (int hn = 0; hn < 4; ++hn)
#pragma unroll
    for (int e = 0; e < 4; ++e) out0[hn][e] = 0.f, out1[hn][e] = 0.f;
  for (int i = t; i < p.nt; ++i) {
    __syncthreads();
    load_tile_(s, act, dos, base, i * AT_ROWS, S, TA_Q, -1, true, true, true);
    __syncthreads();
#pragma unroll 1
    for (int qc = 0; qc < AT_ROWS; qc += 16) {
      const int qb = i * AT_ROWS + qc;
      if (qb + 15 < k0) continue;   // every query of the chunk is before every key of the warp
      if (qb >= S) break;
      float st[2][4], dpt[2][4];
      mma_rows_(fa, s.ra, qc, st);    // S^T = k q^T
      mma_rows_(fb, s.rb, qc, dpt);   // dP^T = v dO^T
      uint32_t pa[4], dsa[4];
#pragma unroll
      for (int nt = 0; nt < 2; ++nt) {
        float pv[4], dv[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const int k = k0 + g + (e >> 1) * 8, ql = qc + nt * 8 + 2 * c + (e & 1), q = i * AT_ROWS + ql;
          const float pr = (q >= k && q < S) ? __expf(st[nt][e] - s.lse[ql]) : 0.f;
          pv[e] = pr, dv[e] = pr * (dpt[nt][e] - s.dd[ql]);
        }
        pa[2 * nt] = bf2_(pv[0], pv[1]), pa[2 * nt + 1] = bf2_(pv[2], pv[3]);
        dsa[2 * nt] = bf2_(dv[0], dv[1]), dsa[2 * nt + 1] = bf2_(dv[2], dv[3]);
      }
      mma_cols_(pa, s.tb, qc, out1);    // dv += P^T dO
      mma_cols_(dsa, s.ta, qc, out0);   // dk += dS^T q
    }
  }
  store_rows_(grec + GR_DQKV + 32, k0, S, out0, 1.0f);
  store_rows_(grec + GR_DQKV + 64, k0, S, out1, 1.0f);
}

// ---- host side ----
struct TrainLayout {
  int L, S, din, du, NC, CH, P;
  size_t NR, act, fin, grec, gfin, part, wimg, dos, total;   // offsets in floats (wimg, dos: precision 1 only)
};

static int params_per_slot(int L, int din, int du) {
  const int per_layer = 32 * 96 + 96 + 32 * 32 + 32 + 32 * 128 + 128 + 128 * 32 + 32 + 4 * 32;
  const int p = L * per_layer + 32 * du + du + 2 * 32 + 32 * din + 32;
  return (p + 3) & ~3;
}

static TrainLayout train_layout(int L, int din, int du, int B, int T, int precision = 0) {
  TrainLayout t{};
  t.L = L, t.S = T + 1, t.din = din, t.du = du;
  t.NR = (size_t)B * t.S;
  // chunks of >= 256 rows, at most 256 of them; the chunking depends on the shape only (determinism)
  t.NC = (int)std::min<size_t>(256, (t.NR + 255) / 256);
  if (t.NC < 1) t.NC = 1;
  t.CH = (int)((((t.NR + t.NC - 1) / t.NC) + 31) / 32 * 32);
  t.NC = (int)((t.NR + t.CH - 1) / t.CH);
  if (t.NC < 1) t.NC = 1;
  t.P = params_per_slot(L, din, du);
  size_t o = 0;
  t.act = o, o += (size_t)L * t.NR * TA_STRIDE;
  t.fin = o, o += t.NR * TF_STRIDE;
  t.grec = o, o += (size_t)L * t.NR * GR_STRIDE;
  t.gfin = o, o += t.NR * GF_STRIDE;
  t.part = o, o += (size_t)t.NC * t.P;
  if (precision == 1) {
    t.wimg = o, o += (size_t)L * WIMG_BYTES / sizeof(float);
    t.dos = o, o += t.NR * DOS_STRIDE;
  }
  t.total = o;
  return t;
}

// `mem`: the member's index in a population call (its messages name it), -1 for the one-model entry points
static int check_model(const char* fn, int mem, const dpt_gpt2_weights_t* w, int B, int T) {
  char who[96];
  if (mem < 0) snprintf(who, sizeof who, "%s", fn);
  else snprintf(who, sizeof who, "%s: member %d", fn, mem);
  DPT_CHECK_ARG(w, "%s: null weights", who);
  if (w->n_embd != G_E) {
    set_error("%s: n_embd=%d, training supports n_embd == %d", who, w->n_embd, G_E);
    return DPT_ERR_UNSUPPORTED;
  }
  if (w->n_layer < 1 || w->n_layer > G_MAX_L) {
    set_error("%s: n_layer=%d outside [1,%d]", who, w->n_layer, G_MAX_L);
    return DPT_ERR_UNSUPPORTED;
  }
  const int din = 2 * w->state_dim + w->action_dim + 1;
  DPT_CHECK_ARG(w->state_dim >= 1 && w->action_dim >= 1 && din <= 32,
                "%s: token width 2*state_dim+action_dim+1 = %d must be <= 32", who, din);
  DPT_CHECK_ARG(B >= 0 && T >= 0, "%s: B=%d T=%d", who, B, T);
  if (T + 1 > 512) {
    set_error("%s: T=%d, training supports sequences of <= 512 tokens (T <= 511)", who, T);
    return DPT_ERR_UNSUPPORTED;
  }
  DPT_CHECK_ARG(T + 1 <= w->n_positions, "%s: sequence %d exceeds n_positions %d", who, T + 1, w->n_positions);
  DPT_CHECK_ARG(w->wpe && w->embed_w && w->embed_b && w->pred_w && w->pred_b && w->lnf_w && w->lnf_b && w->ln1_w && w->ln1_b &&
                    w->attn_w && w->attn_b && w->proj_w && w->proj_b && w->ln2_w && w->ln2_b && w->fc_w && w->fc_b &&
                    w->fc2_w && w->fc2_b,
                "%s: null weight pointer", who);
  for (int l = 0; l < w->n_layer; ++l)
    DPT_CHECK_ARG(w->ln1_w[l] && w->ln1_b[l] && w->attn_w[l] && w->attn_b[l] && w->proj_w[l] && w->proj_b[l] && w->ln2_w[l] &&
                      w->ln2_b[l] && w->fc_w[l] && w->fc_b[l] && w->fc2_w[l] && w->fc2_b[l],
                  "%s: null layer %d weight", who, l);
  return DPT_OK;
}

// The checks of a population call: 0 <= n <= TRAIN_POP_MAX, every member valid (check_model) and of member 0's shape.
// Returns DPT_OK with *done = true when there is nothing to compute (n = 0 or B = 0).
static int check_population(const char* fn, const dpt_gpt2_weights_t* w, int n, int B, int T, bool* done, int precision = 0) {
  *done = true;
  if (precision != 0 && precision != 1) {
    set_error("%s: precision=%d, training supports 0 (fp32) and 1 (bf16 tensor cores)", fn, precision);
    return DPT_ERR_UNSUPPORTED;
  }
  DPT_CHECK_ARG(n >= 0 && n <= TRAIN_POP_MAX, "%s: n_models=%d outside [0,%d]", fn, n, TRAIN_POP_MAX);
  if (n == 0) return DPT_OK;
  DPT_CHECK_ARG(w, "%s: null weights", fn);
  for (int i = 0; i < n; ++i) {
    const int rc = check_model(fn, n == 1 ? -1 : i, w + i, B, T);
    if (rc != DPT_OK) return rc;
    const struct { const char* name; int v, v0; } f[] = {{"n_layer", w[i].n_layer, w[0].n_layer},
                                                         {"state_dim", w[i].state_dim, w[0].state_dim},
                                                         {"action_dim", w[i].action_dim, w[0].action_dim},
                                                         {"n_positions", w[i].n_positions, w[0].n_positions}};
    for (const auto& x : f)
      DPT_CHECK_ARG(x.v == x.v0, "%s: member %d has %s=%d, member 0 has %d (members must share one shape)", fn, i, x.name,
                    x.v, x.v0);
  }
  *done = B == 0;
  return DPT_OK;
}

static TrainW train_w(const dpt_gpt2_weights_t* w) {
  TrainW d{};
  d.wpe = w->wpe, d.embed_w = w->embed_w, d.embed_b = w->embed_b, d.pred_w = w->pred_w, d.pred_b = w->pred_b;
  d.lnf_w = w->lnf_w, d.lnf_b = w->lnf_b;
  for (int l = 0; l < w->n_layer; ++l) {
    TrainLayerW& lw = d.layer[l];
    lw.ln1_w = w->ln1_w[l], lw.ln1_b = w->ln1_b[l], lw.attn_w = w->attn_w[l], lw.attn_b = w->attn_b[l];
    lw.proj_w = w->proj_w[l], lw.proj_b = w->proj_b[l], lw.ln2_w = w->ln2_w[l], lw.ln2_b = w->ln2_b[l];
    lw.fc_w = w->fc_w[l], lw.fc_b = w->fc_b[l], lw.fc2_w = w->fc2_w[l], lw.fc2_b = w->fc2_b[l];
  }
  return d;
}

static uint64_t member_bytes(const dpt_gpt2_weights_t* w, int B, int T, int precision = 0) {
  return train_layout(w->n_layer, 2 * w->state_dim + w->action_dim + 1, w->action_dim, B, T, precision).total * sizeof(float);
}

template <int NM>
static int population_forward(const char* fn, const dpt_gpt2_weights_t* w, int n, const float* const* query,
                              const float* const* cs, const float* const* ca, const float* const* cns, const float* const* cr,
                              int B, int T, int T_stride, int test, float* const* out, float* ws, cudaStream_t st) {
  const TrainLayout lay = train_layout(w->n_layer, 2 * w->state_dim + w->action_dim + 1, w->action_dim, B, T);
  TrainFwdParams<NM> p{};
  p.L = w->n_layer, p.dx = w->state_dim, p.du = w->action_dim, p.din = lay.din;
  p.B = B, p.T = T, p.Ts = T_stride, p.test = test ? 1 : 0;
  for (int i = 0; i < n; ++i) {
    TrainFwdMember& m = p.mem[i];
    m.w = train_w(w + i);
    for (int l = 0; l < p.L; ++l) {
      const TrainLayerW& lw = m.w.layer[l];
      DPT_CHECK_ARG(aligned16(lw.attn_w) && aligned16(lw.proj_w) && aligned16(lw.fc_w) && aligned16(lw.fc2_w),
                    "%s: layer %d matrices must be 16 B aligned", fn, l);
    }
    m.query = query[i], m.cs = T ? cs[i] : nullptr, m.ca = T ? ca[i] : nullptr, m.cns = T ? cns[i] : nullptr;
    m.cr = T ? cr[i] : nullptr, m.out = out[i];
    float* mws = ws + (size_t)i * lay.total;
    m.sv = TrainSave{mws + lay.act, mws + lay.fin};
  }
  return gpt2_train_forward_launch<NM>(p, n, st);
}

template <int NM>
static int population_forward16(const char* fn, const dpt_gpt2_weights_t* w, int n, const float* const* query,
                                const float* const* cs, const float* const* ca, const float* const* cns, const float* const* cr,
                                int B, int T, int T_stride, int test, float* const* out, float* ws, cudaStream_t st) {
  const TrainLayout lay = train_layout(w->n_layer, 2 * w->state_dim + w->action_dim + 1, w->action_dim, B, T, 1);
  TrainFwd16Params<NM> p{};
  WimgPackParams<NM> pk{};
  p.L = w->n_layer, p.dx = w->state_dim, p.du = w->action_dim, p.din = lay.din;
  p.B = B, p.T = T, p.Ts = T_stride, p.test = test ? 1 : 0;
  for (int i = 0; i < n; ++i) {
    TrainFwdMember& m = p.mem[i];
    m.w = train_w(w + i);
    m.query = query[i], m.cs = T ? cs[i] : nullptr, m.ca = T ? ca[i] : nullptr, m.cns = T ? cns[i] : nullptr;
    m.cr = T ? cr[i] : nullptr, m.out = out[i];
    float* mws = ws + (size_t)i * lay.total;
    m.sv = TrainSave{mws + lay.act, mws + lay.fin};
    p.wimg[i] = reinterpret_cast<const uint4*>(mws + lay.wimg);
    pk.img[i] = reinterpret_cast<unsigned char*>(mws + lay.wimg);
    for (int l = 0; l < p.L; ++l) {
      const TrainLayerW& lw = m.w.layer[l];
      pk.w[i][l][0] = lw.attn_w, pk.w[i][l][1] = lw.proj_w, pk.w[i][l][2] = lw.fc_w, pk.w[i][l][3] = lw.fc2_w;
    }
  }
  const int rc = gpt2_pack_train_wimg<NM>(pk, p.L, n, st);
  if (rc != DPT_OK) return rc;
  return gpt2_train_forward_bf16_launch<NM>(p, n, st);
}

template <int THREADS, int NM>
static cudaError_t launch_back(const BackParams<NM>& p, int n, cudaStream_t st) {
  const int smem = db_floats(THREADS) * (int)sizeof(float);
  cudaError_t e = cudaFuncSetAttribute(gpt2_train_backward_kernel<THREADS, NM>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
  if (e != cudaSuccess) return e;
  gpt2_train_backward_kernel<THREADS, NM><<<dim3(p.B, n), THREADS, smem, st>>>(p);
  return cudaGetLastError();
}

template <int NM>
static int population_backward(const char* fn, const dpt_gpt2_weights_t* w, int n, const float* const* dout, int B, int T,
                               int test, const dpt_gpt2_grads_t* grads, float* ws, cudaStream_t st, int precision) {
  const int L = w->n_layer;
  const TrainLayout lay = train_layout(L, 2 * w->state_dim + w->action_dim + 1, w->action_dim, B, T, precision);
  const size_t NR = lay.NR;
  BackParams<NM> bp{};
  bp.L = L, bp.du = w->action_dim, bp.B = B, bp.T = T, bp.test = test ? 1 : 0;
  for (int i = 0; i < n; ++i) {
    BackMember& m = bp.mem[i];
    float* mws = ws + (size_t)i * lay.total;
    m.w = train_w(w + i);
    m.dout = dout[i];
    m.act = mws + lay.act, m.fin = mws + lay.fin, m.grec = mws + lay.grec, m.gfin = mws + lay.gfin;
  }
  const int S = T + 1;
  cudaError_t e;
  if (precision == 0) {
    e = S <= 128 ? launch_back<128>(bp, n, st) : S <= 256 ? launch_back<256>(bp, n, st) : launch_back<512>(bp, n, st);
  } else {
    Rows16Params<NM> rp{};
    Attn16Params<NM> ap{};
    rp.b = bp;
    ap.B = B, ap.S = S, ap.nt = (S + AT_ROWS - 1) / AT_ROWS, ap.NR = NR;
    for (int i = 0; i < n; ++i) {
      float* mws = ws + (size_t)i * lay.total;
      rp.dos[i] = mws + lay.dos;
      ap.act[i] = mws + lay.act, ap.grec[i] = mws + lay.grec, ap.dos[i] = mws + lay.dos;
    }
    const int smem = RB_FLOATS * (int)sizeof(float);
    e = cudaFuncSetAttribute(gpt2_train_rows_bf16_kernel<NM>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    const dim3 rows_grid((unsigned)((NR + 127) / 128), n), attn_grid((unsigned)(B * ap.nt), n);
    for (int l = L - 1; l >= -1 && e == cudaSuccess; --l) {
      rp.l = l;
      gpt2_train_rows_bf16_kernel<NM><<<rows_grid, 128, smem, st>>>(rp);
      if (l >= 0) {
        ap.l = l;
        gpt2_train_attn_bf16_kernel<NM><<<attn_grid, 128, 0, st>>>(ap);
      }
      e = cudaGetLastError();
    }
  }
  if (e != cudaSuccess) {
    set_error("%s: backward launch failed: %s", fn, cudaGetErrorString(e));
    return DPT_ERR_CUDA;
  }

  // weight-gradient jobs (operands in member 0's workspace region) and, per member, the gradient tensors they reduce into
  RParams rp{};
  RSegs<NM> rs{};
  WpeParams<NM> wp{};
  int nj = 0, nt = 0, ns = 0, off = 0;
  auto job = [&](const float* A, int sa, const float* G, int sg, int nin, int nout, int diag, int trans) {
    RJob& j = rp.job[nj];
    j.A = A, j.G = G, j.sa = sa, j.sg = sg, j.nin = nin, j.nout = nout, j.diag = diag, j.trans = trans;
    const int nw = diag ? nout : nin * nout;
    j.woff = off, rs.seg[ns++] = RSeg{off, nw}, off += nw;
    j.boff = off, rs.seg[ns++] = RSeg{off, nout}, off += nout;
    if (diag) {
      rp.tile[nt++] = RTile{(short)nj, 0, 0};
    } else {
      for (int i0 = 0; i0 < nin; i0 += 32)
        for (int o0 = 0; o0 < nout; o0 += 32) rp.tile[nt++] = RTile{(short)nj, (short)i0, (short)o0};
    }
    ++nj;
  };
  for (int l = 0; l < L; ++l) {
    const float* a = ws + lay.act + (size_t)l * NR * TA_STRIDE;
    const float* gr = ws + lay.grec + (size_t)l * NR * GR_STRIDE;
    job(gr + GR_G, GR_STRIDE, gr + GR_DX, GR_STRIDE, G_FF, G_E, 0, 0);
    job(gr + GR_Y2, GR_STRIDE, gr + GR_DH, GR_STRIDE, G_E, G_FF, 0, 0);
    job(gr + GR_XH2, GR_STRIDE, gr + GR_DY2, GR_STRIDE, G_E, G_E, 1, 0);
    job(a + TA_O, TA_STRIDE, gr + GR_DXM, GR_STRIDE, G_E, G_E, 0, 0);
    job(gr + GR_Y1, GR_STRIDE, gr + GR_DQKV, GR_STRIDE, G_E, 3 * G_E, 0, 0);
    job(gr + GR_XH1, GR_STRIDE, gr + GR_DY1, GR_STRIDE, G_E, G_E, 1, 0);
  }
  const float* gf = ws + lay.gfin;
  job(gf + GF_YF, GF_STRIDE, gf + GF_DLOG, GF_STRIDE, G_E, lay.du, 0, 1);
  job(gf + GF_XHF, GF_STRIDE, gf + GF_DYF, GF_STRIDE, G_E, G_E, 1, 0);
  job(ws + lay.fin + TF_TOK, TF_STRIDE, gf + GF_DX0, GF_STRIDE, lay.din, G_E, 0, 1);
  if (off > lay.P) {
    set_error("%s: internal: %d gradient entries exceed the partial slot of %d", fn, off, lay.P);
    return DPT_ERR_CUDA;
  }
  for (int i = 0; i < n; ++i) {   // the segments in job order: per layer fc2, fc, ln_2, proj, attn, ln_1 (w, b), then the top
    const dpt_gpt2_grads_t* g = grads + i;
    float** d = rs.dst[i];
    int k = 0;
    for (int l = 0; l < L; ++l) {
      d[k++] = g->fc2_w[l], d[k++] = g->fc2_b[l], d[k++] = g->fc_w[l], d[k++] = g->fc_b[l];
      d[k++] = g->ln2_w[l], d[k++] = g->ln2_b[l], d[k++] = g->proj_w[l], d[k++] = g->proj_b[l];
      d[k++] = g->attn_w[l], d[k++] = g->attn_b[l], d[k++] = g->ln1_w[l], d[k++] = g->ln1_b[l];
    }
    d[k++] = g->pred_w, d[k++] = g->pred_b, d[k++] = g->lnf_w, d[k++] = g->lnf_b, d[k++] = g->embed_w, d[k++] = g->embed_b;
    wp.dwpe[i] = g->wpe;
  }
  rp.NR = (int)NR, rp.CH = lay.CH, rp.P = lay.P, rp.mstride = lay.total, rp.part = ws + lay.part;
  weight_grad_partial_kernel<<<dim3(nt, lay.NC, n), 256, 0, st>>>(rp);
  int maxn = 0;
  for (int s = 0; s < ns; ++s) maxn = std::max(maxn, rs.seg[s].n);
  rs.NC = lay.NC, rs.P = lay.P, rs.mstride = lay.total, rs.part = ws + lay.part;
  weight_grad_reduce_kernel<NM><<<dim3((maxn + 255) / 256, ns, n), 256, 0, st>>>(rs);
  wp.gfin = ws + lay.gfin, wp.mstride = lay.total, wp.B = B, wp.S = S, wp.n_pos = w->n_positions;
  wpe_grad_kernel<NM><<<dim3((w->n_positions * G_E + 255) / 256, n), 256, 0, st>>>(wp);
  DPT_LAUNCH_CHECK();
  return DPT_OK;
}

// the argument checks and launches shared by the one-model and the population entry points (one = the one-model call)
static int train_forward(const char* fn, bool one, const dpt_gpt2_weights_t* w, int n, const float* const* query,
                         const float* const* cs, const float* const* ca, const float* const* cns, const float* const* cr, int B,
                         int T, int T_stride, int test, float* const* out, void* workspace, uint64_t workspace_bytes,
                         void* stream, int precision = 0) {
  bool done;
  int rc = check_population(fn, w, n, B, T, &done, precision);
  if (rc != DPT_OK) return rc;
  if (n == 0) return DPT_OK;
  DPT_CHECK_ARG(T_stride >= T, "%s: T_stride=%d < T=%d", fn, T_stride, T);
  if (done) return DPT_OK;
  DPT_CHECK_ARG(query && out && (T == 0 || (cs && ca && cns && cr)), "%s: null input or output pointer array", fn);
  for (int i = 0; i < n; ++i)
    DPT_CHECK_ARG(query[i] && out[i] && (T == 0 || (cs[i] && ca[i] && cns[i] && cr[i])),
                  one ? "%s: null input or output pointer" : "%s: member %d: null input or output pointer", fn, i);
  const uint64_t need = (uint64_t)n * member_bytes(w, B, T, precision);
  DPT_CHECK_ARG(workspace && workspace_bytes >= need && aligned16(workspace), "%s: workspace of %llu B, needs %llu B (16 B aligned)",
                fn, (unsigned long long)workspace_bytes, (unsigned long long)need);
  float* ws = static_cast<float*>(workspace);
  cudaStream_t st = (cudaStream_t)stream;
  if (precision == 1)
    return n == 1 ? population_forward16<1>(fn, w, n, query, cs, ca, cns, cr, B, T, T_stride, test, out, ws, st)
                  : population_forward16<TRAIN_POP_MAX>(fn, w, n, query, cs, ca, cns, cr, B, T, T_stride, test, out, ws, st);
  return n == 1 ? population_forward<1>(fn, w, n, query, cs, ca, cns, cr, B, T, T_stride, test, out, ws, st)
                : population_forward<TRAIN_POP_MAX>(fn, w, n, query, cs, ca, cns, cr, B, T, T_stride, test, out, ws, st);
}

static int train_backward(const char* fn, bool one, const dpt_gpt2_weights_t* w, int n, const float* const* dout, int B, int T,
                          int test, const dpt_gpt2_grads_t* grads, void* workspace, uint64_t workspace_bytes, void* stream,
                          int precision = 0) {
  bool done;
  int rc = check_population(fn, w, n, B, T, &done, precision);
  if (rc != DPT_OK || done) return rc;
  DPT_CHECK_ARG(dout && grads, "%s: null dout or grads", fn);
  const uint64_t need = (uint64_t)n * member_bytes(w, B, T, precision);
  DPT_CHECK_ARG(workspace && workspace_bytes >= need && aligned16(workspace), "%s: workspace of %llu B, needs %llu B (16 B aligned)",
                fn, (unsigned long long)workspace_bytes, (unsigned long long)need);
  const int L = w->n_layer;
  for (int i = 0; i < n; ++i) {
    const dpt_gpt2_grads_t* g = grads + i;
    DPT_CHECK_ARG(dout[i], one ? "%s: null dout or grads" : "%s: member %d: null dout", fn, i);
    DPT_CHECK_ARG(g->wpe && g->embed_w && g->embed_b && g->pred_w && g->pred_b && g->lnf_w && g->lnf_b && g->ln1_w && g->ln1_b &&
                      g->attn_w && g->attn_b && g->proj_w && g->proj_b && g->ln2_w && g->ln2_b && g->fc_w && g->fc_b &&
                      g->fc2_w && g->fc2_b,
                  one ? "%s: null gradient pointer" : "%s: member %d: null gradient pointer", fn, i);
    for (int l = 0; l < L; ++l)
      DPT_CHECK_ARG(g->ln1_w[l] && g->ln1_b[l] && g->attn_w[l] && g->attn_b[l] && g->proj_w[l] && g->proj_b[l] && g->ln2_w[l] &&
                        g->ln2_b[l] && g->fc_w[l] && g->fc_b[l] && g->fc2_w[l] && g->fc2_b[l],
                    "%s: member %d: null layer %d gradient", fn, i, l);
  }
  float* ws = static_cast<float*>(workspace);
  cudaStream_t st = (cudaStream_t)stream;
  return n == 1 ? population_backward<1>(fn, w, n, dout, B, T, test, grads, ws, st, precision)
                : population_backward<TRAIN_POP_MAX>(fn, w, n, dout, B, T, test, grads, ws, st, precision);
}

}  // namespace dpt

using namespace dpt;

extern "C" uint64_t dpt_gpt2_train_population_workspace_bytes_ex(const dpt_gpt2_weights_t* w, int n_models, int B, int T,
                                                                  int precision) {
  if (!w || n_models <= 0 || n_models > TRAIN_POP_MAX || B <= 0 || T < 0 || w->n_layer < 1 || (precision != 0 && precision != 1))
    return 0;
  return (uint64_t)n_models * member_bytes(w, B, T, precision);
}

extern "C" uint64_t dpt_gpt2_train_population_workspace_bytes(const dpt_gpt2_weights_t* w, int n_models, int B, int T) {
  return dpt_gpt2_train_population_workspace_bytes_ex(w, n_models, B, T, 0);
}

extern "C" uint64_t dpt_gpt2_train_workspace_bytes(const dpt_gpt2_weights_t* w, int B, int T) {
  return dpt_gpt2_train_population_workspace_bytes(w, 1, B, T);
}

extern "C" int dpt_gpt2_train_population_forward(const dpt_gpt2_weights_t* w, int n_models, const float* const* query_states,
                                                 const float* const* ctx_states, const float* const* ctx_actions,
                                                 const float* const* ctx_next_states, const float* const* ctx_rewards, int B,
                                                 int T, int T_stride, int test, float* const* out, void* workspace,
                                                 uint64_t workspace_bytes, void* stream) {
  return train_forward("dpt_gpt2_train_population_forward", false, w, n_models, query_states, ctx_states, ctx_actions,
                       ctx_next_states, ctx_rewards, B, T, T_stride, test, out, workspace, workspace_bytes, stream);
}

extern "C" int dpt_gpt2_train_forward(const dpt_gpt2_weights_t* w, const float* query_states, const float* ctx_states,
                                      const float* ctx_actions, const float* ctx_next_states, const float* ctx_rewards, int B,
                                      int T, int T_stride, int test, float* out, void* workspace, uint64_t workspace_bytes,
                                      void* stream) {
  return train_forward("dpt_gpt2_train_forward", true, w, 1, &query_states, &ctx_states, &ctx_actions, &ctx_next_states,
                       &ctx_rewards, B, T, T_stride, test, &out, workspace, workspace_bytes, stream);
}

extern "C" int dpt_gpt2_train_population_forward_ex(const dpt_gpt2_weights_t* w, int n_models, const float* const* query_states,
                                                    const float* const* ctx_states, const float* const* ctx_actions,
                                                    const float* const* ctx_next_states, const float* const* ctx_rewards, int B,
                                                    int T, int T_stride, int test, int precision, float* const* out,
                                                    void* workspace, uint64_t workspace_bytes, void* stream) {
  return train_forward("dpt_gpt2_train_population_forward_ex", n_models == 1, w, n_models, query_states, ctx_states,
                       ctx_actions, ctx_next_states, ctx_rewards, B, T, T_stride, test, out, workspace, workspace_bytes, stream,
                       precision);
}

extern "C" int dpt_gpt2_train_population_backward_ex(const dpt_gpt2_weights_t* w, int n_models, const float* const* dout, int B,
                                                     int T, int test, int precision, const dpt_gpt2_grads_t* grads,
                                                     void* workspace, uint64_t workspace_bytes, void* stream) {
  return train_backward("dpt_gpt2_train_population_backward_ex", n_models == 1, w, n_models, dout, B, T, test, grads, workspace,
                        workspace_bytes, stream, precision);
}

extern "C" int dpt_gpt2_train_population_backward(const dpt_gpt2_weights_t* w, int n_models, const float* const* dout, int B,
                                                  int T, int test, const dpt_gpt2_grads_t* grads, void* workspace,
                                                  uint64_t workspace_bytes, void* stream) {
  return train_backward("dpt_gpt2_train_population_backward", false, w, n_models, dout, B, T, test, grads, workspace,
                        workspace_bytes, stream);
}

extern "C" int dpt_gpt2_train_backward(const dpt_gpt2_weights_t* w, const float* dout, int B, int T, int test,
                                       const dpt_gpt2_grads_t* grads, void* workspace, uint64_t workspace_bytes, void* stream) {
  return train_backward("dpt_gpt2_train_backward", true, w, 1, &dout, B, T, test, grads, workspace, workspace_bytes, stream);
}
