// Dense Transformer.forward(x) on the 5th-generation tensor cores (precision = 1; this kernel: <= 128 tokens,
// the multi-tile kernel below: 129..512 tokens).
//
// One CTA = one sequence; thread t owns token row t (128 threads = 128 TMEM lanes).  Every contraction of
// the GPT-2 block is ONE tcgen05.mma chain with M = 128 tokens, bf16 operands in shared memory (K-major,
// 128 B swizzle) and the fp32 accumulator in tensor memory; the element-wise work between contractions
// (LayerNorm, bias, causal softmax, gelu_new, residual) is done by the row's thread on fp32 registers
// after a tcgen05.ld of its TMEM lane:
//
//   Xn  = LN1(x)            -> smem A            QKV[128,96] = Xn   Wqkv      (N = 96,  K = 32)
//   q,k,v (+bias)           -> smem A / B / B^T  S  [128,128] = Q    K^T       (N = 128, K = 32)
//   P   = softmax(mask(S))  -> smem A            O  [128,32]  = P    V         (N = 32,  K = 128)
//   o   = O / rowsum        -> smem A            Y  [128,32]  = o    Wproj     (N = 32,  K = 32)   x += Y + b
//   Xn  = LN2(x)            -> smem A            F  [128,128] = Xn   Wfc       (N = 128, K = 32)
//   g   = gelu_new(F + b)   -> smem A            Y2 [128,32]  = g    Wfc2      (N = 32,  K = 128)  x += Y2 + b
//
// Weights are pre-transposed / pre-swizzled into bf16 B-operand images at model creation (40 KB per layer)
// and copied into shared memory per layer.  The residual stream x stays in fp32 registers (32 per thread).
// This is the dense path of SURVEY.md §8(d) ("the only place tensor cores are the relevant pipe"); it is
// opt-in (precision = 1, 2e-2 logit bar) because the 1e-5 bar of the default path excludes bf16 operands.
//
// The short pipeline is one row body, dense_short_rows<SAVE>.  SAVE = false is inference (gpt2_dense_kernel).  SAVE = true
// is the forward of bf16 training (gpt2_train_forward_bf16_kernel, called from gpt2_train.cu): the same rows on the
// parameter tensors and on weight images packed from them, so the logits are bit-identical to inference, and every row
// also stores what the backward needs in fp32 (TrainSave, layout TA_* / TF_* in gpt2_model.cuh).  The long pipeline has a
// training copy, dense_long_rows (see there).  A training launch covers a population of same-shape models: CTA (b,
// member = blockIdx.y).  pack_wimg_kernel writes the weight images of inference and training.
#include "common.cuh"
#include "gpt2_model.cuh"
#include "umma.cuh"
#include "gpt2_fp32.cuh"

namespace dpt {

constexpr int DN_THREADS = 128;
// dynamic shared memory layout (bytes, every tile 1024 B-aligned)
constexpr int SM_A0 = 0;                    // A tile, k 0..63      [128 x 64] 16 KB
constexpr int SM_A1 = 16384;                // A tile, k 64..127
constexpr int SM_K = 32768;                 // K as B operand       [128 x 64] 16 KB
constexpr int SM_VT0 = 49152;               // V^T as B operand     [32 x 64]   4 KB (keys 0..63)
constexpr int SM_VT1 = 53248;               //                                       (keys 64..127)
constexpr int SM_W = 57344;                 // weight image of the current layer, WIMG_BYTES
constexpr int SM_TOTAL = SM_W + WIMG_BYTES; // 98304
constexpr int TM_COLS = 256;

__device__ __forceinline__ void ln_row(const float* x, const float* w, const float* b, float* y) {
  float mean = 0.f;
#pragma unroll
  for (int c = 0; c < G_E; ++c) mean += x[c];
  mean *= (1.0f / G_E);
  float var = 0.f;
#pragma unroll
  for (int c = 0; c < G_E; ++c) var = fmaf(x[c] - mean, x[c] - mean, var);
  const float rs = 1.0f / sqrtf(var * (1.0f / G_E) + 1e-5f);
#pragma unroll
  for (int c = 0; c < G_E; ++c) y[c] = (x[c] - mean) * rs * __ldg(w + c) + __ldg(b + c);
}

// bf16-operand path (2e-2 bar): hardware approximations are far below the operand rounding (2^-9)
__device__ __forceinline__ float tanh_fast(float x) {
  float y;
  asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float exp_fast(float x) {   // e^x = 2^(x log2 e)
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x * 1.4426950408889634f));
  return y;
}
__device__ __forceinline__ float gelu_new_d(float x) {
  return 0.5f * x * (1.0f + tanh_fast(0.7978845608028654f * (x + 0.044715f * x * x * x)));
}

// write a 32-wide fp32 row as bf16 into chunks 0..3 of row m of a K64 tile
__device__ __forceinline__ void st_row32(unsigned char* tile, int m, const float* v) {
#pragma unroll
  for (int c = 0; c < 4; ++c) umma::st_chunk(tile, m, c, v + 8 * c);
}

struct Pipe {   // mbarrier + phase bookkeeping (uniform over the CTA)
  uint64_t* bar;
  uint32_t phase;
};

// all threads: make smem operand writes visible, sync; thread 0 issues `nk` K-steps and commits; all wait.
template <typename IssueFn>
__device__ __forceinline__ void run_mma(Pipe& pp, int tid, IssueFn issue) {
  umma::fence_async_smem();
  umma::fence_before_sync();
  __syncthreads();
  umma::fence_after_sync();
  if (tid == 0) {
    issue();
    umma::mma_commit(pp.bar);
  }
  umma::mbar_wait(pp.bar, pp.phase);
  pp.phase ^= 1;
  umma::fence_after_sync();
}

// rec[at..at+31] = x, rec[st] = mean, rec[st + 1] = 1 / std of x (the statistics of ln_row)
__device__ __forceinline__ void save_ln_(float* rec, int at, int st, const float* x) {
  store32_(rec + at, x);
  float mean = 0.f;
#pragma unroll
  for (int c = 0; c < G_E; ++c) mean += x[c];
  mean *= (1.0f / G_E);
  float var = 0.f;
#pragma unroll
  for (int c = 0; c < G_E; ++c) var = fmaf(x[c] - mean, x[c] - mean, var);
  rec[st] = mean, rec[st + 1] = 1.0f / sqrtf(var * (1.0f / G_E) + 1e-5f);
}
// dst[0..31] = y + bias
__device__ __forceinline__ void save_bias_(float* dst, const float* y, const float* bias) {
  float v[G_E];
#pragma unroll
  for (int c = 0; c < G_E; ++c) v[c] = y[c] + __ldg(bias + c);
  store32_(dst, v);
}

// The rows of sequence b = blockIdx.x (<= 128 tokens), thread t = row t.  SAVE = false: m = sh = the handle (Gpt2Dev), with
// its transposed embed / pred copies and the layer images m.layer[l].wimg.  SAVE = true: m = TrainW, the parameter tensors
// as they are (embed_transition.weight [E, din], pred_actions.weight [du, E]); sh gives L, dx, du, din and the images
// sh.wimg + l * WIMG_BYTES; every row also stores its activations in sv.  p: the inputs, the output and B, T, Ts, test, share.
template <bool SAVE, class W, class Sh, class P>
__device__ __forceinline__ void dense_short_rows(const W& m, const Sh& sh, const P& p, const TrainSave& sv) {
  extern __shared__ __align__(1024) unsigned char smem_raw[];
  __shared__ uint64_t bar;
  __shared__ uint32_t tmem_base_s;
  // dynamic smem base is only guaranteed 16 B-aligned: round up to 1024 B (the launch adds 1 KB of slack)
  unsigned char* smem = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const int tid = threadIdx.x, warp = tid >> 5;
  const int b = blockIdx.x;
  const int S = p.T + 1;                // tokens in the sequence (<= 128)
  const bool valid = tid < S;
  const int dx = sh.dx, du = sh.du, din = sh.din;

  if (warp == 0) umma::tmem_alloc(&tmem_base_s, TM_COLS);
  if (tid == 0) umma::mbar_init(&bar, 1);
  Pipe pp{&bar, 0};

  // ---- token embedding (models/net.py:45-54): row 0 = query state, rows 1..T = context transitions ----
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
  umma::fence_before_sync();
  __syncthreads();
  umma::fence_after_sync();
  const uint32_t tb = tmem_base_s;
  const uint32_t aA0 = umma::smem_u32(smem + SM_A0), aA1 = umma::smem_u32(smem + SM_A1), aK = umma::smem_u32(smem + SM_K);
  const uint32_t aVT0 = umma::smem_u32(smem + SM_VT0), aVT1 = umma::smem_u32(smem + SM_VT1), aW = umma::smem_u32(smem + SM_W);
  const uint32_t id32 = umma::make_idesc_bf16(128, 32), id96 = umma::make_idesc_bf16(128, 96), id128 = umma::make_idesc_bf16(128, 128);

  for (int l = 0; l < sh.L; ++l) {
    const auto& w = m.layer[l];
    float* const rec = SAVE && valid ? sv.act + (((size_t)l * p.B + b) * S + tid) * TA_STRIDE : nullptr;   // SAVE: this row's record
    // weight image of this layer -> smem (all MMAs that read the previous image have completed)
    {
      const uint4* src;
      if constexpr (SAVE) src = sh.wimg + (size_t)l * (WIMG_BYTES / 16);
      else src = w.wimg;
      uint4* dst = reinterpret_cast<uint4*>(smem + SM_W);
      for (int i = tid; i < WIMG_BYTES / 16; i += DN_THREADS) dst[i] = __ldg(src + i);
    }
    float y[G_E];
    // ---- LN1 -> A ; QKV = Xn Wqkv ----
    if (SAVE && valid) save_ln_(rec, TA_XIN, TA_MU1, x);
    ln_row(x, w.ln1_w, w.ln1_b, y);
    st_row32(smem + SM_A0, tid, y);
    run_mma(pp, tid, [&] {
#pragma unroll
      for (int ks = 0; ks < 2; ++ks)
        umma::mma_bf16(tb + 0, umma::make_desc_k64(aA0 + ks * 32), umma::make_desc_k64(aW + WIMG_QKV + ks * 32), id96, ks > 0);
    });
    // ---- q (scaled) -> A, k -> B, v -> B^T ----
    umma::tmem_ld32(umma::tmem_addr(tb, warp, 0), y);
#pragma unroll
    for (int c = 0; c < G_E; ++c) y[c] = (y[c] + __ldg(w.attn_b + c)) * 0.17677669529663687f;
    if (SAVE && valid) store32_(rec + TA_Q, y);
    st_row32(smem + SM_A0, tid, y);
    umma::tmem_ld32(umma::tmem_addr(tb, warp, 32), y);
#pragma unroll
    for (int c = 0; c < G_E; ++c) y[c] += __ldg(w.attn_b + G_E + c);
    if (SAVE && valid) store32_(rec + TA_K, y);
    st_row32(smem + SM_K, tid, y);
    umma::tmem_ld32(umma::tmem_addr(tb, warp, 64), y);
    if (SAVE && valid) save_bias_(rec + TA_V, y, w.attn_b + 2 * G_E);
    {
      unsigned char* vt = smem + (tid < 64 ? SM_VT0 : SM_VT1);
      const int kk = tid & 63;
#pragma unroll
      for (int c = 0; c < G_E; ++c)
        *reinterpret_cast<__nv_bfloat16*>(vt + umma::k64_offset(c, kk)) = __float2bfloat16_rn(y[c] + __ldg(w.attn_b + 2 * G_E + c));
    }
    // ---- S = Q K^T ----
    run_mma(pp, tid, [&] {
#pragma unroll
      for (int ks = 0; ks < 2; ++ks)
        umma::mma_bf16(tb + 128, umma::make_desc_k64(aA0 + ks * 32), umma::make_desc_k64(aK + ks * 32), id128, ks > 0);
    });
    // ---- causal softmax of row tid (keys <= tid), two passes over the TMEM row ----
    float mx = -INFINITY;
#pragma unroll
    for (int c0 = 0; c0 < 128; c0 += 32) {
      umma::tmem_ld32(umma::tmem_addr(tb, warp, 128 + c0), y);
#pragma unroll
      for (int i = 0; i < 32; ++i)
        if (c0 + i <= tid) mx = fmaxf(mx, y[i]);
    }
    float sum = 0.f;
#pragma unroll
    for (int c0 = 0; c0 < 128; c0 += 32) {
      umma::tmem_ld32(umma::tmem_addr(tb, warp, 128 + c0), y);
#pragma unroll
      for (int i = 0; i < 32; ++i) {
        const float pr = (c0 + i <= tid) ? exp_fast(y[i] - mx) : 0.f;
        // the normaliser uses the bf16-rounded probabilities that the tensor core will see
        y[i] = __bfloat162float(__float2bfloat16_rn(pr));
        sum += y[i];
      }
      unsigned char* tile = smem + (c0 < 64 ? SM_A0 : SM_A1);
#pragma unroll
      for (int c = 0; c < 4; ++c) umma::st_chunk(tile, tid, ((c0 & 63) >> 3) + c, y + 8 * c);
    }
    const float inv = 1.0f / sum;
    if (SAVE && valid) rec[TA_LSE] = mx + logf(sum);
    // ---- O = P V ----
    run_mma(pp, tid, [&] {
#pragma unroll
      for (int ks = 0; ks < 8; ++ks)
        umma::mma_bf16(tb + 0, umma::make_desc_k64((ks < 4 ? aA0 : aA1) + (ks & 3) * 32),
                       umma::make_desc_k64((ks < 4 ? aVT0 : aVT1) + (ks & 3) * 32), id32, ks > 0);
    });
    umma::tmem_ld32(umma::tmem_addr(tb, warp, 0), y);
#pragma unroll
    for (int c = 0; c < G_E; ++c) y[c] *= inv;
    if (SAVE && valid) store32_(rec + TA_O, y);
    st_row32(smem + SM_A0, tid, y);
    // ---- x += o Wproj + b ----
    run_mma(pp, tid, [&] {
#pragma unroll
      for (int ks = 0; ks < 2; ++ks)
        umma::mma_bf16(tb + 32, umma::make_desc_k64(aA0 + ks * 32), umma::make_desc_k64(aW + WIMG_PROJ + ks * 32), id32, ks > 0);
    });
    umma::tmem_ld32(umma::tmem_addr(tb, warp, 32), y);
#pragma unroll
    for (int c = 0; c < G_E; ++c) x[c] += y[c] + __ldg(w.proj_b + c);
    // ---- LN2 -> A ; F = Xn Wfc ----
    if (SAVE && valid) save_ln_(rec, TA_XMID, TA_MU2, x);
    ln_row(x, w.ln2_w, w.ln2_b, y);
    st_row32(smem + SM_A0, tid, y);
    run_mma(pp, tid, [&] {
#pragma unroll
      for (int ks = 0; ks < 2; ++ks)
        umma::mma_bf16(tb + 128, umma::make_desc_k64(aA0 + ks * 32), umma::make_desc_k64(aW + WIMG_FC + ks * 32), id128, ks > 0);
    });
#pragma unroll
    for (int c0 = 0; c0 < 128; c0 += 32) {
      umma::tmem_ld32(umma::tmem_addr(tb, warp, 128 + c0), y);
      if (SAVE && valid) save_bias_(rec + TA_H + c0, y, w.fc_b + c0);
#pragma unroll
      for (int i = 0; i < 32; ++i) y[i] = gelu_new_d(y[i] + __ldg(w.fc_b + c0 + i));
      unsigned char* tile = smem + (c0 < 64 ? SM_A0 : SM_A1);
#pragma unroll
      for (int c = 0; c < 4; ++c) umma::st_chunk(tile, tid, ((c0 & 63) >> 3) + c, y + 8 * c);
    }
    // ---- x += g Wfc2 + b ----
    run_mma(pp, tid, [&] {
#pragma unroll
      for (int ks = 0; ks < 8; ++ks)
        umma::mma_bf16(tb + 0, umma::make_desc_k64((ks < 4 ? aA0 : aA1) + (ks & 3) * 32),
                       umma::make_desc_k64(aW + WIMG_FC2 + (ks < 4 ? 0 : 4096) + (ks & 3) * 32), id32, ks > 0);
    });
    umma::tmem_ld32(umma::tmem_addr(tb, warp, 0), y);
#pragma unroll
    for (int c = 0; c < G_E; ++c) x[c] += y[c] + __ldg(w.fc2_b + c);
    umma::fence_before_sync();
    __syncthreads();   // every thread has drained its TMEM loads and smem reads before the next layer's image copy
  }

  // ---- ln_f + pred_actions ----
  if (SAVE && valid) save_ln_(sv.fin + ((size_t)b * S + tid) * TF_STRIDE, TF_X, TF_MU, x);
  if (p.test ? (tid == p.T) : (tid >= 1 && tid <= p.T)) {
    float y[G_E];
    ln_row(x, m.lnf_w, m.lnf_b, y);
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
  umma::fence_before_sync();
  __syncthreads();
  if (warp == 0) umma::tmem_dealloc(tb, TM_COLS);
}

__global__ void __launch_bounds__(DN_THREADS) gpt2_dense_kernel(const DenseParams p) {
  dense_short_rows<false>(p.m, p.m, p, TrainSave{});
}

int gpt2_dense_launch(const DenseParams& p, cudaStream_t st) {
  const int smem = SM_TOTAL + 1024;
  cudaError_t e = cudaFuncSetAttribute(gpt2_dense_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
  if (e != cudaSuccess) {
    set_error("gpt2_dense: cannot reserve %d B of shared memory: %s", smem, cudaGetErrorString(e));
    return DPT_ERR_CUDA;
  }
  gpt2_dense_kernel<<<p.B, DN_THREADS, smem, st>>>(p);
  e = cudaGetLastError();
  if (e != cudaSuccess) {
    set_error("gpt2_dense launch failed: %s", cudaGetErrorString(e));
    return DPT_ERR_CUDA;
  }
  return DPT_OK;
}

}  // namespace dpt

// =============================================================================================
// Long sequences (129..512 tokens): the same tensor-core pipeline over NT = 2..4 token tiles of 128 rows.
// Thread t owns row t of EVERY tile (residual streams x[NT][32] in registers).  Per layer the tiles are
// processed in causal order; tile i writes its K rows / V^T columns into sequence-wide shared-memory
// operand buffers and then attends to key tiles j = 0..i flash-style: S_ij = Q_i K_j^T (UMMA, N = 128) ->
// running row maximum / rescale in registers -> P_ij (bf16) -> O_ij = P_ij V_j (UMMA, N = 32) -> acc.  The
// MMA of S_i,j+1 is issued together with the P V MMA of tile j (different TMEM columns), so a tile costs
// i + 2 synchronisation stages for attention plus 4 for QKV / proj / fc / fc2.
// =============================================================================================
namespace dpt {

constexpr int LG_A0 = 0;                       // A tile k 0..63        16 KB
constexpr int LG_A1 = 16384;                   // A tile k 64..127      16 KB
constexpr int LG_Q = 32768;                    // Q_i as A operand      16 KB
constexpr int LG_K = 49152;                    // K of the whole sequence: 4 tiles x 16 KB
constexpr int LG_VT = LG_K + 4 * 16384;        // V^T: 8 K64 tiles of [32 rows x 64 keys], 4 KB each
constexpr int LG_W = LG_VT + 8 * 4096;         // weight image
constexpr int LG_TOTAL = LG_W + WIMG_BYTES;    // 188416 B

template <int NT>
__global__ void __launch_bounds__(DN_THREADS) gpt2_dense_long_kernel(const DenseParams p) {
  extern __shared__ __align__(1024) unsigned char smem_raw[];
  __shared__ uint64_t bar;
  __shared__ uint32_t tmem_base_s;
  unsigned char* smem = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const int tid = threadIdx.x, warp = tid >> 5;
  const int b = blockIdx.x;
  const Gpt2Dev& m = p.m;
  const int S = p.T + 1;
  const int dx = m.dx, du = m.du, din = m.din;

  if (warp == 0) umma::tmem_alloc(&tmem_base_s, TM_COLS);
  if (tid == 0) umma::mbar_init(&bar, 1);
  Pipe pp{&bar, 0};

  float x[NT][G_E];
#pragma unroll
  for (int i = 0; i < NT; ++i) {
    const int row = 128 * i + tid;             // token index of this thread in tile i
    const bool valid = row < S;
    float tok[32];
#pragma unroll
    for (int q = 0; q < 32; ++q) tok[q] = 0.f;
    if (valid) {
      if (row == 0) {
        for (int q = 0; q < dx; ++q) tok[q] = p.query[(size_t)b * dx + q];
      } else {
        const size_t r = (size_t)(b / p.share) * p.Ts + (row - 1);
        for (int q = 0; q < dx; ++q) tok[q] = p.cs[r * dx + q];
        for (int q = 0; q < du; ++q) tok[dx + q] = p.ca[r * du + q];
        for (int q = 0; q < dx; ++q) tok[dx + du + q] = p.cns[r * dx + q];
        tok[2 * dx + du] = p.cr[r];
      }
    }
#pragma unroll
    for (int c = 0; c < G_E; ++c) x[i][c] = valid ? __ldg(m.embed_b + c) + __ldg(m.wpe + (size_t)row * G_E + c) : 0.f;
    for (int q = 0; q < din; ++q) {
      const float tv = tok[q];
#pragma unroll
      for (int c = 0; c < G_E; ++c) x[i][c] = fmaf(tv, __ldg(m.embed_wT + q * G_E + c), x[i][c]);
    }
  }
  umma::fence_before_sync();
  __syncthreads();
  umma::fence_after_sync();
  const uint32_t tb = tmem_base_s;
  const uint32_t aA0 = umma::smem_u32(smem + LG_A0), aA1 = umma::smem_u32(smem + LG_A1), aQ = umma::smem_u32(smem + LG_Q);
  const uint32_t aK = umma::smem_u32(smem + LG_K), aVT = umma::smem_u32(smem + LG_VT), aW = umma::smem_u32(smem + LG_W);
  const uint32_t id32 = umma::make_idesc_bf16(128, 32), id96 = umma::make_idesc_bf16(128, 96), id128 = umma::make_idesc_bf16(128, 128);

  auto issue_S = [&](int j) {                  // S = Q_i K_j^T -> TMEM cols 128..255
#pragma unroll
    for (int ks = 0; ks < 2; ++ks)
      umma::mma_bf16(tb + 128, umma::make_desc_k64(aQ + ks * 32), umma::make_desc_k64(aK + j * 16384 + ks * 32), id128, ks > 0);
  };

  for (int l = 0; l < m.L; ++l) {
    const LayerW& w = m.layer[l];
    {
      const uint4* src = w.wimg;
      uint4* dst = reinterpret_cast<uint4*>(smem + LG_W);
      for (int q = tid; q < WIMG_BYTES / 16; q += DN_THREADS) dst[q] = __ldg(src + q);
    }
#pragma unroll
    for (int i = 0; i < NT; ++i) {
      float y[G_E];
      // ---- LN1 -> A0 ; QKV ----
      ln_row(x[i], w.ln1_w, w.ln1_b, y);
      st_row32(smem + LG_A0, tid, y);
      run_mma(pp, tid, [&] {
#pragma unroll
        for (int ks = 0; ks < 2; ++ks)
          umma::mma_bf16(tb + 0, umma::make_desc_k64(aA0 + ks * 32), umma::make_desc_k64(aW + WIMG_QKV + ks * 32), id96, ks > 0);
      });
      umma::tmem_ld32(umma::tmem_addr(tb, warp, 0), y);
#pragma unroll
      for (int c = 0; c < G_E; ++c) y[c] = (y[c] + __ldg(w.attn_b + c)) * 0.17677669529663687f;
      st_row32(smem + LG_Q, tid, y);
      umma::tmem_ld32(umma::tmem_addr(tb, warp, 32), y);
#pragma unroll
      for (int c = 0; c < G_E; ++c) y[c] += __ldg(w.attn_b + G_E + c);
      st_row32(smem + LG_K + i * 16384, tid, y);
      umma::tmem_ld32(umma::tmem_addr(tb, warp, 64), y);
      {
        unsigned char* vt = smem + LG_VT + (2 * i + (tid >> 6)) * 4096;
        const int kk = tid & 63;
#pragma unroll
        for (int c = 0; c < G_E; ++c)
          *reinterpret_cast<__nv_bfloat16*>(vt + umma::k64_offset(c, kk)) = __float2bfloat16_rn(y[c] + __ldg(w.attn_b + 2 * G_E + c));
      }
      // ---- flash attention over key tiles 0..i ----
      float acc[G_E];
#pragma unroll
      for (int c = 0; c < G_E; ++c) acc[c] = 0.f;
      float mx = -INFINITY, lsum = 0.f;
      run_mma(pp, tid, [&] { issue_S(0); });
      for (int j = 0; j <= i; ++j) {
        const bool diag = (j == i);
        // new running maximum over this key tile
        float mnew = mx;
#pragma unroll
        for (int c0 = 0; c0 < 128; c0 += 32) {
          umma::tmem_ld32(umma::tmem_addr(tb, warp, 128 + c0), y);
#pragma unroll
          for (int q = 0; q < 32; ++q)
            if (!diag || c0 + q <= tid) mnew = fmaxf(mnew, y[q]);
        }
        const float sc = exp_fast(mx - mnew);     // 0 when mx == -inf
        mx = mnew;
        lsum *= sc;
#pragma unroll
        for (int c = 0; c < G_E; ++c) acc[c] *= sc;
#pragma unroll
        for (int c0 = 0; c0 < 128; c0 += 32) {
          umma::tmem_ld32(umma::tmem_addr(tb, warp, 128 + c0), y);
#pragma unroll
          for (int q = 0; q < 32; ++q) {
            const float pr = (!diag || c0 + q <= tid) ? exp_fast(y[q] - mx) : 0.f;
            y[q] = __bfloat162float(__float2bfloat16_rn(pr));
            lsum += y[q];
          }
          unsigned char* tile = smem + (c0 < 64 ? LG_A0 : LG_A1);
#pragma unroll
          for (int c = 0; c < 4; ++c) umma::st_chunk(tile, tid, ((c0 & 63) >> 3) + c, y + 8 * c);
        }
        // O_ij = P_ij V_j (cols 0..31); the next tile's S is issued in the same stage (cols 128..255)
        run_mma(pp, tid, [&] {
#pragma unroll
          for (int ks = 0; ks < 8; ++ks)
            umma::mma_bf16(tb + 0, umma::make_desc_k64((ks < 4 ? aA0 : aA1) + (ks & 3) * 32),
                           umma::make_desc_k64(aVT + (2 * j + (ks >> 2)) * 4096 + (ks & 3) * 32), id32, ks > 0);
          if (j < i) issue_S(j + 1);
        });
        umma::tmem_ld32(umma::tmem_addr(tb, warp, 0), y);
#pragma unroll
        for (int c = 0; c < G_E; ++c) acc[c] += y[c];
      }
      const float inv = 1.0f / lsum;
#pragma unroll
      for (int c = 0; c < G_E; ++c) y[c] = acc[c] * inv;
      st_row32(smem + LG_A0, tid, y);
      // ---- proj ----
      run_mma(pp, tid, [&] {
#pragma unroll
        for (int ks = 0; ks < 2; ++ks)
          umma::mma_bf16(tb + 32, umma::make_desc_k64(aA0 + ks * 32), umma::make_desc_k64(aW + WIMG_PROJ + ks * 32), id32, ks > 0);
      });
      umma::tmem_ld32(umma::tmem_addr(tb, warp, 32), y);
#pragma unroll
      for (int c = 0; c < G_E; ++c) x[i][c] += y[c] + __ldg(w.proj_b + c);
      // ---- MLP ----
      ln_row(x[i], w.ln2_w, w.ln2_b, y);
      st_row32(smem + LG_A0, tid, y);
      run_mma(pp, tid, [&] {
#pragma unroll
        for (int ks = 0; ks < 2; ++ks)
          umma::mma_bf16(tb + 128, umma::make_desc_k64(aA0 + ks * 32), umma::make_desc_k64(aW + WIMG_FC + ks * 32), id128, ks > 0);
      });
#pragma unroll
      for (int c0 = 0; c0 < 128; c0 += 32) {
        umma::tmem_ld32(umma::tmem_addr(tb, warp, 128 + c0), y);
#pragma unroll
        for (int q = 0; q < 32; ++q) y[q] = gelu_new_d(y[q] + __ldg(w.fc_b + c0 + q));
        unsigned char* tile = smem + (c0 < 64 ? LG_A0 : LG_A1);
#pragma unroll
        for (int c = 0; c < 4; ++c) umma::st_chunk(tile, tid, ((c0 & 63) >> 3) + c, y + 8 * c);
      }
      run_mma(pp, tid, [&] {
#pragma unroll
        for (int ks = 0; ks < 8; ++ks)
          umma::mma_bf16(tb + 0, umma::make_desc_k64((ks < 4 ? aA0 : aA1) + (ks & 3) * 32),
                         umma::make_desc_k64(aW + WIMG_FC2 + (ks < 4 ? 0 : 4096) + (ks & 3) * 32), id32, ks > 0);
      });
      umma::tmem_ld32(umma::tmem_addr(tb, warp, 0), y);
#pragma unroll
      for (int c = 0; c < G_E; ++c) x[i][c] += y[c] + __ldg(w.fc2_b + c);
    }
    umma::fence_before_sync();
    __syncthreads();
  }

#pragma unroll
  for (int i = 0; i < NT; ++i) {
    const int row = 128 * i + tid;
    if (p.test ? (row == p.T) : (row >= 1 && row <= p.T)) {
      float y[G_E];
      ln_row(x[i], m.lnf_w, m.lnf_b, y);
      float* o = p.test ? p.out + (size_t)b * du : p.out + ((size_t)b * p.T + (row - 1)) * du;
      for (int j = 0; j < du; ++j) {
        float lg = __ldg(m.pred_b + j);
#pragma unroll
        for (int c = 0; c < G_E; ++c) lg = fmaf(y[c], __ldg(m.pred_wT + c * du + j), lg);
        o[j] = lg;
      }
    }
  }
  umma::fence_before_sync();
  __syncthreads();
  if (warp == 0) umma::tmem_dealloc(tb, TM_COLS);
}

template <int NT>
static cudaError_t launch_long(const DenseParams& p, cudaStream_t st) {
  const int smem = LG_TOTAL + 1024;
  cudaError_t e = cudaFuncSetAttribute(gpt2_dense_long_kernel<NT>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
  if (e != cudaSuccess) return e;
  gpt2_dense_long_kernel<NT><<<p.B, DN_THREADS, smem, st>>>(p);
  return cudaGetLastError();
}

int gpt2_dense_long_launch(const DenseParams& p, cudaStream_t st) {
  const int S = p.T + 1;
  cudaError_t e = S <= 256 ? launch_long<2>(p, st) : S <= 384 ? launch_long<3>(p, st) : launch_long<4>(p, st);
  if (e != cudaSuccess) {
    set_error("gpt2_dense_long launch failed: %s", cudaGetErrorString(e));
    return DPT_ERR_CUDA;
  }
  return DPT_OK;
}

// The rows of sequence b (129..512 tokens) for the forward of bf16 training: gpt2_dense_long_kernel's pipeline on the
// parameter tensors, saving the activations; m, sh, p and sv as in dense_short_rows with SAVE = true.  Unlike the short
// pipeline, this one is not shared with the inference kernel: compiled from one SAVE-templated body,
// gpt2_dense_long_kernel<2> ran 1.1 % slower at B = 1024 x 201 tokens (one B200 at 1000 W).  A change to the pipeline
// is made in both copies, and the training logits stay bit-identical to gpt2_dense_long_kernel's.
template <int NT, class W, class Sh, class P>
__device__ __forceinline__ void dense_long_rows(const W& m, const Sh& sh, const P& p, const TrainSave& sv) {
  extern __shared__ __align__(1024) unsigned char smem_raw[];
  __shared__ uint64_t bar;
  __shared__ uint32_t tmem_base_s;
  unsigned char* smem = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const int tid = threadIdx.x, warp = tid >> 5;
  const int b = blockIdx.x;
  const int S = p.T + 1;
  const int dx = sh.dx, du = sh.du, din = sh.din;

  if (warp == 0) umma::tmem_alloc(&tmem_base_s, TM_COLS);
  if (tid == 0) umma::mbar_init(&bar, 1);
  Pipe pp{&bar, 0};

  float x[NT][G_E];
#pragma unroll
  for (int i = 0; i < NT; ++i) {
    const int row = 128 * i + tid;             // token index of this thread in tile i
    const bool valid = row < S;
    float tok[32];
#pragma unroll
    for (int q = 0; q < 32; ++q) tok[q] = 0.f;
    if (valid) {
      if (row == 0) {
        for (int q = 0; q < dx; ++q) tok[q] = p.query[(size_t)b * dx + q];
      } else {
        const size_t r = (size_t)(b / p.share) * p.Ts + (row - 1);
        for (int q = 0; q < dx; ++q) tok[q] = p.cs[r * dx + q];
        for (int q = 0; q < du; ++q) tok[dx + q] = p.ca[r * du + q];
        for (int q = 0; q < dx; ++q) tok[dx + du + q] = p.cns[r * dx + q];
        tok[2 * dx + du] = p.cr[r];
      }
    }
    if (valid) store32_(sv.fin + ((size_t)b * S + row) * TF_STRIDE + TF_TOK, tok);
#pragma unroll
    for (int c = 0; c < G_E; ++c) x[i][c] = valid ? __ldg(m.embed_b + c) + __ldg(m.wpe + (size_t)row * G_E + c) : 0.f;
    for (int q = 0; q < din; ++q) {
      const float tv = tok[q];
#pragma unroll
      for (int c = 0; c < G_E; ++c) x[i][c] = fmaf(tv, __ldg(m.embed_w + c * din + q), x[i][c]);
    }
  }
  umma::fence_before_sync();
  __syncthreads();
  umma::fence_after_sync();
  const uint32_t tb = tmem_base_s;
  const uint32_t aA0 = umma::smem_u32(smem + LG_A0), aA1 = umma::smem_u32(smem + LG_A1), aQ = umma::smem_u32(smem + LG_Q);
  const uint32_t aK = umma::smem_u32(smem + LG_K), aVT = umma::smem_u32(smem + LG_VT), aW = umma::smem_u32(smem + LG_W);
  const uint32_t id32 = umma::make_idesc_bf16(128, 32), id96 = umma::make_idesc_bf16(128, 96), id128 = umma::make_idesc_bf16(128, 128);

  auto issue_S = [&](int j) {                  // S = Q_i K_j^T -> TMEM cols 128..255
#pragma unroll
    for (int ks = 0; ks < 2; ++ks)
      umma::mma_bf16(tb + 128, umma::make_desc_k64(aQ + ks * 32), umma::make_desc_k64(aK + j * 16384 + ks * 32), id128, ks > 0);
  };

  for (int l = 0; l < sh.L; ++l) {
    const auto& w = m.layer[l];
    {
      const uint4* src = sh.wimg + (size_t)l * (WIMG_BYTES / 16);
      uint4* dst = reinterpret_cast<uint4*>(smem + LG_W);
      for (int q = tid; q < WIMG_BYTES / 16; q += DN_THREADS) dst[q] = __ldg(src + q);
    }
#pragma unroll
    for (int i = 0; i < NT; ++i) {
      float y[G_E];
      const bool valid = 128 * i + tid < S;
      float* const rec = valid ? sv.act + (((size_t)l * p.B + b) * S + 128 * i + tid) * TA_STRIDE : nullptr;
      // ---- LN1 -> A0 ; QKV ----
      if (valid) save_ln_(rec, TA_XIN, TA_MU1, x[i]);
      ln_row(x[i], w.ln1_w, w.ln1_b, y);
      st_row32(smem + LG_A0, tid, y);
      run_mma(pp, tid, [&] {
#pragma unroll
        for (int ks = 0; ks < 2; ++ks)
          umma::mma_bf16(tb + 0, umma::make_desc_k64(aA0 + ks * 32), umma::make_desc_k64(aW + WIMG_QKV + ks * 32), id96, ks > 0);
      });
      umma::tmem_ld32(umma::tmem_addr(tb, warp, 0), y);
#pragma unroll
      for (int c = 0; c < G_E; ++c) y[c] = (y[c] + __ldg(w.attn_b + c)) * 0.17677669529663687f;
      if (valid) store32_(rec + TA_Q, y);
      st_row32(smem + LG_Q, tid, y);
      umma::tmem_ld32(umma::tmem_addr(tb, warp, 32), y);
#pragma unroll
      for (int c = 0; c < G_E; ++c) y[c] += __ldg(w.attn_b + G_E + c);
      if (valid) store32_(rec + TA_K, y);
      st_row32(smem + LG_K + i * 16384, tid, y);
      umma::tmem_ld32(umma::tmem_addr(tb, warp, 64), y);
      if (valid) save_bias_(rec + TA_V, y, w.attn_b + 2 * G_E);
      {
        unsigned char* vt = smem + LG_VT + (2 * i + (tid >> 6)) * 4096;
        const int kk = tid & 63;
#pragma unroll
        for (int c = 0; c < G_E; ++c)
          *reinterpret_cast<__nv_bfloat16*>(vt + umma::k64_offset(c, kk)) = __float2bfloat16_rn(y[c] + __ldg(w.attn_b + 2 * G_E + c));
      }
      // ---- flash attention over key tiles 0..i ----
      float acc[G_E];
#pragma unroll
      for (int c = 0; c < G_E; ++c) acc[c] = 0.f;
      float mx = -INFINITY, lsum = 0.f;
      run_mma(pp, tid, [&] { issue_S(0); });
      for (int j = 0; j <= i; ++j) {
        const bool diag = (j == i);
        // new running maximum over this key tile
        float mnew = mx;
#pragma unroll
        for (int c0 = 0; c0 < 128; c0 += 32) {
          umma::tmem_ld32(umma::tmem_addr(tb, warp, 128 + c0), y);
#pragma unroll
          for (int q = 0; q < 32; ++q)
            if (!diag || c0 + q <= tid) mnew = fmaxf(mnew, y[q]);
        }
        const float sc = exp_fast(mx - mnew);     // 0 when mx == -inf
        mx = mnew;
        lsum *= sc;
#pragma unroll
        for (int c = 0; c < G_E; ++c) acc[c] *= sc;
#pragma unroll
        for (int c0 = 0; c0 < 128; c0 += 32) {
          umma::tmem_ld32(umma::tmem_addr(tb, warp, 128 + c0), y);
#pragma unroll
          for (int q = 0; q < 32; ++q) {
            const float pr = (!diag || c0 + q <= tid) ? exp_fast(y[q] - mx) : 0.f;
            y[q] = __bfloat162float(__float2bfloat16_rn(pr));
            lsum += y[q];
          }
          unsigned char* tile = smem + (c0 < 64 ? LG_A0 : LG_A1);
#pragma unroll
          for (int c = 0; c < 4; ++c) umma::st_chunk(tile, tid, ((c0 & 63) >> 3) + c, y + 8 * c);
        }
        // O_ij = P_ij V_j (cols 0..31); the next tile's S is issued in the same stage (cols 128..255)
        run_mma(pp, tid, [&] {
#pragma unroll
          for (int ks = 0; ks < 8; ++ks)
            umma::mma_bf16(tb + 0, umma::make_desc_k64((ks < 4 ? aA0 : aA1) + (ks & 3) * 32),
                           umma::make_desc_k64(aVT + (2 * j + (ks >> 2)) * 4096 + (ks & 3) * 32), id32, ks > 0);
          if (j < i) issue_S(j + 1);
        });
        umma::tmem_ld32(umma::tmem_addr(tb, warp, 0), y);
#pragma unroll
        for (int c = 0; c < G_E; ++c) acc[c] += y[c];
      }
      const float inv = 1.0f / lsum;
#pragma unroll
      for (int c = 0; c < G_E; ++c) y[c] = acc[c] * inv;
      if (valid) store32_(rec + TA_O, y), rec[TA_LSE] = mx + logf(lsum);
      st_row32(smem + LG_A0, tid, y);
      // ---- proj ----
      run_mma(pp, tid, [&] {
#pragma unroll
        for (int ks = 0; ks < 2; ++ks)
          umma::mma_bf16(tb + 32, umma::make_desc_k64(aA0 + ks * 32), umma::make_desc_k64(aW + WIMG_PROJ + ks * 32), id32, ks > 0);
      });
      umma::tmem_ld32(umma::tmem_addr(tb, warp, 32), y);
#pragma unroll
      for (int c = 0; c < G_E; ++c) x[i][c] += y[c] + __ldg(w.proj_b + c);
      // ---- MLP ----
      if (valid) save_ln_(rec, TA_XMID, TA_MU2, x[i]);
      ln_row(x[i], w.ln2_w, w.ln2_b, y);
      st_row32(smem + LG_A0, tid, y);
      run_mma(pp, tid, [&] {
#pragma unroll
        for (int ks = 0; ks < 2; ++ks)
          umma::mma_bf16(tb + 128, umma::make_desc_k64(aA0 + ks * 32), umma::make_desc_k64(aW + WIMG_FC + ks * 32), id128, ks > 0);
      });
#pragma unroll
      for (int c0 = 0; c0 < 128; c0 += 32) {
        umma::tmem_ld32(umma::tmem_addr(tb, warp, 128 + c0), y);
        if (valid) save_bias_(rec + TA_H + c0, y, w.fc_b + c0);
#pragma unroll
        for (int q = 0; q < 32; ++q) y[q] = gelu_new_d(y[q] + __ldg(w.fc_b + c0 + q));
        unsigned char* tile = smem + (c0 < 64 ? LG_A0 : LG_A1);
#pragma unroll
        for (int c = 0; c < 4; ++c) umma::st_chunk(tile, tid, ((c0 & 63) >> 3) + c, y + 8 * c);
      }
      run_mma(pp, tid, [&] {
#pragma unroll
        for (int ks = 0; ks < 8; ++ks)
          umma::mma_bf16(tb + 0, umma::make_desc_k64((ks < 4 ? aA0 : aA1) + (ks & 3) * 32),
                         umma::make_desc_k64(aW + WIMG_FC2 + (ks < 4 ? 0 : 4096) + (ks & 3) * 32), id32, ks > 0);
      });
      umma::tmem_ld32(umma::tmem_addr(tb, warp, 0), y);
#pragma unroll
      for (int c = 0; c < G_E; ++c) x[i][c] += y[c] + __ldg(w.fc2_b + c);
    }
    umma::fence_before_sync();
    __syncthreads();
  }

#pragma unroll
  for (int i = 0; i < NT; ++i) {
    const int row = 128 * i + tid;
    if (row < S) save_ln_(sv.fin + ((size_t)b * S + row) * TF_STRIDE, TF_X, TF_MU, x[i]);
    if (p.test ? (row == p.T) : (row >= 1 && row <= p.T)) {
      float y[G_E];
      ln_row(x[i], m.lnf_w, m.lnf_b, y);
      float* o = p.test ? p.out + (size_t)b * du : p.out + ((size_t)b * p.T + (row - 1)) * du;
      for (int j = 0; j < du; ++j) {
        float lg = __ldg(m.pred_b + j);
#pragma unroll
        for (int c = 0; c < G_E; ++c) lg = fmaf(y[c], __ldg(m.pred_w + j * G_E + c), lg);
        o[j] = lg;
      }
    }
  }
  umma::fence_before_sync();
  __syncthreads();
  if (warp == 0) umma::tmem_dealloc(tb, TM_COLS);
}


// ---- the forward of bf16 training: CTA (b, member = blockIdx.y), on the member's parameters ----
struct TrainShape16 {
  int L, dx, du, din;
  const uint4* wimg;
};
template <int NM>
__device__ __forceinline__ void train16_member(const TrainFwd16Params<NM>& p, const TrainFwdMember*& mb, TrainShape16& sh) {
  const int z = NM == 1 ? 0 : blockIdx.y;
  mb = &p.mem[z];
  sh = TrainShape16{p.L, p.dx, p.du, p.din, p.wimg[z]};
}
struct TrainIo {
  const float *query, *cs, *ca, *cns, *cr;
  float* out;
  int B, T, Ts, test, share;
};

template <int NM>
__global__ void __launch_bounds__(DN_THREADS) gpt2_train_forward_bf16_kernel(const __grid_constant__ TrainFwd16Params<NM> p) {
  const TrainFwdMember* mb;
  TrainShape16 sh;
  train16_member(p, mb, sh);
  const TrainIo io{mb->query, mb->cs, mb->ca, mb->cns, mb->cr, mb->out, p.B, p.T, p.Ts, p.test, 1};
  dense_short_rows<true>(mb->w, sh, io, mb->sv);
}

template <int NT, int NM>
__global__ void __launch_bounds__(DN_THREADS) gpt2_train_forward_long_bf16_kernel(const __grid_constant__ TrainFwd16Params<NM> p) {
  const TrainFwdMember* mb;
  TrainShape16 sh;
  train16_member(p, mb, sh);
  const TrainIo io{mb->query, mb->cs, mb->ca, mb->cns, mb->cr, mb->out, p.B, p.T, p.Ts, p.test, 1};
  dense_long_rows<NT>(mb->w, sh, io, mb->sv);
}

template <class K, class P>
static cudaError_t launch_train16(K kern, int smem, const P& p, int n, cudaStream_t st) {
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
  if (e != cudaSuccess) return e;
  kern<<<dim3(p.B, n), DN_THREADS, smem, st>>>(p);
  return cudaGetLastError();
}

template <int NM>
int gpt2_train_forward_bf16_launch(const TrainFwd16Params<NM>& p, int n, cudaStream_t st) {
  const int S = p.T + 1;
  cudaError_t e = S <= 128   ? launch_train16(gpt2_train_forward_bf16_kernel<NM>, SM_TOTAL + 1024, p, n, st)
                  : S <= 256 ? launch_train16(gpt2_train_forward_long_bf16_kernel<2, NM>, LG_TOTAL + 1024, p, n, st)
                  : S <= 384 ? launch_train16(gpt2_train_forward_long_bf16_kernel<3, NM>, LG_TOTAL + 1024, p, n, st)
                             : launch_train16(gpt2_train_forward_long_bf16_kernel<4, NM>, LG_TOTAL + 1024, p, n, st);
  if (e != cudaSuccess) {
    set_error("gpt2_train_forward (bf16) launch failed: %s", cudaGetErrorString(e));
    return DPT_ERR_CUDA;
  }
  return DPT_OK;
}
template int gpt2_train_forward_bf16_launch<1>(const TrainFwd16Params<1>&, int, cudaStream_t);
template int gpt2_train_forward_bf16_launch<TRAIN_POP_MAX>(const TrainFwd16Params<TRAIN_POP_MAX>&, int, cudaStream_t);

// The weight images (layout WIMG_* in gpt2_model.cuh) of members 0 .. n-1, layers 0 .. L-1, one launch: CTA (element
// block, layer, member).  Every byte of an image is written; k beyond In is zero.
template <int NM>
__global__ void pack_wimg_kernel(const __grid_constant__ WimgPackParams<NM> p) {
  const int z = NM == 1 ? 0 : blockIdx.z, l = blockIdx.y;
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= WIMG_BYTES / 2) return;
  // segments of the image: [rows Out] x [Kpad = max(64, In)] elements each
  int i = e, seg = 0;
  const int Out[4] = {3 * G_E, G_E, G_FF, G_E}, In[4] = {G_E, G_E, G_E, G_FF}, Off[4] = {WIMG_QKV, WIMG_PROJ, WIMG_FC, WIMG_FC2};
  while (i >= Out[seg] * max(64, In[seg])) i -= Out[seg] * max(64, In[seg]), ++seg;
  const int kp = max(64, In[seg]), n = i / kp, k = i % kp;
  const float v = k < In[seg] ? p.w[z][l][seg][k * Out[seg] + n] : 0.f;
  unsigned char* tile = p.img[z][l] + Off[seg] + (k >> 6) * (Out[seg] * 128);
  *reinterpret_cast<__nv_bfloat16*>(tile + umma::k64_offset(n, k & 63)) = __float2bfloat16_rn(v);
}
static_assert(sizeof(WimgPackParams<TRAIN_POP_MAX>) <= 32764 && sizeof(TrainFwd16Params<TRAIN_POP_MAX>) <= 32764,
              "the per-member tables of TRAIN_POP_MAX members must fit the kernel parameter limit");

template <int NM>
int gpt2_pack_wimg(const WimgPackParams<NM>& p, int L, int n, cudaStream_t st) {
  pack_wimg_kernel<NM><<<dim3((WIMG_BYTES / 2 + 255) / 256, L, n), 256, 0, st>>>(p);
  const cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) {
    set_error("pack_wimg launch failed: %s", cudaGetErrorString(e));
    return DPT_ERR_CUDA;
  }
  return DPT_OK;
}
template int gpt2_pack_wimg<1>(const WimgPackParams<1>&, int, int, cudaStream_t);
template int gpt2_pack_wimg<TRAIN_POP_MAX>(const WimgPackParams<TRAIN_POP_MAX>&, int, int, cudaStream_t);

}  // namespace dpt
