// GPT-2 trunk of the DPT Transformer (reference models/net.py:9-60 over transformers GPT2Model with
// n_head = 1): embed_transition -> +wpe -> L x [LN -> c_attn -> causal softmax(QK^T/sqrt(E)) V ->
// c_proj -> +res; LN -> c_fc -> gelu_new -> c_proj -> +res] -> ln_f -> pred_actions.
//
// Both entry points run the model one token at a time with a per-sequence K/V cache, one WARP per
// sequence, lane = channel (n_embd = 32 = warp width, head_dim = 32):
//   dpt_gpt2_online_loop : the bandit in-context evaluation loop (evals/eval_bandit.py:56-103 +
//       ctrls/ctrl_bandit.py:383-444 + env step) fused into one launch.  The reference re-runs the
//       whole (h+1)-token forward at every step (O(H^2) token-forwards, plus a full host->device copy
//       of the context each step); because the bandit query token is constant and sits at position 0
//       of a causal model, appending one token per step to a K/V cache is mathematically identical
//       (SURVEY.md §3.3), so a step is ONE token-forward + softmax/categorical draw + env step.
//   dpt_gpt2_forward     : Transformer.forward(x) for an arbitrary context (dense semantics, computed
//       causally token by token with a scratch K/V cache).
// Layout: K and V are both [layer][t][channel] (128 B rows, appended coalesced).  Attention maps a
// lane to (key group lane/8, channel quad lane%8): one LDG.128 instruction covers 4 keys x 32 channels,
// 8 are kept in flight per lane (32 keys), the 8-lane dot products are combined by a 7-shuffle
// butterfly transpose-reduce, softmax is a warp reduction, and PV accumulates float4 channel quads.  The
// fp32 attention (attention_f32) is one body for both stagings of the K/V tiles: register-staged global
// loads (GlobalKv) or bulk-async copies through a per-warp shared-memory ring (KvRing, small batches of
// the online loop).  K/V reads bypass L1 (ld.global.cg) so L1 keeps the ~200 KB of weights that
// every warp re-reads; weights are read through the read-only path.  fp32 everywhere, accurate
// expf/tanhf/sqrtf (the 1e-5 logit parity bar excludes TF32 and .approx forms).
// Bound: K/V bytes read per token-forward = n_layer * 2 * t * 32 * 4 (HBM once the in-flight caches
// exceed L2), ~0.9 FLOP/B -- HBM-bound, not tensor-bound (SURVEY.md §8d).
#include <cuda_bf16.h>

#include <algorithm>
#include <type_traits>

#include "common.cuh"
#include "philox.cuh"

#include "gpt2_model.cuh"

namespace dpt {

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// L2 prefetch of one 128 B line per lane (a warp covers 4 KB): issued a few iterations ahead of the
// demand loads of the K/V streams so that DRAM latency is paid off the critical path.
__device__ __forceinline__ void prefetch_l2(const void* p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }

__device__ __forceinline__ float layer_norm(float x, const float* w, const float* b, int lane) {
  const float mean = warp_sum(x) * (1.0f / G_E);
  const float dv = x - mean;
  const float var = warp_sum(dv * dv) * (1.0f / G_E);
  return dv * (1.0f / sqrtf(var + 1e-5f)) * __ldg(w + lane) + __ldg(b + lane);
}

__device__ __forceinline__ float2 ffma2(float2 a, float2 b, float2 c) {
  float2 d;
  asm("fma.rn.f32x2 %0, %1, %2, %3;"
      : "=l"(reinterpret_cast<unsigned long long&>(d))
      : "l"(reinterpret_cast<unsigned long long&>(a)), "l"(reinterpret_cast<unsigned long long&>(b)),
        "l"(reinterpret_cast<unsigned long long&>(c)));
  return d;
}

// out[g] = bias[g*32 + lane] + sum_i xs[i] * W[i][g*32 + lane]  for g < G, W packed as described at LayerW.
// Two float2 accumulators per output (4 partial sums) keep the dependent FFMA2 chain at IN/4.
template <int IN, int G>
__device__ __forceinline__ void matvec_packed(const float* xs, const float4* wP, const float* bias, int lane, float* out) {
  float2 acc[G][2];
#pragma unroll
  for (int g = 0; g < G; ++g) acc[g][0] = make_float2(__ldg(bias + g * 32 + lane), 0.f), acc[g][1] = make_float2(0.f, 0.f);
#pragma unroll 4
  for (int iq = 0; iq < IN / 4; ++iq) {
    const float4 xv = reinterpret_cast<const float4*>(xs)[iq];
#pragma unroll
    for (int g = 0; g < G; ++g) {
      const float4 wv = __ldg(wP + (size_t)(iq * G + g) * 32 + lane);
      acc[g][0] = ffma2(make_float2(xv.x, xv.y), make_float2(wv.x, wv.y), acc[g][0]);
      acc[g][1] = ffma2(make_float2(xv.z, xv.w), make_float2(wv.z, wv.w), acc[g][1]);
    }
  }
#pragma unroll
  for (int g = 0; g < G; ++g) out[g] = (acc[g][0].x + acc[g][0].y) + (acc[g][1].x + acc[g][1].y);
}

__device__ __forceinline__ float gelu_new(float x) {  // transformers NewGELUActivation
  return 0.5f * x * (1.0f + tanhf(0.7978845608028654f * (x + 0.044715f * x * x * x)));
}

constexpr int PF_AHEAD = 3;      // K/V L2 prefetch distance in 32-key iterations (fp32 cache: 4 KB each)
constexpr int PF_MAX_POS = 192;  // only short (latency-bound) sequences prefetch: +20 % at H=100, -2 % at H=500 without the cap

// D[16x8] += A[16x16] B[16x8], bf16 operands, fp32 accumulate (legacy tensor-core path; tcgen05 needs M = 128 rows
// that a one-row-per-env decode does not have)
__device__ __forceinline__ void mma_bf16_16816(float (&d)[4], uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t b0,
                                               uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
               : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
}
__device__ __forceinline__ uint32_t pack_bf16(float lo, float hi) {   // lo -> bits 0..15 (the lower k / n index)
  const __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<const uint32_t*>(&v);
}

// y[N] = x[K] W on the tensor cores, one warp, weights as pre-arranged bf16 B fragments in shared memory (WF_* layout
// in gpt2_model.cuh).  xin / yout: 8 B-aligned, distinct buffers.
template <int K, int N>
__device__ __forceinline__ void matvec_mma(const uint4* wf, const float* xin, float* yout, int lane) {
  const int c = lane & 3;
  uint32_t a0[K / 16], a2[K / 16];
#pragma unroll
  for (int ks = 0; ks < K / 16; ++ks) {
    a0[ks] = a2[ks] = 0u;
    if (lane < 4) {
      const float2 u = *reinterpret_cast<const float2*>(xin + 16 * ks + 2 * c);
      const float2 w = *reinterpret_cast<const float2*>(xin + 16 * ks + 8 + 2 * c);
      a0[ks] = pack_bf16(u.x, u.y), a2[ks] = pack_bf16(w.x, w.y);
    }
  }
  // transposed product y^T = W^T x^T: the 16 x 16 weight tile is the A operand (16 outputs per HMMA), x is column 0 of
  // B (lanes 0..3), the outputs are column 0 of the accumulator: lanes with c == 0 hold outputs g and g + 8
#pragma unroll
  for (int ntp = 0; ntp < N / 16; ++ntp) {
    float d[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int ks = 0; ks < K / 16; ++ks) {
      const uint4 bw = wf[(ks * (N / 16) + ntp) * 32 + lane];
      mma_bf16_16816(d, bw.x, bw.z, bw.y, bw.w, a0[ks], a2[ks]);
    }
    if (c == 0) yout[16 * ntp + (lane >> 2)] = d[0], yout[16 * ntp + 8 + (lane >> 2)] = d[2];
  }
}

// W[K][N] fp32 -> WF_* fragment image (one thread per (group, lane))
__global__ void pack_wfrag_kernel(const float* __restrict__ W, uint4* __restrict__ dst, int K, int N) {
  const int id = blockIdx.x * blockDim.x + threadIdx.x;
  if (id >= (K / 16) * (N / 16) * 32) return;
  const int lane = id & 31, grp = id >> 5;
  const int ks = grp / (N / 16), ntp = grp - ks * (N / 16);
  const int c = lane & 3, n0 = 16 * ntp + (lane >> 2), n1 = n0 + 8, k0 = 16 * ks + 2 * c;
  auto w = [&](int k, int n) { return W[(size_t)k * N + n]; };
  dst[id] = make_uint4(pack_bf16(w(k0, n0), w(k0 + 1, n0)), pack_bf16(w(k0 + 8, n0), w(k0 + 9, n0)),
                       pack_bf16(w(k0, n1), w(k0 + 1, n1)), pack_bf16(w(k0 + 8, n1), w(k0 + 9, n1)));
}

// resident CTAs per SM the online-loop kernels are compiled for (register cap = 65536 / (128 * n)); measured on B200
constexpr int GPT2_MINB_F32 = 9;   // 56 registers: 221 ms at C4 against 241 ms (8) / 226 ms (7) / 270 ms (10)
constexpr int GPT2_MINB_BF16 = 6;

// Bytes of one sequence's K/V cache: [L][K, V][Tpad][32 channels], fp32 or bf16 (precision 1)
__host__ __device__ __forceinline__ size_t kv_seq_bytes(int L, int Tpad, bool bf16) {
  return (size_t)L * 2 * G_E * Tpad * (bf16 ? 2 : 4);
}

// Keys 0..pos-1 in tiles of TILE: f(k0, std::false_type) for every full tile, then f(k0, std::true_type) for the last,
// partial one if there is one.  MASK_ALL: every tile takes the masked (std::true_type) form -- one copy of the tile code
template <int TILE, bool MASK_ALL = false, class F>
__device__ __forceinline__ void for_each_key_tile(int pos, F&& f) {
  if constexpr (MASK_ALL) {
    for (int k0 = 0; k0 < pos; k0 += TILE) f(k0, std::true_type{});
  } else {
    int k0 = 0;
    for (; k0 + TILE <= pos; k0 += TILE) f(k0, std::false_type{});
    if (k0 < pos) f(k0, std::true_type{});
  }
}

// ---------------------------------------------------------------------------------------------
// Sources of the fp32 attention's 32-key K / V tiles.  tile(X, k0, pos, lane) returns this lane's channel quad of the
// tile (X = the layer's K or V cache), load(t, k0, r) reads row r of it (row stride = 8 float4), consumed(lane) follows
// the last read of a tile, begin_token / end_token bracket each token.
// ---------------------------------------------------------------------------------------------
// Register-staged: ld.global.cg straight from the cache, 8 rows in flight per lane; short sequences prefetch to L2 ahead.
struct GlobalKv {
  static constexpr bool MASK_ALL = false;
  __device__ __forceinline__ void begin_token(int, int) {}
  __device__ __forceinline__ void end_token() {}
  __device__ __forceinline__ const float4* tile(const float* X, int k0, int pos, int lane) {
    if (pos <= PF_MAX_POS && k0 + PF_AHEAD * 32 < pos) prefetch_l2(X + (size_t)(k0 + PF_AHEAD * 32 + lane) * G_E);
    return reinterpret_cast<const float4*>(X) + (lane & 7);
  }
  __device__ __forceinline__ float4 load(const float4* t, int k0, int r) const { return __ldcg(t + (size_t)(k0 + r) * 8); }
  __device__ __forceinline__ void consumed(int) {}
};

// Bulk-async (TMA engine) staging: cp.async.bulk global -> shared, completion on an mbarrier.  A warp's cached keys of one
// layer are ONE contiguous run per tensor ([t][32 channels] fp32, 128 B rows), so a tile of 32 keys is a single <= 4 KB
// bulk copy of exactly the live rows (no padded rows are read).  Each warp owns a ring of KV_STAGES such tiles and walks
// the token's tile sequence  layer 0 K tiles, layer 0 V tiles, layer 1 K tiles, ...: the copy of tile j + KV_STAGES is
// issued (one lane, one instruction) the moment tile j has been consumed, so the stream keeps flowing through the softmax
// between the K and the V pass and through the projections / MLP between layers -- with register-staged loads a warp has
// nothing in flight during those phases.
constexpr int TMA_WARPS = 4;
constexpr int TMA_MINB = 5;   // 96 registers: 20 warps per SM with a 2-deep ring (measured best at 10k envs: 210 ms; 4 CTAs / 128 regs: 257 ms)
constexpr int KV_STAGES = 2;  // ring depth: measured at 1250 and 10000 envs, 2 stages beat 3, 4 and 6 (DESIGN.md)
constexpr int KV_TILE_BYTES = 32 * G_E * 4;   // 32 keys x 32 channels fp32

__device__ __forceinline__ uint32_t smem_addr(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

struct KvRing {
  static constexpr bool MASK_ALL = true;   // every tile masked, K rows past the last key read stale (fewer registers than the split)
  uint32_t stage0, bar0;        // shared addresses: stage s at stage0 + s * KV_TILE_BYTES, its mbarrier at bar0 + 8 s
  uint32_t is;                  // stage the next issued tile goes to
  uint32_t cs, cp;              // stage of the next tile to consume, and the parity of its mbarrier phase
  int cl, ckv, ct;              // cursor of the next tile to issue: layer, K (0) / V (1), tile
  int nt, pos, L, Tpad;
  const float* kv;

  __device__ __forceinline__ void issue_next(int lane) {
    if (cl >= L) return;
    if (lane == 0) {
      const uint32_t s = is;
      const int nkeys = min(32, pos - 32 * ct);
      const uint32_t bytes = (uint32_t)nkeys * (G_E * 4);
      const float* src = kv + ((size_t)(cl * 2 + ckv) * Tpad + (size_t)ct * 32) * G_E;
      const uint32_t bar = bar0 + 8 * s, dst = stage0 + s * KV_TILE_BYTES;
      asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
      asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst), "l"(src), "r"(bytes),
                   "r"(bar)
                   : "memory");
    }
    if (++is == KV_STAGES) is = 0;
    if (++ct == nt) {
      ct = 0;
      if (++ckv == 2) ckv = 0, ++cl;
    }
  }
  // start of a token at position `pos` (keys 0 .. pos-1 are cached): fill the ring
  __device__ __forceinline__ void begin_token(int pos_, int lane) {
    pos = pos_, nt = (pos_ + 31) >> 5;
    cl = nt ? 0 : L, ckv = 0, ct = 0;
    for (int i = 0; i < KV_STAGES; ++i) issue_next(lane);
  }
  // this token's appended K/V rows (generic-proxy stores of all lanes) must be visible to the bulk copies (async proxy)
  // that the next token issues
  __device__ __forceinline__ void end_token() {
    __syncwarp();
    asm volatile("fence.proxy.async;" ::: "memory");
  }
  // wait for the next tile in sequence (tiles arrive in the order the attention asks for them; X, k0 and pos are implied)
  __device__ __forceinline__ const float4* tile(const float*, int, int, int lane) {
    const uint32_t s = cs, par = cp;
    const uint32_t bar = bar0 + 8 * s;
    asm volatile(
        "{\n\t.reg .pred p;\n\tKVWAIT_%=:\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t@!p bra KVWAIT_%=;\n\t}" ::"r"(bar), "r"(par)
        : "memory");
    return reinterpret_cast<const float4*>(__cvta_shared_to_generic((size_t)(stage0 + s * KV_TILE_BYTES))) + (lane & 7);
  }
  __device__ __forceinline__ float4 load(const float4* t, int, int r) const { return t[r * 8]; }   // rows past the last key: stale
  // every lane has finished reading the tile: its stage is free for the next copy
  __device__ __forceinline__ void consumed(int lane) {
    __syncwarp();
    if (++cs == KV_STAGES) cs = 0, cp ^= 1u;
    issue_next(lane);
  }
};

// fp32 attention of the token at `pos` (query q, key k, value v: this lane's channel) over the cached keys 0..pos-1 and
// itself; appends k and v to the layer's caches K and V first.  Returns this lane's channel of the attention output.
// A lane maps to (key group g = lane/8, channel quad b8 = lane%8): one 16 B load covers 4 keys x 32 channels, 8 are kept
// in flight per lane (32 keys), the 8-lane dot products are combined by a 7-shuffle butterfly transpose-reduce, softmax
// is a warp reduction, and PV accumulates float4 channel quads.
template <class Src>
__device__ __forceinline__ float attention_f32(float q, float k, float v, int pos, float* K, float* V, float* sx, float* ssc,
                                               int lane, Src& src) {
  K[(size_t)pos * G_E + lane] = k;   // both caches are [t][channel]: appends are coalesced 128 B rows
  V[(size_t)pos * G_E + lane] = v;
  q *= 0.17677669529663687f;  // 1/sqrt(head_dim = 32)
  sx[lane] = q;
  __syncwarp();
  const int g = lane >> 3, b8 = lane & 7;
  const float4 q4 = reinterpret_cast<const float4*>(sx)[b8];
  __syncwarp();
  // TAIL = the last, partial tile: load instruction i covers keys k0 + 4 i .. k0 + 4 i + 3 of all key groups, so
  // instructions past the last key are skipped with a WARP-UNIFORM predicate (round 2: the padded rows of the last tile
  // were 4.7 % of the kernel's DRAM traffic; per-lane predication of every tile, which skips 3-5 % of the K/V traffic at
  // H = 500, cost more issue than the bytes saved)
  float lmax = -INFINITY;
  for_each_key_tile<32, Src::MASK_ALL>(pos, [&](const int k0, auto tail_tag) {
    constexpr bool TAIL = decltype(tail_tag)::value;
    const int r = pos - k0;
    const float4* t = src.tile(K, k0, pos, lane);
    float4 kk[8];
#pragma unroll
    for (int i = 0; i < 8; ++i)
      kk[i] = (!TAIL || Src::MASK_ALL || 4 * i < r) ? src.load(t, k0, 4 * i + g) : make_float4(0.f, 0.f, 0.f, 0.f);   // in bounds (Tpad % 32 == 0)
    float pv[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) pv[i] = fmaf(q4.x, kk[i].x, fmaf(q4.y, kk[i].y, fmaf(q4.z, kk[i].z, q4.w * kk[i].w)));
    src.consumed(lane);
    // butterfly transpose-reduce over the 8 lanes of a key group: lane b8 ends with the full dot of chunk i = b8
    float w4[4], w2[2];
    const bool u4 = b8 & 4, u2 = b8 & 2, u1 = b8 & 1;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float send = u4 ? pv[j] : pv[j + 4], keep = u4 ? pv[j + 4] : pv[j];
      w4[j] = keep + __shfl_xor_sync(0xffffffffu, send, 4);
    }
#pragma unroll
    for (int j = 0; j < 2; ++j) {
      const float send = u2 ? w4[j] : w4[j + 2], keep = u2 ? w4[j + 2] : w4[j];
      w2[j] = keep + __shfl_xor_sync(0xffffffffu, send, 2);
    }
    const float sc = (u1 ? w2[1] : w2[0]) + __shfl_xor_sync(0xffffffffu, u1 ? w2[0] : w2[1], 1);
    const int key = k0 + 4 * b8 + g;
    if (!TAIL || key < pos) {
      ssc[key] = sc;
      lmax = fmaxf(lmax, sc);
    }
  });
  const float s_self = warp_sum(q * k);  // the token attends to itself (causal mask keeps keys <= pos)
  lmax = fmaxf(warp_max(lmax), s_self);
  __syncwarp();
  float lsum = 0.f;
  for (int key = lane; key < pos; key += 32) {
    const float pr = expf(ssc[key] - lmax);
    ssc[key] = pr;
    lsum += pr;
  }
  const float p_self = expf(s_self - lmax);
  const float inv = 1.0f / (warp_sum(lsum) + p_self);
  __syncwarp();
  float4 oa = make_float4(0.f, 0.f, 0.f, 0.f);
  for_each_key_tile<32, Src::MASK_ALL>(pos, [&](const int k0, auto tail_tag) {
    constexpr bool TAIL = decltype(tail_tag)::value;
    const float4* t = src.tile(V, k0, pos, lane);
    float4 vv[8];
    float pr[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int key = k0 + 4 * i + g;
      const bool ok = !TAIL || key < pos;        // rows >= pos are uninitialised or stale: never touch them
      vv[i] = ok ? src.load(t, k0, 4 * i + g) : make_float4(0.f, 0.f, 0.f, 0.f);
      pr[i] = ok ? ssc[key] : 0.f;
    }
    src.consumed(lane);
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      oa.x = fmaf(pr[i], vv[i].x, oa.x);
      oa.y = fmaf(pr[i], vv[i].y, oa.y);
      oa.z = fmaf(pr[i], vv[i].z, oa.z);
      oa.w = fmaf(pr[i], vv[i].w, oa.w);
    }
  });
  // sum the 4 key groups (lanes with equal b8), then hand channel `lane` its value
#pragma unroll
  for (int o_ = 8; o_ <= 16; o_ <<= 1) {
    oa.x += __shfl_xor_sync(0xffffffffu, oa.x, o_);
    oa.y += __shfl_xor_sync(0xffffffffu, oa.y, o_);
    oa.z += __shfl_xor_sync(0xffffffffu, oa.z, o_);
    oa.w += __shfl_xor_sync(0xffffffffu, oa.w, o_);
  }
  __syncwarp();
  if (lane < 8) reinterpret_cast<float4*>(sx)[lane] = oa;
  __syncwarp();
  return (sx[lane] + p_self * v) * inv;
}

// bf16 cache on the tensor cores (mma.sync m16n8k16, fp32 accumulate); same contract as attention_f32.  The decode is a
// GEMV per env (one query against that env's private keys), so the products are formed transposed -- keys / channels /
// outputs are the 16 rows of the A tile and the single query (or probability, or activation) vector is column 0 of B;
// what the MMA buys is instruction count: 2 HMMA replace ~180 unpack / FMA / shuffle instructions per 16 keys.
//   K cache: one 64 B row per key, channels permuted so that lane (g = lane/4, c = lane%4) reads the B
//            fragments of key g for both k-steps with ONE 16 B load (kperm below).
//   V cache: blocks of 16 keys x 32 channels (1 KB) stored as [channel-in-octet g][key pair c][octet j]
//            [keys 2c, 2c+1, 2c+8, 2c+9]: lane (g, c) reads the B fragments of all four channel octets with
//            two 16 B loads; a block is zeroed when its first key is appended (P = 0 must meet finite V).

// One token through all layers.  x: this lane's channel of the embedded token (+wpe).  kv: this sequence's cache
// (kv_seq_bytes).  sx[32], sh[128], ssc[Tpad]: per-warp shared scratch.  WS: the projections run on the tensor cores
// from bf16 weight fragments in shared memory (`wf`, all layers).  src: where the fp32 attention's K/V tiles come from.
template <bool BF16, bool WS = false, class Src = GlobalKv>
__device__ __forceinline__ float token_forward(const Gpt2Dev& m, float x, int pos, void* kv_, int Tpad, float* sx,
                                               float* sh, float* ssc, int lane, const uint4* wf = nullptr, Src&& src = {}) {
  using KvT = std::conditional_t<BF16, __nv_bfloat16, float>;
  src.begin_token(pos, lane);
  for (int l = 0; l < m.L; ++l) {
    const LayerW& w = m.layer[l];
    // ---- attention ----
    sx[lane] = layer_norm(x, w.ln1_w, w.ln1_b, lane);
    __syncwarp();
    float qkv[3];
    if constexpr (WS) {
      matvec_mma<G_E, 3 * G_E>(wf + l * WF_UINT4 + WF_QKV, sx, sh, lane);
      __syncwarp();
#pragma unroll
      for (int i = 0; i < 3; ++i) qkv[i] = sh[32 * i + lane] + __ldg(w.attn_b + 32 * i + lane);
    } else {
      matvec_packed<G_E, 3>(sx, w.attn_wP, w.attn_b, lane, qkv);
    }
    __syncwarp();
    KvT* K = reinterpret_cast<KvT*>(kv_) + (size_t)(l * 2) * G_E * Tpad;
    KvT* V = K + (size_t)G_E * Tpad;
    float o;
    if constexpr (BF16)
    {
      float q = qkv[0];
      const float k = qkv[1], v = qkv[2];
      const int g = lane >> 2, c = lane & 3;
      {
        const int r = lane & 15;
        const int kperm = ((r & 7) >> 1) * 8 + (lane >> 4) * 4 + (r >> 3) * 2 + (r & 1);
        K[(size_t)pos * G_E + kperm] = __float2bfloat16_rn(k);
        __nv_bfloat16* vb = V + (size_t)(pos >> 4) * 512;
        if ((pos & 15) == 0) {
          reinterpret_cast<uint4*>(vb)[2 * lane] = make_uint4(0, 0, 0, 0);
          reinterpret_cast<uint4*>(vb)[2 * lane + 1] = make_uint4(0, 0, 0, 0);
          __syncwarp();
        }
        const int kk = pos & 15;
        vb[(((lane & 7) * 4 + ((kk & 7) >> 1)) * 4 + (lane >> 3)) * 4 + (kk >> 3) * 2 + (kk & 1)] = __float2bfloat16_rn(v);
      }
      q *= 0.17677669529663687f;
      sx[lane] = q;
      __syncwarp();
      uint32_t qa0 = 0, qa1 = 0, qa2 = 0, qa3 = 0;   // q as column 0 of the B tile: k-step 0 (b0, b1), k-step 1 (b0, b1)
      if (lane < 4) {
        qa0 = pack_bf16(sx[2 * c], sx[2 * c + 1]), qa1 = pack_bf16(sx[2 * c + 8], sx[2 * c + 9]);
        qa2 = pack_bf16(sx[2 * c + 16], sx[2 * c + 17]), qa3 = pack_bf16(sx[2 * c + 24], sx[2 * c + 25]);
      }
      const uint4* K8 = reinterpret_cast<const uint4*>(K) + c;   // row stride = 4 uint4
      __syncwarp();
      // 64 keys per tile; TAIL = the last, partial tile: load instruction i covers keys k0 + 8 i .. k0 + 8 i + 7, instructions
      // past the last key are skipped with a warp-uniform predicate (the padded rows were 6.2 % of the DRAM traffic)
      float lmax = -INFINITY;
      for_each_key_tile<64>(pos, [&](const int k0, auto tail_tag) {
        constexpr bool TAIL = decltype(tail_tag)::value;
        const int r = pos - k0;
        uint4 kk[8];
    #pragma unroll
        for (int i = 0; i < 8; ++i)
          kk[i] = (!TAIL || 8 * i < r) ? __ldcg(K8 + (size_t)(k0 + 8 * i + g) * 4) : make_uint4(0u, 0u, 0u, 0u);   // in bounds (Tpad % 64 == 0)
        // (an L2 prefetch of the same 64 keys' V blocks here was measured slower: 161 ms with, 155 ms without, C4)
        // scores^T = K q^T: 16 keys are the rows of the A tile (octets 2m and 2m + 1), q is column 0 of B
    #pragma unroll
        for (int mt = 0; mt < 4; ++mt) {
          if (TAIL && 16 * mt >= r) break;        // (warp-uniform)
          float d[4] = {0.f, 0.f, 0.f, 0.f};
          mma_bf16_16816(d, kk[2 * mt].x, kk[2 * mt + 1].x, kk[2 * mt].y, kk[2 * mt + 1].y, qa0, qa1);
          mma_bf16_16816(d, kk[2 * mt].z, kk[2 * mt + 1].z, kk[2 * mt].w, kk[2 * mt + 1].w, qa2, qa3);
          const int key = k0 + 16 * mt + g;       // column 0 of the tile: lanes with c == 0 hold keys g and g + 8
          if (c == 0) {
            if (!TAIL || key < pos) ssc[key] = d[0], lmax = fmaxf(lmax, d[0]);
            if (!TAIL || key + 8 < pos) ssc[key + 8] = d[2], lmax = fmaxf(lmax, d[2]);
          }
        }
      });
      const float s_self = warp_sum(q * k);
      lmax = fmaxf(warp_max(lmax), s_self);
      __syncwarp();
      float lsum = 0.f;
      for (int key = lane; key < pos; key += 32) {
        // the normaliser uses the bf16-rounded probabilities that the tensor core will see
        const float pr = __bfloat162float(__float2bfloat16_rn(expf(ssc[key] - lmax)));
        ssc[key] = pr;
        lsum += pr;
      }
      for (int key = pos + lane; key < ((pos + 15) & ~15); key += 32) ssc[key] = 0.f;   // tail of the last key block
      const float p_self = expf(s_self - lmax);
      const float inv = 1.0f / (warp_sum(lsum) + p_self);
      __syncwarp();
      float oa[2][4];   // out^T = V^T p^T: channel tiles 0..15 and 16..31 are the rows, p is column 0 of B
    #pragma unroll
      for (int jn = 0; jn < 2; ++jn) oa[jn][0] = oa[jn][1] = oa[jn][2] = oa[jn][3] = 0.f;
      const uint4* VB = reinterpret_cast<const uint4*>(V) + 2 * lane;   // block stride = 64 uint4
      for (int k0 = 0; k0 < pos; k0 += 64) {
        uint4 va[4], vc[4];
    #pragma unroll
        for (int i = 0; i < 4; ++i) {
          const bool ok = k0 + 16 * i < pos;          // blocks past the last key are uninitialised: never touch them
          va[i] = ok ? __ldcg(VB + (size_t)((k0 >> 4) + i) * 64) : make_uint4(0, 0, 0, 0);
          vc[i] = ok ? __ldcg(VB + (size_t)((k0 >> 4) + i) * 64 + 1) : make_uint4(0, 0, 0, 0);
        }
    #pragma unroll
        for (int i = 0; i < 4; ++i) {
          uint32_t pa0 = 0, pa2 = 0;
          if (lane < 4 && k0 + 16 * i < pos) {
            const float2 p0 = *reinterpret_cast<const float2*>(ssc + k0 + 16 * i + 2 * c);
            const float2 p1 = *reinterpret_cast<const float2*>(ssc + k0 + 16 * i + 8 + 2 * c);
            pa0 = pack_bf16(p0.x, p0.y), pa2 = pack_bf16(p1.x, p1.y);
          }
          mma_bf16_16816(oa[0], va[i].x, va[i].z, va[i].y, va[i].w, pa0, pa2);
          mma_bf16_16816(oa[1], vc[i].x, vc[i].z, vc[i].y, vc[i].w, pa0, pa2);
        }
      }
      __syncwarp();
      if (c == 0) {   // column 0 of the output tiles: lane (g, 0) holds channels 16 jn + g and 16 jn + g + 8
    #pragma unroll
        for (int jn = 0; jn < 2; ++jn) sx[16 * jn + g] = oa[jn][0], sx[16 * jn + 8 + g] = oa[jn][2];
      }
      __syncwarp();
      o = (sx[lane] + p_self * v) * inv;
    }
    else
      o = attention_f32(qkv[0], qkv[1], qkv[2], pos, K, V, sx, ssc, lane, src);
    __syncwarp();
    sx[lane] = o;
    __syncwarp();
    float y;
    if constexpr (WS) {
      matvec_mma<G_E, G_E>(wf + l * WF_UINT4 + WF_PROJ, sx, sh, lane);
      __syncwarp();
      y = sh[lane] + __ldg(w.proj_b + lane);
    } else {
      matvec_packed<G_E, 1>(sx, w.proj_wP, w.proj_b, lane, &y);
    }
    x += y;
    __syncwarp();
    // ---- MLP ----
    sx[lane] = layer_norm(x, w.ln2_w, w.ln2_b, lane);
    __syncwarp();
    float hh[4];
    if constexpr (WS) {
      matvec_mma<G_E, G_FF>(wf + l * WF_UINT4 + WF_FC, sx, sh, lane);
      __syncwarp();
#pragma unroll
      for (int i = 0; i < 4; ++i) hh[i] = sh[32 * i + lane] + __ldg(w.fc_b + 32 * i + lane);
    } else {
      matvec_packed<G_E, 4>(sx, w.fc_wP, w.fc_b, lane, hh);
    }
    sh[lane] = gelu_new(hh[0]), sh[32 + lane] = gelu_new(hh[1]), sh[64 + lane] = gelu_new(hh[2]), sh[96 + lane] = gelu_new(hh[3]);
    __syncwarp();
    float y2;
    if constexpr (WS) {
      matvec_mma<G_FF, G_E>(wf + l * WF_UINT4 + WF_FC2, sh, sx, lane);
      __syncwarp();
      y2 = sx[lane] + __ldg(w.fc2_b + lane);
    } else {
      matvec_packed<G_FF, 1>(sh, w.fc2_wP, w.fc2_b, lane, &y2);
    }
    x += y2;
    __syncwarp();
  }
  src.end_token();
  return x;
}

// ln_f + pred_actions: returns logit[lane] for lane < du (others 0)
__device__ __forceinline__ float head_logits(const Gpt2Dev& m, float x, float* sx, int lane) {
  sx[lane] = layer_norm(x, m.lnf_w, m.lnf_b, lane);
  __syncwarp();
  float lg = 0.f;
  if (lane < m.du) {
    lg = __ldg(m.pred_b + lane);
    for (int c = 0; c < G_E; ++c) lg = fmaf(sx[c], __ldg(m.pred_wT + c * m.du + lane), lg);
  }
  __syncwarp();
  return lg;
}

struct WarpScratch {
  float* sx;
  float* sh;
  float* ssc;
};
__host__ __device__ __forceinline__ size_t warp_scratch_bytes(int Tpad) { return (size_t)(G_E + G_FF + Tpad) * sizeof(float); }
__device__ __forceinline__ WarpScratch warp_scratch(float* smem, int warp, int Tpad) {
  float* base = smem + (size_t)warp * (G_E + G_FF + Tpad);
  return WarpScratch{base, base + G_E, base + G_E + G_FF};
}

// ---------------------------------------------------------------------------------------------
// Transformer.forward(x)
// ---------------------------------------------------------------------------------------------
struct ForwardParams {
  Gpt2Dev m;
  const float *query, *cs, *ca, *cns, *cr;
  int B, T, Ts, test, Tpad, share;
  float* out;
  void* kv;
};

template <bool BF16>
__global__ void __launch_bounds__(G_THREADS) gpt2_forward_kernel(const ForwardParams p) {
  extern __shared__ __align__(16) float g_smem[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int b = blockIdx.x * G_WARPS + warp;
  if (b >= p.B) return;
  const Gpt2Dev& m = p.m;
  const WarpScratch ws = warp_scratch(g_smem, warp, p.Tpad);
  char* kv = reinterpret_cast<char*>(p.kv) + (size_t)b * kv_seq_bytes(m.L, p.Tpad, BF16);
  const int dx = m.dx, du = m.du, din = m.din;
  for (int pos = 0; pos <= p.T; ++pos) {
    // token = [state | action | next_state | reward]; position 0 = query state, zeros elsewhere (models/net.py:45-53)
    float tok = 0.f;
    if (lane < din) {
      if (pos == 0) {
        tok = lane < dx ? p.query[(size_t)b * dx + lane] : 0.f;
      } else {
        const size_t row = (size_t)(b / p.share) * p.Ts + (pos - 1);
        if (lane < dx)
          tok = p.cs[row * dx + lane];
        else if (lane < dx + du)
          tok = p.ca[row * du + (lane - dx)];
        else if (lane < 2 * dx + du)
          tok = p.cns[row * dx + (lane - dx - du)];
        else
          tok = p.cr[row];
      }
    }
    float x = __ldg(m.embed_b + lane) + __ldg(m.wpe + (size_t)pos * G_E + lane);
    for (int i = 0; i < din; ++i) x = fmaf(__shfl_sync(0xffffffffu, tok, i), __ldg(m.embed_wT + i * G_E + lane), x);
    x = token_forward<BF16>(m, x, pos, kv, p.Tpad, ws.sx, ws.sh, ws.ssc, lane);
    if (p.test ? (pos == p.T) : (pos >= 1)) {
      const float lg = head_logits(m, x, ws.sx, lane);
      if (lane < du) {
        if (p.test)
          p.out[(size_t)b * du + lane] = lg;
        else
          p.out[((size_t)b * p.T + (pos - 1)) * du + lane] = lg;
      }
    }
  }
}

// ---------------------------------------------------------------------------------------------
// One decode step for callers that drive their own loop (interactive trainers' rollout half): append the token of
// position `pos` to each sequence's K/V cache and return the logits at that position.
// ---------------------------------------------------------------------------------------------
struct StepParams {
  Gpt2Dev m;
  const float* tokens;   // [N, din]: [state | action | next_state | reward]; position 0 = [query state, 0, ...]
  int N, pos, Tpad;
  float* out;            // [N, du]
  void* kv;
};

template <bool BF16>
__global__ void __launch_bounds__(G_THREADS) gpt2_decode_step_kernel(const StepParams p) {
  extern __shared__ __align__(16) float g_smem[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int b = blockIdx.x * G_WARPS + warp;
  if (b >= p.N) return;
  const Gpt2Dev& m = p.m;
  const WarpScratch ws = warp_scratch(g_smem, warp, p.Tpad);
  char* kv = reinterpret_cast<char*>(p.kv) + (size_t)b * kv_seq_bytes(m.L, p.Tpad, BF16);
  const float tok = lane < m.din ? p.tokens[(size_t)b * m.din + lane] : 0.f;
  float x = __ldg(m.embed_b + lane) + __ldg(m.wpe + (size_t)p.pos * G_E + lane);
  for (int i = 0; i < m.din; ++i) x = fmaf(__shfl_sync(0xffffffffu, tok, i), __ldg(m.embed_wT + i * G_E + lane), x);
  x = token_forward<BF16>(m, x, p.pos, kv, p.Tpad, ws.sx, ws.sh, ws.ssc, lane);
  const float lg = head_logits(m, x, ws.sx, lane);
  if (lane < m.du) p.out[(size_t)b * m.du + lane] = lg;
}

// ---------------------------------------------------------------------------------------------
// Fused bandit online loop with the transformer controller
// ---------------------------------------------------------------------------------------------
// The online loop's launch parameters.  NM: member capacity of the launch -- 1 for a one-model dpt_gpt2_online_loop call,
// ONLINE_POP_MAX for a population call, whose CTA (env block, member = blockIdx.y) takes its member's weights, K/V region
// and outputs from a table in the kernel parameters (no upload, graph-capturable).  The means, noise and inject arrays
// are shared: member i computes exactly what a one-model call on its own weights would.
constexpr int ONLINE_POP_MAX = DPT_GPT2_ONLINE_POPULATION_MAX;
struct OnlineMember {   // what differs between the members of a population launch
  Gpt2Dev m;
  void* kv;
  float *ctx_s, *ctx_a, *ctx_ns, *ctx_r, *cum_means;
  double* regret;
  dpt_gpt2_online_dump_t out;
};
template <int NM>
struct OnlineGptParams {
  const float* means;
  double var;
  int rtype;   // DPT_REWARD_*
  int sample;
  Key key;
  uint64_t env_id0;
  int N, H, Tpad;
  dpt_gpt2_online_inject_t in;
  OnlineMember mem[NM];
  __device__ __forceinline__ const OnlineMember& member() const { return mem[blockIdx.y]; }
  OnlineMember& slot(int i) { return mem[i]; }
};
static_assert(sizeof(OnlineGptParams<ONLINE_POP_MAX>) <= 32764, "population table exceeds the kernel parameter limit");
// one model: the fields of OnlineMember and the shared ones in one block (the layout the one-model kernels were tuned with)
template <>
struct OnlineGptParams<1> {
  Gpt2Dev m;
  const float* means;
  double var;
  int rtype;   // DPT_REWARD_*
  int sample;
  Key key;
  uint64_t env_id0;
  int N, H, Tpad;
  void* kv;
  float *ctx_s, *ctx_a, *ctx_ns, *ctx_r, *cum_means;
  double* regret;
  dpt_gpt2_online_inject_t in;
  dpt_gpt2_online_dump_t out;
  __device__ __forceinline__ const OnlineGptParams& member() const { return *this; }
  OnlineGptParams& slot(int) { return *this; }
};

// WS (precision 1): ONE CTA of GW_WARPS warps per SM shares the bf16 weight fragments of all layers in shared memory
// (24 KB per layer) and every warp runs its env's projections on the tensor cores from there.
constexpr int GW_WARPS = 24;
constexpr int GW_THREADS = GW_WARPS * 32;

// TMA (precision 0 only): the fp32 K/V stream is staged through a per-warp ring of bulk-async copies (KvRing)
template <bool BF16, bool WS, bool TMA = false, int NM = 1>
__global__ void __launch_bounds__(WS ? GW_THREADS : (TMA ? TMA_WARPS * 32 : G_THREADS),
                                  WS ? 1 : (TMA ? TMA_MINB : (BF16 ? GPT2_MINB_BF16 : GPT2_MINB_F32)))
    gpt2_online_kernel(const __grid_constant__ OnlineGptParams<NM> p) {
  extern __shared__ __align__(128) float g_smem[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const auto& mb = p.member();   // this CTA's member
  const Gpt2Dev& m = mb.m;
  const uint4* wf = nullptr;
  float* scratch = g_smem;
  std::conditional_t<TMA, KvRing, GlobalKv> kv_src;
  if constexpr (TMA) {   // [warps][KV_STAGES] tiles of 4 KB | [warps][KV_STAGES] mbarriers | per-warp scratch
    const int nw = blockDim.x >> 5;
    unsigned char* base = reinterpret_cast<unsigned char*>(g_smem);
    uint64_t* bars = reinterpret_cast<uint64_t*>(base + (size_t)nw * KV_STAGES * KV_TILE_BYTES);
    if (threadIdx.x < nw * KV_STAGES)
      asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_addr(bars + threadIdx.x)) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    __syncthreads();
    kv_src.stage0 = smem_addr(base + (size_t)warp * KV_STAGES * KV_TILE_BYTES);
    kv_src.bar0 = smem_addr(bars + warp * KV_STAGES);
    kv_src.is = kv_src.cs = kv_src.cp = 0;
    kv_src.L = m.L, kv_src.Tpad = p.Tpad;
    scratch = reinterpret_cast<float*>(bars + ((nw * KV_STAGES + 1) & ~1));   // keep the per-warp scratch 16 B aligned
  }
  if constexpr (WS) {
    uint4* dst = reinterpret_cast<uint4*>(g_smem);
    for (int l = 0; l < m.L; ++l)
      for (int i = threadIdx.x; i < WF_UINT4; i += blockDim.x) dst[l * WF_UINT4 + i] = __ldg(m.layer[l].wfrag + i);
    wf = dst;
    scratch = g_smem + (size_t)m.L * WF_UINT4 * 4;
    __syncthreads();
  }
  const int env = blockIdx.x * (int)(blockDim.x >> 5) + warp;   // WS: the host picks <= GW_WARPS warps per CTA
  if (env >= p.N) return;
  const WarpScratch ws = warp_scratch(scratch, warp, p.Tpad);
  char* kv = reinterpret_cast<char*>(mb.kv) + (size_t)env * kv_seq_bytes(m.L, p.Tpad, BF16);
  if constexpr (TMA) kv_src.kv = reinterpret_cast<const float*>(kv);
  const int du = m.du, H = p.H, N = p.N;
  const uint64_t gid = p.env_id0 + (uint64_t)env;
  const float mean_l = lane < du ? p.means[(size_t)env * du + lane] : -INFINITY;
  const float mmax = warp_max(mean_l);
  if (mb.ctx_s) {
    for (int h = lane; h < H; h += 32) {
      mb.ctx_s[(size_t)env * H + h] = 1.0f;
      mb.ctx_ns[(size_t)env * H + h] = 1.0f;
    }
  }
  // constant part of every token: bias + state (== 1) column (+ next_state column for context tokens)
  const float e_state = __ldg(m.embed_wT + 0 * G_E + lane);
  const float e_next = __ldg(m.embed_wT + (1 + du) * G_E + lane);
  const float e_rew = __ldg(m.embed_wT + (2 + du) * G_E + lane);
  const float e_bias = __ldg(m.embed_b + lane);
  int a_prev = 0;
  float r_prev = 0.f, z_next = 0.f;
  double creg = 0.0;
  for (int h = 0; h < H; ++h) {
    float x = e_bias + e_state + __ldg(m.wpe + (size_t)h * G_E + lane);
    if (h > 0) x += __ldg(m.embed_wT + (1 + a_prev) * G_E + lane) + e_next + e_rew * r_prev;
    x = token_forward<BF16, WS>(m, x, h, kv, p.Tpad, ws.sx, ws.sh, ws.ssc, lane, wf, kv_src);
    const float lg = head_logits(m, x, ws.sx, lane);
    if (mb.out.logits && lane < du) mb.out.logits[((size_t)h * N + env) * du + lane] = lg;
    int a;
    if (p.sample) {
      // scipy.special.softmax (float64) + np.random.choice(p): cdf = cumsum(p) / cdf[-1]; searchsorted(u, 'right')
      const float lm = warp_max(lane < du ? lg : -INFINITY);
      const double pe = lane < du ? exp((double)lg - (double)lm) : 0.0;
      double tot = 0.0;
      for (int j = 0; j < du; ++j) tot = __dadd_rn(tot, __shfl_sync(0xffffffffu, pe, j));
      const double pj = __ddiv_rn(pe, tot);
      double acc = 0.0, cdf = 0.0;
      for (int j = 0; j < du; ++j) {
        const double v = __shfl_sync(0xffffffffu, pj, j);
        acc = (j == 0) ? v : __dadd_rn(acc, v);
        if (j == lane) cdf = acc;
      }
      const double last = __shfl_sync(0xffffffffu, cdf, du - 1);
      cdf = __ddiv_rn(cdf, last);
      double u;
      if (p.in.ctrl_u) {
        u = p.in.ctrl_u[(size_t)h * N + env];
      } else {  // 53-bit uniform in [0,1) from two words, like numpy's random_sample
        const uint4 w = philox_words(p.key, gid, (uint32_t)h, STREAM_CTRL);
        u = ((double)(w.x >> 5) * 67108864.0 + (double)(w.y >> 6)) * (1.0 / 9007199254740992.0);
      }
      if (mb.out.ctrl_u && lane == 0) mb.out.ctrl_u[(size_t)h * N + env] = u;
      a = __popc(__ballot_sync(0xffffffffu, lane < du - 1 && cdf <= u));
    } else {  // np.argmax: first maximum
      const float lm = warp_max(lane < du ? lg : -INFINITY);
      a = __ffs(__ballot_sync(0xffffffffu, lane < du && lg == lm)) - 1;
    }
    float z;
    if (p.in.reward_z) {
      z = p.in.reward_z[(size_t)h * N + env];
    } else if ((h & 1) == 0) {
      const uint4 w = philox_words(p.key, gid, (uint32_t)(h >> 1), STREAM_ENV_REWARD);
      if (p.rtype == DPT_REWARD_GAUSSIAN)
        box_muller(w.z, w.w, z, z_next);
      else
        z = u24(w.z), z_next = u24(w.w);
    } else {
      z = z_next;
    }
    const float ma = __shfl_sync(0xffffffffu, mean_l, a);
    const float r = p.rtype == DPT_REWARD_GAUSSIAN ? (float)((double)ma + (0.0 + p.var * (double)z))   // envs/bandit_env.py:59
                                                   : (z < ma ? 1.f : 0.f);                             // :61 Bernoulli(mean)
    if (lane == 0) {
      if (mb.out.reward_z) mb.out.reward_z[(size_t)h * N + env] = z;
      if (mb.cum_means) mb.cum_means[(size_t)h * N + env] = ma;
      if (mb.regret) {
        const double reg = (double)mmax - (double)ma;
        creg += reg;
        double* dst = mb.regret + 4 * (size_t)h;
        atomicAdd(dst, reg), atomicAdd(dst + 1, reg * reg), atomicAdd(dst + 2, creg), atomicAdd(dst + 3, creg * creg);
      }
      if (mb.ctx_r) mb.ctx_r[(size_t)env * H + h] = r;
    }
    if (mb.ctx_a && lane < du) mb.ctx_a[((size_t)env * H + h) * du + lane] = (lane == a) ? 1.f : 0.f;
    a_prev = a;
    r_prev = r;
  }
}

// ---------------------------------------------------------------------------------------------
// Fused explorer / exploiter rollout (the no-grad half of an episode of train_explorer_exploiter.py:110-166): ONE launch for all
// K steps.  One warp per env, two models with their own K/V caches.  Per step t both models score the context so far (token t =
// query token at t = 0, else transition t - 1), the explorer's sampled arm is what gets RECORDED in the context (:131-136, :155)
// while the env is stepped with a uniformly random arm (:137-152), and the advantage of step t - 1 is the change of the
// exploiter's cross-entropy against the optimal arm (:158-164).  The exploiter's own sample (:141-146) is never used by the
// reference and is not drawn.  Draws: Philox block (step t, STREAM_CTRL): words x, y -> the 53-bit uniform of the explorer's
// categorical draw (same float64 cdf rule as the online loop), word z -> the random arm (z * du) >> 32; reward noise as in the
// online loop (one block per step pair on STREAM_ENV_REWARD).
// ---------------------------------------------------------------------------------------------
struct ExploreParams {
  Gpt2Dev me, mx;   // explorer, exploiter
  const float* means;
  double var;
  int rtype;
  Key key;
  uint64_t env_id0;
  int N, K, Tpad;
  void *kv_e, *kv_x;
  float *ctx_s, *ctx_a, *ctx_ns, *ctx_r;
  float* adv;       // [N, K - 1]
  dpt_explore_inject_t in;
  dpt_explore_dump_t out;
};

__global__ void __launch_bounds__(G_THREADS, GPT2_MINB_F32) gpt2_explore_exploit_kernel(const ExploreParams p) {
  extern __shared__ __align__(128) float g_smem[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int env = blockIdx.x * G_WARPS + warp;
  if (env >= p.N) return;
  const Gpt2Dev& me = p.me;
  const Gpt2Dev& mx = p.mx;
  const WarpScratch ws = warp_scratch(g_smem, warp, p.Tpad);
  char* kve = reinterpret_cast<char*>(p.kv_e) + (size_t)env * kv_seq_bytes(me.L, p.Tpad, false);
  char* kvx = reinterpret_cast<char*>(p.kv_x) + (size_t)env * kv_seq_bytes(mx.L, p.Tpad, false);
  const int du = me.du, K = p.K, N = p.N;
  const uint64_t gid = p.env_id0 + (uint64_t)env;
  const float mean_l = lane < du ? p.means[(size_t)env * du + lane] : -INFINITY;
  const float mmax = warp_max(mean_l);
  const int target = __ffs(__ballot_sync(0xffffffffu, lane < du && mean_l == mmax)) - 1;   // opt_a_index: first maximum
  for (int h = lane; h < K; h += 32) {
    p.ctx_s[(size_t)env * K + h] = 1.0f;
    p.ctx_ns[(size_t)env * K + h] = 1.0f;
  }
  // constant parts of a token, per model: bias + state (== 1) column (+ next_state column for transition tokens)
  const float ee_state = __ldg(me.embed_wT + lane), ee_next = __ldg(me.embed_wT + (1 + du) * G_E + lane);
  const float ee_rew = __ldg(me.embed_wT + (2 + du) * G_E + lane), ee_bias = __ldg(me.embed_b + lane);
  const float ex_state = __ldg(mx.embed_wT + lane), ex_next = __ldg(mx.embed_wT + (1 + du) * G_E + lane);
  const float ex_rew = __ldg(mx.embed_wT + (2 + du) * G_E + lane), ex_bias = __ldg(mx.embed_b + lane);
  int a_prev = 0;
  float r_prev = 0.f, z_next = 0.f, loss_prev = 0.f;
  for (int h = 0; h < K; ++h) {
    // ---- explorer: logits at position h, sampled arm (recorded) -----------------------------
    float x = ee_bias + ee_state + __ldg(me.wpe + (size_t)h * G_E + lane);
    if (h > 0) x += __ldg(me.embed_wT + (1 + a_prev) * G_E + lane) + ee_next + ee_rew * r_prev;
    x = token_forward<false>(me, x, h, kve, p.Tpad, ws.sx, ws.sh, ws.ssc, lane);
    const float lge = head_logits(me, x, ws.sx, lane);
    if (p.out.logits_explorer && lane < du) p.out.logits_explorer[((size_t)h * N + env) * du + lane] = lge;
    const uint4 w = philox_words(p.key, gid, (uint32_t)h, STREAM_CTRL);
    int a;
    {
      const float lm = warp_max(lane < du ? lge : -INFINITY);
      const double pe = lane < du ? exp((double)lge - (double)lm) : 0.0;
      double tot = 0.0;
      for (int j = 0; j < du; ++j) tot = __dadd_rn(tot, __shfl_sync(0xffffffffu, pe, j));
      const double pj = __ddiv_rn(pe, tot);
      double acc = 0.0, cdf = 0.0;
      for (int j = 0; j < du; ++j) {
        const double v = __shfl_sync(0xffffffffu, pj, j);
        acc = (j == 0) ? v : __dadd_rn(acc, v);
        if (j == lane) cdf = acc;
      }
      const double last = __shfl_sync(0xffffffffu, cdf, du - 1);
      cdf = __ddiv_rn(cdf, last);
      const double u = p.in.ctrl_u ? p.in.ctrl_u[(size_t)h * N + env]
                                   : ((double)(w.x >> 5) * 67108864.0 + (double)(w.y >> 6)) * (1.0 / 9007199254740992.0);
      if (p.out.ctrl_u && lane == 0) p.out.ctrl_u[(size_t)h * N + env] = u;
      a = __popc(__ballot_sync(0xffffffffu, lane < du - 1 && cdf <= u));
    }
    // ---- exploiter: logits at position h, cross-entropy against the optimal arm --------------
    float y = ex_bias + ex_state + __ldg(mx.wpe + (size_t)h * G_E + lane);
    if (h > 0) y += __ldg(mx.embed_wT + (1 + a_prev) * G_E + lane) + ex_next + ex_rew * r_prev;
    y = token_forward<false>(mx, y, h, kvx, p.Tpad, ws.sx, ws.sh, ws.ssc, lane);
    const float lgx = head_logits(mx, y, ws.sx, lane);
    if (p.out.logits_exploiter && lane < du) p.out.logits_exploiter[((size_t)h * N + env) * du + lane] = lgx;
    const float lmx = warp_max(lane < du ? lgx : -INFINITY);
    const float loss = lmx + logf(warp_sum(lane < du ? expf(lgx - lmx) : 0.f)) - __shfl_sync(0xffffffffu, lgx, target);
    if (h > 0 && lane == 0) p.adv[(size_t)env * (K - 1) + (h - 1)] = loss - loss_prev;   // :160-164
    loss_prev = loss;
    // ---- env step with a uniformly random arm -----------------------------------------------
    const int ar = p.in.random_arm ? p.in.random_arm[(size_t)h * N + env] : (int)bounded(w.z, (uint32_t)du);
    float z;
    if (p.in.reward_z) {
      z = p.in.reward_z[(size_t)h * N + env];
    } else if ((h & 1) == 0) {
      const uint4 wr = philox_words(p.key, gid, (uint32_t)(h >> 1), STREAM_ENV_REWARD);
      if (p.rtype == DPT_REWARD_GAUSSIAN)
        box_muller(wr.z, wr.w, z, z_next);
      else
        z = u24(wr.z), z_next = u24(wr.w);
    } else {
      z = z_next;
    }
    const float ma = __shfl_sync(0xffffffffu, mean_l, ar);
    const float r = p.rtype == DPT_REWARD_GAUSSIAN ? (float)((double)ma + (0.0 + p.var * (double)z)) : (z < ma ? 1.f : 0.f);
    if (lane == 0) {
      if (p.out.reward_z) p.out.reward_z[(size_t)h * N + env] = z;
      if (p.out.random_arm) p.out.random_arm[(size_t)h * N + env] = ar;
      p.ctx_r[(size_t)env * K + h] = r;
    }
    if (lane < du) p.ctx_a[((size_t)env * K + h) * du + lane] = (lane == a) ? 1.f : 0.f;   // the EXPLORER's arm is recorded (:155)
    a_prev = a;
    r_prev = r;
  }
}

__global__ void transpose_kernel(const float* src, float* dst, int rows, int cols) {  // dst[c][r] = src[r][c]
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < rows * cols) dst[(i % cols) * rows + i / cols] = src[i];
}

// dst[((iq * G + g) * 32 + lane) * 4 + r] = src[(4 iq + r) * Out + g * 32 + lane],  G = Out / 32
__global__ void pack_quads_kernel(const float* src, float* dst, int In, int Out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= In * Out) return;
  const int r = i & 3, lane = (i >> 2) & 31, rest = i >> 7;
  const int G = Out / 32, g = rest % G, iq = rest / G;
  dst[i] = src[(size_t)(4 * iq + r) * Out + g * 32 + lane];
}

static int tpad_for(int T1, int precision) { return precision ? (T1 + 63) & ~63 : (T1 + 31) & ~31; }

}  // namespace dpt

using namespace dpt;

extern "C" int dpt_gpt2_create(const dpt_gpt2_weights_t* w, dpt_gpt2_t** out, void* stream) {
  DPT_CHECK_ARG(w && out, "dpt_gpt2_create: null argument");
  DPT_CHECK_ARG(w->n_embd == G_E, "dpt_gpt2_create: n_embd=%d, this build supports n_embd == %d (head_dim == warp width)",
                w->n_embd, G_E);
  DPT_CHECK_ARG(w->n_layer >= 1 && w->n_layer <= G_MAX_L, "dpt_gpt2_create: n_layer=%d outside [1,%d]", w->n_layer, G_MAX_L);
  const int din = 2 * w->state_dim + w->action_dim + 1;
  DPT_CHECK_ARG(w->state_dim >= 1 && w->action_dim >= 1 && din <= 32,
                "dpt_gpt2_create: token width 2*state_dim+action_dim+1 = %d must be <= 32", din);
  DPT_CHECK_ARG(w->n_positions >= 1 && w->wpe && w->embed_w && w->embed_b && w->pred_w && w->pred_b && w->lnf_w && w->lnf_b,
                "dpt_gpt2_create: null weight pointer");
  cudaStream_t st = (cudaStream_t)stream;
  const int L = w->n_layer, du = w->action_dim;
  const size_t per_layer = 4 * G_E + G_E * 3 * G_E + 3 * G_E + G_E * G_E + G_E + G_E * G_FF + G_FF + G_FF * G_E + G_E;
  const size_t total = (size_t)w->n_positions * G_E + (size_t)din * G_E + G_E + (size_t)G_E * du + du + 2 * G_E + L * (2 * per_layer + WIMG_BYTES / 4 + WF_UINT4 * 4) + 4 * (16 + 18 * (size_t)L);
  struct Guard {   // frees the half-built model on every early return below
    dpt_gpt2* m;
    ~Guard() {
      if (m) {
        cudaFree(m->blob);
        delete m;
      }
    }
  } guard{new dpt_gpt2()};
  dpt_gpt2* m = guard.m;
  m->blob = nullptr;
  DPT_CUDA(cudaMalloc(&m->blob, total * sizeof(float)));
  float* cur = m->blob;
  auto take = [&](size_t n) {
    float* p = cur;
    cur += (n + 3) & ~size_t(3);
    return p;
  };
  auto copy = [&](const float* src, size_t n) {
    float* d = take(n);
    cudaMemcpyAsync(d, src, n * sizeof(float), cudaMemcpyDeviceToDevice, st);
    return (const float*)d;
  };
  Gpt2Dev& d = m->dev;
  d.L = L, d.dx = w->state_dim, d.du = du, d.din = din, d.H = w->horizon, d.n_pos = w->n_positions;
  d.wpe = copy(w->wpe, (size_t)w->n_positions * G_E);
  float* ewT = take((size_t)din * G_E);  // embed_transition.weight [E, din] -> [din, E]
  transpose_kernel<<<(G_E * din + 255) / 256, 256, 0, st>>>(w->embed_w, ewT, G_E, din);
  d.embed_wT = ewT;
  d.embed_b = copy(w->embed_b, G_E);
  float* pwT = take((size_t)G_E * du);   // pred_actions.weight [du, E] -> [E, du]
  transpose_kernel<<<(G_E * du + 255) / 256, 256, 0, st>>>(w->pred_w, pwT, du, G_E);
  d.pred_wT = pwT;
  d.pred_b = copy(w->pred_b, du);
  d.lnf_w = copy(w->lnf_w, G_E);
  d.lnf_b = copy(w->lnf_b, G_E);
  WimgPackParams<1> pk{};
  for (int l = 0; l < L; ++l) {
    LayerW& lw = d.layer[l];
    DPT_CHECK_ARG(w->ln1_w[l] && w->attn_w[l] && w->proj_w[l] && w->fc_w[l] && w->fc2_w[l], "dpt_gpt2_create: null layer %d weight", l);
    lw.ln1_w = copy(w->ln1_w[l], G_E), lw.ln1_b = copy(w->ln1_b[l], G_E);
    auto pack = [&](const float* src, int In, int Out) {
      float* d = take((size_t)In * Out);
      pack_quads_kernel<<<(In * Out + 255) / 256, 256, 0, st>>>(src, d, In, Out);
      return reinterpret_cast<const float4*>(d);
    };
    lw.attn_wP = pack(w->attn_w[l], G_E, 3 * G_E), lw.attn_b = copy(w->attn_b[l], 3 * G_E);
    lw.proj_wP = pack(w->proj_w[l], G_E, G_E), lw.proj_b = copy(w->proj_b[l], G_E);
    lw.ln2_w = copy(w->ln2_w[l], G_E), lw.ln2_b = copy(w->ln2_b[l], G_E);
    lw.fc_wP = pack(w->fc_w[l], G_E, G_FF), lw.fc_b = copy(w->fc_b[l], G_FF);
    lw.fc2_wP = pack(w->fc2_w[l], G_FF, G_E), lw.fc2_b = copy(w->fc2_b[l], G_E);
    lw.attn_w = copy(w->attn_w[l], G_E * 3 * G_E), lw.proj_w = copy(w->proj_w[l], G_E * G_E);
    lw.fc_w = copy(w->fc_w[l], G_E * G_FF), lw.fc2_w = copy(w->fc2_w[l], G_FF * G_E);
    unsigned char* img = reinterpret_cast<unsigned char*>(take(WIMG_BYTES / 4));   // tcgen05 B-operand image (bf16)
    pk.w[0][l][0] = w->attn_w[l], pk.w[0][l][1] = w->proj_w[l], pk.w[0][l][2] = w->fc_w[l], pk.w[0][l][3] = w->fc2_w[l];
    pk.img[0][l] = img;
    lw.wimg = reinterpret_cast<const uint4*>(img);
    uint4* frag = reinterpret_cast<uint4*>(take((size_t)WF_UINT4 * 4));                // mma.sync B fragments (bf16)
    auto packf = [&](const float* src, int K, int N, int off) {
      const int n = (K / 16) * (N / 16) * 32;
      pack_wfrag_kernel<<<(n + 255) / 256, 256, 0, st>>>(src, frag + off, K, N);
    };
    packf(w->attn_w[l], G_E, 3 * G_E, WF_QKV), packf(w->proj_w[l], G_E, G_E, WF_PROJ);
    packf(w->fc_w[l], G_E, G_FF, WF_FC), packf(w->fc2_w[l], G_FF, G_E, WF_FC2);
    lw.wfrag = frag;
  }
  const int rc = gpt2_pack_wimg<1>(pk, L, 1, st);   // every layer's image in one launch
  if (rc != DPT_OK) return rc;
  DPT_LAUNCH_CHECK();
  guard.m = nullptr;
  *out = m;
  return DPT_OK;
}

extern "C" int dpt_gpt2_destroy(dpt_gpt2_t* m) {
  if (!m) return DPT_OK;
  cudaFree(m->blob);
  delete m;
  return DPT_OK;
}

extern "C" uint64_t dpt_gpt2_forward_workspace_bytes(const dpt_gpt2_t* m, int B, int T, int precision) {
  if (!m || B <= 0 || T < 0) return 0;
  return (uint64_t)B * kv_seq_bytes(m->dev.L, tpad_for(T + 1, precision), precision);
}

// Launch `kern` (one instantiation of a kernel template) with `smem` bytes of dynamic shared memory, raising the
// kernel's shared-memory limit first when that is over the default 48 KB
template <class P>
static int launch(void (*kern)(P), dim3 blocks, int threads, size_t smem, void* stream, const P& p) {
  if (smem > 48 * 1024) {
    cudaError_t e = cudaFuncSetAttribute((const void*)kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) {
      set_error("sequence too long for the per-warp score scratch (%zu B of shared memory): %s", smem, cudaGetErrorString(e));
      return DPT_ERR_INVALID_ARG;
    }
  }
  kern<<<blocks, threads, smem, (cudaStream_t)stream>>>(p);
  DPT_LAUNCH_CHECK();
  return DPT_OK;
}

extern "C" int dpt_gpt2_forward(dpt_gpt2_t* m, const float* query_states, const float* ctx_states,
                                const float* ctx_actions, const float* ctx_next_states, const float* ctx_rewards, int B,
                                int T, int T_stride, int ctx_share, int test, int precision, float* out, void* workspace,
                                uint64_t workspace_bytes, void* stream) {
  DPT_CHECK_ARG(m, "dpt_gpt2_forward: null model");
  DPT_CHECK_ARG(precision == 0 || precision == 1, "dpt_gpt2_forward: precision %d (0 = fp32, 1 = bf16 K/V cache)", precision);
  DPT_CHECK_ARG(B >= 0 && T >= 0 && T_stride >= T, "dpt_gpt2_forward: B=%d T=%d T_stride=%d", B, T, T_stride);
  DPT_CHECK_ARG(ctx_share >= 1, "dpt_gpt2_forward: ctx_share=%d must be >= 1", ctx_share);
  DPT_CHECK_ARG(T + 1 <= m->dev.n_pos, "dpt_gpt2_forward: sequence %d exceeds n_positions %d", T + 1, m->dev.n_pos);
  if (B == 0 || (!test && T == 0)) return DPT_OK;
  DPT_CHECK_ARG(query_states && out && (T == 0 || (ctx_states && ctx_actions && ctx_next_states && ctx_rewards)),
                "dpt_gpt2_forward: null pointer");
  if (T + 1 <= 512) {   // dense path, one CTA per sequence, no K/V scratch:
    // precision 1: tcgen05 (bf16 operands; 1 tile of 128 tokens or 2..4 tiles); precision 0: CUDA-core fp32
    DenseParams dp{};
    dp.m = m->dev;
    dp.query = query_states, dp.cs = ctx_states, dp.ca = ctx_actions, dp.cns = ctx_next_states, dp.cr = ctx_rewards;
    dp.B = B, dp.T = T, dp.Ts = T_stride, dp.test = test, dp.share = ctx_share, dp.out = out;
    if (precision == 1) return T + 1 <= 128 ? gpt2_dense_launch(dp, (cudaStream_t)stream) : gpt2_dense_long_launch(dp, (cudaStream_t)stream);
    return gpt2_dense_fp32_launch(dp, (cudaStream_t)stream);
  }
  DPT_CHECK_ARG(workspace && workspace_bytes >= dpt_gpt2_forward_workspace_bytes(m, B, T, precision),
                "dpt_gpt2_forward: workspace too small");
  ForwardParams p{};
  p.m = m->dev;
  p.query = query_states, p.cs = ctx_states, p.ca = ctx_actions, p.cns = ctx_next_states, p.cr = ctx_rewards;
  p.B = B, p.T = T, p.Ts = T_stride, p.test = test, p.Tpad = tpad_for(T + 1, precision), p.share = ctx_share;
  p.out = out, p.kv = workspace;
  return launch(precision ? gpt2_forward_kernel<true> : gpt2_forward_kernel<false>, (B + G_WARPS - 1) / G_WARPS, G_THREADS,
                G_WARPS * warp_scratch_bytes(p.Tpad), stream, p);
}

extern "C" int dpt_gpt2_decode_step(dpt_gpt2_t* m, const float* tokens, int N, int pos, int T_max, int precision, void* kv_cache,
                                    uint64_t kv_bytes, float* logits, void* stream) {
  DPT_CHECK_ARG(m, "dpt_gpt2_decode_step: null model");
  DPT_CHECK_ARG(precision == 0 || precision == 1, "dpt_gpt2_decode_step: precision %d (0 = fp32, 1 = bf16 K/V cache)", precision);
  DPT_CHECK_ARG(N >= 0 && T_max >= 1 && pos >= 0 && pos < T_max, "dpt_gpt2_decode_step: N=%d pos=%d T_max=%d", N, pos, T_max);
  DPT_CHECK_ARG(T_max <= m->dev.n_pos, "dpt_gpt2_decode_step: %d positions exceed n_positions %d", T_max, m->dev.n_pos);
  if (N == 0) return DPT_OK;
  DPT_CHECK_ARG(tokens && logits && kv_cache && kv_bytes >= dpt_gpt2_online_kv_bytes(m, N, T_max, precision),
                "dpt_gpt2_decode_step: null pointer or kv cache too small");
  StepParams p{};
  p.m = m->dev;
  p.tokens = tokens, p.N = N, p.pos = pos, p.Tpad = tpad_for(T_max, precision), p.out = logits, p.kv = kv_cache;
  return launch(precision ? gpt2_decode_step_kernel<true> : gpt2_decode_step_kernel<false>, (N + G_WARPS - 1) / G_WARPS, G_THREADS,
                G_WARPS * warp_scratch_bytes(p.Tpad), stream, p);
}

extern "C" uint64_t dpt_gpt2_online_kv_bytes(const dpt_gpt2_t* m, int N, int H, int precision) {
  if (!m || N <= 0 || H <= 0) return 0;
  return (uint64_t)N * kv_seq_bytes(m->dev.L, tpad_for(H, precision), precision);
}

// Launch the online loop for members 0 .. n-1 of `p` (n = 1: the one-model call).  The kernel variant and the CTA size
// follow from the launch's total env-warps n * N: WS when the bf16 weight fragments fit, the bulk-copy ring at <= 24 fp32
// env-warps per SM, register-staged loads otherwise.  Every draw is keyed by (seed, env id, step), so a member's result
// does not depend on the variant.  Grid: (env blocks, member).
template <int NM>
static int online_launch(const OnlineGptParams<NM>& p, int n, int L, int precision, void* stream) {
  const long N = p.N, total = (long)n * p.N;
  const size_t per_warp = warp_scratch_bytes(p.Tpad);
  const size_t smem_ws = (size_t)L * WF_UINT4 * 16 + GW_WARPS * per_warp;
  if (precision && smem_ws <= 227 * 1024) {   // weight fragments of all layers + 24 warps' scratch fit one SM
    // one CTA per SM: keep the wave count of 24-warp CTAs but spread the envs evenly over those waves
    const long per_wave = (long)sm_count() * GW_WARPS, waves = (total + per_wave - 1) / per_wave;
    const int nw = (int)std::min<long>(GW_WARPS, std::max<long>(1, (total + waves * sm_count() - 1) / (waves * sm_count())));
    return launch(gpt2_online_kernel<true, true, false, NM>, dim3((N + nw - 1) / nw, n), nw * 32, smem_ws, stream, p);
  }
  // fp32 K/V staged by bulk-async copies (cp.async.bulk + mbarrier ring per warp) when the batch leaves warp slots empty
  // (fewer than ~36 env-warps per SM): there the register-staged kernel cannot keep enough bytes in flight (0.43 of the HBM
  // bound at 1250 envs) and a ring can (0.8+)
  const long env_warps_per_sm = (total + sm_count() - 1) / sm_count();
  if (!precision && env_warps_per_sm <= 24) {
    // CTA size: small batches get small CTAs so that the SMs carry equal numbers of warps (1250 envs = 8.4 warps per SM:
    // 4-warp CTAs would put 12 warps on some SMs and 8 on the others)
    const int nw = env_warps_per_sm <= 12 ? 1 : (env_warps_per_sm <= 20 ? 2 : TMA_WARPS);
    const size_t smem_tma = (size_t)nw * (KV_STAGES * (KV_TILE_BYTES + 8) + per_warp) + 8;
    return launch(gpt2_online_kernel<false, false, true, NM>, dim3((N + nw - 1) / nw, n), nw * 32, smem_tma, stream, p);
  }
  return launch(precision ? gpt2_online_kernel<true, false, false, NM> : gpt2_online_kernel<false, false, false, NM>,
                dim3((N + G_WARPS - 1) / G_WARPS, n), G_THREADS, G_WARPS * per_warp, stream, p);
}

extern "C" int dpt_gpt2_online_loop(dpt_gpt2_t* const* models, int n_models, const float* means, double var, int reward_type,
                                    int sample, uint64_t seed, uint64_t env_id0, int N, int H, int precision, void* kv_cache,
                                    uint64_t kv_bytes, float* const* ctx_states, float* const* ctx_actions,
                                    float* const* ctx_next_states, float* const* ctx_rewards, float* const* cum_means,
                                    double* const* regret_sums, const dpt_gpt2_online_inject_t* inject,
                                    const dpt_gpt2_online_dump_t* dump, void* stream) {
  const char* fn = "dpt_gpt2_online_loop";
  DPT_CHECK_ARG(n_models >= 0 && n_models <= ONLINE_POP_MAX, "%s: n_models=%d outside [0,%d]", fn, n_models, ONLINE_POP_MAX);
  if (n_models == 0) return DPT_OK;
  DPT_CHECK_ARG(models, "%s: null models array", fn);
  DPT_CHECK_ARG(reward_type == DPT_REWARD_GAUSSIAN || reward_type == DPT_REWARD_BERNOULLI,
                "%s: unknown reward_type %d (0 uniform/gaussian, 1 bernoulli)", fn, reward_type);
  DPT_CHECK_ARG(precision == 0 || precision == 1, "%s: precision %d (0 = fp32, 1 = bf16 K/V cache)", fn, precision);
  DPT_CHECK_ARG(N >= 0 && H >= 0, "%s: N=%d H=%d", fn, N, H);
  auto at = [](auto* const* a, int i) { return a ? a[i] : nullptr; };
  for (int i = 0; i < n_models; ++i) {
    DPT_CHECK_ARG(models[i], "%s: member %d is a null model", fn, i);
    const Gpt2Dev &d = models[i]->dev, &d0 = models[0]->dev;
    DPT_CHECK_ARG(d.dx == 1, "%s: member %d has state_dim=%d, the bandit loop needs 1", fn, i, d.dx);
    const struct { const char* name; int v, v0; } f[] = {{"n_layer", d.L, d0.L}, {"action_dim", d.du, d0.du}};
    for (const auto& x : f)
      DPT_CHECK_ARG(x.v == x.v0, "%s: member %d has %s=%d, member 0 has %d (members must share one shape)", fn, i, x.name, x.v,
                    x.v0);
    DPT_CHECK_ARG(H <= d.n_pos, "%s: member %d: H=%d exceeds n_positions %d", fn, i, H, d.n_pos);
    const int set = !!at(ctx_states, i) + !!at(ctx_actions, i) + !!at(ctx_next_states, i) + !!at(ctx_rewards, i);
    DPT_CHECK_ARG(set == 0 || set == 4, "%s: member %d: context pointers must be all NULL or all non-NULL", fn, i);
  }
  if (N == 0 || H == 0) return DPT_OK;
  const uint64_t per = dpt_gpt2_online_kv_bytes(models[0], N, H, precision);
  DPT_CHECK_ARG(means && kv_cache && kv_bytes / n_models >= per, "%s: null means, or kv cache of %llu B below %d x %llu B", fn,
                (unsigned long long)kv_bytes, n_models, (unsigned long long)per);
  auto fill = [&](auto& p) {
    p.means = means, p.var = var, p.rtype = reward_type, p.sample = sample;
    p.key = Key{(uint32_t)seed, (uint32_t)(seed >> 32)};
    p.env_id0 = env_id0;
    p.N = N, p.H = H, p.Tpad = tpad_for(H, precision);
    if (inject) p.in = *inject;
    for (int i = 0; i < n_models; ++i) {
      auto& mb = p.slot(i);
      mb.m = models[i]->dev;
      mb.kv = static_cast<char*>(kv_cache) + i * per;
      mb.ctx_s = at(ctx_states, i), mb.ctx_a = at(ctx_actions, i), mb.ctx_ns = at(ctx_next_states, i), mb.ctx_r = at(ctx_rewards, i);
      mb.cum_means = at(cum_means, i), mb.regret = at(regret_sums, i);
      if (dump) mb.out = dump[i];
    }
    return online_launch(p, n_models, models[0]->dev.L, precision, stream);
  };
  if (n_models == 1) {   // the one-model kernels and parameter block
    OnlineGptParams<1> p{};
    return fill(p);
  }
  OnlineGptParams<ONLINE_POP_MAX> p{};
  return fill(p);
}

extern "C" int dpt_gpt2_explore_exploit_rollout(dpt_gpt2_t* explorer, dpt_gpt2_t* exploiter, const float* means, double var, int reward_type,
                                                uint64_t seed, uint64_t env_id0, int N, int K, void* kv_explorer, void* kv_exploiter,
                                                uint64_t kv_bytes_each, float* ctx_states, float* ctx_actions, float* ctx_next_states,
                                                float* ctx_rewards, float* advantages, const dpt_explore_inject_t* inject,
                                                const dpt_explore_dump_t* dump, void* stream) {
  DPT_CHECK_ARG(explorer && exploiter, "dpt_gpt2_explore_exploit_rollout: null model");
  DPT_CHECK_ARG(reward_type == DPT_REWARD_GAUSSIAN || reward_type == DPT_REWARD_BERNOULLI,
                "dpt_gpt2_explore_exploit_rollout: unknown reward_type %d (0 uniform/gaussian, 1 bernoulli)", reward_type);
  DPT_CHECK_ARG(explorer->dev.dx == 1 && exploiter->dev.dx == 1 && explorer->dev.du == exploiter->dev.du,
                "dpt_gpt2_explore_exploit_rollout: both models need state_dim == 1 and the same action_dim");
  DPT_CHECK_ARG(N >= 0 && K >= 0, "dpt_gpt2_explore_exploit_rollout: N=%d K=%d", N, K);
  DPT_CHECK_ARG(K <= explorer->dev.n_pos && K <= exploiter->dev.n_pos, "dpt_gpt2_explore_exploit_rollout: K=%d exceeds n_positions", K);
  if (N == 0 || K == 0) return DPT_OK;
  const uint64_t need = std::max(dpt_gpt2_online_kv_bytes(explorer, N, K, 0), dpt_gpt2_online_kv_bytes(exploiter, N, K, 0));
  DPT_CHECK_ARG(means && kv_explorer && kv_exploiter && kv_explorer != kv_exploiter && kv_bytes_each >= need,
                "dpt_gpt2_explore_exploit_rollout: null means, or K/V caches missing / shared / too small");
  DPT_CHECK_ARG(ctx_states && ctx_actions && ctx_next_states && ctx_rewards && (advantages || K < 2),
                "dpt_gpt2_explore_exploit_rollout: null output pointer");
  ExploreParams p{};
  p.me = explorer->dev, p.mx = exploiter->dev;
  p.means = means, p.var = var, p.rtype = reward_type;
  p.key = Key{(uint32_t)seed, (uint32_t)(seed >> 32)};
  p.env_id0 = env_id0;
  p.N = N, p.K = K, p.Tpad = tpad_for(K, 0);
  p.kv_e = kv_explorer, p.kv_x = kv_exploiter;
  p.ctx_s = ctx_states, p.ctx_a = ctx_actions, p.ctx_ns = ctx_next_states, p.ctx_r = ctx_rewards, p.adv = advantages;
  if (inject) p.in = *inject;
  if (dump) p.out = *dump;
  return launch(gpt2_explore_exploit_kernel, (N + G_WARPS - 1) / G_WARPS, G_THREADS, G_WARPS * warp_scratch_bytes(p.Tpad), stream, p);
}
