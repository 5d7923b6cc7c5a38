// Model handle shared by the GPT-2 kernels (gpt2.cu: token-sequential; gpt2_dense.cu: tcgen05 dense).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/dpt_b200.h"

namespace dpt {

constexpr int G_E = 32;
constexpr int G_FF = 128;
constexpr int G_MAX_L = 8;
constexpr int G_WARPS = 4;
constexpr int G_THREADS = G_WARPS * 32;

// Weight matrices [in][out] are repacked at create time into per-lane quads:
//   P[(in/4)][out/32][lane][in%4]  so that one LDG.128 gives a lane the 4 consecutive-input weights of its
//   output (out = group*32 + lane), consumed by two FFMA2 (fma.rn.f32x2) against an LDS.128 of the inputs.
struct LayerW {
  const float *ln1_w, *ln1_b, *attn_b, *proj_b, *ln2_w, *ln2_b, *fc_b, *fc2_b;
  const float4 *attn_wP, *proj_wP, *fc_wP, *fc2_wP;
  const float *attn_w, *proj_w, *fc_w, *fc2_w;   // original [in][out] layouts (dense fp32 kernel)
  const uint4* wimg;  // bf16 B-operand image for the tcgen05 dense forward (see gpt2_dense.cu), 40 KB
  const uint4* wfrag; // bf16 mma.sync B fragments for the KV-cached decode (see gpt2.cu, WF_*), 24 KB
};

struct Gpt2Dev {
  int L, dx, du, din, H, n_pos;
  const float *wpe, *embed_wT, *embed_b, *pred_wT, *pred_b, *lnf_w, *lnf_b;
  LayerW layer[G_MAX_L];
};

}  // namespace dpt

struct dpt_gpt2 {
  dpt::Gpt2Dev dev;
  float* blob;
};

namespace dpt {
// LayerW::wfrag, in uint4 units: for every Conv1D weight W[K][N] and every (k-step ks of 16 inputs, pair ntp of two
// 8-output tiles) one uint4 per lane = {b0, b1 of tile 2 ntp, b0, b1 of tile 2 ntp + 1} of mma.m16n8k16 (col-major B):
// lane (g = lane / 4, c = lane % 4): b0 = W[16 ks + 2c, +1][n], b1 = W[16 ks + 2c + 8, +9][n], n = 8 tile + g.
constexpr int WF_QKV = 0;      // K = 32, N = 96 : 2 x 6 groups of 32 lanes
constexpr int WF_PROJ = 384;   // K = 32, N = 32 : 2 x 2
constexpr int WF_FC = 512;     // K = 32, N = 128: 2 x 8
constexpr int WF_FC2 = 1024;   // K = 128, N = 32: 8 x 2
constexpr int WF_UINT4 = 1536; // 24576 B per layer
// byte layout of LayerW::wimg (K64 tiles, see umma.cuh): B[n][k] = W[k][n] for every Conv1D weight W[in][out]
constexpr int WIMG_QKV = 0;            // [96 rows x 64]   12288 B
constexpr int WIMG_PROJ = 12288;       // [32 rows x 64]    4096 B
constexpr int WIMG_FC = 16384;         // [128 rows x 64]  16384 B
constexpr int WIMG_FC2 = 32768;        // 2 x [32 rows x 64] 8192 B (k 0..63, 64..127)
constexpr int WIMG_BYTES = 40960;

struct DenseParams {
  Gpt2Dev m;
  const float *query, *cs, *ca, *cns, *cr;
  int B, T, Ts, test, share;   // share: sequences per context row
  float* out;
};
int gpt2_dense_launch(const DenseParams& p, cudaStream_t st);        // gpt2_dense.cu (tcgen05, bf16 operands)
int gpt2_dense_long_launch(const DenseParams& p, cudaStream_t st);   // gpt2_dense.cu (tcgen05, 129..512 tokens)
int gpt2_dense_fp32_launch(const DenseParams& p, cudaStream_t st);   // gpt2_dense_fp32.cu (CUDA cores, fp32)

// Activations the training forward saves for the backward (gpt2_train.cu), fp32.  act: [L][B][S][TA_STRIDE], one record
// per layer and row (S = T + 1 rows, row 0 = query token); fin: [B][S][TF_STRIDE], the input token, the final residual
// and the ln_f statistics.
constexpr int TA_XIN = 0;      // residual input of the layer [32]
constexpr int TA_Q = 32;       // q * 1/sqrt(32) [32]
constexpr int TA_K = 64;       // [32]
constexpr int TA_V = 96;       // [32]
constexpr int TA_O = 128;      // attention output (input of attn.c_proj) [32]
constexpr int TA_XMID = 160;   // residual after attention [32]
constexpr int TA_H = 192;      // mlp.c_fc pre-activation [128]
constexpr int TA_MU1 = 320, TA_RS1 = 321, TA_LSE = 322, TA_MU2 = 323, TA_RS2 = 324;
constexpr int TA_STRIDE = 328;
constexpr int TF_X = 0, TF_TOK = 32, TF_MU = 64, TF_RS = 65, TF_STRIDE = 68;   // TF_TOK: the input token, zero-padded
struct TrainSave {
  float *act, *fin;
};

// Training reads the parameter tensors in place (reference layouts: embed_w = embed_transition.weight [E, din], pred_w =
// pred_actions.weight [du, E]).  A population of same-shape models runs in one launch: CTA (b, member = blockIdx.y).
// The per-member tables travel in the kernel parameters, so a launch needs no upload and stays graph-capturable; at
// ~0.9 KB per member, TRAIN_POP_MAX members fit the 32 764 B parameter limit.
constexpr int TRAIN_POP_MAX = DPT_GPT2_POPULATION_MAX;
struct TrainLayerW {
  const float *ln1_w, *ln1_b, *attn_w, *attn_b, *proj_w, *proj_b, *ln2_w, *ln2_b, *fc_w, *fc_b, *fc2_w, *fc2_b;
};
struct TrainW {
  const float *wpe, *embed_w, *embed_b, *pred_w, *pred_b, *lnf_w, *lnf_b;
  TrainLayerW layer[G_MAX_L];
};
struct TrainFwdMember {
  TrainW w;
  const float *query, *cs, *ca, *cns, *cr;
  float* out;
  TrainSave sv;
};
template <int NM>   // NM: member capacity of the launch (1 for the one-model entry points, else TRAIN_POP_MAX)
struct TrainFwdParams {
  int L, dx, du, din, B, T, Ts, test;
  TrainFwdMember mem[NM];
};
// the dense fp32 forward that also saves the activations (gpt2_dense_fp32.cu), members mem[0 .. n)
template <int NM>
int gpt2_train_forward_launch(const TrainFwdParams<NM>& p, int n, cudaStream_t st);
void gpt2_pack_wimg(const float* attn_w, const float* proj_w, const float* fc_w, const float* fc2_w, unsigned char* img,
                    cudaStream_t st);

// bf16 training (precision 1): the tcgen05 dense forward (gpt2_dense.cu, SAVE = true) on the parameter tensors, with the
// weight images of member i, layer l at wimg[i] + l * WIMG_BYTES (packed from the parameters by gpt2_pack_train_wimg in
// the same call).  It saves the same fp32 records (TA_* / TF_*) as the fp32 forward of training.
template <int NM>
struct TrainFwd16Params {
  int L, dx, du, din, B, T, Ts, test;
  TrainFwdMember mem[NM];
  const uint4* wimg[NM];
};
template <int NM>
int gpt2_train_forward_bf16_launch(const TrainFwd16Params<NM>& p, int n, cudaStream_t st);
template <int NM>
struct WimgPackParams {
  const float* w[NM][G_MAX_L][4];   // attn_w, proj_w, fc_w, fc2_w of member i, layer l
  unsigned char* img[NM];
};
template <int NM>
int gpt2_pack_train_wimg(const WimgPackParams<NM>& p, int L, int n, cudaStream_t st);
}  // namespace dpt
