"""Helpers of the sharp-attention tests (test_sharp_attention_cpu.py, test_sharp_attention_gpu.py): a model and batches at
which attention looks like a trained DPT's, and the statistics that show it.

At the weights of the other numerical tests (initialisation plus 0.05-0.15 * randn) every query row spreads its attention
almost evenly over its keys: a row's scores span well under one nat and its largest probability is ~1 / S.  There the
kernels' running-maximum rescale multiplies by ~1, so a rescale that is skipped or applied to the wrong sum moves the
output by little.  Here the q and k blocks of every layer's c_attn weight are multiplied by ``alpha`` (scores grow as
alpha^2), and "landmark" tokens, context rows whose reward lies far outside [0, 1) and grows with the position, pull the
row maximum forward across the 64- and 128-key tile edges, into the last partial tile and into the query's own tile.

Everything here is plain torch and runs on the CPU or the GPU."""
import torch

import kernel_structure as KS
import train_oracle as TO

# alpha of the fp32 and of the bf16 cases, side by side.  At fp32, alpha = 3 keeps the float32 torch restatement within
# 4e-6 of float64 (2.5x under the 1e-5 bar).  At bf16 the rounding of q, k, v, P and the projection operands grows with the
# scores: a restatement that rounds them stays within 1e-2 of float64 (normwise, half the 2e-2 bar) at alpha = 2, not at
# 3.  Both are asserted in test_sharp_attention_cpu.py.
ALPHA_FP32 = 3.0
ALPHA_BF16 = 2.0

# (dx, seed of the model): bandit and darkroom token layouts, 4 layers, 5 actions.  The seeds are ones whose layer 0
# meets the regime statistics at every length of TS (asserted in test_sharp_attention_cpu.py).
CASES = [(1, 0), (2, 2)]
DU, L = 5, 4
TS = (63, 64, 127, 128, 129, 255, 256, 383, 384, 511, 540)   # transitions: tokens S = T + 1 around the tile edges

HORIZON = 540          # n_positions = 4 * (1 + horizon) covers every length of the tests
REWARD0, REWARD_SLOPE = 2.0, 4.0   # landmark reward at token j of S: REWARD0 + REWARD_SLOPE * j / 512
LAST_EXTRA = 2.0                   # added to the last context row's reward, so that the last tile holds a row maximum


def model(dx, du, L, test, alpha, horizon=HORIZON, seed=0):
    """kernel_structure.model (scale 0.15) with columns 0..63 (q and k) of every c_attn weight multiplied by alpha."""
    m = KS.model(dx, du, L, horizon, test, seed=seed)
    with torch.no_grad():
        for blk in m.transformer.h:
            blk.attn.c_attn.weight[:, :64] *= alpha
    return m


def landmarks(S):
    """Token positions (context row + 1) of the landmarks of a sequence of S tokens: both sides of the 64- and 128-key
    edges (kernel_structure.probes) and the last tokens, which lie in the last, partial tile."""
    return [j for j in KS.probes(S, edges=(62, 63, 64, 65, 126, 127, 128, 129, 254, 255, 256, 257, 382, 383, 384, 385,
                                           510, 511)) if j >= 1]


def batch(dx, du, B, T, seed, device="cpu"):
    """kernel_structure.base_batch with the landmark rewards of landmarks(T + 1)."""
    b = KS.base_batch(dx, du, B, T, seed)
    for j in landmarks(T + 1):
        b["context_rewards"][:, j - 1] = REWARD0 + REWARD_SLOPE * j / 512
    if T:
        b["context_rewards"][:, T - 1] += LAST_EXTRA
    return {k: v.to(device) for k, v in b.items()}


def forward(P, L, x, test, **kw):
    """train_oracle.forward on a batch dict, in the dtype of P."""
    return TO.forward(P, L, x["query_states"], x["context_states"], x["context_actions"], x["context_next_states"],
                      x["context_rewards"], test, **kw)


def params(m, dtype=torch.float64, device="cpu"):
    return {k: p.detach().to(device=device, dtype=dtype).clone() for k, p in m.named_parameters() if "wte" not in k}


def layer_stats(m, L, x):
    """Per layer, the float64 scores and probabilities ([B, S, S]) of the model on batch x, and their statistics:
    - range: median over query rows 1.. of (max - min) of the row's scores, in nats;
    - top: median over query rows 1.. of the row's largest probability;
    - moved: among rows past token 128, the fraction whose argmax key lies in a later 128-key tile than the argmax of
      its first tile (keys 0..127), so that the running maximum of every kernel must move past tile 0;
    - last_tile: per sequence, whether some row's argmax key lies in the last 128-key tile when that tile is partial
      (S not a multiple of 128), else in the last 64 keys."""
    rec = []
    with torch.no_grad():
        forward(params(m, device=x["context_rewards"].device), L, {k: v.double() for k, v in x.items()}, False,
                record=rec)
    out = []
    for s, p in rec:
        S = s.shape[-1]
        lo = s.masked_fill(torch.isinf(s), float("inf")).amin(-1)
        am = p.argmax(-1)                                                  # first maximum, as the kernels' softmax
        last0 = (S - 1) // 128 * 128 if S % 128 else S - 64
        moved = (am[:, 128:] >= 128).double().mean().item() if S > 128 else float("nan")
        out.append({"scores": s, "probs": p, "range": (s.amax(-1) - lo)[:, 1:].median().item(),
                    "top": p.amax(-1)[:, 1:].median().item(), "moved": moved,
                    "last_tile": (am >= last0).any(-1).tolist()})
    return out


def rel_err(a, b):
    """max |a - b| / max(1, |b|) elementwise: the measure of the 1e-5 and 2e-2 logit bars."""
    a, b = a.double(), b.double()
    return ((a - b).abs() / b.abs().clamp_min(1.0)).max().item()


def bf16(t):
    return t.to(torch.bfloat16).to(t.dtype)
