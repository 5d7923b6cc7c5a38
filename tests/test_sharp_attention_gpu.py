"""GPU tier of the sharp-attention tests: the GPT-2 kernels against float64 where attention is as sharp as a trained DPT's
(tests/sharp_attention.py; the regime and the conditioning of the reference are asserted in test_sharp_attention_cpu.py).

At the weights of the other numerical tests every row attends almost uniformly, so the kernels' running-maximum rescale
(fp32 dense rows on every new maximum, the tcgen05 long pipeline once per 128-key tile) multiplies by ~1 and a skipped or
misplaced rescale hides under the bars.  Here the running maximum moves by nats across the tile edges, at the project's
unchanged bars: fp32 logits within 1e-5 (elementwise, max(1, |ref|)), fp32 gradients within GRAD_BAR = 2e-4 of
max(1, max|g64|) per tensor and per wpe row; bf16 logits within 2e-2 normwise (max|d| / max(1, max|ref|), as the bf16
training tests), bf16 gradients within 2e-2 normwise per tensor.

- forward: precision 0 (dense fp32 rows in their 128-, 256- and 512-thread CTAs, the token-sequential kernel past 512
  tokens) and precision 1 (short tcgen05 kernel, long kernel with 2, 3 and 4 tiles), test=True and False.
- forward_train gradients at both precisions against float64 autograd.
- Transformer.decoder at both precisions (bandit layout), step by step, across the 32- and 64-key tiles of the decode.
- online_loop in each of its six kernel instantiations (kernel_structure.online_cases): dumped logits against float64
  and the recorded arms against the dumped logits and uniforms.  The loop draws its own rewards, so only alpha sharpens
  it (median largest arm probability 0.33-0.40).
- The offline evaluation's learner rows at both precisions.

Worst errors measured on a B200 (1000 W power limit), bandit / darkroom: forward fp32 2.6e-6 / 3.1e-6, bf16 6.6e-3 /
8.1e-3 normwise (elementwise 1.95e-2 / 2.11e-2); gradients fp32 7.8e-6 / 3.4e-6 (wpe rows 3.4e-5 / 8.4e-6), bf16 1.32e-2 /
1.11e-2; decoder fp32 9.1e-7, bf16 1.1e-3 (elementwise 2.7e-3); online loop fp32 1.35e-6 in all four fp32 variants, bf16
6.2e-3 warp-specialised and 4.7e-3 fallback (elementwise 9.5e-3 / 5.1e-3); offline learner rows fp32 1.3e-6, bf16 5.0e-3
(elementwise 1.2e-2).  Elementwise, the bf16 forward is at the 2e-2 bar of test_transformer_gpu._close, and past it for
darkroom.  That is the size of bf16 rounding itself: a float64 restatement that rounds the same operands to bf16 is off by
1e-2 to 2.7e-2 elementwise here, and by 1.5e-2 at plain initialisation (test_sharp_attention_cpu.py).  So the bf16 logits
are held to the normwise bar of the bf16 training tests.  The bf16 gradient error of the bandit case is the closest to
its bar.

Planted defects.  A running-maximum rescale whose exponent is clamped at -4 nats is exact wherever the maximum moves by
less than 4 nats, which is every row of the older tests.  In the long tcgen05 pipeline (gpt2_dense_long_kernel) the whole
older GPU suite passes with it, and this file fails (bf16 forward, darkroom).  In the fp32 dense rows only the explorer /
exploiter rollout test (weights + 0.2 * randn) of the older suite fails, and this file fails five tests: fp32 forward and
gradients in both layouts, and the fp32 offline learner rows.  Cruder defects (no ``lsum *= sc`` in the long pipeline,
acc rescaled without lsum in the fp32 rows, lse0 for both row halves of the bf16 attention backward, s_self left out of
the bf16 decode's maximum, P recomputed with the running maximum in the fp32 backward) fail both this file and the older
tests."""
import pytest
import torch
import torch.nn.functional as F

import kernel_structure as KS
import sharp_attention as SA
import train_oracle as TO

pytestmark = pytest.mark.gpu

LOGIT_BAR = {0: 1e-5, 1: 2e-2}
GRAD_BAR = {0: 2e-4, 1: 2e-2}


def _alpha(precision):
    return SA.ALPHA_FP32 if precision == 0 else SA.ALPHA_BF16


def _logit_err(out, ref, precision):
    """(error under the bar of the precision, elementwise error): at fp32 both are the elementwise max |d| / max(1, |ref|);
    at bf16 the first is normwise, max |d| / max(1, max |ref|), and the elementwise one is reported beside it."""
    ew = SA.rel_err(out, ref)
    if precision == 0:
        return ew, ew
    return ((out.double() - ref).abs().max() / ref.abs().max().clamp_min(1.0)).item(), ew


def _ref(m, x, test):
    with torch.no_grad():
        return SA.forward(SA.params(m, device="cuda"), len(m.transformer.h), {k: v.double() for k, v in x.items()}, test)


@pytest.mark.parametrize("precision", [0, 1])
@pytest.mark.parametrize("dx,seed", SA.CASES)
def test_forward(dpt, dx, seed, precision):
    m = SA.model(dx, SA.DU, SA.L, False, _alpha(precision), seed=seed).cuda()
    m.precision = precision
    worst, worst_ew = 0.0, 0.0
    for T in SA.TS:
        x = SA.batch(dx, SA.DU, 4, T, seed=T, device="cuda")
        for test in (False, True):
            m.test = test
            err, ew = _logit_err(m(x), _ref(m, x, test), precision)
            worst, worst_ew = max(worst, err), max(worst_ew, ew)
            assert err <= LOGIT_BAR[precision], (T, test, err)
    print("forward precision %d dx=%d: worst logit error %.3g (elementwise %.3g)" % (precision, dx, worst, worst_ew))


def _loss(pred, b):
    t = b["optimal_actions"][:, None].expand(-1, pred.shape[1], -1)
    return F.cross_entropy(pred.reshape(-1, SA.DU), t.reshape(-1, SA.DU).to(pred.dtype), reduction="sum")


@pytest.mark.parametrize("precision", [0, 1])
@pytest.mark.parametrize("dx,seed", SA.CASES)
def test_gradients(dpt, dx, seed, precision):
    """Every parameter's gradient against float64 autograd; at fp32 also each wpe.grad row, so that the rows of the
    landmark positions are checked on their own rather than inside a tensor's norm."""
    m = SA.model(dx, SA.DU, SA.L, False, _alpha(precision), seed=seed).cuda()
    worst, worst_row = 0.0, 0.0
    for T in [t for t in SA.TS if t < 512]:
        x = SA.batch(dx, SA.DU, 2, T, seed=T, device="cuda")
        m.zero_grad(set_to_none=True)
        _loss(m.forward_train(x, precision), x).backward()
        P = TO.params64(m, "cuda")
        _loss(SA.forward(P, SA.L, {k: v.double() for k, v in x.items()}, False), x).backward()
        params = dict(m.named_parameters())
        for k, p64 in P.items():
            g, g64 = params[k].grad.double(), p64.grad
            if precision == 0:
                scale = max(1.0, g64.abs().max().item())
                err = (g - g64).abs().max().item() / scale
            else:
                err = ((g - g64).norm() / g64.norm().clamp_min(1e-30)).item()
            worst = max(worst, err)
            assert err <= GRAD_BAR[precision], (T, k, err)
        if precision == 0:
            g, g64 = params["transformer.wpe.weight"].grad.double(), P["transformer.wpe.weight"].grad
            row = ((g - g64).abs().amax(-1) / g64.abs().amax(-1).clamp_min(1.0)).max().item()
            worst_row = max(worst_row, row)
            assert row <= GRAD_BAR[0], (T, row)
    print("gradients precision %d dx=%d: worst tensor error %.3g, worst wpe row error %.3g" % (precision, dx, worst,
                                                                                                worst_row))


@pytest.mark.parametrize("precision", [0, 1])
def test_decoder(dpt, precision):
    """Bandit layout only (a decoder keeps one query state per sequence; darkroom's query state changes every step):
    logits at steps around the decode's key tiles (32 keys at fp32, 64 at bf16) against float64 over the context
    appended so far."""
    H = 300
    m = SA.model(1, SA.DU, SA.L, True, _alpha(precision), seed=SA.CASES[0][1]).cuda()
    m.precision = precision
    x = SA.batch(1, SA.DU, 4, H, seed=H, device="cuda")
    dec = m.decoder(4, H)
    steps = {0, 1, 31, 32, 33, 63, 64, 65, 127, 128, 129, 191, 192, 255, 256, 257, H}
    worst, worst_ew = 0.0, 0.0
    for t in range(H + 1):
        if t == 0:
            lg = dec.query(x["query_states"])
        else:
            lg = dec.append(*(x[k][:, t - 1] for k in ("context_states", "context_actions", "context_next_states",
                                                       "context_rewards")))
        if t in steps:
            xt = {k: (v[:, :t] if k.startswith("context") else v) for k, v in x.items()}
            err, ew = _logit_err(lg, _ref(m, xt, True), precision)
            worst, worst_ew = max(worst, err), max(worst_ew, ew)
            assert err <= LOGIT_BAR[precision], (t, err)
    print("decoder precision %d: worst logit error %.3g (elementwise %.3g)" % (precision, worst, worst_ew))


CTX = ("context_states", "context_actions", "context_next_states", "context_rewards")


@pytest.mark.parametrize("case", range(6))
def test_online_loop(dpt, case):
    """online_loop with dump=True in every instantiation of gpt2_online_kernel (kernel_structure.online_cases), at the
    sharpened weights (the loop draws its own rewards, so there are no landmarks): the logits the loop saw at steps
    around the decode's key tiles against float64 over the context it built (envs spread over the grid, the last one in
    a partial CTA), and every recorded arm is the categorical draw (float64 cdf of the dumped logits, searchsorted
    'right') of the dumped uniform."""
    import numpy as np
    precision, L, N, H, variant = KS.online_cases()[case]
    m = SA.model(1, SA.DU, L, True, _alpha(precision), horizon=H).cuda()
    m.precision = precision
    means, _, _ = dpt.kernels.bandit_sample_means(N, SA.DU, 7, 0)
    out = m.online_loop(means, H, 0.3, True, 7, 0, dump=True)
    logits = out["noise"]["logits"]
    idx = torch.tensor(sorted({0, 1, N // 3, N // 2, N - 2, N - 1} & set(range(N))), device="cuda")
    worst, worst_ew = 0.0, 0.0
    for h in sorted({0, 1, 31, 32, 33, 63, 64, 65, 127, 128, 129, 700, H - 1} & set(range(H))):
        x = {k: out[k][idx][:, :h] for k in CTX}
        x["query_states"] = torch.ones(len(idx), 1, device="cuda")
        err, ew = _logit_err(logits[h][idx], _ref(m, x, True), precision)
        worst, worst_ew = max(worst, err), max(worst_ew, ew)
        assert err <= LOGIT_BAR[precision], (variant, h, err)
    lg = logits.double().cpu().numpy()                                   # [H, N, d]
    pr = np.exp(lg - lg.max(-1, keepdims=True))
    cdf = np.cumsum(pr / pr.sum(-1, keepdims=True), -1)
    cdf /= cdf[..., -1:]
    u = out["noise"]["ctrl_u"].double().cpu().numpy()                  # [H, N]
    arm = (cdf[..., :-1] <= u[..., None]).sum(-1)
    assert np.array_equal(arm.T, out["context_actions"].argmax(-1).cpu().numpy()), variant
    top = np.median(np.exp(lg - lg.max(-1, keepdims=True)).max(-1) / np.exp(lg - lg.max(-1, keepdims=True)).sum(-1))
    print("online_loop %s: worst logit error %.3g (elementwise %.3g), median top arm probability %.2f"
          % (variant, worst, worst_ew, top))


@pytest.mark.parametrize("precision", [0, 1])
def test_offline_learner_rows(dpt, precision):
    """The learner rows of the offline evaluation (one test=False forward over max(horizons) rows, eval_bandit.
    learner_logits) at the sharpened weights and with landmark rewards in the context: row h - 1 against float64 over
    the first h transitions, at horizons on both sides of the tile edges; the learner's reward is the mean of the arm
    that is the first maximum of the kernel's row, and of the float64 row wherever its top-two gap exceeds the bar."""
    import numpy as np
    from dpt_b200.evals import eval_bandit
    N, H, var = 64, 300, 0.3
    m = SA.model(1, SA.DU, SA.L, True, _alpha(precision), horizon=H).cuda()
    m.precision = precision
    means, _, _ = dpt.kernels.bandit_sample_means(N, SA.DU, 77, 0)
    ctx = dpt.collect_data.collect_bandit(N, SA.DU, H, var, seed=77, means=means)
    for j in SA.landmarks(H + 1):
        ctx["context_rewards"][:, j - 1] = SA.REWARD0 + SA.REWARD_SLOPE * j / 512
    hz = [H, 1, 2, 63, 64, 65, 127, 128, 129, 255, 256, 257, H - 1]
    out = eval_bandit.offline_device(ctx, means, hz, m, var, seed=5)
    lg = eval_bandit.learner_logits(m, {k: ctx[k] for k in CTX}, H)
    assert m.test is True
    x = {k: ctx[k] for k in CTX}
    x["query_states"] = torch.ones(N, 1, device="cuda")
    ref = _ref(m, x, False)                                              # [N, H, d]: row h - 1 = test=True on h rows
    lnr = out["rewards"][:, dpt.kernels.OFFLINE_SLOTS.index("lnr")].cpu().numpy()
    m64, lgn, refn = means.double().cpu().numpy(), lg.double().cpu().numpy(), ref.cpu().numpy()
    worst, worst_ew = 0.0, 0.0
    for k, h in enumerate(hz):
        err, ew = _logit_err(lg[:, h - 1], ref[:, h - 1], precision)
        worst, worst_ew = max(worst, err), max(worst_ew, ew)
        assert err <= LOGIT_BAR[precision], (h, err)
        assert np.array_equal(lnr[k], m64[np.arange(N), lgn[:, h - 1].argmax(1)]), h
        top2 = np.sort(refn[:, h - 1], axis=1)[:, -2:]
        ok = (top2[:, 1] - top2[:, 0]) >= 2 * LOGIT_BAR[precision] * np.maximum(1.0, np.abs(refn[:, h - 1]).max())
        assert np.array_equal(lnr[k][ok], m64[np.arange(N), refn[:, h - 1].argmax(1)][ok]), h
    print("offline learner rows precision %d: worst logit error %.3g (elementwise %.3g)" % (precision, worst, worst_ew))
