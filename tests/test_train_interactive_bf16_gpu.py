"""GPU tier of bf16 interactive training (train.train_interactive(..., precision=1)): an iteration against its composition
from public pieces (bit for bit, at both rollout precisions), micro-batched gradients against float64 autograd of the
whole batch (tests/train_oracle.py) and against one micro-batch, determinism, exact resume, and learning next to fp32."""
import numpy as np
import pytest
import torch

import train_oracle as TO

pytestmark = pytest.mark.gpu

GRAD_BAR = 2e-2   # as tests/test_train_bf16_gpu.py: ||g - g64|| <= GRAD_BAR * ||g64||, per parameter tensor
CTX = ("context_states", "context_actions", "context_next_states", "context_rewards")


def _model(d, L, H, seed=0, scale=0.15):
    from dpt_b200.models.net import Transformer
    torch.manual_seed(seed)
    m = Transformer({"horizon": H, "state_dim": 1, "action_dim": d, "n_layer": L, "n_embd": 32, "n_head": 1, "dropout": 0.0,
                     "test": True}).cuda()
    with torch.no_grad():
        for k, p in m.named_parameters():
            if "wte" not in k:
                p.add_(scale * torch.randn_like(p))
    return m


def _rollout(m, d, N, K, var, seed, it):
    from dpt_b200 import rng
    from dpt_b200.envs.gpu_bandit_env import GPUBanditEnv
    ro = GPUBanditEnv(d, N, K, var, "uniform", seed=rng.key_for(seed, it)).rollout(m, K)
    b = {k: ro[k][:, :K - 1] for k in CTX}
    b["query_states"] = torch.ones((N, 1), device="cuda")
    return b, ro["target"]


def _normwise(g, g64):
    return ((g.double() - g64).norm() / g64.norm().clamp_min(1e-30)).item()


@pytest.mark.parametrize("rollout_precision", [0, 1])
def test_one_microbatch_iteration_is_its_composition(dpt, rollout_precision):
    from dpt_b200 import train as TR
    d, L, N, K, var, seed = 5, 2, 300, 30, 0.3, 7
    m1, m2 = _model(d, L, K, seed=1), _model(d, L, K, seed=1)
    m1.precision = m2.precision = rollout_precision
    m1.test = False                      # the trainer takes the last logits whatever the model's test flag says
    losses, _ = TR.train_interactive(m1, d, N, K, 1, mb=512, var=var, seed=seed, precision=1)
    b, target = _rollout(m2, d, N, K, var, seed, 0)
    opt2 = torch.optim.AdamW(m2.parameters(), lr=1e-3, weight_decay=1e-4)
    opt2.zero_grad()
    pred = m2.forward_train(b, precision=1)
    loss = TR.interactive_loss(pred, target, N)
    loss.backward()
    opt2.step()
    assert len(losses) == 1 and losses[0] == loss.item()
    for (k, p1), p2 in zip(m1.named_parameters(), m2.parameters()):
        assert torch.equal(p1, p2), k
        if p2.grad is not None:
            assert torch.equal(p1.grad, p2.grad), k
    assert m1.transformer.wte.weight.grad is None


def _frozen_iteration(m, d, N, K, mb, var, seed):
    """One precision-1 iteration whose AdamW step changes nothing: (loss, {name: gradient})."""
    from dpt_b200 import train as TR
    frozen = torch.optim.AdamW(m.parameters(), lr=0.0, weight_decay=0.0)
    before = [p.detach().clone() for p in m.parameters()]
    losses, _ = TR.train_interactive(m, d, N, K, 1, mb=mb, var=var, seed=seed, optimizer=frozen, precision=1)
    assert all(torch.equal(a, p) for a, p in zip(before, m.parameters()))
    return losses[0], {k: p.grad.clone() for k, p in m.named_parameters() if p.grad is not None}


# micro-batches of 256, 256, 256 and 232 envs; and 512 tokens, the limit, in micro-batches of 48 and 16 envs
@pytest.mark.parametrize("N,K,mb,H", [(1000, 40, 256, 40), (64, 512, 48, 512)])
def test_microbatched_gradient_matches_float64_and_one_microbatch(dpt, N, K, mb, H):
    from dpt_b200 import train as TR
    d, L, var, seed = 5, 2, 0.3, 3
    m = _model(d, L, H, seed=2)
    loss, grads = _frozen_iteration(m, d, N, K, mb, var, seed)
    b, target = _rollout(m, d, N, K, var, seed, 0)                     # the iteration's rollout, rebuilt
    P = TO.params64(m, "cuda")
    b64 = {k: v.double() for k, v in b.items()}
    out64 = TO.forward(P, L, b64["query_states"], *(b64[k] for k in CTX), test=True)
    loss64 = TR.interactive_loss(out64, target, N)
    loss64.backward()
    assert abs(loss - loss64.item()) <= GRAD_BAR * max(1.0, abs(loss64.item()))
    worst = 0.0
    assert grads.keys() == P.keys()
    for k, p64 in P.items():
        assert grads[k].shape == p64.grad.shape, k
        err = _normwise(grads[k], p64.grad)
        worst = max(worst, err)
        assert err <= GRAD_BAR, (k, err)
    print("N=%d K=%d mb=%d: largest normwise gradient error against float64: %.3g, loss %.6f vs %.6f"
          % (N, K, mb, worst, loss, loss64.item()))
    # the same iteration in one micro-batch: the slots' sum is that gradient up to the order of the sums
    loss1, grads1 = _frozen_iteration(_model(d, L, H, seed=2), d, N, K, N, var, seed)
    assert abs(loss - loss1) <= 1e-5 * abs(loss1)
    worst = max(_normwise(grads[k], grads1[k].double()) for k in grads1)
    print("largest normwise difference to one micro-batch: %.3g" % worst)
    assert worst <= GRAD_BAR


def test_same_seed_same_weights(dpt):
    from dpt_b200 import train as TR
    runs = []
    for _ in range(2):
        m = _model(5, 2, 24, seed=4)
        losses, _ = TR.train_interactive(m, 5, 2000, 24, 3, mb=512, var=0.3, seed=11, precision=1)
        runs.append((losses, [p.detach().clone() for p in m.parameters()]))
    assert runs[0][0] == runs[1][0] and len(runs[0][0]) == 3
    assert all(torch.equal(a, b) for a, b in zip(runs[0][1], runs[1][1]))
    m = _model(5, 2, 24, seed=4)
    other, _ = TR.train_interactive(m, 5, 2000, 24, 3, mb=512, var=0.3, seed=12, precision=1)
    assert other != runs[0][0]            # another seed draws other envs


def test_resumed_is_the_uninterrupted_run_and_precision_checked(dpt, tmp_path):
    from dpt_b200 import train as TR
    d, N, K, mb, var, seed, n = 5, 1000, 24, 256, 0.3, 4, 4
    full = _model(d, 2, K, seed=1)
    losses, opt = TR.train_interactive(full, d, N, K, n, mb=mb, var=var, seed=seed, precision=1)
    path = str(tmp_path / "it.pt")
    first, _ = TR.train_interactive(_model(d, 2, K, seed=1), d, N, K, n // 2, mb=mb, var=var, seed=seed, precision=1,
                                    state_path=path)
    assert first == losses[:n // 2]
    res = _model(d, 2, K, seed=3)          # other initial weights: everything comes from the file
    lr_, optr = TR.train_interactive(res, d, N, K, n, mb=mb, var=var, seed=seed, precision=1, state_path=path, resume=True)
    assert lr_ == losses
    for p, q in zip(full.parameters(), res.parameters()):
        assert torch.equal(p, q)
        if p in opt.state:
            assert all(torch.equal(opt.state[p][k], optr.state[q][k]) for k in opt.state[p])
    assert len(optr.state) == len(full._train_params())
    m = _model(d, 2, K, seed=5)
    before = [p.detach().clone() for p in m.parameters()]
    with pytest.raises(ValueError, match="^precision=0, the checkpoint 1$"):
        TR.train_interactive(m, d, N, K, n, mb=mb, var=var, seed=seed, state_path=path, resume=True)
    assert all(torch.equal(a, p) for a, p in zip(before, m.parameters()))


# bf16's mean loss over the last 5 iterations may differ from fp32's by at most this fraction
LEARN_REL_TOL = 0.03


def test_loss_falls_like_fp32(dpt):
    from dpt_b200 import train as TR
    tail = {}
    for prec in (0, 1):
        m = _model(5, 2, 20, seed=5, scale=0.0)
        losses, _ = TR.train_interactive(m, 5, 4096, 20, 30, mb=1024, var=0.3, seed=1, lr=3e-3, precision=prec)
        print("precision", prec, "interactive losses", np.round(losses, 4).tolist())
        assert all(np.isfinite(losses))
        assert np.mean(losses[-5:]) < np.mean(losses[:5]) - 0.05
        tail[prec] = np.mean(losses[-5:])
    gap = tail[1] / tail[0] - 1
    print("mean of the last 5 losses: fp32 %.5f bf16 %.5f, relative gap %+.4f" % (tail[0], tail[1], gap))
    assert abs(gap) <= LEARN_REL_TOL
