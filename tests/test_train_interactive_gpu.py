"""GPU tier of the interactive trainer (train.train_interactive, train_interactive.py:97-139): an iteration against its
composition from public pieces (bit for bit), micro-batched gradients against float64 autograd of the whole batch
(tests/train_oracle.py), determinism, learning, and the error / empty cases."""
import numpy as np
import pytest
import torch

import train_oracle as TO

pytestmark = pytest.mark.gpu

GRAD_BAR = 2e-4   # as tests/test_train_gpu.py: max|g - g64| <= GRAD_BAR * max(1, max|g64|), per parameter tensor
CTX = ("context_states", "context_actions", "context_next_states", "context_rewards")


def _model(d, L, H, seed=0, scale=0.15, dropout=0.0):
    from dpt_b200.models.net import Transformer
    torch.manual_seed(seed)
    m = Transformer({"horizon": H, "state_dim": 1, "action_dim": d, "n_layer": L, "n_embd": 32, "n_head": 1, "dropout": dropout,
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


def test_one_microbatch_iteration_is_its_composition(dpt):
    from dpt_b200 import train as TR
    d, L, N, K, var, seed = 5, 2, 300, 30, 0.3, 7
    m1, m2 = _model(d, L, K, seed=1), _model(d, L, K, seed=1)
    m1.test = False                      # the trainer takes the last logits whatever the model's test flag says
    losses, opt1 = TR.train_interactive(m1, d, N, K, 1, mb=512, var=var, seed=seed)
    b, target = _rollout(m2, d, N, K, var, seed, 0)
    opt2 = torch.optim.AdamW(m2.parameters(), lr=1e-3, weight_decay=1e-4)
    opt2.zero_grad()
    pred = m2.forward_train(b)
    loss = TR.interactive_loss(pred, target, N)
    loss.backward()
    opt2.step()
    assert len(losses) == 1 and losses[0] == loss.item()
    assert abs(loss.item() - torch.nn.functional.cross_entropy(pred.detach(), target).item()) < 1e-6   # torch's mean
    for (k, p1), p2 in zip(m1.named_parameters(), m2.parameters()):
        assert torch.equal(p1, p2), k
        if p2.grad is not None:
            assert torch.equal(p1.grad, p2.grad), k
    assert m1.transformer.wte.weight.grad is None
    assert isinstance(opt1, torch.optim.AdamW) and len(opt1.state) == len(m1._train_params())


def test_microbatched_gradient_matches_float64_autograd(dpt):
    from dpt_b200 import train as TR
    d, L, N, K, mb, var, seed = 5, 2, 1000, 40, 256, 0.3, 3          # micro-batches of 256, 256, 256 and 232 envs
    m = _model(d, L, K, seed=2)
    frozen = torch.optim.AdamW(m.parameters(), lr=0.0, weight_decay=0.0)   # the step leaves the weights as they were
    before = [p.detach().clone() for p in m.parameters()]
    losses, _ = TR.train_interactive(m, d, N, K, 1, mb=mb, var=var, seed=seed, optimizer=frozen)
    assert all(torch.equal(a, p) for a, p in zip(before, m.parameters()))
    b, target = _rollout(m, d, N, K, var, seed, 0)                     # the iteration's rollout, rebuilt
    P = TO.params64(m, "cuda")
    b64 = {k: v.double() for k, v in b.items()}
    out64 = TO.forward(P, L, b64["query_states"], *(b64[k] for k in CTX), test=True)
    loss64 = TR.interactive_loss(out64, target, N)
    loss64.backward()
    assert abs(losses[0] - loss64.item()) <= 1e-5 * max(1.0, abs(loss64.item()))
    params, worst = dict(m.named_parameters()), 0.0
    for k, p64 in P.items():
        g, g64 = params[k].grad, p64.grad
        assert g is not None and g.shape == g64.shape, k
        scale = max(1.0, g64.abs().max().item())
        err = (g.double() - g64).abs().max().item()
        worst = max(worst, err / scale)
        assert err <= GRAD_BAR * scale, (k, err, scale)
    print("largest gradient error / max(1, max|g64|) over 4 micro-batches: %.3g" % worst)


def test_same_seed_same_weights(dpt):
    from dpt_b200 import train as TR
    runs = []
    for _ in range(2):
        m = _model(5, 2, 24, seed=4)
        losses, _ = TR.train_interactive(m, 5, 2000, 24, 3, mb=512, var=0.3, seed=11)
        runs.append((losses, [p.detach().clone() for p in m.parameters()]))
    assert runs[0][0] == runs[1][0] and len(runs[0][0]) == 3
    assert all(torch.equal(a, b) for a, b in zip(runs[0][1], runs[1][1]))
    m = _model(5, 2, 24, seed=4)
    other, _ = TR.train_interactive(m, 5, 2000, 24, 3, mb=512, var=0.3, seed=12)
    assert other != runs[0][0]            # another seed draws other envs


def test_loss_falls(dpt):
    from dpt_b200 import train as TR
    m = _model(5, 2, 20, seed=5, scale=0.0)
    losses, opt = TR.train_interactive(m, 5, 4096, 20, 30, mb=1024, var=0.3, seed=1, lr=3e-3)
    print("interactive losses", np.round(losses, 4).tolist())
    assert all(np.isfinite(losses))
    assert np.mean(losses[-5:]) < np.mean(losses[:5]) - 0.05
    assert opt.param_groups[0]["lr"] == 3e-3


def test_errors_and_empty_batch(dpt):
    from dpt_b200 import train as TR
    m = _model(5, 2, 600, dropout=0.1)
    with pytest.raises(NotImplementedError, match="dropout"):
        TR.train_interactive(m, 5, 64, 10, 1)
    m.dropout = 0.0
    before = [p.detach().clone() for p in m.parameters()]
    with pytest.raises(NotImplementedError, match="512 tokens"):
        TR.train_interactive(m, 5, 64, 513, 1)          # 513 tokens: the limit of forward_train, checked before the rollout
    with pytest.raises(ValueError, match="micro-batch"):
        TR.train_interactive(m, 5, 64, 10, 1, mb=0)
    losses, opt = TR.train_interactive(m, 5, 0, 10, 3)   # no envs: nothing runs
    assert losses == [] and not opt.state
    assert all(torch.equal(a, p) for a, p in zip(before, m.parameters()))
    losses, _ = TR.train_interactive(m, 5, 64, 512, 1, mb=48)   # 512 tokens is the limit
    assert np.isfinite(losses[0])
