"""GPU tier of training: Transformer.forward_train (dpt_gpt2_train_forward / _backward) against forward() and against
float64 autograd of the restatement in tests/train_oracle.py; determinism, graph capture, errors, and train.train end
to end on collect_bandit's device-resident data."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

import train_oracle as TO

pytestmark = pytest.mark.gpu

TS = [1, 7, 31, 127, 128, 255, 500, 511]
GRAD_BAR = 2e-4   # max|g - g64| <= GRAD_BAR * max(1, max|g64|), per parameter tensor


def _model(dx, du, L, H, test, seed=0, scale=0.15):
    from dpt_b200.models.net import Transformer
    torch.manual_seed(seed)
    m = Transformer({"horizon": H, "state_dim": dx, "action_dim": du, "n_layer": L, "n_embd": 32, "n_head": 1, "dropout": 0.0,
                     "test": test}).cuda()
    with torch.no_grad():
        for k, p in m.named_parameters():
            if "wte" not in k:
                p.add_(scale * torch.randn_like(p))
    return m


def _batch(dx, du, B, H, T, seed):
    """Strided [:, :T] views of [B,H,.] buffers; bandit: constant states, darkroom (dx = 2): varying integer states."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    if dx == 1:
        cs = torch.ones(B, H, 1, device="cuda")
        q = torch.ones(B, 1, device="cuda")
    else:
        cs = torch.randint(0, 10, (B, H, dx), generator=g, device="cuda").float()
        q = torch.randint(0, 10, (B, dx), generator=g, device="cuda").float()
    ca = torch.eye(du, device="cuda")[torch.randint(0, du, (B, H), generator=g, device="cuda")]
    cns = cs if dx == 1 else torch.randint(0, 10, (B, H, dx), generator=g, device="cuda").float()
    cr = torch.rand(B, H, 1, generator=g, device="cuda")
    b = {"query_states": q, "context_states": cs[:, :T], "context_actions": ca[:, :T], "context_next_states": cns[:, :T],
         "context_rewards": cr[:, :T]}
    b["optimal_actions"] = torch.eye(du, device="cuda")[torch.randint(0, du, (B,), generator=g, device="cuda")]
    return b


SHAPES = [(1, 5, 2), (1, 5, 4), (2, 5, 3)]   # (dx, du, L): bandit L = 2, 4; darkroom L = 3


@pytest.mark.parametrize("dx,du,L", SHAPES)
def test_forward_train_logits_bit_identical(dpt, dx, du, L):
    m = _model(dx, du, L, 511, True)
    for T in TS:
        b = _batch(dx, du, 5, 511, T, T)
        for test in (True, False):
            m.test = test
            ref = m(b)
            out = m.forward_train(b)
            assert out.requires_grad and out.grad_fn is not None
            assert torch.equal(out.detach(), ref), (T, test)


def _losses(du):
    w = None

    def ce_sum(pred, b):
        t = b["optimal_actions"][:, None].expand(-1, pred.shape[1], -1)
        return F.cross_entropy(pred.reshape(-1, du), t.reshape(-1, du), reduction="sum")

    def ce_last(pred, b):
        return F.cross_entropy(pred, b["optimal_actions"], reduction="sum")

    def ce_weighted(pred, b):
        nonlocal w
        if w is None or w.shape != pred.shape[:2]:
            w = torch.linspace(-1.0, 2.0, pred.shape[0] * pred.shape[1], device=pred.device, dtype=torch.float64).reshape(pred.shape[:2])
        t = b["optimal_actions"][:, None].expand(-1, pred.shape[1], -1)
        ce = F.cross_entropy(pred.reshape(-1, du), t.reshape(-1, du).to(pred.dtype), reduction="none").reshape(pred.shape[:2])
        return (ce * w.to(pred.dtype)).sum()
    return [("ce_sum", False, ce_sum), ("ce_last", True, ce_last), ("ce_weighted", False, ce_weighted)]


WORST = {}


@pytest.mark.parametrize("dx,du,L", SHAPES)
def test_gradients_match_float64_autograd(dpt, dx, du, L):
    m = _model(dx, du, L, 511, False)
    worst = 0.0
    for T in TS:
        b = _batch(dx, du, 3 if T > 255 else 5, 511, T, 100 + T)
        for name, test, loss_fn in _losses(du):
            m.test = test
            m.zero_grad(set_to_none=True)
            loss_fn(m.forward_train(b), b).backward()
            P = TO.params64(m, "cuda")
            b64 = {k: v.double() for k, v in b.items()}
            out64 = TO.forward(P, L, b64["query_states"], b64["context_states"], b64["context_actions"],
                               b64["context_next_states"], b64["context_rewards"], test)
            loss_fn(out64, b64).backward()
            assert m.transformer.wte.weight.grad is None
            params = dict(m.named_parameters())
            for k, p64 in P.items():
                g, g64 = params[k].grad, p64.grad
                assert g is not None and g.shape == g64.shape, k
                scale = max(1.0, g64.abs().max().item())
                err = (g.double() - g64).abs().max().item()
                worst = max(worst, err / scale)
                assert err <= GRAD_BAR * scale, (T, name, k, err, scale)
            assert torch.count_nonzero(m.transformer.wpe.weight.grad[T + 1:]) == 0
    WORST[(dx, du, L)] = worst
    print("largest gradient error / max(1, max|g64|) at dx=%d du=%d L=%d: %.3g" % (dx, du, L, worst))


def test_backward_deterministic_and_graph_capturable(dpt):
    from dpt_b200 import train as TR
    m = _model(1, 5, 4, 500, False, seed=3)
    b = _batch(1, 5, 64, 500, 500, 7)
    grads = []
    for _ in range(2):
        m.zero_grad(set_to_none=True)
        TR.ce_sum_loss(m.forward_train(b), b).backward()
        grads.append([p.grad.clone() for p in m._train_params()])
    for g1, g2 in zip(*grads):
        assert torch.equal(g1, g2)
    # a whole training step in one CUDA graph: no host round trip inside forward_train / backward / AdamW
    opt = torch.optim.AdamW(m.parameters(), lr=1e-3, weight_decay=1e-4, capturable=True)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for _ in range(2):
            TR.train_step(m, opt, b)
    torch.cuda.current_stream().wait_stream(s)
    before = [p.detach().clone() for p in m.parameters()]
    graph = torch.cuda.CUDAGraph()
    opt.zero_grad(set_to_none=False)
    with torch.cuda.graph(graph):
        pred = m.forward_train(b)
        loss = TR.ce_sum_loss(pred, b)
        loss.backward()
        opt.step()
    assert all(torch.equal(a, p) for a, p in zip(before, m.parameters()))   # captured, not run
    graph.replay()
    torch.cuda.synchronize()
    assert not all(torch.equal(a, p) for a, p in zip(before, m.parameters()))
    assert torch.isfinite(loss).item()


def test_errors_and_empty_batch(dpt):
    from dpt_b200.models.net import Transformer
    cfg = {"horizon": 600, "state_dim": 1, "action_dim": 5, "n_layer": 2, "n_embd": 32, "n_head": 1, "dropout": 0.1, "test": False}
    m = Transformer(cfg).cuda()
    b = _batch(1, 5, 2, 600, 10, 0)
    with pytest.raises(NotImplementedError):
        m.forward_train(b)
    m.dropout = 0.0
    with pytest.raises(NotImplementedError):
        m.forward_train(_batch(1, 5, 2, 600, 512, 0))        # T + 1 = 513 tokens
    m.forward_train(_batch(1, 5, 2, 600, 511, 0))           # 512 tokens is the limit
    e = {k: v[:0] for k, v in b.items()}
    out = m.forward_train(e)
    assert out.shape == (0, 10, 5)
    out.sum().backward()
    assert all(float(p.grad.abs().sum()) == 0.0 for p in m._train_params())


def test_train_end_to_end_on_collected_bandit_data(dpt):
    from dpt_b200 import collect_data, train as TR
    from dpt_b200.dataset import Dataset
    from dpt_b200.evals import eval_bandit
    H, d = 50, 5
    batch = collect_data.collect_bandit(4096, d, H, 0.3, seed=5)
    cfg = {"horizon": H, "state_dim": 1, "action_dim": d, "shuffle": True, "store_gpu": True}
    n_tr = 3584
    tr = Dataset.from_batch({k: v[:n_tr] for k, v in batch.items()}, cfg)
    te = Dataset.from_batch({k: v[n_tr:] for k, v in batch.items()}, cfg)
    torch.manual_seed(0)
    from dpt_b200.models.net import Transformer
    m = Transformer({"horizon": H, "state_dim": 1, "action_dim": d, "n_layer": 2, "n_embd": 32, "n_head": 1, "dropout": 0.0,
                     "test": False}).cuda()
    train_loss, test_loss, opt = TR.train(m, tr, te, 12, seed=0)
    print("train", train_loss, "test", test_loss)
    assert all(np.isfinite(train_loss)) and all(np.isfinite(test_loss))
    assert test_loss[-1] < 0.85 * test_loss[0]   # the first entry is the untrained model (test loss before each epoch)
    assert set(opt.state_dict()["state"]) and opt.state_dict()["param_groups"][0]["weight_decay"] == 1e-4
    # the handle follows the trained weights: forward() equals forward_train on them
    b = {k: v[:64] for k, v in te.dataset.items()}
    for test in (False, True):
        m.test = test
        assert torch.equal(m(b), m.forward_train(b).detach())
    # and the trained model runs in the evaluations without a stale handle
    m.test = True
    ol = m.online_loop(batch["means"][:256], H, 0.3, False, 1, 0)
    assert torch.isfinite(ol["cum_means"]).all()
    with torch.no_grad():
        m.pred_actions.bias.add_(0.5)
    m.test = False
    assert torch.equal(m(b), m.forward_train(b).detach())


def test_train_step_for_interactive_last_logit_loss(dpt):
    """train_interactive.py's step: CE on the last logits after a GPUBanditEnv rollout, through train.train_step."""
    from dpt_b200 import train as TR
    m = _model(1, 5, 2, 40, True, seed=9, scale=0.0)
    opt = torch.optim.AdamW(m.parameters(), lr=1e-3, weight_decay=1e-4)
    b = _batch(1, 5, 32, 40, 40, 3)
    losses = [TR.train_step(m, opt, b, lambda pred, bb: F.cross_entropy(pred, bb["optimal_actions"], reduction="sum"))
              for _ in range(30)]
    assert losses[0].dim() == 0 and losses[0].is_cuda
    assert losses[-1].item() < losses[0].item()
