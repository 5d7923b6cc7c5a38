"""GPU tier of bf16 training (forward_train(x, precision=1)): logits bit-identical to forward() at model.precision = 1
and within 2e-2 of fp32 training; gradients against float64 autograd of the restatement in tests/train_oracle.py;
determinism; population members bit-identical to training alone; exact resume; learning on collected bandit data next
to fp32; and a training step in a CUDA graph."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

import train_oracle as TO

pytestmark = pytest.mark.gpu

LOGIT_BAR = 2e-2   # max|bf16 - fp32| <= LOGIT_BAR * max(1, max|fp32|)  (DESIGN §5)
GRAD_BAR = 2e-2    # ||g - g64|| <= GRAD_BAR * ||g64||, per parameter tensor


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


def _loss(pred, b):
    du = pred.shape[-1]
    t = b["optimal_actions"] if pred.dim() == 2 else b["optimal_actions"][:, None].expand(-1, pred.shape[1], -1)
    return F.cross_entropy(pred.reshape(-1, du), t.reshape(-1, du), reduction="sum")


def _grads(m, b, precision=1):
    m.zero_grad(set_to_none=True)
    out = m.forward_train(b, precision)
    _loss(out, b).backward()
    return out.detach(), [p.grad.clone() for p in m._train_params()]


@pytest.mark.parametrize("dx", [1, 2])
def test_logits_bit_identical_to_forward_and_near_fp32(dpt, dx):
    m = _model(dx, 5, 3, 511, False)
    for T in (10, 100, 127, 200, 511):
        b = _batch(dx, 5, 6, 511, T, T)
        for test in (False, True):
            m.test, m.precision = test, 1
            ref = m(b)
            got = m.forward_train(b, precision=1)
            assert got.grad_fn is not None
            assert torch.equal(got.detach(), ref), (T, test)
            m.precision = 0
            f32 = m.forward_train(b).detach()
            assert (got.detach() - f32).abs().max().item() <= LOGIT_BAR * max(1.0, f32.abs().max().item()), (T, test)


@pytest.mark.parametrize("dx,du,L", [(1, 5, 2), (1, 5, 4), (2, 5, 3)])
def test_gradients_match_float64_autograd(dpt, dx, du, L):
    m = _model(dx, du, L, 511, False)
    worst = 0.0
    # ragged T (not a multiple of the 64-row tile), the last-tile edges 63 / 64 / 65 and 127 / 128, B = 1
    for T, B in ((1, 4), (7, 1), (62, 3), (63, 2), (64, 3), (127, 2), (200, 1), (320, 2), (511, 2)):
        b = _batch(dx, du, B, 511, T, 100 + T)
        for test in (False, True):
            m.test = test
            _grads(m, b)
            P = TO.params64(m, "cuda")
            b64 = {k: v.double() for k, v in b.items()}
            out64 = TO.forward(P, L, b64["query_states"], b64["context_states"], b64["context_actions"],
                               b64["context_next_states"], b64["context_rewards"], test)
            _loss(out64, b64).backward()
            assert m.transformer.wte.weight.grad is None
            params = dict(m.named_parameters())
            for k, p64 in P.items():
                g, g64 = params[k].grad, p64.grad
                assert g is not None and g.shape == g64.shape, k
                err = ((g.double() - g64).norm() / g64.norm().clamp_min(1e-30)).item()
                worst = max(worst, err)
                assert err <= GRAD_BAR, (T, B, test, k, err)
            assert torch.count_nonzero(m.transformer.wpe.weight.grad[T + 1:]) == 0
    print("largest normwise gradient error at dx=%d du=%d L=%d: %.3g" % (dx, du, L, worst))


def test_deterministic(dpt):
    m = _model(1, 5, 4, 500, False, seed=3)
    b = _batch(1, 5, 64, 500, 500, 7)
    o1, g1 = _grads(m, b)
    o2, g2 = _grads(m, b)
    assert torch.equal(o1, o2) and all(torch.equal(a, c) for a, c in zip(g1, g2))


@pytest.mark.parametrize("k", [1, 3, 33])
def test_population_members_bit_identical_to_alone(dpt, k):
    from dpt_b200.models.net import forward_train_population
    T = 130 if k == 33 else 77
    ms = [_model(1, 5, 2, 200, False, seed=10 + i) for i in range(k)]
    bs = [_batch(1, 5, 5, 200, T, 50 + i) for i in range(k)]
    ref = [_grads(m, b) for m, b in zip(ms, bs)]
    for m in ms:
        m.zero_grad(set_to_none=True)
    outs = forward_train_population(ms, bs, precision=1)
    sum(_loss(o, b) for o, b in zip(outs, bs)).backward()
    for m, o, (ro, rg) in zip(ms, outs, ref):
        assert torch.equal(o.detach(), ro)
        assert all(torch.equal(p.grad, g) for p, g in zip(m._train_params(), rg))


def _datasets(seed, n_items=424, H=40):
    from dpt_b200 import collect_data
    from dpt_b200.dataset import Dataset
    batch = collect_data.collect_bandit(n_items, 5, H, 0.3, seed=seed)
    cfg = {"horizon": H, "state_dim": 1, "action_dim": 5, "shuffle": True, "store_gpu": True}
    n_tr = n_items * 3 // 4
    return (Dataset.from_batch({k: v[:n_tr] for k, v in batch.items()}, cfg),
            Dataset.from_batch({k: v[n_tr:] for k, v in batch.items()}, cfg))


def _same(ma, oa, mb, ob):
    for p, q in zip(ma.parameters(), mb.parameters()):
        assert torch.equal(p, q)
        sa, sb = oa.state[p], ob.state[q]
        assert sa.keys() == sb.keys() and all(torch.equal(sa[n], sb[n]) for n in sa)


def test_train_population_bit_identical_to_train(dpt):
    from dpt_b200 import train as TR
    tr, te = _datasets(1)
    pop = [_model(1, 5, 2, 40, False, seed=20 + i, scale=0.02) for i in range(3)]
    alone = [_model(1, 5, 2, 40, False, seed=20 + i, scale=0.02) for i in range(3)]
    _, _, opt = TR.train_population(pop, tr, te, 2, seeds=[1, 2, 3], precision=1)
    for i, m in enumerate(alone):
        _, _, o = TR.train(m, tr, te, 2, seed=i + 1, precision=1)
        for p, q in zip(pop[i].parameters(), m.parameters()):
            assert torch.equal(p, q)
            assert all(torch.equal(opt.state[p][n], o.state[q][n]) for n in o.state[q])


def test_resume_bit_identical_and_precision_checked(dpt, tmp_path):
    from dpt_b200 import train as TR
    tr, te = _datasets(2)
    a = _model(1, 5, 2, 40, False, seed=30, scale=0.02)
    la, ta, oa = TR.train(a, tr, te, 3, seed=4, precision=1)
    path = str(tmp_path / "state.pt")
    b = _model(1, 5, 2, 40, False, seed=30, scale=0.02)
    TR.train(b, tr, te, 1, seed=4, precision=1, state_path=path, save_every=1)
    c = _model(1, 5, 2, 40, False, seed=30, scale=0.02)
    lc, tc, oc = TR.train(c, tr, te, 3, seed=4, precision=1, state_path=path, save_every=1, resume=True)
    assert la == lc and ta == tc
    _same(a, oa, c, oc)
    d = _model(1, 5, 2, 40, False, seed=30, scale=0.02)
    before = [p.detach().clone() for p in d.parameters()]
    with pytest.raises(ValueError, match="precision=0, the checkpoint 1"):
        TR.train(d, tr, te, 4, seed=4, state_path=path, resume=True)
    assert all(torch.equal(p, q) for p, q in zip(before, d.parameters()))


# bf16's final test loss may exceed fp32's by at most this fraction.  Measured on one B200: fp32 1.39410, bf16 1.39351
# after 12 epochs (relative gap -0.04 %); the bar leaves room for other builds' rounding without hiding a real regression.
LEARN_REL_TOL = 0.02


def test_learns_like_fp32_on_collected_bandit_data(dpt):
    from dpt_b200 import collect_data, train as TR
    from dpt_b200.dataset import Dataset
    from dpt_b200.models.net import Transformer
    H, d = 50, 5
    batch = collect_data.collect_bandit(4096, d, H, 0.3, seed=5)
    cfg = {"horizon": H, "state_dim": 1, "action_dim": d, "shuffle": True, "store_gpu": True}
    tr = Dataset.from_batch({k: v[:3584] for k, v in batch.items()}, cfg)
    te = Dataset.from_batch({k: v[3584:] for k, v in batch.items()}, cfg)
    final = {}
    for prec in (0, 1):
        torch.manual_seed(0)
        m = Transformer({"horizon": H, "state_dim": 1, "action_dim": d, "n_layer": 2, "n_embd": 32, "n_head": 1,
                         "dropout": 0.0, "test": False}).cuda()
        train_loss, test_loss, _ = TR.train(m, tr, te, 12, seed=0, precision=prec)
        print("precision", prec, "train", train_loss, "test", test_loss)
        assert all(np.isfinite(train_loss)) and all(np.isfinite(test_loss))
        assert test_loss[-1] < 0.85 * test_loss[0]
        final[prec] = test_loss[-1]
    gap = final[1] / final[0] - 1
    print("final test loss fp32 %.5f bf16 %.5f, relative gap %+.4f" % (final[0], final[1], gap))
    assert gap <= LEARN_REL_TOL


def test_train_step_graph_capturable(dpt):
    from dpt_b200 import train as TR
    m = _model(1, 5, 4, 500, False, seed=3)
    b = _batch(1, 5, 64, 500, 500, 7)
    opt = torch.optim.AdamW(m.parameters(), lr=1e-3, weight_decay=1e-4, capturable=True)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for _ in range(2):
            TR.train_step(m, opt, b, precision=1)
    torch.cuda.current_stream().wait_stream(s)
    before = [p.detach().clone() for p in m.parameters()]
    graph = torch.cuda.CUDAGraph()
    opt.zero_grad(set_to_none=False)
    with torch.cuda.graph(graph):
        loss = TR.train_step(m, opt, b, precision=1)
    assert all(torch.equal(a, p) for a, p in zip(before, m.parameters()))   # captured, not run
    graph.replay()
    torch.cuda.synchronize()
    assert not all(torch.equal(a, p) for a, p in zip(before, m.parameters()))
    assert torch.isfinite(loss).item()
