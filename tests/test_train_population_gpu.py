"""GPU tier of population training: forward_train_population / train_population against each member trained alone
(forward_train, backward, train), bit for bit; determinism, graph capture and the limits."""
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

TS = [1, 7, 127, 128, 255, 500, 511]


def _model(dx, du, L, H, test, seed, scale=0.15):
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


SHAPES = [(1, 5, 4), (2, 5, 3)]   # (dx, du, L): bandit, darkroom


@pytest.mark.parametrize("dx,du,L", SHAPES)
def test_population_logits_bit_identical(dpt, dx, du, L):
    from dpt_b200.models.net import forward_train_population
    ms = [_model(dx, du, L, 511, True, seed) for seed in (0, 1, 2)]
    for T in TS:
        bs = [_batch(dx, du, 5, 511, T, 10 * T + i) for i in range(3)]
        for test in (True, False):
            for m in ms:
                m.test = test
            outs = forward_train_population(ms, bs)
            for m, b, out in zip(ms, bs, outs):
                assert out.requires_grad and out.grad_fn is not None
                assert torch.equal(out.detach(), m(b)), (T, test)
                assert torch.equal(out.detach(), m.forward_train(b).detach()), (T, test)


def _losses(du):
    def ce_sum(pred, b):
        t = b["optimal_actions"][:, None].expand(-1, pred.shape[1], -1)
        return F.cross_entropy(pred.reshape(-1, du), t.reshape(-1, du), reduction="sum")

    def ce_last(pred, b):
        return F.cross_entropy(pred[:, -1], b["optimal_actions"], reduction="sum")

    def ce_weighted(pred, b):
        w = torch.linspace(-1.0, 2.0, pred.shape[0] * pred.shape[1], device=pred.device).reshape(pred.shape[:2])
        t = b["optimal_actions"][:, None].expand(-1, pred.shape[1], -1)
        ce = F.cross_entropy(pred.reshape(-1, du), t.reshape(-1, du), reduction="none").reshape(pred.shape[:2])
        return (ce * w).sum()
    return [ce_sum, ce_last, ce_weighted]


@pytest.mark.parametrize("dx,du,L", SHAPES)
def test_population_gradients_bit_identical(dpt, dx, du, L):
    from dpt_b200.models.net import forward_train_population
    ms = [_model(dx, du, L, 511, False, seed) for seed in range(4)]
    losses = _losses(du)
    for T in (7, 128, 500):
        bs = [_batch(dx, du, 6, 511, T, 100 * T + i) for i in range(4)]
        ref = []
        for i, (m, b) in enumerate(zip(ms, bs)):
            m.zero_grad(set_to_none=True)
            if i < 3:   # member 3's logits get no gradient
                losses[i](m.forward_train(b), b).backward()
            ref.append([None if p.grad is None else p.grad.clone() for p in m.parameters()])
            m.zero_grad(set_to_none=True)
        outs = forward_train_population(ms, bs)
        sum(losses[i](outs[i], bs[i]) for i in range(3)).backward()
        for i, m in enumerate(ms):
            for (name, p), g in zip(m.named_parameters(), ref[i]):
                if g is None:
                    assert p.grad is None, (T, i, name)
                else:
                    assert torch.equal(p.grad, g), (T, i, name)
            assert m.transformer.wte.weight.grad is None


def _datasets(H, n_items, seed):
    from dpt_b200 import collect_data
    from dpt_b200.dataset import Dataset
    batch = collect_data.collect_bandit(n_items, 5, H, 0.3, seed=seed)
    cfg = {"horizon": H, "state_dim": 1, "action_dim": 5, "shuffle": True, "store_gpu": True}
    n_tr = n_items * 3 // 4
    return (Dataset.from_batch({k: v[:n_tr] for k, v in batch.items()}, cfg),
            Dataset.from_batch({k: v[n_tr:] for k, v in batch.items()}, cfg))


def _state(opt, m):
    return [{k: v.clone() for k, v in opt.state[p].items()} for p in m.parameters() if p in opt.state]


@pytest.mark.parametrize("k", [3, 1])
def test_train_population_bit_identical_to_train(dpt, k):
    from dpt_b200 import train as TR
    H = 40
    tr_a, te_a = _datasets(H, 424, 5)        # 318 train items: a ragged last batch of 62
    tr_b, te_b = _datasets(H, 424, 6)
    seeds, lrs = [11, 12, 13][:k], [1e-3, 3e-3, 1e-3][:k]
    trs, tes = [tr_a, tr_a, tr_b][:k], [te_a, te_a, te_b][:k]

    def models():
        return [_model(1, 5, 2, H, False, 20 + i, scale=0.02) for i in range(k)]
    alone = []
    for i, m in enumerate(models()):
        tl, vl, opt = TR.train(m, trs[i], tes[i], 2, lr=lrs[i], seed=seeds[i])
        alone.append((m, tl, vl, _state(opt, m)))
    ms = models()
    tl, vl, opt = TR.train_population(ms, trs if k > 1 else trs[0], tes if k > 1 else tes[0], 2, lr=lrs, seeds=seeds)
    for i, m in enumerate(ms):
        ma, tla, vla, sa = alone[i]
        for p, q in zip(m.parameters(), ma.parameters()):
            assert torch.equal(p, q), i
        for s, t in zip(_state(opt, m), sa):
            assert s.keys() == t.keys() and all(torch.equal(s[n], t[n]) for n in s), i
        assert vl[i] == vla, i                                                     # test losses: bit for bit
        assert all(abs(a - b) <= 1e-6 * abs(b) for a, b in zip(tl[i], tla)), i     # train losses: 1e-6 relative
        if k == 1:
            assert tl[i] == tla


def test_population_deterministic_and_graph_capturable(dpt):
    from dpt_b200 import train as TR
    bs = [_batch(1, 5, 64, 500, 500, 7 + i) for i in range(2)]
    runs = []
    for _ in range(2):
        ms = [_model(1, 5, 4, 500, False, 3 + i) for i in range(2)]
        opt = torch.optim.AdamW([p for m in ms for p in m.parameters()], lr=1e-3, weight_decay=1e-4)
        for _ in range(2):
            TR.train_population_step(ms, opt, bs)
        runs.append([p.detach().clone() for m in ms for p in m.parameters()])
    assert all(torch.equal(a, b) for a, b in zip(*runs))
    # a whole population step in one CUDA graph
    opt = torch.optim.AdamW([p for m in ms for p in m.parameters()], lr=1e-3, weight_decay=1e-4, capturable=True)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for _ in range(2):
            TR.train_population_step(ms, opt, bs)
    torch.cuda.current_stream().wait_stream(s)
    before = [p.detach().clone() for m in ms for p in m.parameters()]
    graph = torch.cuda.CUDAGraph()
    opt.zero_grad(set_to_none=False)
    with torch.cuda.graph(graph):
        from dpt_b200.models.net import forward_train_population
        preds = forward_train_population(ms, bs)
        loss = sum(TR.ce_sum_loss(p, b) for p, b in zip(preds, bs))
        loss.backward()
        opt.step()
    after = [p for m in ms for p in m.parameters()]
    assert all(torch.equal(a, p) for a, p in zip(before, after))   # captured, not run
    graph.replay()
    torch.cuda.synchronize()
    assert not all(torch.equal(a, p) for a, p in zip(before, after))
    assert torch.isfinite(loss).item()


def test_population_limits(dpt):
    from dpt_b200.models.net import forward_train_population
    ms = [_model(1, 5, 2, 600, False, i) for i in range(2)]
    with pytest.raises(NotImplementedError, match="512 tokens"):
        forward_train_population(ms, [_batch(1, 5, 2, 600, 512, i) for i in range(2)])   # T + 1 = 513 tokens
    forward_train_population(ms, [_batch(1, 5, 2, 600, 511, i) for i in range(2)])      # 512 tokens is the limit
    ms[1].dropout = 0.1
    with pytest.raises(NotImplementedError, match="dropout"):
        forward_train_population(ms, [_batch(1, 5, 2, 600, 10, i) for i in range(2)])
    ms[1].dropout = 0.0
    assert forward_train_population([], []) == []
    e = [{k: v[:0] for k, v in _batch(1, 5, 2, 600, 10, i).items()} for i in range(2)]
    outs = forward_train_population(ms, e)
    assert [o.shape for o in outs] == [(0, 10, 5)] * 2
    sum(o.sum() for o in outs).backward()
    assert all(float(p.grad.abs().sum()) == 0.0 for m in ms for p in m._train_params())
    # more members than one launch takes: cut into launches, still each member's own logits
    many = [_model(1, 5, 2, 600, False, i, scale=0.05) for i in range(34)]
    bs = [_batch(1, 5, 2, 600, 9, i) for i in range(34)]
    for m, b, o in zip(many, bs, forward_train_population(many, bs)):
        assert torch.equal(o.detach(), m(b))
