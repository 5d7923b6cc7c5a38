"""GPU tier of population evaluation: every member of an online_loop_population call computes bit for bit what its own
online_loop computes alone -- cum_means, the four context tensors and the dumped logits, reward noise and uniforms (the
regret sums are float64 atomics: equal within 1e-9 relative) -- whichever kernel variant the population's total env-warps
select, across launches cut by member capacity or by the K/V bound, eagerly or replayed from a CUDA graph; and
online_population equals online per member from the same rng state."""
import ctypes

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

CTX = ("context_states", "context_actions", "context_next_states", "context_rewards")
NOISE = ("logits", "reward_z", "ctrl_u")


def _member(seed, **over):
    from dpt_b200.models.net import Transformer
    cfg = {"horizon": 500, "state_dim": 1, "action_dim": 5, "n_layer": 4, "n_embd": 32, "n_head": 1, "dropout": 0.0, "test": True}
    cfg.update(over)
    torch.manual_seed(seed)
    m = Transformer(cfg)
    with torch.no_grad():   # move off the init so that the softmax is far from uniform, differently for every member
        for k, p in m.named_parameters():
            if "wte" not in k:
                p.add_(0.15 * torch.randn_like(p))
    return m.cuda()


@pytest.fixture(scope="module")
def members(dpt):
    """members(k, precision): k distinct same-shape models (made once, shared by the tests of this module)."""
    cache = []

    def get(k, precision=0):
        while len(cache) < k:
            cache.append(_member(100 + len(cache)))
        for m in cache[:k]:
            m.precision = precision
        return cache[:k]
    return get


def _same(got, ref, what=""):
    assert torch.equal(got["cum_means"], ref["cum_means"]), what
    for k in CTX:
        if k in ref:
            assert torch.equal(got[k], ref[k]), (what, k)
    if "noise" in ref:
        for k in NOISE:
            assert torch.equal(got["noise"][k], ref["noise"][k]), (what, k)
    if "regret_sums" in ref:
        assert torch.allclose(got["regret_sums"], ref["regret_sums"], rtol=1e-9, atol=1e-12), what


def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


@pytest.mark.parametrize("regime", ["ring", "ring_alone", "staged"])
@pytest.mark.parametrize("precision", [0, 1])
@pytest.mark.parametrize("H", [77, 500])
@pytest.mark.parametrize("reward_type", ["uniform", "bernoulli"])
@pytest.mark.parametrize("sample", [True, False])
def test_members_equal_their_own_loop(dpt, members, sample, reward_type, H, precision, regime):
    """ring: 100 envs, the fp32 ring alone and in the population; ring_alone: 8 env-warps per SM and k = 4, the ring alone
    and register-staged loads in the population; staged: 32 per SM, register-staged both ways (bf16: WS CTA sizes)."""
    from dpt_b200.models.net import online_loop_population
    N, k = {"ring": (100, 3), "ring_alone": (8 * _sms(), 4), "staged": (32 * _sms(), 3)}[regime]
    ms = members(k, precision)
    means, _, _ = dpt.kernels.bandit_sample_means(N, 5, 31, 11)
    kw = dict(env_id0=11, dump=True, reward_type=reward_type)
    pop = online_loop_population(ms, means, H, 0.3, sample, 31, **kw)
    for i, m in enumerate(ms):
        _same(pop[i], m.online_loop(means, H, 0.3, sample, 31, **kw), "member %d" % i)
    assert not torch.equal(pop[0]["noise"]["logits"], pop[1]["noise"]["logits"])   # the members do differ


def test_injected_noise_is_shared(dpt, members):
    from dpt_b200.models.net import online_loop_population
    N, H = 300, 60
    ms = members(3)
    means, _, _ = dpt.kernels.bandit_sample_means(N, 5, 4, 0)
    g = torch.Generator(device="cuda").manual_seed(5)
    inject = {"reward_z": torch.randn((H, N), device="cuda", generator=g),
              "ctrl_u": torch.rand((H, N), device="cuda", dtype=torch.float64, generator=g)}
    pop = online_loop_population(ms, means, H, 0.3, True, 9, inject=inject, dump=True)
    for i, m in enumerate(ms):
        ref = m.online_loop(means, H, 0.3, True, 9, inject=inject, dump=True)
        _same(pop[i], ref, "member %d" % i)
        assert torch.equal(ref["noise"]["reward_z"], inject["reward_z"]) and torch.equal(ref["noise"]["ctrl_u"], inject["ctrl_u"])


def _c_online_loop(dpt, m, means, H, seed, env_id0):
    """The one-model C entry point called directly (Transformer.online_loop goes through the population entry point)."""
    from dpt_b200._lib import lib, ptr, stream_ptr
    N, d = means.shape
    out = {"cum_means": torch.empty((H, N), device="cuda"), "regret_sums": torch.zeros((H, 4), dtype=torch.float64, device="cuda"),
           "context_states": torch.empty((N, H, 1), device="cuda"), "context_actions": torch.empty((N, H, d), device="cuda"),
           "context_next_states": torch.empty((N, H, 1), device="cuda"), "context_rewards": torch.empty((N, H, 1), device="cuda"),
           "noise": {"reward_z": torch.empty((H, N), device="cuda"), "ctrl_u": torch.zeros((H, N), dtype=torch.float64, device="cuda"),
                     "logits": torch.empty((H, N, d), device="cuda")}}
    h = m.handle()
    nb = lib().dpt_gpt2_online_kv_bytes(h, N, H, m.precision)
    kv = torch.empty((nb,), dtype=torch.uint8, device="cuda")
    dump = dpt._lib.Gpt2OnlineDump(**{k: ptr(t) for k, t in out["noise"].items()})
    dpt._lib.check(lib().dpt_gpt2_online_loop(h, ptr(means), 0.3, 0, 1, seed, env_id0, N, H, m.precision, ptr(kv), nb,
                                              *[ptr(out[k]) for k in CTX], ptr(out["cum_means"]), ptr(out["regret_sums"]), None,
                                              ctypes.byref(dump), stream_ptr()), "dpt_gpt2_online_loop")
    return out


@pytest.mark.parametrize("precision", [0, 1])
def test_one_member_equals_the_one_model_entry_point(dpt, members, precision):
    from dpt_b200.models.net import online_loop_population
    m = members(1, precision)[0]
    means, _, _ = dpt.kernels.bandit_sample_means(500, 5, 3, 2)
    ref = _c_online_loop(dpt, m, means, 90, 3, 2)
    _same(online_loop_population([m], means, 90, 0.3, True, 3, 2, dump=True)[0], ref)
    _same(m.online_loop(means, 90, 0.3, True, 3, 2, dump=True), ref)


def test_population_above_one_launch(dpt, members):
    from dpt_b200.models import net
    k = net.ONLINE_POPULATION_MAX + 2
    ms = members(k)
    means, _, _ = dpt.kernels.bandit_sample_means(100, 5, 8, 0)
    pop = net.online_loop_population(ms, means, 77, 0.3, True, 8, dump=True)
    assert len(pop) == k
    for i in (0, net.ONLINE_POPULATION_MAX - 1, net.ONLINE_POPULATION_MAX, k - 1):
        _same(pop[i], ms[i].online_loop(means, 77, 0.3, True, 8, dump=True), "member %d" % i)


def test_split_by_kv_bound_changes_nothing(dpt, members, monkeypatch):
    from dpt_b200.models import net
    ms = members(5)
    means, _, _ = dpt.kernels.bandit_sample_means(200, 5, 6, 0)
    whole = net.online_loop_population(ms, means, 120, 0.3, True, 6, dump=True)
    per = dpt._lib.lib().dpt_gpt2_online_kv_bytes(ms[0].handle(), 200, 120, 0)
    monkeypatch.setattr(net, "ONLINE_KV_LAUNCH_BYTES", 2 * per)
    assert net.online_launch_groups(5, per) == [(0, 2), (2, 4), (4, 5)]
    split = net.online_loop_population(ms, means, 120, 0.3, True, 6, dump=True)
    for i in range(5):
        _same(split[i], whole[i], "member %d" % i)


def test_deterministic_and_graph_capturable(dpt, members):
    from dpt_b200.models.net import online_loop_population
    ms = members(3)
    means, _, _ = dpt.kernels.bandit_sample_means(400, 5, 12, 0)
    run = lambda: online_loop_population(ms, means, 64, 0.3, True, 12, dump=True)   # noqa: E731
    eager = run()
    again = run()
    for a, b in zip(eager, again):
        _same(a, b)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):   # warm-up on a side stream before capture
        run()
    torch.cuda.current_stream().wait_stream(side)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        captured = run()
    g.replay()
    torch.cuda.synchronize()
    for a, b in zip(captured, eager):
        _same(a, b)


def test_empty_population_and_empty_shapes(dpt, members):
    from dpt_b200.models.net import online_loop_population
    ms = members(2)
    means, _, _ = dpt.kernels.bandit_sample_means(16, 5, 1, 0)
    assert online_loop_population([], means, 10, 0.3, True, 1) == []
    lib = dpt._lib.lib()
    assert lib.dpt_gpt2_online_loop_population(None, 0, None, 0.3, 0, 1, 1, 0, 16, 10, 0, None, 0, None, None, None, None, None,
                                               None, None, None, None) == 0
    zero_n = online_loop_population(ms, means[:0], 10, 0.3, True, 1)
    assert [o["cum_means"].shape for o in zero_n] == [(10, 0)] * 2
    zero_h = online_loop_population(ms, means, 0, 0.3, True, 1)
    assert [o["cum_means"].shape for o in zero_h] == [(0, 16)] * 2
    torch.cuda.synchronize()


def test_mismatched_members_raise_in_python_and_c(dpt, members):
    from dpt_b200.models.net import online_loop_population
    from dpt_b200._lib import lib, ptr
    ms = members(2)
    means, _, _ = dpt.kernels.bandit_sample_means(16, 5, 1, 0)
    for field, over in (("action_dim", {"action_dim": 4}), ("n_layer", {"n_layer": 3})):
        odd = _member(7, **over)
        with pytest.raises(ValueError, match="member 2 has %s" % field):
            online_loop_population(ms + [odd], means, 10, 0.3, True, 1)
        hs = (ctypes.c_void_p * 3)(*[m.handle() for m in ms + [odd]])
        kv = torch.empty((1 << 24,), dtype=torch.uint8, device="cuda")
        rc = lib().dpt_gpt2_online_loop_population(hs, 3, ptr(means), 0.3, 0, 1, 1, 0, 16, 10, 0, ptr(kv), kv.numel(), None, None,
                                                   None, None, None, None, None, None, None)
        assert rc == dpt._lib.ERR_INVALID_ARG and ("member 2 has %s" % field) in lib().dpt_last_error().decode()
    hs = (ctypes.c_void_p * 2)(*[m.handle() for m in ms])
    per = lib().dpt_gpt2_online_kv_bytes(ms[0].handle(), 16, 10, 0)
    kv = torch.empty((2 * per,), dtype=torch.uint8, device="cuda")
    args = (ptr(means), 0.3, 0, 1, 1, 0, 16, 10, 0, ptr(kv))
    assert lib().dpt_gpt2_online_loop_population(hs, 2, *args, 2 * per - 1, None, None, None, None, None, None, None, None,
                                                 None) == dpt._lib.ERR_INVALID_ARG
    assert "kv cache" in lib().dpt_last_error().decode()
    cs = (ctypes.c_void_p * 2)(None, ptr(torch.empty(16 * 10, device="cuda")))
    assert lib().dpt_gpt2_online_loop_population(hs, 2, *args, 2 * per, cs, None, None, None, None, None, None, None,
                                                 None) == dpt._lib.ERR_INVALID_ARG
    assert "member 1: context pointers" in lib().dpt_last_error().decode()


def test_online_population_equals_online_per_member(dpt, members):
    from dpt_b200.evals import eval_bandit
    ms = members(3)
    rs = np.random.RandomState(3)
    trajs = [{"means": rs.uniform(0, 1, 5)} for _ in range(100)]
    dpt.rng.seed(77)
    pop_means, pop_stats = eval_bandit.online_population(trajs, ms, 100, 120, 0.3)
    for i, m in enumerate(ms):
        dpt.rng.seed(77)
        ref_means, ref_stats = eval_bandit.online(trajs, m, 100, 120, 0.3)
        assert list(pop_means[i]) == list(ref_means) == ["opt", "Lnr", "Emp", "UCB1.0", "Thomp"]
        for k in ref_means:
            assert np.array_equal(pop_means[i][k], ref_means[k]), (i, k)
            for s in ref_stats[k]:
                assert np.array_equal(pop_stats[i][k][s], ref_stats[k][s]), (i, k, s)
    assert not np.array_equal(pop_means[0]["Lnr"], pop_means[1]["Lnr"])
