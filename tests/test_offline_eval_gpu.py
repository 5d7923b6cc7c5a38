"""GPU tier of the offline evaluation (dpt_offline_eval, eval_bandit / eval_linear_bandit offline_device and
offline_graph(fused=True)): the reference's golden run, the numpy restatement on the device's own normals, the learner
rows of the single test=False forward, shard independence and the public functions."""
import numpy as np
import pytest
import torch

from conftest import golden
from oracle import dpt_oracle as O
import offline_oracle as OO

pytestmark = pytest.mark.gpu

SLOT = {n: i for i, n in enumerate(("opt", "emp", "lcb", "thmp", "linreg", "lnr"))}


def _np(t):
    return t.detach().cpu().numpy()


def _model(d, H, n_layer=2, sd=None, seed=0):
    from dpt_b200.models.net import Transformer
    torch.manual_seed(seed)
    m = Transformer({"horizon": H, "state_dim": 1, "action_dim": d, "n_layer": n_layer, "n_embd": 32, "n_head": 1,
                     "dropout": 0.0, "test": True})
    if sd is not None:
        m.load_state_dict(sd, strict=False)
    return m


@pytest.fixture(scope="module")
def offline_golden():
    g = golden("offline_bandit")
    d, H = int(g["d"]), int(g["H"])
    N = g["means"].shape[0]
    trajs = [{"means": g["means"][i], "context_states": np.ones((H, 1)), "context_actions": np.eye(d)[g["context_actions"][i]],
              "context_next_states": np.ones((H, 1)), "context_rewards": g["context_rewards"][i]} for i in range(N)]
    sd = {k[3:]: torch.tensor(g[k]) for k in g.files if k.startswith("sd/")}
    return g, trajs, _model(d, H, int(g["n_layer"]), sd)


def test_golden_all_five_controllers(dpt, offline_golden):
    """One launch over horizons [20, 10, 1] with the reference's Thompson normals injected reproduces the per-env
    rewards of the reference's offline() for opt / emp / lnr / lcb / thmp."""
    from dpt_b200.evals import eval_bandit
    g, trajs, m = offline_golden
    N, d, H, var, seed = len(trajs), int(g["d"]), int(g["H"]), float(g["var"]), int(g["seed"])
    horizons = [H, H // 2, 1]
    zs = []
    for h in horizons:
        np.random.seed(seed + h)
        np.random.standard_normal(4 * N)               # the deploy_eval of opt, emp, lnr, lcb
        zs.append(np.random.standard_normal((100, N, d)))
    out = eval_bandit.offline_device(trajs, None, horizons, m, var, inject={"z": np.stack(zs)})
    rew = _np(out["rewards"])
    for k, h in enumerate(horizons):
        for name in ("opt", "emp", "lnr", "lcb", "thmp"):
            assert np.allclose(rew[k, SLOT[name]], g["h%d_%s" % (h, name)], rtol=0, atol=1e-6), (h, name)
    assert np.all(rew[:, SLOT["linreg"]] == 0)         # unselected slots are not written


SWEEP = [(1, 31, 33), (2, 33, 32), (5, 257, 200), (10, 33, 31), (32, 31, 200), (5, 1, 1), (10, 257, 33), (32, 1, 31),
         (2, 257, 1), (1, 1, 200)]


@pytest.mark.parametrize("reward_type", ["uniform", "bernoulli"])
@pytest.mark.parametrize("d,N,H", SWEEP)
def test_oracle_sweep(dpt, d, N, H, reward_type):
    """Contexts from dpt_bandit_rollin, an unsorted horizon list with duplicates, Thompson normals from dump replayed
    through the oracle: every controller's arm is the oracle's and the sums match to 1e-9."""
    var, seed = 0.3, 1000 * d + N + H
    means, _, _ = dpt.kernels.bandit_sample_means(N, d, seed, 0)
    ctx = dpt.kernels.bandit_rollin(means, H, var, seed, 0, reward_type=reward_type)
    hz = np.linspace(1, H, 50, dtype=int)
    np.random.RandomState(seed).shuffle(hz)
    out = dpt.kernels.offline_eval(means, ctx["context_actions"], ctx["context_rewards"], hz, ("opt", "emp", "lcb", "thmp"),
                                   thmp_std=var, seed=seed, dump=True)
    m64 = _np(means).astype(np.float64)
    ca, cr = _np(ctx["context_actions"]).astype(np.float64), _np(ctx["context_rewards"])[:, :, 0].astype(np.float64)
    z = _np(out["noise"]["z"])
    assert np.isfinite(z).all() and z.shape == (50, 100, N, d)
    ctrls = {"opt": O.OptCtrl(m64), "emp": O.EmpMeanCtrl(d, online=False), "lcb": OO.PessMeanCtrl(d, .8),
             "thmp": O.ThompsonCtrl(d, std=var, sample=False, prior_mean=.5, prior_var=1 / 12.0)}
    rew, sums = OO.offline_eval(m64, ca, cr, list(hz), ctrls, O.ReplayNoise({"thompson_z": z.reshape(-1, N, d)}))
    got, gs = _np(out["rewards"]), _np(out["sums"])
    for name in ctrls:
        assert np.array_equal(got[:, SLOT[name]], rew[name]), name
        assert np.allclose(gs[:, SLOT[name]], sums[name], rtol=1e-9, atol=1e-12), name


@pytest.mark.parametrize("lin_d", [2, 5, 8])
def test_linreg_sweep(dpt, lin_d):
    """LinReg on linear-bandit contexts (generate_linear_bandit_histories) against O.LinUCBCtrl(arms, 0.0)."""
    from dpt_b200 import collect_data
    dpt.seed(lin_d)
    N, d, H, var = 70, 10, 40, 0.3
    trajs = collect_data.generate_linear_bandit_histories(N, d, lin_d, H, var, n_hists=1, n_samples=1, cov=0.0, data_type="thompson")
    arms = trajs[0]["arms"]
    m64 = np.stack([t["means"] for t in trajs]).astype(np.float32).astype(np.float64)
    ca = np.stack([t["context_actions"] for t in trajs])
    cr = np.stack([np.asarray(t["context_rewards"]) for t in trajs]).astype(np.float32).astype(np.float64)
    hz = [40, 1, 7, 7, 20, 33, 2]
    out = dpt.kernels.offline_eval(torch.tensor(m64, dtype=torch.float32), torch.tensor(ca, dtype=torch.float32),
                                   torch.tensor(cr, dtype=torch.float32), hz, ("opt", "linreg"), arms=arms)
    rew, sums = OO.offline_eval(m64, ca, cr, hz, {"linreg": O.LinUCBCtrl(arms, 0.0)}, None)
    assert np.array_equal(_np(out["rewards"])[:, SLOT["linreg"]], rew["linreg"])
    assert np.allclose(_np(out["sums"])[:, SLOT["linreg"]], sums["linreg"], rtol=1e-9, atol=1e-12)


@pytest.mark.parametrize("precision,tol", [(0, 1e-5), (1, 2e-2)])
def test_learner_rows(dpt, precision, tol):
    """Row h-1 of the one test=False forward equals the test=True forward on context[:, :h], and the learner's arm is
    its argmax (envs whose top-two gap is within the logit tolerance are exempt, and must be rare)."""
    from dpt_b200.evals import eval_bandit
    N, d, H, var = 96, 5, 40, 0.3
    means, _, _ = dpt.kernels.bandit_sample_means(N, d, 77, 0)
    ctx = dpt.collect_data.collect_bandit(N, d, H, var, seed=77, means=means)
    m = _model(d, H, seed=3)
    m.precision = precision
    hz = [40, 1, 2, 17, 31, 39, 17]
    out = eval_bandit.offline_device(ctx, means, hz, m, var, seed=5)
    lg = _np(eval_bandit.learner_logits(m, {k: ctx[k] for k in ("context_states", "context_actions", "context_next_states",
                                                                  "context_rewards")}, max(hz)))
    assert m.test is True
    lnr, m64 = _np(out["rewards"])[:, SLOT["lnr"]], _np(means).astype(np.float64)
    exempt = 0
    for k, h in enumerate(hz):
        x = {kk: ctx[kk][:, :h] for kk in ("context_states", "context_actions", "context_next_states", "context_rewards")}
        x["query_states"] = torch.ones((N, 1), device="cuda")
        ref = _np(m(x)).astype(np.float64)
        assert np.abs(lg[:, h - 1] - ref).max() <= tol * max(1.0, np.abs(ref).max()), h
        assert np.array_equal(lnr[k], m64[np.arange(N), lg[:, h - 1].argmax(1)]), h      # the kernel's first-max argmax
        top2 = np.sort(ref, axis=1)[:, -2:]
        ok = (top2[:, 1] - top2[:, 0]) >= (1e-5 if precision == 0 else 2 * tol) * np.maximum(1.0, np.abs(top2[:, 1]))
        exempt += int((~ok).sum())
        assert np.array_equal(lnr[k][ok], m64[np.arange(N), ref.argmax(1)][ok]), h
    if precision == 0:   # at the bf16 bar a top-two gap below 4e-2 is common for an untrained model
        assert exempt <= 0.02 * N * len(hz), exempt


def test_shard_independence(dpt):
    """Two launches over env halves (env_id0 = 0, N/2) give the full launch's per-env rewards and normals bit for bit;
    their sums add up to the full launch's."""
    N, d, H, var, seed = 200, 5, 60, 0.3, 31
    means, _, _ = dpt.kernels.bandit_sample_means(N, d, seed, 0)
    ctx = dpt.kernels.bandit_rollin(means, H, var, seed, 0)
    ca, cr = ctx["context_actions"], ctx["context_rewards"]
    hz = [60, 3, 3, 45, 12]
    kw = dict(ctrls=("opt", "emp", "lcb", "thmp"), thmp_std=var, seed=seed, dump=True)
    full = dpt.kernels.offline_eval(means, ca, cr, hz, **kw)
    h = N // 2
    parts = [dpt.kernels.offline_eval(means[s], ca[s], cr[s], hz, env_id0=s.start, **kw) for s in (slice(0, h), slice(h, N))]
    assert torch.equal(torch.cat([p["rewards"] for p in parts], 2), full["rewards"])
    assert torch.equal(torch.cat([p["noise"]["z"] for p in parts], 2), full["noise"]["z"])
    tot = _np(parts[0]["sums"] + parts[1]["sums"])
    assert np.allclose(tot, _np(full["sums"]), rtol=1e-12, atol=0)


def test_offline_graph_fused_bandit(dpt, offline_golden):
    from dpt_b200.evals import eval_bandit
    g, trajs, m = offline_golden
    N, var = len(trajs), float(g["var"])
    hs0, reg0 = eval_bandit.offline_graph(trajs, None, N, 6, var)
    hs1, reg1 = eval_bandit.offline_graph(trajs, None, N, 6, var, fused=True)
    assert np.array_equal(hs0, hs1) and list(reg0) == list(reg1)
    for k in reg0:
        assert reg1[k].shape == reg0[k].shape == (50,) and reg1[k].dtype == reg0[k].dtype and np.all(reg1[k] >= -1e-9), k
    assert np.allclose(reg1["emp"], reg0["emp"], atol=1e-9) and np.allclose(reg1["lcb"], reg0["lcb"], atol=1e-9)
    _, regm = eval_bandit.offline_graph(trajs, m, N, 20, var, fused=True)
    assert list(regm) == ["emp", "lnr", "lcb", "thmp"]
    # an injected run: the regrets of the sums are the ones recomputed from the per-env rewards
    hz = np.linspace(1, 20, 50, dtype=int)
    z = np.random.RandomState(0).standard_normal((50, 100, N, int(g["d"])))
    out = eval_bandit.offline_device(trajs, None, hz, m, var, inject={"z": z})
    rew, s = _np(out["rewards"]), _np(out["sums"])
    for name in ("emp", "lnr", "lcb", "thmp"):
        assert np.allclose(s[:, SLOT[name], 0] / N, (rew[:, 0] - rew[:, SLOT[name]]).mean(1), rtol=1e-12, atol=1e-15), name


def test_offline_graph_fused_linear(dpt):
    from dpt_b200 import collect_data
    from dpt_b200.evals import eval_linear_bandit
    dpt.seed(21)
    N, d, lin_d, H, var = 12, 10, 2, 9, 0.3
    trajs = collect_data.generate_linear_bandit_histories(N, d, lin_d, H, var, n_hists=1, n_samples=1, cov=0.0, data_type="thompson")
    for n in (N, 1):
        hs0, sub0 = eval_linear_bandit.offline_graph(trajs[:n], None, n, H, var)
        hs1, sub1 = eval_linear_bandit.offline_graph(trajs[:n], None, n, H, var, fused=True)
        assert np.array_equal(hs0, hs1) and list(sub0) == list(sub1) == ["thmp", "linreg"]
        for k in sub0:
            for a, b in zip(sub0[k], sub1[k]):
                assert a.shape == b.shape == (H,) and a.dtype == b.dtype, k
            assert np.all(sub1[k][0] >= -1e-9)
            if n == 1:
                assert np.all(np.isnan(sub1[k][1]))
            else:
                assert np.all(sub1[k][1] >= 0)
        assert np.allclose(sub0["linreg"][0], sub1["linreg"][0], atol=1e-6)


def test_offline_device_on_collected_batch_stays_on_device(dpt, monkeypatch):
    """offline_device takes collect_bandit's dict as is: no device tensor comes back to the host during the call."""
    from dpt_b200.evals import eval_bandit
    batch = dpt.collect_data.collect_bandit(300, 5, 64, 0.3, seed=8)
    m = _model(5, 64, seed=1)
    m.handle()                        # the weights are packed once, before the call

    def forbid(name):
        orig = getattr(torch.Tensor, name)

        def f(self, *a, **k):
            if self.is_cuda:
                raise AssertionError("host round trip: Tensor.%s on a device tensor" % name)
            return orig(self, *a, **k)
        monkeypatch.setattr(torch.Tensor, name, f)
    for name in ("cpu", "numpy", "tolist", "item"):
        forbid(name)
    out = eval_bandit.offline_device(batch, None, [64, 1, 32], m, 0.3, seed=2)
    monkeypatch.undo()
    assert out["rewards"].is_cuda and out["sums"].is_cuda
    rew = _np(out["rewards"])
    assert np.all(rew[:, 0] == _np(batch["means"]).max(1)[None])
    assert np.all(rew[:, 1:4] <= rew[:, :1]) and np.all(rew[:, SLOT["lnr"]] > 0)
