"""GPU tier: the GPT-2 forward (dpt_gpt2_forward) and the fused KV-cached online loop
(dpt_gpt2_online_loop) against golden logits from the reference's own Transformer (HF GPT2Model)
and against the float64 oracle.  Bar (north_star): fp32 logits within 1e-5 relative, arms bit-exact
given identical injected noise."""
import numpy as np
import pytest
import torch

from conftest import golden
from oracle import dpt_oracle as O

pytestmark = pytest.mark.gpu
TOL = 1e-5


def _np(t):
    return t.detach().cpu().numpy()


def _close(a, b, tol=TOL):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    assert a.shape == b.shape, (a.shape, b.shape)
    err = np.abs(a - b) / np.maximum(1.0, np.abs(b))
    assert err.max() <= tol, err.max()


def _model(dpt, g, test=True):
    from dpt_b200.models.net import Transformer
    cfg = {"horizon": int(g["H"]), "state_dim": 1, "action_dim": int(g["d"]), "n_layer": int(g["n_layer"]),
           "n_embd": int(g["n_embd"]), "n_head": 1, "dropout": 0.0, "test": test}
    m = Transformer(cfg)
    sd = {k[3:]: torch.tensor(g[k]) for k in g.files if k.startswith("sd/")}
    res = m.load_state_dict(sd, strict=False)
    assert list(res.missing_keys) == ["transformer.wte.weight"] and not res.unexpected_keys
    return m, {k: v.numpy() for k, v in sd.items()}


def _batch(g, t, device="cuda"):
    d = int(g["d"])
    acts, rew = g["fwd_actions"].astype(np.int64), g["fwd_rewards"]
    B, H = acts.shape
    f = lambda a: torch.tensor(a, dtype=torch.float32, device=device)   # noqa: E731
    full = {"context_states": f(np.ones((B, H, 1))), "context_actions": f(np.eye(d)[acts]),
            "context_next_states": f(np.ones((B, H, 1))), "context_rewards": f(rew)}
    b = {k: v[:, :t] for k, v in full.items()}            # views of the [B,H,.] buffers, like eval_bandit.py:71-76
    b["query_states"] = f(np.ones((B, 1)))
    b["zeros"] = torch.zeros(B, 1 + d + 1, device=device)
    return b


@pytest.mark.parametrize("name", ["transformer_l2", "transformer_l4"])
def test_forward_matches_reference_logits(dpt, name):
    g = golden(name)
    m, sd = _model(dpt, g)
    H, L, d = int(g["H"]), int(g["n_layer"]), int(g["d"])
    for t in (0, 1, 5, H):
        b = _batch(g, t)
        m.test = True
        out = m(b)
        assert out.shape == (6, d)
        _close(_np(out), g["logits_t%d" % t])
        o64 = O.transformer_forward(sd, _np(b["query_states"]), _np(b["context_states"]), _np(b["context_actions"]),
                                    _np(b["context_next_states"]), _np(b["context_rewards"]), L, test=True)
        _close(_np(out), o64)
        if t > 0:
            m.test = False
            out = m(b)
            assert out.shape == (6, t, d)
            _close(_np(out), g["logits_all_t%d" % t])
            # contiguous copies give the same answer as strided views
            bc = {k: v.contiguous() for k, v in b.items()}
            assert torch.equal(out, m(bc))
    # state_dict round trip with the reference's extra mask buffers (transformers 4.5.1 checkpoints)
    sd2 = dict(m.state_dict())
    sd2["transformer.h.0.attn.bias"] = torch.ones(1, 1, 4, 4)
    sd2["transformer.h.0.attn.masked_bias"] = torch.tensor(-1e4)
    m.load_state_dict(sd2)
    m.test = True
    _close(_np(m(_batch(g, 5))), g["logits_t5"])
    # a weight update invalidates the packed handle
    with torch.no_grad():
        m.pred_actions.bias.add_(1.0)
    _close(_np(m(_batch(g, 5))), g["logits_t5"] + 1.0)


def test_forward_darkroom_shapes_match_oracle(dpt):
    """state_dim=2 / action_dim=5 (darkroom token layout, query state varies) against the float64 oracle."""
    from dpt_b200.models.net import Transformer
    torch.manual_seed(0)
    cfg = {"horizon": 20, "state_dim": 2, "action_dim": 5, "n_layer": 3, "n_embd": 32, "n_head": 1, "dropout": 0.0, "test": True}
    m = Transformer(cfg)
    with torch.no_grad():
        for k, p in m.named_parameters():
            if "wte" not in k:
                p.add_(0.15 * torch.randn_like(p))
    sd = {k: v.cpu().numpy() for k, v in m.state_dict().items()}
    rs = np.random.RandomState(0)
    B, T = 9, 20
    q = rs.randint(0, 10, (B, 2)).astype(np.float64)
    cs, cns = rs.randint(0, 10, (B, T, 2)).astype(np.float64), rs.randint(0, 10, (B, T, 2)).astype(np.float64)
    ca, cr = np.eye(5)[rs.randint(0, 5, (B, T))], rs.randint(0, 2, (B, T, 1)).astype(np.float64)
    f = lambda a: torch.tensor(a, dtype=torch.float32, device="cuda")   # noqa: E731
    for t in (0, 7, 20):
        out = m({"query_states": f(q), "zeros": torch.zeros(B, 10), "context_states": f(cs[:, :t]), "context_actions": f(ca[:, :t]),
                 "context_next_states": f(cns[:, :t]), "context_rewards": f(cr[:, :t])})
        _close(_np(out), O.transformer_forward(sd, q, cs[:, :t], ca[:, :t], cns[:, :t], cr[:, :t], 3, test=True), 2e-5)
    with pytest.raises(ValueError):
        Transformer(dict(cfg, n_embd=64)).handle()


@pytest.mark.parametrize("name", ["transformer_l2", "transformer_l4"])
def test_online_loop_injected_matches_reference(dpt, name):
    """The reference's own deploy_online_vec + BanditTransformerController(sample=True) run (full recompute
    every step) is reproduced by the fused KV-cached loop fed the same uniforms / normals."""
    g = golden(name)
    m, sd = _model(dpt, g)
    H, var = int(g["H"]), float(g["var"])
    out = m.online_loop(torch.tensor(g["online_means"], dtype=torch.float32), H, var, True, 0,
                        inject={"reward_z": g["online_reward_z"], "ctrl_u": g["online_ctrl_u"]}, dump=True)
    assert np.array_equal(_np(out["context_actions"]).argmax(-1), g["online_actions"])
    _close(_np(out["context_rewards"])[:, :, 0], g["online_rewards"])
    _close(_np(out["cum_means"]), g["online_cum_means"])
    assert bool((out["context_states"] == 1).all()) and bool((out["context_next_states"] == 1).all())
    reg = g["online_means"].max(1)[None] - g["online_cum_means"]
    _close(_np(out["regret_sums"])[:, 0], reg.sum(1), 1e-6)
    _close(_np(out["regret_sums"])[:, 3], (np.cumsum(reg, axis=0) ** 2).sum(1), 1e-6)
    # KV-cached logits at step h == dense forward over the first h context rows
    for h in (0, 3, H - 1):
        b = {k: out[k][:, :h] for k in ("context_states", "context_actions", "context_next_states", "context_rewards")}
        b["query_states"] = torch.ones(out["cum_means"].shape[1], 1, device="cuda")
        _close(_np(out["noise"]["logits"][h]), _np(m(b)), 2e-6)


@pytest.mark.parametrize("sample", [True, False])
def test_online_loop_philox_matches_oracle(dpt, sample):
    g = golden("transformer_l4")
    m, sd = _model(dpt, g)
    N, H, d, L, var, seed = 24, 40, 5, 4, 0.3, 11
    means, _, _ = dpt.kernels.bandit_sample_means(N, d, seed, 0)
    out = m.online_loop(means, H, var, sample, seed, 0, dump=True)
    nz = {k: _np(v).astype(np.float64) for k, v in out["noise"].items()}
    if sample:
        assert nz["ctrl_u"].min() >= 0 and nz["ctrl_u"].max() < 1
    dev_logits = iter(nz["logits"])

    def logits_fn(cs, ca, cns, cr):
        lg = O.transformer_forward(sd, np.ones((N, 1)), cs, ca, cns, cr.astype(np.float32).astype(np.float64), L, test=True)
        _close(next(dev_logits), lg)                                   # device logits within 1e-5 of float64
        return lg
    cum, meta = O.deploy_online_vec(_np(means).astype(np.float64), var, H, O.TransformerCtrl(logits_fn, d, sample=sample),
                                    O.ReplayNoise({"reward_z": nz["reward_z"], "ctrl_u": nz["ctrl_u"].reshape(-1)}))
    assert np.array_equal(_np(out["context_actions"]).astype(np.float64), meta["context_actions"])
    _close(_np(out["context_rewards"]), meta["context_rewards"])
    _close(_np(out["cum_means"]), cum)
    # shard independence + no materialisation
    out2 = m.online_loop(means[7:], H, var, sample, seed, 7, materialise=False)
    assert torch.equal(out["cum_means"][:, 7:], out2["cum_means"])


def test_online_loop_sampling_statistics(dpt):
    """At h = 0 every env sees the same query-only sequence: arm frequencies follow softmax(logits)."""
    g = golden("transformer_l2")
    m, _ = _model(dpt, g)
    N = 40000
    means, _, _ = dpt.kernels.bandit_sample_means(N, 5, 3, 0)
    out = m.online_loop(means, 2, 0.3, True, 3, 0, dump=True)
    lg = out["noise"]["logits"][0]
    assert float((lg - lg[0]).abs().max()) == 0.0
    p = torch.softmax(lg[0].double(), -1)
    freq = out["context_actions"][:, 0].double().mean(0)
    assert float((freq - p).abs().max()) < 5 * 0.5 / N ** 0.5


def test_transformer_controller_dropin(dpt):
    from dpt_b200.ctrls.ctrl_bandit import BanditTransformerController
    from dpt_b200.envs.bandit_env import BanditEnv, BanditEnvVec
    from dpt_b200.evals import eval_bandit
    g = golden("transformer_l2")
    m, _ = _model(dpt, g)
    dpt.seed(0)
    N, H = 32, 12
    rs = np.random.RandomState(0)
    envs = [BanditEnv(rs.uniform(0, 1, 5), H, var=0.3) for _ in range(N)]
    vec = BanditEnvVec(envs)
    ctrl = BanditTransformerController(m, sample=True, batch_size=N)
    cm, meta = eval_bandit.deploy_online_vec(vec, ctrl, H, include_meta=True)          # fused path
    assert cm.shape == (H, N) and meta["context_actions"].shape == (N, H, 5) and np.all(meta["context_actions"].sum(-1) == 1)
    # generic per-step path (set_batch_numpy_vec + act_numpy_vec, full forward per step like the reference)
    ctrl2 = BanditTransformerController(m, sample=False, batch_size=N)
    ctrl2.fused_spec = None
    cm2, meta2 = eval_bandit.deploy_online_vec(vec, ctrl2, 6, include_meta=True)
    assert cm2.shape == (6, N)
    ctrl2.set_batch_numpy_vec({k: v[:, :5] for k, v in meta2.items()})
    a = ctrl2.act_numpy_vec(vec.reset())
    assert np.array_equal(a, meta2["context_actions"][:, 5])                             # deterministic (argmax) controller
    all_means, stats = eval_bandit.online([{"means": e.means} for e in envs], m, N, H, 0.3)
    assert set(all_means) == {"opt", "Lnr", "Emp", "UCB1.0", "Thomp"}


def test_online_loop_config4_size(dpt):
    """BASELINE config 4: 10k envs x H=500, embd 32, 4 layers, sample=True (random-init weights)."""
    from dpt_b200.models.net import Transformer
    torch.manual_seed(0)
    m = Transformer({"horizon": 500, "state_dim": 1, "action_dim": 5, "n_layer": 4, "n_embd": 32, "n_head": 1, "dropout": 0.0, "test": True})
    N, H = 10000, 500
    means, _, _ = dpt.kernels.bandit_sample_means(N, 5, 0, 0)
    out = m.online_loop(means, H, 0.3, True, 0, 0, dump=True)
    torch.cuda.synchronize()
    ca = out["context_actions"]
    assert bool(((ca == 0) | (ca == 1)).all()) and bool((ca.sum(-1) == 1).all())
    assert torch.equal(out["cum_means"].T, (means[:, None, :] * ca).sum(-1))
    resid = (out["context_rewards"][:, :, 0] - out["cum_means"].T) / 0.3
    assert torch.allclose(resid, out["noise"]["reward_z"].T, atol=2e-5)
    # spot-check the KV-cached logits of the last step against the dense forward on the same context
    idx = torch.arange(0, N, 1250, device="cuda")
    b = {k: out[k][idx][:, :H - 1] for k in ("context_states", "context_actions", "context_next_states", "context_rewards")}
    b["query_states"] = torch.ones(len(idx), 1, device="cuda")
    _close(_np(out["noise"]["logits"][H - 1][idx]), _np(m(b)), 5e-6)


@pytest.mark.parametrize("name", ["darkroom_online", "darkroom_online_perm"])
def test_darkroom_online_eval_matches_reference(dpt, name):
    """SURVEY §8(f) row 1: evals/eval_darkroom.py deploy_online_vec with DarkroomTransformerController
    (sample=True) reproduces the reference's per-episode returns from the same np.random seed."""
    from dpt_b200.models.net import Transformer
    from dpt_b200.ctrls.ctrl_darkroom import DarkroomOptPolicy, DarkroomTransformerController
    from dpt_b200.envs.darkroom_env import DarkroomEnv, DarkroomEnvPermuted, DarkroomEnvVec
    from dpt_b200.evals import eval_darkroom
    g = golden(name)
    dim, horizon, H, Heps = int(g["dim"]), int(g["horizon"]), int(g["H"]), int(g["Heps"])
    m = Transformer({"horizon": H, "state_dim": 2, "action_dim": 5, "n_layer": int(g["n_layer"]), "n_embd": 32, "n_head": 1,
                     "dropout": 0.0, "test": True})
    m.load_state_dict({k[3:]: torch.tensor(g[k]) for k in g.files if k.startswith("sd/")}, strict=False)
    if len(g["perm_indices"]):
        envs = [DarkroomEnvPermuted(dim, int(pi), horizon) for pi in g["perm_indices"]]
    else:
        envs = [DarkroomEnv(dim, goal, horizon) for goal in g["goals"]]
    N = len(envs)
    np.random.seed(int(g["seed"]))
    slow = DarkroomTransformerController(m, batch_size=N, sample=True)
    slow.fused = False                                 # the reference's step-by-step loop, same np.random stream
    ret = eval_darkroom.deploy_online_vec(DarkroomEnvVec(envs), slow, Heps, H, horizon)
    assert ret.shape == (N, Heps) and np.array_equal(ret, g["ref_returns"])
    # fused device path (one batched dense forward over all dim*dim query states + one rollout kernel per episode)
    # fed the uniforms the reference consumed: same returns
    fo = eval_darkroom.deploy_online_vec_device(DarkroomEnvVec(envs), m, Heps, H, horizon, sample=True, seed=1, inject_u=g["ctrl_u"])
    assert np.array_equal(_np(fo["returns"]).astype(np.float64), g["ref_returns"])
    # Philox mode: dump the uniforms, replay them through the oracle loop (float64 oracle forward)
    fo = eval_darkroom.deploy_online_vec_device(DarkroomEnvVec(envs), m, Heps, H, horizon, sample=True, seed=7, dump=True)
    sd = {k[3:]: g[k] for k in g.files if k.startswith("sd/")}
    pidx = g["perm_indices"] if len(g["perm_indices"]) else None
    want, _ = O.deploy_online_vec_darkroom(g["goals"], dim, Heps, H, horizon,
                                           lambda q, cs, ca, cns, cr: O.transformer_forward(sd, q, cs, ca, cns, cr, int(g["n_layer"]), test=True),
                                           O.ReplayNoise({"ctrl_u": _np(fo["u"]).reshape(-1)}), pidx)
    assert np.array_equal(_np(fo["returns"]).astype(np.float64), want)
    fused = eval_darkroom.deploy_online_vec(DarkroomEnvVec(envs), DarkroomTransformerController(m, batch_size=N, sample=False), Heps, H, horizon)
    assert fused.shape == (N, Heps)
    # the optimal policy reaches the goal and stays (ctrls/ctrl_darkroom.py:10-20)
    env = envs[0]
    obs, acts, nobs, rews = env.deploy(DarkroomOptPolicy(env))
    gx, gy = int(env.goal[0]), int(env.goal[1])
    assert rews.shape == (horizon,) and rews.sum() == max(0, horizon - max(gx + gy, 1) + 1)
    trajs = [{"goal": e.goal, "perm_index": getattr(e, "perm_index", 0)} for e in envs]
    allm, mean, sem = eval_darkroom.online(trajs, m, Heps, H, N, dim, horizon, permuted=bool(len(g["perm_indices"])))
    assert allm.shape == (N, Heps) and mean.shape == (Heps,) and sem.shape == (Heps,)


@pytest.mark.parametrize("name", ["transformer_l2", "transformer_l4"])
def test_bf16_kv_mode_within_2e2(dpt, name):
    """precision = 1 (bf16 K/V cache, fp32 arithmetic): logits within 2e-2 relative (north_star bf16 bar)
    of the reference's fp32 logits; the loop's arms are consistent with the logits it dumped."""
    g = golden(name)
    m, sd = _model(dpt, g)
    m.precision = 1
    H, L, d = int(g["H"]), int(g["n_layer"]), int(g["d"])
    for t in (0, 1, 5, H):
        b = _batch(g, t)
        m.test = True
        out = m(b)
        _close(_np(out), g["logits_t%d" % t], 2e-2)
        assert t == 0 or not np.array_equal(_np(out), g["logits_t%d" % t])
    N, var, seed = 16, 0.3, 5
    means, _, _ = dpt.kernels.bandit_sample_means(N, d, seed, 0)
    out = m.online_loop(means, H, var, True, seed, 0, dump=True)
    nz = {k: _np(v).astype(np.float64) for k, v in out["noise"].items()}
    ca, cr = _np(out["context_actions"]).astype(np.float64), _np(out["context_rewards"]).astype(np.float64)
    ones = np.ones((N, H, 1))
    for h in range(H):
        ref = O.transformer_forward(sd, np.ones((N, 1)), ones[:, :h], ca[:, :h], ones[:, :h], cr[:, :h], L, test=True)
        _close(nz["logits"][h], ref, 2e-2)
        lg = nz["logits"][h]
        e = np.exp(lg - lg.max(-1, keepdims=True))
        pr = e / e.sum(-1, keepdims=True)
        a = np.array([int(O.choice_cdf(p).searchsorted(u, side="right")) for p, u in zip(pr, nz["ctrl_u"][h])])
        assert np.array_equal(a, ca[:, h].argmax(-1))


@pytest.mark.parametrize("dx,du,L", [(2, 5, 4), (1, 5, 3), (1, 10, 2)])
def test_dense_tensor_core_forward(dpt, dx, du, L):
    """precision = 1: the tcgen05 dense kernels (bf16 operands, fp32 accumulate in TMEM; <= 128 tokens one
    tile, 129..512 tokens the flash-style multi-tile kernel) against the fp32 path and the float64 oracle at
    the 2e-2 bar."""
    from dpt_b200.models.net import Transformer
    torch.manual_seed(dx * 100 + du)
    cfg = {"horizon": 160, "state_dim": dx, "action_dim": du, "n_layer": L, "n_embd": 32, "n_head": 1, "dropout": 0.0, "test": True}
    m = Transformer(cfg)
    with torch.no_grad():
        for k, p in m.named_parameters():
            if "wte" not in k:
                p.add_(0.1 * torch.randn_like(p))
    sd = {k: v.cpu().numpy() for k, v in m.state_dict().items()}
    rs = np.random.RandomState(1)
    B, Tmax = 37, 160
    q = rs.randint(0, 10, (B, dx)).astype(np.float64) if dx == 2 else np.ones((B, dx))
    cs = rs.randint(0, 10, (B, Tmax, dx)).astype(np.float64) if dx == 2 else np.ones((B, Tmax, dx))
    cns = rs.randint(0, 10, (B, Tmax, dx)).astype(np.float64) if dx == 2 else np.ones((B, Tmax, dx))
    ca, cr = np.eye(du)[rs.randint(0, du, (B, Tmax))], rs.normal(0.5, 0.5, (B, Tmax, 1))
    f = lambda a: torch.tensor(a, dtype=torch.float32, device="cuda")   # noqa: E731
    full = {"context_states": f(cs), "context_actions": f(ca), "context_next_states": f(cns), "context_rewards": f(cr)}
    for t in (0, 1, 17, 63, 64, 100, 127, 128, 150):
        x = {k: v[:, :t] for k, v in full.items()}
        x["query_states"] = f(q)
        for test in (True, False):
            if not test and t == 0:
                continue
            m.test = test
            m.precision = 0
            ref = m(x)
            m.precision = 1
            out = m(x)
            assert out.shape == ref.shape
            _close(_np(out), _np(ref), 2e-2)
            assert not torch.equal(out, ref)                   # precision 1 is the bf16 tensor-core path
        if t in (17, 127, 128, 150):
            o64 = O.transformer_forward(sd, q, cs[:, :t], ca[:, :t], cns[:, :t], cr[:, :t], L, test=False)
            _close(_np(out), o64, 2e-2)
    m.precision = 1
    m.test = True
    big = {k: v[:1, :100].expand(300, -1, -1) for k, v in full.items()}     # many CTAs, identical sequences
    big["query_states"] = f(q)[:1].expand(300, -1)
    o = m(big)
    assert float((o - o[0]).abs().max()) == 0.0


def test_forward_long_sequences(dpt):
    """Dense fp32 kernel with 256 / 512 token rows, and the token-sequential kernel (> 512 tokens: fp32 and bf16
    K/V cache) against the float64 oracle."""
    from dpt_b200.models.net import Transformer
    torch.manual_seed(3)
    H, d, L = 560, 5, 2
    m = Transformer({"horizon": H, "state_dim": 1, "action_dim": d, "n_layer": L, "n_embd": 32, "n_head": 1, "dropout": 0.0, "test": True})
    with torch.no_grad():
        for k, p in m.named_parameters():
            if "wte" not in k:
                p.add_(0.05 * torch.randn_like(p))
    sd = {k: v.cpu().numpy() for k, v in m.state_dict().items()}
    rs = np.random.RandomState(2)
    B = 5
    ca, cr = np.eye(d)[rs.randint(0, d, (B, H))], rs.normal(0.5, 0.5, (B, H, 1))
    ones = np.ones((B, H, 1))
    f = lambda a: torch.tensor(a, dtype=torch.float32, device="cuda")   # noqa: E731
    for t in (200, 255, 256, 400, 511, 512, 540):
        x = {"query_states": torch.ones(B, 1, device="cuda"), "context_states": f(ones[:, :t]), "context_actions": f(ca[:, :t]),
             "context_next_states": f(ones[:, :t]), "context_rewards": f(cr[:, :t])}
        ref = O.transformer_forward(sd, np.ones((B, 1)), ones[:, :t], ca[:, :t], ones[:, :t], cr[:, :t], L, test=True)
        m.precision = 0
        _close(_np(m(x)), ref, 1e-5)
        m.precision = 1
        _close(_np(m(x)), ref, 2e-2)
    m.test = False
    for t in (300, 383, 384, 511):      # every row's logits: 3- and 4-tile tensor-core kernels, 512-thread fp32 kernel
        x = {"query_states": torch.ones(B, 1, device="cuda"), "context_states": f(ones[:, :t]), "context_actions": f(ca[:, :t]),
             "context_next_states": f(ones[:, :t]), "context_rewards": f(cr[:, :t])}
        ref = O.transformer_forward(sd, np.ones((B, 1)), ones[:, :t], ca[:, :t], ones[:, :t], cr[:, :t], L, test=False)
        m.precision = 0
        _close(_np(m(x)), ref, 1e-5)
        m.precision = 1
        _close(_np(m(x)), ref, 2e-2)
    m.precision = 0


def test_interactive_bandit_rows(dpt):
    """SURVEY §8(f) row 4 (rollout half of train_interactive.py:97-134) and evals/eval_interactive_bandit.py
    run_online_eval: fused K-step interactive rollout on GPUBanditEnv; the logits it reports at step t are
    the dense forward's logits on context[:, :t]."""
    from dpt_b200.envs.gpu_bandit_env import GPUBanditEnv
    from dpt_b200.evals import eval_interactive_bandit
    g = golden("transformer_l2")
    m, _ = _model(dpt, g)
    env = GPUBanditEnv(5, 300, 12, var=0.3, seed=4)
    ro = env.rollout(m, K=12, sample=True)
    assert ro["context_actions"].shape == (300, 12, 5) and ro["logits"].shape == (12, 300, 5) and ro["target"].shape == (300,)
    assert torch.equal(ro["target"], env.means.argmax(1))
    for t in (0, 5, 11):
        b = {k: ro[k][:, :t] for k in ("context_states", "context_actions", "context_next_states", "context_rewards")}
        b["query_states"] = env.reset()
        _close(_np(ro["logits"][t]), _np(m(b)), 5e-6)
    resid = (ro["context_rewards"][:, :, 0] - (env.means[:, None, :] * ro["context_actions"]).sum(-1)) / 0.3
    assert abs(float(resid.mean())) < 0.1 and abs(float(resid.std()) - 1) < 0.1
    rs = np.random.RandomState(0)
    trajs = [{"means": rs.uniform(0, 1, 5)} for _ in range(64)]
    res = eval_interactive_bandit.run_online_eval(trajs, m, 64, 12, 0.3, "uniform", sample_model=True)
    assert set(res) == {"means", "sems", "regret_means", "regret_sems", "all_means", "all_means_diff"}
    assert set(res["means"]) == {"opt", "Interactive", "Emp", "UCB1.0", "Thomp"}
    assert res["regret_means"]["Thomp"].shape == (12,) and np.all(res["regret_means"]["opt"] == 0)


@pytest.mark.parametrize("name", ["darkroom_online", "darkroom_online_perm"])
def test_darkroom_offline_eval(dpt, name):
    """evals/eval_darkroom.py:124-190 `offline`: Opt / Learner / Learner (greedy) returns of one H-step episode with
    each eval trajectory's own context.  The fused path (policy table from one batched forward + one rollout
    launch) must equal the reference-shaped step-by-step path (DarkroomEnvVec.deploy_eval with the controller
    classes); the sampled learner is replayed through the oracle loop on the dumped uniforms."""
    from dpt_b200 import collect_data
    from dpt_b200.models.net import Transformer
    from dpt_b200.ctrls.ctrl_darkroom import DarkroomOptPolicy, DarkroomTransformerController
    from dpt_b200.envs.darkroom_env import DarkroomEnv, DarkroomEnvPermuted, DarkroomEnvVec
    from dpt_b200.evals import eval_darkroom
    g = golden(name)
    dim, H, nl = int(g["dim"]), int(g["horizon"]), int(g["n_layer"])
    permuted = bool(len(g["perm_indices"]))
    m = Transformer({"horizon": int(g["H"]), "state_dim": 2, "action_dim": 5, "n_layer": nl, "n_embd": 32, "n_head": 1,
                     "dropout": 0.0, "test": True})
    m.load_state_dict({k[3:]: torch.tensor(g[k]) for k in g.files if k.startswith("sd/")}, strict=False)
    dpt.seed(4)
    if permuted:
        trajs = collect_data.generate_darkroom_permuted_histories(g["perm_indices"], dim, H, n_hists=1, n_samples=1, rollin_type="uniform")
        envs = [DarkroomEnvPermuted(dim, int(t["perm_index"]), H) for t in trajs]
    else:
        trajs = collect_data.generate_darkroom_histories(g["goals"], dim, H, n_hists=1, n_samples=1, rollin_type="uniform")
        envs = [DarkroomEnv(dim, t["goal"], H) for t in trajs]
    N = len(trajs)
    res = eval_darkroom.offline(trajs, m, N, H, dim, permuted=permuted)
    assert set(res) == {"Opt", "Learner", "Learner (greedy)"} and all(v.shape == (N,) for v in res.values())
    # Opt: DarkroomOptPolicy deployed on each env (:151-155)
    want_opt = [np.sum(e.deploy_eval(DarkroomOptPolicy(e))[3]) for e in envs]
    assert np.array_equal(res["Opt"], np.array(want_opt, dtype=np.float64))
    # greedy learner: the step-by-step controller path on the same batch
    batch = {"context_states": torch.tensor(np.stack([t["context_states"] for t in trajs]), dtype=torch.float32),
             "context_actions": torch.tensor(np.stack([t["context_actions"] for t in trajs]), dtype=torch.float32),
             "context_next_states": torch.tensor(np.stack([t["context_next_states"] for t in trajs]), dtype=torch.float32),
             "context_rewards": torch.tensor(np.stack([np.asarray(t["context_rewards"])[:, None] for t in trajs]), dtype=torch.float32)}
    greedy = DarkroomTransformerController(m, batch_size=N, sample=False)
    greedy.set_batch(batch)
    rs = DarkroomEnvVec(envs).deploy_eval(greedy)[3]
    assert np.array_equal(res["Learner (greedy)"], np.sum(rs, axis=-1).astype(np.float64))
    # sampled learner: dump the uniforms and replay them through the oracle's episode loop on the same logits
    out = eval_darkroom.offline_device(trajs, m, N, H, dim, permuted=permuted, seed=9, dump=True)
    sd = {k[3:]: g[k] for k in g.files if k.startswith("sd/")}
    cs, ca, cns, cr = (batch[k].numpy().astype(np.float64) for k in ("context_states", "context_actions", "context_next_states", "context_rewards"))
    goals = np.stack([e.goal for e in envs])
    want = O.darkroom_episode(goals, dim, H, lambda q: O.transformer_forward(sd, q, cs, ca, cns, cr, nl, test=True),
                              _np(out["sample"]["u"]), [int(t["perm_index"]) for t in trajs] if permuted else None, sample=True)
    assert np.array_equal(_np(out["returns_sample"]).astype(np.float64), want)
    assert np.all(res["Learner"] <= res["Opt"]) and np.all(res["Learner (greedy)"] <= res["Opt"])


def test_bf16_decode_fallback_geometry(dpt):
    """precision = 1 beyond what one SM's shared memory holds (weight fragments of all layers + 24 warps of score
    scratch): the loop falls back to 4-warp CTAs with the weights read through L1.  Same 2e-2 bar: the logits the loop
    saw at the last steps against a fp32 forward (token-sequential kernel, > 512 tokens) over the context it built.
    At L = 4 the fallback starts at Tpad = 1280 (H > 1216): 4 x 24 KB of fragments + 24 x (160 + Tpad) x 4 B > 227 KB."""
    from dpt_b200.models.net import Transformer
    torch.manual_seed(11)
    H, d, L, N = 1300, 5, 4, 6
    m = Transformer({"horizon": H, "state_dim": 1, "action_dim": d, "n_layer": L, "n_embd": 32, "n_head": 1, "dropout": 0.0, "test": True})
    with torch.no_grad():
        for k, p in m.named_parameters():
            if "wte" not in k:
                p.add_(0.05 * torch.randn_like(p))
    means, _, _ = dpt.kernels.bandit_sample_means(N, d, 3, 0)
    m.precision = 1
    out = m.online_loop(means, H, 0.3, True, 3, 0, dump=True)
    m.precision = 0
    for h in (H - 1, 700, 64):
        b = {k: out[k][:, :h] for k in ("context_states", "context_actions", "context_next_states", "context_rewards")}
        b["query_states"] = torch.ones(N, 1, device="cuda")
        _close(_np(out["noise"]["logits"][h]), _np(m(b)), 2e-2)
    assert float(out["context_actions"].sum(-1).min()) == 1.0


@pytest.mark.parametrize("precision,tol", [(0, 1e-5), (1, 2e-2)])
def test_decoder_step_by_step(dpt, precision, tol):
    """Transformer.decoder: K/V-cached step-by-step logits (arm chosen outside the kernel, as in the interactive
    trainers' rollouts) equal the dense forward over the context appended so far, step by step."""
    from dpt_b200.models.net import Transformer
    torch.manual_seed(5)
    K, d, L, N = 40, 5, 3, 37
    m = Transformer({"horizon": K, "state_dim": 1, "action_dim": d, "n_layer": L, "n_embd": 32, "n_head": 1, "dropout": 0.0, "test": True})
    with torch.no_grad():
        for k, p in m.named_parameters():
            if "wte" not in k:
                p.add_(0.1 * torch.randn_like(p))
    rs = np.random.RandomState(0)
    acts = torch.tensor(np.eye(d)[rs.randint(0, d, (N, K))], dtype=torch.float32, device="cuda")
    rews = torch.tensor(rs.normal(0.5, 0.4, (N, K, 1)), dtype=torch.float32, device="cuda")
    ones = torch.ones(N, K, 1, device="cuda")
    m.precision = precision
    dec = m.decoder(N)
    m.precision = 0                       # dense fp32 reference
    for t in range(K + 1):
        lg = dec.query(torch.ones(N, 1)) if t == 0 else dec.append(ones[:, t - 1], acts[:, t - 1], ones[:, t - 1], rews[:, t - 1])
        ref = m({"query_states": torch.ones(N, 1, device="cuda"), "context_states": ones[:, :t], "context_actions": acts[:, :t],
                 "context_next_states": ones[:, :t], "context_rewards": rews[:, :t]})
        _close(_np(lg), _np(ref), tol)
    with pytest.raises(AssertionError):
        dec.append(ones[:, 0], acts[:, 0], ones[:, 0], rews[:, 0])       # cache full


def test_explorer_exploiter_rollout(dpt):
    """train_explorer_exploiter.py:110-166, no-grad half: two models score the same growing context through their own
    K/V-cached decoders; the recorded logits equal dense forwards over the recorded context, the advantages are the
    exploiter's cross-entropy differences, and the recorded arm is the explorer's (the env is stepped with a random arm)."""
    from dpt_b200.models.net import Transformer
    from dpt_b200.envs.gpu_bandit_env import GPUBanditEnv
    torch.manual_seed(9)
    K, d, N = 12, 5, 70
    cfg = {"horizon": K, "state_dim": 1, "action_dim": d, "n_layer": 2, "n_embd": 32, "n_head": 1, "dropout": 0.0, "test": True}
    explorer, exploiter = Transformer(cfg), Transformer(cfg)
    with torch.no_grad():
        for mdl in (explorer, exploiter):
            for k, p in mdl.named_parameters():
                if "wte" not in k:
                    p.add_(0.2 * torch.randn_like(p))
    for fused in (True, False):
        env = GPUBanditEnv(d, N, K, var=0.3, seed=4)
        out = env.rollout_explorer_exploiter(explorer, exploiter, fused=fused, dump=fused)
        assert out["context_actions"].shape == (N, K, d) and float(out["context_actions"].sum(-1).min()) == 1.0
        assert out["advantages"].shape == (N, K - 1, 1) and out["explorer_logits"].shape == (K, N, d)
        assert bool((out["context_states"] == 1).all()) and bool((out["context_next_states"] == 1).all())
        names = ("context_states", "context_actions", "context_next_states", "context_rewards")
        losses = []
        for t in range(K):
            b = {k: out[k][:, :t] for k in names}
            b["query_states"] = torch.ones(N, 1, device="cuda")
            _close(_np(out["exploiter_logits"][t]), _np(exploiter(b)), 1e-5)
            _close(_np(out["explorer_logits"][t]), _np(explorer(b)), 1e-5)
            losses.append(torch.nn.functional.cross_entropy(out["exploiter_logits"][t], out["target"], reduction="none"))
        for t in range(1, K):
            assert torch.allclose(out["advantages"][:, t - 1, 0], losses[t] - losses[t - 1], atol=1e-5 if fused else 1e-6)
        with pytest.raises(ValueError):
            env.step(out["context_actions"][:, 0])       # the episode of K steps is over (:59-61)
        if not fused:
            continue
        # the fused launch: recorded arm = categorical draw from the explorer's logits on the dumped uniform (float64 softmax
        # cdf, searchsorted 'right'), reward = means[random arm] + var * z, and a replay on the dumped draws is identical
        nz = {k: _np(v) for k, v in out["noise"].items()}
        means = _np(env.means).astype(np.float64)
        assert nz["random_arm"].min() >= 0 and nz["random_arm"].max() < d and len(np.unique(nz["random_arm"])) == d
        for t in range(K):
            lg = _np(out["explorer_logits"][t]).astype(np.float64)
            pr = np.exp(lg - lg.max(1, keepdims=True))
            pr /= pr.sum(1, keepdims=True)
            cdf = np.cumsum(pr, 1)
            cdf /= cdf[:, -1:]
            arm = (cdf[:, :-1] <= nz["ctrl_u"][t][:, None]).sum(1)
            assert np.array_equal(_np(out["context_actions"][:, t]).argmax(1), arm), t
            want_r = means[np.arange(N), nz["random_arm"][t]] + 0.3 * nz["reward_z"][t].astype(np.float64)
            assert np.allclose(_np(out["context_rewards"][:, t, 0]), want_r, atol=1e-6)
        env2 = GPUBanditEnv(d, N, K, var=0.3, seed=4)
        rep = env2.rollout_explorer_exploiter(explorer, exploiter, inject=out["noise"])
        for k in names + ("advantages", "explorer_logits", "exploiter_logits"):
            assert torch.equal(rep[k], out[k]), k
        # a re-used env object does not replay its noise
        again = env2.rollout_explorer_exploiter(explorer, exploiter)
        assert not torch.equal(again["context_rewards"], rep["context_rewards"])
    # the single-model fused rollout also serves bernoulli envs now
    benv = GPUBanditEnv(d, N, K, var=0.3, type="bernoulli", seed=4)
    r = benv.rollout(explorer, K)
    assert set(np.unique(_np(r["context_rewards"]))) <= {0.0, 1.0}


@pytest.mark.parametrize("du,H,L,N", [(2, 17, 1, 50), (10, 65, 3, 29), (5, 130, 4, 25)])
def test_bf16_decode_shapes(dpt, du, H, L, N):
    """precision = 1 loop (tensor-core attention + projections, 16-key V blocks, 64-key K tiles) at horizons that are not
    multiples of the block sizes, other arm counts and depths, env counts that do not fill a CTA: logits the loop saw
    against the fp32 dense / token-sequential forward over the context it built (2e-2), one-hot actions throughout."""
    from dpt_b200.models.net import Transformer
    torch.manual_seed(du * 7 + H)
    m = Transformer({"horizon": H, "state_dim": 1, "action_dim": du, "n_layer": L, "n_embd": 32, "n_head": 1, "dropout": 0.0, "test": True})
    with torch.no_grad():
        for k, p in m.named_parameters():
            if "wte" not in k:
                p.add_(0.08 * torch.randn_like(p))
    means, _, _ = dpt.kernels.bandit_sample_means(N, du, 3, 0)
    m.precision = 1
    out = m.online_loop(means, H, 0.3, True, 3, 0, dump=True)
    m.precision = 0
    for h in sorted({0, 1, 15, 16, 17, 63, 64, H - 1} & set(range(H))):
        b = {k: out[k][:, :h] for k in ("context_states", "context_actions", "context_next_states", "context_rewards")}
        b["query_states"] = torch.ones(N, 1, device="cuda")
        _close(_np(out["noise"]["logits"][h]), _np(m(b)), 2e-2)
    assert float(out["context_actions"].sum(-1).min()) == 1.0 and float(out["context_actions"].sum(-1).max()) == 1.0
