"""GPU tier: parity of the CUDA rollout kernels (through the C ABI) against the golden vectors
from the live reference and against the oracle on identical noise.

Bars: integer / index outputs (actions, states, next states, darkroom rewards) bit-exact;
fp32 bandit rewards within 1e-5 relative of the float64 reference (north_star)."""
import numpy as np
import pytest
import torch

from conftest import golden
from oracle import dpt_oracle as O
from oracle import philox as P

pytestmark = pytest.mark.gpu
RTOL = 1e-5


def _close(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    assert a.shape == b.shape
    assert np.all(np.abs(a - b) <= RTOL * np.maximum(1.0, np.abs(b))), np.abs(a - b).max()


def _np(t):
    return t.detach().cpu().numpy()


# ------------------------------------------------------------------ bandit rollin -------------
@pytest.mark.parametrize("name", ["bandit_rollin_d5", "bandit_rollin_d10", "bandit_rollin_d3"])
def test_bandit_rollin_injected_matches_reference(dpt, name):
    """Identical injected noise -> the reference's own outputs (fast path d5 H=24, generic d10 H=37)."""
    g = golden(name)
    H = int(g["H"])
    inj = {k: g[k] for k in ("cov_idx", "dir_probs", "rand_idx", "u", "z")}
    out = dpt.kernels.bandit_rollin(torch.tensor(g["means"], dtype=torch.float32), H, float(g["var"]), 0, inject=inj)
    assert np.array_equal(_np(out["context_actions"]).astype(np.float64), g["ref_actions"])
    _close(_np(out["context_rewards"])[:, :, 0], g["ref_rewards"])
    assert np.array_equal(_np(out["context_states"]), g["ref_states"].astype(np.float32))
    assert np.array_equal(_np(out["context_next_states"]), g["ref_next_states"].astype(np.float32))
    # action-stream injection gives the same thing
    out2 = dpt.kernels.bandit_rollin(torch.tensor(g["means"], dtype=torch.float32), H, float(g["var"]), 0,
                                     inject={"actions": g["ref_actions"].argmax(-1), "z": g["z"]})
    for k in out:
        assert torch.equal(out[k], out2[k])


@pytest.mark.parametrize("N,d,H", [(64, 5, 500), (33, 10, 200), (7, 3, 61), (5, 16, 36), (3, 24, 17), (2, 1, 9)])
def test_bandit_rollin_philox_matches_oracle(dpt, N, d, H):
    """Philox mode: integer layer bit-exact against oracle/philox.py; outputs against the oracle
    fed with the noise the device dumped."""
    seed, env_id0, var = 1234567, 1000, 0.3
    means, opt_idx, opt_a = dpt.kernels.bandit_sample_means(N, d, seed, env_id0)
    ids = env_id0 + np.arange(N)
    m_or = P.bandit_means(seed, ids, d)
    assert np.array_equal(_np(means).astype(np.float64), m_or)
    assert np.array_equal(_np(opt_idx), m_or.argmax(1))
    assert np.array_equal(_np(opt_a), np.eye(d)[m_or.argmax(1)].astype(np.float32))
    out = dpt.kernels.bandit_rollin(means, H, var, seed, env_id0, dump=True)
    nz = {k: _np(v) for k, v in out["noise"].items()}
    cov_idx, rand_idx = P.rollin_setup_ints(seed, ids, d)
    assert np.array_equal(nz["cov_idx"], cov_idx) and np.array_equal(nz["rand_idx"], rand_idx)
    assert np.array_equal(nz["u"], P.rollin_step_k(seed, ids, H) * 2.0 ** -31)
    assert np.allclose(nz["dir_probs"].sum(1), 1.0, atol=1e-12) and nz["dir_probs"].min() >= 0
    xs, us, xps, rs, acts = O.rollin_bandit_batch(m_or, var, nz["cov_idx"], nz["dir_probs"], nz["rand_idx"], nz["u"], nz["z"])
    assert np.array_equal(nz["actions"], acts)
    assert np.array_equal(_np(out["context_actions"]).astype(np.float64), us)
    _close(_np(out["context_rewards"])[:, :, 0], rs)
    assert np.array_equal(_np(out["context_states"]), xs.astype(np.float32))
    # without dump: identical outputs
    out2 = dpt.kernels.bandit_rollin(means, H, var, seed, env_id0)
    for k in ("context_states", "context_actions", "context_next_states", "context_rewards"):
        assert torch.equal(out[k], out2[k])


def test_bandit_rollin_fast_and_generic_paths_agree(dpt):
    """Same (env, h) -> same draw whatever kernel variant runs: H=64 (fast) vs H=63 (generic)."""
    means, _, _ = dpt.kernels.bandit_sample_means(40, 5, 7, 0)
    a = dpt.kernels.bandit_rollin(means, 64, 0.3, 7, 0)
    b = dpt.kernels.bandit_rollin(means, 63, 0.3, 7, 0)
    for k in a:
        assert torch.equal(a[k][:, :63], b[k])


def test_bandit_rollin_shard_independent(dpt):
    """Contiguous env-range shards with global env ids reproduce the single-call result bit-for-bit."""
    N, d, H, seed = 1000, 5, 100, 99
    means, _, _ = dpt.kernels.bandit_sample_means(N, d, seed, 0)
    full = dpt.kernels.bandit_rollin(means, H, 0.3, seed, 0)
    for lo, hi in [(0, 125), (125, 700), (700, 1000)]:
        m2, _, _ = dpt.kernels.bandit_sample_means(hi - lo, d, seed, lo)
        assert torch.equal(m2, means[lo:hi])
        part = dpt.kernels.bandit_rollin(m2, H, 0.3, seed, lo)
        for k in full:
            assert torch.equal(full[k][lo:hi], part[k])


def test_bandit_rollin_full_size_properties(dpt):
    """BASELINE config 5 per-GPU shard (125k envs x H=500 x d=5, 2 GB): size-independent properties."""
    N, d, H, var, seed = 125000, 5, 500, 0.3, 0
    means, opt_idx, _ = dpt.kernels.bandit_sample_means(N, d, seed, 0)
    out = dpt.kernels.bandit_rollin(means, H, var, seed, 0, dump=True)
    ca, cr = out["context_actions"], out["context_rewards"][:, :, 0]
    assert bool((out["context_states"] == 1).all()) and bool((out["context_next_states"] == 1).all())
    assert bool(((ca == 0) | (ca == 1)).all()) and bool((ca.sum(-1) == 1).all())      # one-hot rows
    acts = ca.argmax(-1)
    assert torch.equal(acts.int(), out["noise"]["actions"])
    resid = (cr - torch.gather(means, 1, acts)) / var                                  # == z
    assert torch.allclose(resid, out["noise"]["z"], atol=2e-5)
    z = out["noise"]["z"].double()
    n = z.numel()
    assert abs(float(z.mean())) < 5 / n ** 0.5 and abs(float(z.var()) - 1) < 5 * (2 / n) ** 0.5
    assert abs(float((z ** 4).mean()) - 3) < 0.01 and abs(float((z ** 3).mean())) < 0.01
    # empirical action frequencies follow the per-env behaviour policy
    cov = torch.tensor(O.COV_GRID, device=ca.device, dtype=torch.float64)[out["noise"]["cov_idx"].long()][:, None]
    probs = (1 - cov) * out["noise"]["dir_probs"] + cov * torch.nn.functional.one_hot(out["noise"]["rand_idx"].long(), d)
    freq = ca.double().mean(1)
    assert float((freq - probs).abs().max()) < 6 * 0.5 / H ** 0.5
    assert abs(float((freq - probs).mean())) < 1e-4
    counts = torch.bincount(out["noise"]["cov_idx"].long(), minlength=11).double() / N
    assert float((counts - 1 / 11).abs().max()) < 0.005
    u = out["noise"]["u"]
    assert float(u.min()) >= 0 and float(u.max()) < 1 and abs(float(u.mean()) - 0.5) < 1e-3


def test_bandit_rollin_edge_cases(dpt):
    k = dpt.kernels
    m = torch.rand(0, 5)
    out = k.bandit_rollin(m.cuda(), 8, 0.3, 0)
    assert out["context_actions"].shape == (0, 8, 5)
    out = k.bandit_rollin(torch.rand(3, 5).cuda(), 0, 0.3, 0)
    assert out["context_rewards"].shape == (3, 0, 1)
    with pytest.raises(ValueError):
        k.bandit_rollin(torch.rand(3, 40).cuda(), 8, 0.3, 0)           # d > 32
    # unaligned output views force the generic path and still agree with the aligned run
    means, _, _ = k.bandit_sample_means(9, 5, 3, 0)
    ref = k.bandit_rollin(means, 20, 0.3, 3, 0)
    pad = {n: torch.empty(t.numel() + 1, device="cuda")[1:].view_as(t) for n, t in ref.items()}
    got = k.bandit_rollin(means, 20, 0.3, 3, 0, out=pad)
    for n in ref:
        assert torch.equal(ref[n], got[n])
    # cov = 1.0 (all mass on rand_index) and cov = 0: cdf entries exactly 0 / 1
    g = golden("bandit_rollin_d5")
    inj = {"cov_idx": np.full(8, 10, np.int32), "dir_probs": g["dir_probs"], "rand_idx": g["rand_idx"], "u": g["u"], "z": g["z"]}
    out = k.bandit_rollin(torch.tensor(g["means"], dtype=torch.float32), 24, 0.3, 0, inject=inj)
    assert np.array_equal(_np(out["context_actions"]).argmax(-1), np.repeat(g["rand_idx"][:, None], 24, 1))


def test_bandit_rollin_host_path(dpt):
    """The e2e entry point (host buffers, pipelined copies) returns exactly the device-path result."""
    N, d, H, seed = 20000, 5, 100, 5
    means, _, _ = dpt.kernels.bandit_sample_means(N, d, seed, 0)
    dev = dpt.kernels.bandit_rollin(means, H, 0.3, seed, 0)
    host, _ = dpt.kernels.bandit_rollin_host(means.cpu().pin_memory(), H, 0.3, seed, 0)
    for k in dev:
        assert torch.equal(dev[k].cpu(), host[k])
    # >= 4 chunks of 8192 envs: the hybrid pipeline (some chunks cross PCIe as arm index + reward and are expanded
    # by host threads, the others arrive fully formed by DMA) must still reproduce the device result bit for bit
    for N, d, H in ((40000, 5, 60), (33000, 10, 22), (35000, 3, 41), (33001, 1, 7), (32769, 32, 5), (70000, 2, 9)):
        means, _, _ = dpt.kernels.bandit_sample_means(N, d, seed, 7)
        dev = dpt.kernels.bandit_rollin(means, H, 0.3, seed, 7)
        host, _ = dpt.kernels.bandit_rollin_host(means.cpu().pin_memory(), H, 0.3, seed, 7)
        for k in dev:
            assert torch.equal(dev[k].cpu(), host[k]), (N, d, H, k)
    # pageable (not pinned) caller buffers: slower copies, same result
    out = {"context_states": torch.empty((N, H, 1)), "context_actions": torch.empty((N, H, d)),
           "context_next_states": torch.empty((N, H, 1)), "context_rewards": torch.empty((N, H, 1))}
    host, _ = dpt.kernels.bandit_rollin_host(means.cpu(), H, 0.3, seed, 7, out=out)
    for k in dev:
        assert torch.equal(dev[k].cpu(), host[k]), ("pageable", k)


# ------------------------------------------------------------------ darkroom ------------------
@pytest.mark.parametrize("name", ["darkroom_uniform", "darkroom_expert", "darkroom_perm_uniform", "darkroom_perm_expert"])
def test_darkroom_injected_matches_reference(dpt, name):
    g = golden(name)
    H, dim, mode = int(g["H"]), int(g["dim"]), str(g["rollin_type"])
    perms = g["perm_indices"] if len(g["perm_indices"]) else None
    inj = {"query": g["query"][:, None, :]}
    if mode == "uniform":
        inj.update(states=g["state"], actions=g["action"])
    out = dpt.kernels.darkroom_rollin(g["goals"], dim, H, mode, 0, 0, perms, 1, inject=inj)
    assert np.array_equal(_np(out["context_states"]), g["ref_states"].astype(np.float32))
    assert np.array_equal(_np(out["context_actions"]), np.eye(5, dtype=np.float32)[g["ref_actions"]])
    assert np.array_equal(_np(out["context_next_states"]), g["ref_next_states"].astype(np.float32))
    assert np.array_equal(_np(out["context_rewards"])[:, :, 0], g["ref_rewards"].astype(np.float32))
    assert np.array_equal(_np(out["query_states"])[:, 0], g["query"].astype(np.float32))
    assert np.array_equal(_np(out["optimal_actions"])[:, 0].argmax(-1), g["ref_optimal_action"])


@pytest.mark.parametrize("N,dim,H,S,perm", [(300, 10, 100, 1, False), (50, 7, 33, 3, True), (17, 256, 64, 2, False),
                                            (9, 300, 12, 1, True), (1000, 10, 100, 1, True)])
def test_darkroom_philox_matches_oracle(dpt, N, dim, H, S, perm):
    """All-integer path: Philox-mode output equals the oracle driven by oracle/philox.py draws."""
    seed, env_id0 = 42, 5000
    rs = np.random.RandomState(1)
    goals = rs.randint(0, dim, (N, 2))
    pidx = rs.randint(0, 120, N) if perm else None
    out = dpt.kernels.darkroom_rollin(goals, dim, H, "uniform", seed, env_id0, pidx, S, dump=True)
    ids = env_id0 + np.arange(N)
    st, ac = P.darkroom_draws(seed, ids, H, dim)
    q = P.darkroom_query(seed, ids, S, dim)
    assert np.array_equal(_np(out["noise"]["states"]), st) and np.array_equal(_np(out["noise"]["actions"]), ac)
    assert np.array_equal(_np(out["noise"]["query"]), q)
    pt = None if pidx is None else np.asarray(O.DARKROOM_PERMS)[pidx][:, None, :]
    ns, r = O.darkroom_transit_batch(st, ac, goals[:, None, :], dim, pt)
    assert np.array_equal(_np(out["context_states"]), st.astype(np.float32))
    assert np.array_equal(_np(out["context_actions"]), np.eye(5, dtype=np.float32)[ac])
    assert np.array_equal(_np(out["context_next_states"]), ns.astype(np.float32))
    assert np.array_equal(_np(out["context_rewards"])[:, :, 0], r.astype(np.float32))
    assert np.array_equal(_np(out["query_states"]), q.astype(np.float32))
    oa = np.array([[O.darkroom_opt_action_index(q[e, s], goals[e], None if pidx is None else O.DARKROOM_PERMS[pidx[e]])
                    for s in range(S)] for e in range(N)])
    assert np.array_equal(_np(out["optimal_actions"]).argmax(-1), oa)


@pytest.mark.parametrize("H", [40, 23])
def test_darkroom_expert_matches_oracle(dpt, H):
    dim = 10
    rs = np.random.RandomState(2)
    goals = rs.randint(0, dim, (60, 2))
    pidx = rs.randint(0, 120, 60)
    for perm in (None, pidx):
        out = dpt.kernels.darkroom_rollin(goals, dim, H, "expert", 0, 0, perm, 0)
        for e in range(60):
            s, a, ns, r = O.rollin_mdp(goals[e], dim, H, "expert", None, None if perm is None else int(perm[e]))
            assert np.array_equal(_np(out["context_states"][e]), s.astype(np.float32))
            assert np.array_equal(_np(out["context_actions"][e]), a.astype(np.float32))
            assert np.array_equal(_np(out["context_next_states"][e]), ns.astype(np.float32))
            assert np.array_equal(_np(out["context_rewards"][e, :, 0]), r.astype(np.float32))


def test_darkroom_exhaustive_transition_table(dpt):
    """All 10x10x5 (state, action) pairs per goal / permutation against the reference's own transit()."""
    g = golden("darkroom_table")
    dim = int(g["dim"])
    xs, ys, acts = np.meshgrid(np.arange(dim), np.arange(dim), np.arange(5), indexing="ij")
    st = np.stack([xs, ys], -1).reshape(-1, 2)
    onehot = np.eye(5, dtype=np.float32)[acts.reshape(-1)]
    st2 = np.stack(np.meshgrid(np.arange(dim), np.arange(dim), indexing="ij"), -1).reshape(-1, 2)
    for i, goal in enumerate(g["goals"]):
        ns, r = dpt.kernels.darkroom_step(st, onehot, np.repeat(goal[None], len(st), 0), dim)
        assert np.array_equal(_np(ns).reshape(dim, dim, 5, 2), g["next_state"][i])
        assert np.array_equal(_np(r).reshape(dim, dim, 5), g["reward"][i])
        oa = dpt.kernels.darkroom_opt_action(st2, np.repeat(goal[None], len(st2), 0))
        assert np.array_equal(_np(oa).argmax(-1).reshape(dim, dim), g["opt_action"][i])
    for i, pi in enumerate(g["perms"]):
        goal = np.array([dim - 1, dim - 1])
        ns, r = dpt.kernels.darkroom_step(st, onehot, np.repeat(goal[None], len(st), 0), dim, np.full(len(st), pi))
        assert np.array_equal(_np(ns).reshape(dim, dim, 5, 2), g["p_next_state"][i])
        assert np.array_equal(_np(r).reshape(dim, dim, 5), g["p_reward"][i])
        oa = dpt.kernels.darkroom_opt_action(st2, np.repeat(goal[None], len(st2), 0), np.full(len(st2), pi))
        assert np.array_equal(_np(oa).argmax(-1).reshape(dim, dim), g["p_opt_action"][i])


def test_darkroom_full_size_config2(dpt):
    """BASELINE config 2: 100k envs, dim 10, H 100 -- bit-exact against the vectorised oracle."""
    N, dim, H, seed = 100000, 10, 100, 0
    goals = np.repeat(np.stack(np.meshgrid(np.arange(dim), np.arange(dim), indexing="ij"), -1).reshape(-1, 2), N // dim ** 2, 0)
    out = dpt.kernels.darkroom_rollin(goals, dim, H, "uniform", seed, 0, None, 1)
    st, ac = P.darkroom_draws(seed, np.arange(N), H, dim)
    ns, r = O.darkroom_transit_batch(st, ac, goals[:, None, :], dim)
    assert np.array_equal(_np(out["context_states"]), st.astype(np.float32))
    assert np.array_equal(_np(out["context_actions"]).argmax(-1), ac)
    assert np.array_equal(_np(out["context_next_states"]), ns.astype(np.float32))
    assert np.array_equal(_np(out["context_rewards"])[:, :, 0], r.astype(np.float32))
    # uniformity of the joint draw
    cnt = np.bincount((st[..., 0] * dim + st[..., 1]).ravel() * 5 + ac.ravel(), minlength=500) / st[..., 0].size
    assert np.abs(cnt - 1 / 500).max() < 5 * (1 / 500 / st[..., 0].size) ** 0.5


# ------------------------------------------------------------------ env classes (drop-in API) --
def test_gpu_bandit_env_matches_reference_semantics(dpt):
    from dpt_b200.envs.gpu_bandit_env import GPUBanditEnv
    env = GPUBanditEnv(5, 1000, 3, var=0.3, seed=11)
    assert env.means.shape == (1000, 5) and env.opt_a.shape == (1000, 5) and env.state.shape == (1000, 1)
    assert torch.equal(env.opt_a_index, env.means.argmax(1)) and env.H == 3 and env.du == 5 and env.dx == 1
    s = env.reset()
    assert torch.equal(s, torch.ones(1000, 1, device=s.device))
    acts = torch.nn.functional.one_hot(torch.randint(0, 5, (1000,)), 5).float().cuda()
    z = torch.randn(1000).cuda()
    _, r = env.transit(env.state, acts, inject=z)                       # r = means[a] + var * z (gpu_bandit_env.py:56-58)
    want = (env.means * acts).sum(1).double() + 0.3 * z.double()
    assert torch.allclose(r.double(), want, rtol=1e-5, atol=1e-6)
    rs = []
    for t in range(3):
        st, r, done, info = env.step(acts)
        assert r.shape == (1000,) and done.dtype == torch.bool and bool(done.all()) == (t == 2) and info == {}
        rs.append(r)
    assert not torch.equal(rs[0], rs[1])                                 # fresh noise every step
    resid = torch.stack(rs) - (env.means * acts).sum(1)
    assert abs(float(resid.std()) - 0.3) < 0.02
    with pytest.raises(ValueError, match="Episode has already ended"):
        env.step(acts)
    assert torch.allclose(env.get_arm_value(acts), (env.means * acts).sum(1))
    b = GPUBanditEnv(5, 20000, 4, type="bernoulli", seed=3)
    a = b.opt_a
    r = torch.stack([b.step(a)[1] for _ in range(4)])
    assert bool(((r == 0) | (r == 1)).all()) and abs(float(r.mean()) - float(b.means.max(1).values.mean())) < 0.01
    with pytest.raises(NotImplementedError):
        GPUBanditEnv(5, 10, 4, type="gaussian")


def test_gpu_bandit_env_golden(dpt):
    """E5 pin: tests/golden/gpu_bandit_env.npz holds the reference's own GPUBanditEnv (envs/gpu_bandit_env.py:12-82) run
    on CPU with torch.randn / torch.bernoulli patched to record their noise (oracle/make_golden.py:gpu_bandit_env)."""
    from dpt_b200.envs.gpu_bandit_env import GPUBanditEnv
    g = golden("gpu_bandit_env")
    N, d, H, var = int(g["N"]), int(g["d"]), int(g["H"]), float(g["var"])
    for typ in ("uniform", "bernoulli"):
        env = GPUBanditEnv(d, N, H, var=var, type=typ, seed=1)
        for k, v in dict(dims=d, dim=d, n_envs=N, H_context=H, H=H, var=var, dx=1, du=d, topk=False, type=typ).items():
            assert getattr(env, k) == v, k
        env.set_means(torch.tensor(g[typ + "_means"]))
        assert np.array_equal(env.opt_a_index.cpu().numpy(), g[typ + "_opt_a_index"])          # int64 argmax: bit-exact
        assert env.opt_a_index.dtype == torch.int64 and np.array_equal(env.opt_a.cpu().numpy(), g[typ + "_opt_a"])
        s0 = env.reset()
        assert s0.shape == (N, 1) and bool((s0 == 1).all())
        for t in range(H):
            a = torch.nn.functional.one_hot(torch.tensor(g[typ + "_actions"][t].astype(np.int64)), d).float().cuda()
            st, r, done, info = env.step(a, inject=torch.tensor(g[typ + "_noise"][t]))
            ref = g[typ + "_rewards"][t].astype(np.float64)
            got = r.cpu().numpy().astype(np.float64)
            if typ == "bernoulli":
                assert np.array_equal(got, ref)                                                 # {0,1}: bit-exact
            else:
                assert np.all(np.abs(got - ref) <= 1e-5 * np.maximum(1.0, np.abs(ref)))
            assert st.shape == (N, 1) and bool((st == 1).all()) and info == {} and done.dtype == torch.bool
            assert np.array_equal(done.cpu().numpy(), g[typ + "_done"][t])
        with pytest.raises(ValueError, match=str(g[typ + "_error"])):
            env.step(a)
        assert np.allclose(env.get_arm_value(a).cpu().numpy(), g[typ + "_arm_value"], rtol=1e-6, atol=0)


def test_gpu_bandit_env_rollout_fresh_noise(dpt):
    """A re-used env object must not replay the noise of its previous fused rollout (ADVICE r1)."""
    from dpt_b200.envs.gpu_bandit_env import GPUBanditEnv
    from dpt_b200.models.net import Transformer
    torch.manual_seed(0)
    net = Transformer({"horizon": 8, "state_dim": 1, "action_dim": 5, "n_layer": 2, "n_embd": 32, "n_head": 1, "dropout": 0.0, "test": True})
    env = GPUBanditEnv(5, 256, 8, var=0.3, seed=5)
    r1 = env.rollout(net)["context_rewards"].clone()
    r2 = env.rollout(net)["context_rewards"].clone()
    assert not torch.equal(r1, r2)


def test_bandit_env_classes(dpt):
    from dpt_b200.envs.bandit_env import BanditEnv, BanditEnvVec, LinearBanditEnv
    dpt.seed(0)
    env = BanditEnv(np.array([0.1, 0.9, 0.5]), 10, var=0.0)
    assert env.opt_a_index == 1 and env.H == 1 and env.H_context == 10 and env.dx == 1 and env.du == 3
    env.reset()
    s, r, done, _ = env.step(np.array([0, 0, 1.0]))
    assert np.array_equal(s, [1]) and abs(r - 0.5) < 1e-6 and done
    with pytest.raises(ValueError, match="Episode has already ended"):
        env.step(np.array([0, 0, 1.0]))
    envs = [BanditEnv(np.random.RandomState(i).rand(5), 10, var=0.3) for i in range(64)]
    vec = BanditEnvVec(envs)

    class Fixed:
        def act_numpy_vec(self, x):
            return np.eye(5)[np.arange(64) % 5]
    xs, us, xps, rs = vec.deploy(Fixed())
    assert xs.shape == (64, 1) and us.shape == (64, 5) and xps.shape == (64, 1) and rs.shape == (64,)
    want = np.array([e.means[i % 5] for i, e in enumerate(envs)])
    assert np.abs(rs - want).std() > 0.1 and np.abs(rs - want).max() < 2.0
    xs, us, xps, rs0 = vec.deploy_eval(Fixed())                                   # zero variance
    assert np.allclose(rs0, want, atol=1e-6) and envs[0].var == 0.3
    assert np.allclose(vec.get_arm_value(us), want, atol=1e-6)
    arms = O.linear_bandit_arms(10, 2)
    le = LinearBanditEnv(np.array([0.3, -0.2]), arms, 5, var=0.1)
    assert np.allclose(le.means, arms @ np.array([0.3, -0.2])) and le.opt_a[le.opt_a_index] == 1


def test_bandit_rollin_host_reference_dtypes(dpt):
    """dpt_bandit_rollin_host_f64 (the reference's own host dtypes, collect_data.py:23-53) == the device path, value for
    value, at ragged sizes (partial chunks, d with and without the lookup table)."""
    for N, H, d in ((1, 1, 5), (37, 23, 5), (9000, 40, 5), (300, 64, 3), (50, 31, 7), (20000, 8, 2)):
        means, _, _ = dpt.kernels.bandit_sample_means(N, d, 17, 3)
        dev = dpt.kernels.bandit_rollin(means, H, 0.3, 99, 3)
        host = dpt.kernels.bandit_rollin_host_ref(means.cpu(), H, 0.3, 99, 3)
        assert host["context_states"].dtype == np.int64 and host["context_actions"].dtype == np.float64
        assert host["context_next_states"].dtype == np.int64 and host["context_rewards"].dtype == np.float64
        assert host["context_rewards"].shape == (N, H) and host["context_states"].shape == (N, H, 1)
        assert np.array_equal(host["context_actions"], dev["context_actions"].cpu().numpy().astype(np.float64))
        assert np.array_equal(host["context_rewards"], dev["context_rewards"][:, :, 0].cpu().numpy().astype(np.float64))
        assert np.all(host["context_states"] == 1) and np.all(host["context_next_states"] == 1)


def test_collect_data_dropin_api(dpt):
    from dpt_b200 import collect_data
    from dpt_b200.envs.bandit_env import BanditEnv
    from dpt_b200.envs.darkroom_env import DarkroomEnv, DarkroomEnvPermuted, DarkroomEnvVec
    dpt.seed(0)
    env = BanditEnv(np.array([0.2, 0.4, 0.6, 0.8, 0.1]), 36, var=0.3)
    xs, us, xps, rs = collect_data.rollin_bandit(env, cov=0.0)
    assert xs.shape == (36, 1) and xs.dtype == np.int64 and us.shape == (36, 5) and us.dtype == np.float64
    assert xps.shape == (36, 1) and rs.shape == (36,) and rs.dtype == np.float64 and np.all(us.sum(1) == 1)
    trajs = collect_data.generate_bandit_histories(50, 5, 20, 0.3, n_hists=2, n_samples=3, cov=0.0, type="uniform")
    assert len(trajs) == 300
    t = trajs[0]
    assert set(t) == {"query_state", "optimal_action", "context_states", "context_actions", "context_next_states",
                      "context_rewards", "means"}
    assert t["context_actions"].shape == (20, 5) and t["context_rewards"].shape == (20,) and t["means"].shape == (5,)
    assert t["optimal_action"].argmax() == t["means"].argmax()
    assert np.array_equal(trajs[0]["context_rewards"], trajs[2]["context_rewards"])       # same history, 3 samples
    assert not np.array_equal(trajs[0]["context_rewards"], trajs[3]["context_rewards"])   # next history
    d = DarkroomEnv(10, [3, 5], 8)
    s, a, ns, r = collect_data.rollin_mdp(d, "uniform")
    assert s.shape == (8, 2) and s.dtype == np.int64 and a.shape == (8, 5) and r.dtype == np.int64
    with pytest.raises(NotImplementedError):
        collect_data.rollin_mdp(d, "bogus")
    d.reset()
    for _ in range(8):
        st, rew, done, _ = d.step(d.opt_action(d.state))
    assert np.array_equal(st, [3, 5]) and rew == 1 and done
    with pytest.raises(ValueError, match="Episode has already ended"):
        d.step(np.eye(5)[4])
    with pytest.raises(AssertionError):
        DarkroomEnvPermuted(10, 120, 8)
    tr = collect_data.generate_darkroom_permuted_histories([0, 5, 119], 10, 12, n_hists=1, n_samples=2, rollin_type="expert")
    assert len(tr) == 6 and tr[2]["perm_index"] == 5 and np.array_equal(tr[0]["goal"], [9, 9])
    vec = DarkroomEnvVec([DarkroomEnv(10, [2, 2], 4), DarkroomEnv(10, [0, 1], 4)])

    class OptCtrl:
        def act(self, obs):
            return [e.opt_action(o) for e, o in zip(vec.envs, obs)]
    obs, acts, nobs, rews = vec.deploy(OptCtrl())
    assert obs.shape == (2, 4, 2) and acts.shape == (2, 4, 5) and rews.shape == (2, 4)
    assert np.array_equal(nobs[:, -1], [[2, 2], [0, 1]]) and rews[1].tolist() == [1, 1, 1, 1]


def test_bandit_rollin_fused_peer_gather_single_rank(dpt):
    """dpt_bandit_rollin_p2p with world = 1: the last CTA publishes the launch's three totals into this rank's
    own CUDA-IPC gather buffer; outputs equal the plain launch, the done-counter resets between launches."""
    from dpt_b200 import dist as D
    N, d, H, var, seed = 20000, 5, 100, 0.3, 8
    means, _, _ = dpt.kernels.bandit_sample_means(N, d, seed, 0)
    ref_stats = torch.zeros(3, dtype=torch.float64, device="cuda")
    ref = dpt.kernels.bandit_rollin(means, H, var, seed, 0, stats=ref_stats)
    pg = D.PeerGather(slots=3)
    try:
        for slot in (0, 2, 1):                                  # three launches: the counter must re-arm itself
            st = torch.zeros(3, dtype=torch.float64, device="cuda")
            out = dpt.kernels.bandit_rollin(means, H, var, seed, 0, stats=st, peer=pg, peer_slot=slot)
            for k in ref:
                assert torch.equal(ref[k], out[k])
            assert torch.equal(st, ref_stats)
        got = pg.read()
        assert got.shape == (3, 1, 3)
        for slot in range(3):
            assert np.array_equal(got[slot, 0], _np(ref_stats))
        batch, stats = D.collect_bandit_sharded(N, d, H, var, seed, peer=pg, peer_slot=0)
        assert abs(stats["mean_reward"] - float(ref_stats[0]) / (N * H)) < 1e-12 and stats["env_steps"] == N * H
    finally:
        pg.close()


@pytest.mark.parametrize("N,d,H", [(64, 5, 500), (9, 10, 61), (40, 3, 37)])
def test_bandit_rollin_bernoulli(dpt, N, d, H):
    """type == 'bernoulli' envs (envs/bandit_env.py:60-61): rewards are Bernoulli(means[a]).  Same action stream
    as the uniform type; rewards exactly [u < mean] on the dumped uniforms (fast and generic kernels), {0,1}
    valued, and their frequency matches the pulled arms' means."""
    seed, env_id0 = 99, 50
    means, _, _ = dpt.kernels.bandit_sample_means(N, d, seed, env_id0)
    m64 = _np(means).astype(np.float64)
    g = dpt.kernels.bandit_rollin(means, H, 0.3, seed, env_id0)
    b = dpt.kernels.bandit_rollin(means, H, 0.3, seed, env_id0, dump=True, reward_type="bernoulli")
    assert torch.equal(g["context_actions"], b["context_actions"]) and torch.equal(g["context_states"], b["context_states"])
    nz = {k: _np(v) for k, v in b["noise"].items()}
    assert nz["z"].min() >= 0.0 and nz["z"].max() < 1.0
    xs, us, xps, rs, acts = O.rollin_bandit_batch(m64, 0.3, nz["cov_idx"], nz["dir_probs"], nz["rand_idx"], nz["u"], nz["z"],
                                                  reward_type="bernoulli")
    r = _np(b["context_rewards"])[:, :, 0]
    assert np.array_equal(r.astype(np.float64), rs) and set(np.unique(r)) <= {0.0, 1.0}
    b2 = dpt.kernels.bandit_rollin(means, H, 0.3, seed, env_id0, reward_type="bernoulli")
    assert torch.equal(b["context_rewards"], b2["context_rewards"])
    # injected uniforms reproduce the rewards
    b3 = dpt.kernels.bandit_rollin(means, H, 0.3, 0, 0, inject={"actions": nz["actions"], "z": nz["z"]}, reward_type="bernoulli")
    assert torch.equal(b["context_rewards"], b3["context_rewards"])
    pm = np.take_along_axis(m64, acts, axis=1)
    se = np.sqrt((pm * (1 - pm)).sum()) / pm.size
    assert abs(r.mean() - pm.mean()) < 5 * se + 1e-9
    with pytest.raises(KeyError):
        dpt.kernels.bandit_rollin(means, H, 0.3, seed, env_id0, reward_type="poisson")


def test_rollin_bandit_follows_env_type(dpt):
    """rollin_bandit / generate_bandit_histories_from_envs take the reward law from env.type (env.transit,
    collect_data.py:45); generate_bandit_histories ignores its `type` kwarg like the reference (:221-225)."""
    from dpt_b200 import collect_data
    from dpt_b200.envs.bandit_env import BanditEnv, sample
    dpt.seed(5)
    env = BanditEnv(np.array([0.2, 0.9, 0.5]), 64, var=0.3, type="bernoulli")
    xs, us, xps, rs = collect_data.rollin_bandit(env, cov=0.0)
    assert rs.shape == (64,) and set(np.unique(rs)) <= {0.0, 1.0} and us.shape == (64, 3)
    envs = [sample(4, 32, 0.3, type="bernoulli") for _ in range(6)]
    trajs = collect_data.generate_bandit_histories_from_envs(envs, n_hists=2, n_samples=1, cov=0.0, type="bernoulli")
    assert len(trajs) == 12 and all(set(np.unique(t["context_rewards"])) <= {0.0, 1.0} for t in trajs)
    trajs = collect_data.generate_bandit_histories(5, 4, 16, 0.3, n_hists=1, n_samples=1, cov=0.0, type="bernoulli")
    assert len(trajs) == 5 and any(len(np.unique(t["context_rewards"])) > 2 for t in trajs)   # gaussian rewards
    with pytest.raises(NotImplementedError):
        collect_data.generate_bandit_histories_from_envs([envs[0], BanditEnv(np.ones(4) * .5, 32, var=0.3)], 1, 1, 0.0, "uniform")


def test_entry_points_are_graph_capturable(dpt):
    """Threads / streams contract (SURVEY §8b): every launch goes to the caller's stream with no hidden synchronisation,
    so the entry points can be captured into a CUDA graph and replayed (one graph = a whole multi-launch rollout)."""
    N, d, H = 4096, 5, 64
    means, _, opt_a = dpt.kernels.bandit_sample_means(N, d, 3, 0)
    ref = dpt.kernels.bandit_rollin(means, H, 0.3, 11, 0)
    out = {k: torch.zeros_like(v) for k, v in ref.items()}
    r = torch.zeros(N, device="cuda")
    acts = torch.eye(d, device="cuda")[torch.arange(N, device="cuda") % d].contiguous()
    r_ref = torch.empty(N, device="cuda")
    dpt.kernels.gpu_bandit_step(means, acts, 0.3, 0, 5, 0, 7, out=r_ref)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        dpt.kernels.bandit_rollin(means, H, 0.3, 11, 0, out=out)       # warm-up outside capture (occupancy queries)
        dpt.kernels.gpu_bandit_step(means, acts, 0.3, 0, 5, 0, 7, out=r)
        ol_ref = dpt.kernels.online_loop("ucb", means, H, 0.3, 5, 0, p0=1.0)   # split pipeline: 4 launches + stream-ordered scratch
    torch.cuda.current_stream().wait_stream(s)
    for v in out.values():
        v.zero_()
    r.zero_()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        dpt.kernels.bandit_rollin(means, H, 0.3, 11, 0, out=out)
        dpt.kernels.gpu_bandit_step(means, acts, 0.3, 0, 5, 0, 7, out=r)
        ol = dpt.kernels.online_loop("ucb", means, H, 0.3, 5, 0, p0=1.0)
    assert float(out["context_actions"].abs().sum()) == 0.0            # captured, not executed
    g.replay()
    torch.cuda.synchronize()
    for k in ref:
        assert torch.equal(out[k], ref[k]), k
    assert torch.equal(r, r_ref)
    for k in ("context_actions", "context_rewards", "context_states", "cum_means"):
        assert torch.equal(ol[k], ol_ref[k]), k
    assert torch.allclose(ol["regret_sums"], ol_ref["regret_sums"], rtol=1e-12)


def test_build_datasets_files(dpt, tmp_path):
    """collect_data.py:352-485 as a function: three pickles with the reference's file names, trajectory keys and splits,
    loadable by the reference-shaped Dataset (dataset.py:11-91)."""
    import pickle
    from dpt_b200 import collect_data
    from dpt_b200.dataset import Dataset
    dpt.seed(0)
    paths = collect_data.build_datasets("bandit", 10, 3, 1, 2, 12, 5, var=0.3, cov=0.0, out_dir=str(tmp_path))
    assert [p.split("datasets/")[1] for p in paths] == ["trajs_bandit_envs10_hists1_samples2_H12_d5_var0.3_cov0.0_train.pkl",
                                                        "trajs_bandit_envs10_hists1_samples2_H12_d5_var0.3_cov0.0_test.pkl",
                                                        "trajs_bandit_envs3_H12_d5_var0.3_cov0.0_eval.pkl"]
    train, test, ev = (pickle.load(open(p, "rb")) for p in paths)
    assert (len(train), len(test), len(ev)) == (8 * 2, 2 * 2, 3 * 2)
    assert set(train[0]) == {"query_state", "optimal_action", "context_states", "context_actions", "context_next_states",
                             "context_rewards", "means"}
    assert train[0]["context_actions"].shape == (12, 5) and train[0]["context_rewards"].shape == (12,)
    ds = Dataset(paths[0], {"horizon": 12, "state_dim": 1, "action_dim": 5, "shuffle": False, "store_gpu": False})
    assert len(ds) == 16 and ds[0]["context_rewards"].shape == (12, 1)
    paths = collect_data.build_datasets("darkroom_heldout", 200, 100, 1, 1, 10, 10, out_dir=str(tmp_path))
    train, test, ev = (pickle.load(open(p, "rb")) for p in paths)
    assert (len(train), len(test), len(ev)) == (160, 40, 100) and paths[2].endswith("trajs_darkroom_heldout_envs100_H10_d10_uniform_eval.pkl")
    goals = np.array([[(j, i) for i in range(10)] for j in range(10)]).reshape(-1, 2)
    np.random.RandomState(seed=0).shuffle(goals)
    assert np.array_equal(np.stack([t["goal"] for t in train]), np.repeat(goals[:80], 2, axis=0))
    assert np.array_equal(np.stack([t["goal"] for t in ev]), np.array(goals[80:].tolist() * 5))
    assert set(train[0]) == {"query_state", "optimal_action", "context_states", "context_actions", "context_next_states",
                             "context_rewards", "goal"}
    paths = collect_data.build_datasets("linear_bandit", 10, 2, 1, 1, 8, 6, var=0.3, cov=0.0, lin_d=2, out_dir=str(tmp_path))
    train = pickle.load(open(paths[0], "rb"))
    assert len(train) == 8 and {"arms", "theta", "var"} <= set(train[0]) and paths[0].endswith("_H8_d6_lind2_var0.3_cov0.0_train.pkl")
    with pytest.raises(NotImplementedError):
        collect_data.build_datasets("miniworld", 10, 2, 1, 1, 8, 6, out_dir=str(tmp_path))


def test_bench_own_arm_contract(dpt):
    """`bench.py` (the arm the driver runs on the GPU box) prints ONE JSON line with the contract's keys."""
    import json
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--gpus", "1", "--steps", "3", "--warmup", "1",
                          "--no-cpu-baseline", "--no-other"], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    r = json.loads(lines[0])
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
              "dtype", "data", "config", "roofline", "e2e", "gpu_launches", "clocks"):
        assert k in r, k
    assert r["n_gpus"] == 1 and r["steps"] == 3 and r["warmup"] >= 3 and r["gpu_launches"] == 3 and r["scaling"] == "weak"
    assert r["unit"] == "env-steps/s" and r["value"] > 1e10 and "workload" in r["config"]
    rf = r["roofline"]
    assert rf["bound"] == "hbm" and rf["unit"] == "GB/s" and abs(rf["frac"] - rf["achieved"] / rf["peak"]) < 1e-9
    e = r["e2e"]
    assert e["unit"] == r["unit"] and 0 < e["value"] < r["value"] and e["h2d_bytes_per_step"] > 0 and e["d2h_bytes_per_step"] > 0
    assert {"sm_mhz", "sm_max_mhz", "reasons"} <= set(r["clocks"])


def test_bench_dump_outputs(dpt, tmp_path):
    """`bench.py --dump-outputs DIR` writes the last timed step's outputs: the sampled envs equal a direct bandit_rollin at
    that step's seed (warm-up + --steps - 1), float32 / float64 only, 64 MB at most."""
    import os
    import subprocess
    import sys
    import bench
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    warmup, steps = 3, 2
    out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--gpus", "1", "--steps", str(steps), "--warmup", str(warmup),
                          "--no-cpu-baseline", "--no-other", "--no-online-eval", "--dump-outputs", str(tmp_path)],
                         capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    files = sorted(os.listdir(tmp_path))
    assert files == ["context_actions.npy", "context_next_states.npy", "context_rewards.npy", "context_states.npy", "return_stats.npy"]
    got = {f[:-4]: np.load(tmp_path / f) for f in files}
    assert all(a.dtype in (np.float32, np.float64) for a in got.values())
    assert sum(a.nbytes for a in got.values()) <= 64 << 20
    N = bench.ENVS_PER_GPU
    idx = np.sort(np.random.RandomState(0).choice(N, min(N, bench.DUMP_ENVS), replace=False))
    means, _, _ = dpt.kernels.bandit_sample_means(N, bench.DIM, 0, 0)
    stats = torch.zeros(3, dtype=torch.float64, device="cuda")
    want = dpt.kernels.bandit_rollin(means, bench.H, bench.VAR, warmup + steps - 1, 0, stats=stats)
    rows = torch.as_tensor(idx, device="cuda")
    for k, t in want.items():
        assert np.array_equal(got[k], _np(t.index_select(0, rows))), k
    assert np.allclose(got["return_stats"], _np(stats), rtol=1e-9)
