"""Tensor-level wrappers of the C ABI (one function per entry point of include/dpt_b200.h).

These allocate outputs with torch (the caller owns all device memory), pass raw pointers and the
current CUDA stream, and map error codes to exceptions.  No computation happens in Python and
nothing here falls back to the CPU.
"""
import ctypes

import torch

from . import _lib
from ._lib import check, lib, ptr, stream_ptr

I32, F32, F64 = torch.int32, torch.float32, torch.float64


def _dev(device=None):
    d = _lib.require_cuda()
    return torch.device(device) if device is not None else d


def _as(t, dtype, device):
    """Tensor / array-like -> contiguous device tensor of ``dtype``."""
    if not torch.is_tensor(t):
        t = torch.as_tensor(t)
    return t.to(device=device, dtype=dtype).contiguous()


def device_info():
    sm, ma, mi = ctypes.c_int(), ctypes.c_int(), ctypes.c_int()
    check(lib().dpt_device_info(ctypes.byref(sm), ctypes.byref(ma), ctypes.byref(mi)), "dpt_device_info")
    return sm.value, ma.value, mi.value


# ------------------------------------------------------------------ bandit task ----------------
def bandit_sample_means(n_envs, dim, seed, env_id0=0, device=None):
    """means ~ U[0,1)^dim, optimal arm index and one-hot (envs/bandit_env.py:10-18, :29-34)."""
    dev = _dev(device)
    means = torch.empty((n_envs, dim), dtype=F32, device=dev)
    opt_idx = torch.empty((n_envs,), dtype=I32, device=dev)
    opt_a = torch.empty((n_envs, dim), dtype=F32, device=dev)
    check(lib().dpt_bandit_sample_means(seed, env_id0, n_envs, dim, ptr(means), ptr(opt_idx), ptr(opt_a), stream_ptr()),
          "dpt_bandit_sample_means")
    return means, opt_idx, opt_a


def bandit_opt_action(means):
    means = _as(means, F32, _dev(means.device if torch.is_tensor(means) and means.is_cuda else None))
    n, d = means.shape
    opt_idx = torch.empty((n,), dtype=I32, device=means.device)
    opt_a = torch.empty((n, d), dtype=F32, device=means.device)
    check(lib().dpt_bandit_opt_action(ptr(means), n, d, ptr(opt_idx), ptr(opt_a), stream_ptr()), "dpt_bandit_opt_action")
    return opt_idx, opt_a


# ------------------------------------------------------------------ rollin_bandit --------------
REWARD_TYPES = {"uniform": 0, "bernoulli": 1}   # envs/bandit_env.py:10-16 type names -> DPT_REWARD_*


def bandit_rollin(means, H, var, seed, env_id0=0, inject=None, dump=False, out=None, stats=None, peer=None, peer_slot=0,
                  reward_type="uniform"):
    """Fused rollin_bandit for all envs (collect_data.py:23-53).  ``means`` [N,d] fp32 device tensor.

    inject: dict with 'z' [N,H] and either 'actions' [N,H] or ('cov_idx' [N], 'dir_probs' [N,d] f64,
    'rand_idx' [N], 'u' [N,H] f64).  dump=True additionally returns the noise that was used.
    stats: optional f64 [3] device tensor, += (sum r, sum r^2, #optimal-arm pulls).
    reward_type: 'uniform' (r = mean + var z) or 'bernoulli' (r = [u < mean]; the 'z' noise arrays then hold u).
    peer: optional dist.PeerGather -- the launch then also stores this rank's three totals into slot
    ``peer_slot`` of every rank's gather buffer over NVLink (``stats`` must be zero before the launch).
    Returns dict: context_states [N,H,1], context_actions [N,H,d], context_next_states [N,H,1],
    context_rewards [N,H,1] (fp32, device) [+ 'noise' dict]."""
    dev = _dev(means.device if torch.is_tensor(means) and means.is_cuda else None)
    means = _as(means, F32, dev)
    N, d = means.shape
    if out is None:
        out = {
            "context_states": torch.empty((N, H, 1), dtype=F32, device=dev),
            "context_actions": torch.empty((N, H, d), dtype=F32, device=dev),
            "context_next_states": torch.empty((N, H, 1), dtype=F32, device=dev),
            "context_rewards": torch.empty((N, H, 1), dtype=F32, device=dev),
        }
    inj_p, dump_p, keep = None, None, []
    if inject is not None:
        s = _lib.BanditInject()
        spec = {"cov_idx": I32, "dir_probs": F64, "rand_idx": I32, "u": F64, "actions": I32, "z": F32}
        for k, dt in spec.items():
            if inject.get(k) is not None:
                t = _as(inject[k], dt, dev)
                keep.append(t)
                setattr(s, k, ptr(t))
        inj_p = ctypes.byref(s)
    noise = None
    if dump:
        noise = {"cov_idx": torch.empty((N,), dtype=I32, device=dev), "dir_probs": torch.empty((N, d), dtype=F64, device=dev),
                 "rand_idx": torch.empty((N,), dtype=I32, device=dev), "u": torch.empty((N, H), dtype=F64, device=dev),
                 "actions": torch.empty((N, H), dtype=I32, device=dev), "z": torch.empty((N, H), dtype=F32, device=dev)}
        s2 = _lib.BanditDump()
        for k, t in noise.items():
            setattr(s2, k, ptr(t))
        dump_p = ctypes.byref(s2)
    if peer is not None:
        assert inject is None and not dump and stats is not None and reward_type == "uniform"
        check(lib().dpt_bandit_rollin_p2p(ptr(means), var, seed, env_id0, N, H, d, ptr(out["context_states"]),
                                          ptr(out["context_actions"]), ptr(out["context_next_states"]),
                                          ptr(out["context_rewards"]), ptr(stats), peer.dst_array(peer_slot), peer.world,
                                          peer.counter_ptr, stream_ptr()), "dpt_bandit_rollin_p2p")
        return out
    check(lib().dpt_bandit_rollin(ptr(means), var, REWARD_TYPES[reward_type], seed, env_id0, N, H, d, ptr(out["context_states"]),
                                  ptr(out["context_actions"]), ptr(out["context_next_states"]),
                                  ptr(out["context_rewards"]), ptr(stats), inj_p, dump_p, stream_ptr()), "dpt_bandit_rollin")
    if noise is not None:
        out = dict(out, noise=noise)
    return out


def bandit_rollin_host(means_host, H, var, seed, env_id0=0, out=None, scratch=None):
    """Host-buffer form (e2e path): ``means_host`` [N,d] fp32 CPU tensor (pinned for full speed);
    returns the four context arrays as pinned CPU tensors.  H2D / kernel / D2H are pipelined."""
    dev = _dev()
    means_host = means_host.contiguous()
    assert means_host.dtype == F32 and not means_host.is_cuda
    N, d = means_host.shape
    if out is None:
        pin = dict(dtype=F32, pin_memory=True)
        out = {"context_states": torch.empty((N, H, 1), **pin), "context_actions": torch.empty((N, H, d), **pin),
               "context_next_states": torch.empty((N, H, 1), **pin), "context_rewards": torch.empty((N, H, 1), **pin)}
    nbytes = lib().dpt_bandit_rollin_host_scratch_bytes(N, H, d)
    if scratch is None or scratch.numel() < nbytes:
        scratch = torch.empty((max(nbytes, 1),), dtype=torch.uint8, device=dev)
    check(lib().dpt_bandit_rollin_host(ptr(means_host), var, seed, env_id0, N, H, d, ptr(out["context_states"]),
                                       ptr(out["context_actions"]), ptr(out["context_next_states"]),
                                       ptr(out["context_rewards"]), ptr(scratch), scratch.numel(), stream_ptr()),
          "dpt_bandit_rollin_host")
    return out, scratch


def bandit_rollin_host_ref(means_host, H, var, seed, env_id0=0, scratch=None):
    """The collection in the REFERENCE's host dtypes (collect_data.py:23-53): returns numpy arrays context_states
    [N,H,1] int64, context_actions [N,H,d] float64, context_next_states [N,H,1] int64, context_rewards [N,H] float64.
    Only arm index + fp32 reward cross PCIe; host threads expand them (dpt_bandit_rollin_host_f64)."""
    import numpy as np
    dev = _dev()
    means_host = means_host.contiguous()
    assert means_host.dtype == F32 and not means_host.is_cuda
    N, d = means_host.shape
    out = {"context_states": np.empty((N, H, 1), dtype=np.int64), "context_actions": np.empty((N, H, d), dtype=np.float64),
           "context_next_states": np.empty((N, H, 1), dtype=np.int64), "context_rewards": np.empty((N, H), dtype=np.float64)}
    nbytes = lib().dpt_bandit_rollin_host_scratch_bytes(N, H, d)
    if scratch is None or scratch.numel() < nbytes:
        scratch = torch.empty((max(nbytes, 1),), dtype=torch.uint8, device=dev)
    check(lib().dpt_bandit_rollin_host_f64(ptr(means_host), var, seed, env_id0, N, H, d, out["context_states"].ctypes.data,
                                           out["context_actions"].ctypes.data, out["context_next_states"].ctypes.data,
                                           out["context_rewards"].ctypes.data, ptr(scratch), scratch.numel(), stream_ptr()),
          "dpt_bandit_rollin_host_f64")
    return out


def host_write_peak(buf=None, nbytes=1 << 30, n_threads=0):
    """GB/s the host cores reach with non-temporal stores (dpt_host_write_peak): into ``buf`` (a CPU tensor, e.g. the
    pinned output arrays of the e2e path) or an internal buffer.  Needs no GPU."""
    if buf is not None:
        nbytes = buf.numel() * buf.element_size()
    v = lib().dpt_host_write_peak(ptr(buf), int(nbytes), int(n_threads))
    if not v > 0.0:
        raise _lib.DptError("dpt_host_write_peak failed")
    return float(v)


# ------------------------------------------------------------------ darkroom -------------------
def darkroom_rollin(goals, dim, H, mode, seed, env_id0=0, perm_index=None, n_samples=1, inject=None, dump=False):
    """Fused rollin_mdp (collect_data.py:83-111, :200-201).  goals [N,2] int; mode 'uniform'|'expert'.
    Returns dict with context_* fp32 [N,H,.], query_states [N,S,2], optimal_actions [N,S,5]."""
    if mode not in ("uniform", "expert"):
        raise NotImplementedError(mode)   # collect_data.py:97
    dev = _dev(goals.device if torch.is_tensor(goals) and goals.is_cuda else None)
    goals = _as(goals, I32, dev)
    N = goals.shape[0]
    perm = None if perm_index is None else _as(perm_index, I32, dev)
    if perm is not None and N and int(perm.max()) >= 120:
        raise AssertionError("perm_index < 120")  # envs/darkroom_env.py:95
    out = {
        "context_states": torch.empty((N, H, 2), dtype=F32, device=dev),
        "context_actions": torch.empty((N, H, 5), dtype=F32, device=dev),
        "context_next_states": torch.empty((N, H, 2), dtype=F32, device=dev),
        "context_rewards": torch.empty((N, H, 1), dtype=F32, device=dev),
        "query_states": torch.empty((N, n_samples, 2), dtype=F32, device=dev),
        "optimal_actions": torch.empty((N, n_samples, 5), dtype=F32, device=dev),
    }
    inj_p, dump_p, keep = None, None, []
    if inject is not None:
        s = _lib.DarkroomInject()
        for k in ("states", "actions", "query"):
            if inject.get(k) is not None:
                t = _as(inject[k], I32, dev)
                keep.append(t)
                setattr(s, k, ptr(t))
        inj_p = ctypes.byref(s)
    noise = None
    if dump:
        noise = {"states": torch.empty((N, H, 2), dtype=I32, device=dev), "actions": torch.empty((N, H), dtype=I32, device=dev),
                 "query": torch.empty((N, n_samples, 2), dtype=I32, device=dev)}
        s2 = _lib.DarkroomDump()
        for k, t in noise.items():
            setattr(s2, k, ptr(t))
        dump_p = ctypes.byref(s2)
    check(lib().dpt_darkroom_rollin(ptr(goals), ptr(perm), dim, 0 if mode == "uniform" else 1, seed, env_id0, N, H,
                                    n_samples, ptr(out["context_states"]), ptr(out["context_actions"]),
                                    ptr(out["context_next_states"]), ptr(out["context_rewards"]),
                                    ptr(out["query_states"]), ptr(out["optimal_actions"]), inj_p, dump_p, stream_ptr()),
          "dpt_darkroom_rollin")
    if noise is not None:
        out["noise"] = noise
    return out


def darkroom_step(states, actions, goals, dim, perm_index=None):
    """Batched DarkroomEnv.transit (envs/darkroom_env.py:37-55): int32 [N,2], fp32 one-hot [N,5]."""
    dev = _dev()
    states, actions, goals = _as(states, I32, dev), _as(actions, F32, dev), _as(goals, I32, dev)
    perm = None if perm_index is None else _as(perm_index, I32, dev)
    N = states.shape[0]
    ns = torch.empty((N, 2), dtype=I32, device=dev)
    r = torch.empty((N,), dtype=I32, device=dev)
    check(lib().dpt_darkroom_step(ptr(states), ptr(actions), ptr(goals), ptr(perm), dim, N, ptr(ns), ptr(r), stream_ptr()),
          "dpt_darkroom_step")
    return ns, r


def darkroom_opt_action(states, goals, perm_index=None):
    dev = _dev()
    states, goals = _as(states, I32, dev), _as(goals, I32, dev)
    perm = None if perm_index is None else _as(perm_index, I32, dev)
    N = states.shape[0]
    a = torch.empty((N, 5), dtype=F32, device=dev)
    check(lib().dpt_darkroom_opt_action(ptr(states), ptr(goals), ptr(perm), N, ptr(a), stream_ptr()), "dpt_darkroom_opt_action")
    return a


# ------------------------------------------------------------------ GPUBanditEnv.step ----------
def gpu_bandit_step(means, actions, var, type_id, seed, env_id0, step, inject=None, dump=False, out=None):
    """envs/gpu_bandit_env.py:53-63 in one launch.  Returns reward [N] (and the noise if dump)."""
    N, d = means.shape
    dev = means.device
    actions = _as(actions, F32, dev)
    reward = out if out is not None else torch.empty((N,), dtype=F32, device=dev)
    inj = None if inject is None else _as(inject, F32, dev)
    dmp = torch.empty((N,), dtype=F32, device=dev) if dump else None
    check(lib().dpt_gpu_bandit_step(ptr(means), ptr(actions), var, type_id, seed, env_id0, step, N, d, ptr(reward),
                                    ptr(inj), ptr(dmp), stream_ptr()), "dpt_gpu_bandit_step")
    return (reward, dmp) if dump else reward


# ------------------------------------------------------------------ controllers ----------------
CTRL_KINDS = {"opt": 0, "emp": 1, "ucb": 2, "thompson": 3, "linucb": 4}


def arm_stats(ctx_actions, ctx_rewards, h=None):
    """Per-(env, arm) reward sums (f64) and pull counts (int32) of the first ``h`` context steps
    (ctrls/ctrl_bandit.py:95-104).  ctx_actions [N,Hs,d], ctx_rewards [N,Hs,1] or [N,Hs] fp32 device."""
    dev = _dev(ctx_actions.device if torch.is_tensor(ctx_actions) and ctx_actions.is_cuda else None)
    ctx_actions, ctx_rewards = _as(ctx_actions, F32, dev), _as(ctx_rewards, F32, dev)
    N, Hs, d = ctx_actions.shape
    h = Hs if h is None else h
    sums = torch.empty((N, d), dtype=F64, device=dev)
    counts = torch.empty((N, d), dtype=I32, device=dev)
    check(lib().dpt_arm_stats(ptr(ctx_actions), ptr(ctx_rewards), N, h, Hs, d, ptr(sums), ptr(counts), stream_ptr()),
          "dpt_arm_stats")
    return sums, counts


def online_loop(kind, means, H, var, seed, env_id0=0, p0=0.0, p1=0.0, p2=0.0, arms=None, materialise=True,
                regret=True, inject=None, dump=False, reward_type="uniform"):
    """Fused deploy_online_vec for a classical controller (evals/eval_bandit.py:56-103).

    Returns dict: cum_means [H,N] fp32, regret_sums [H,4] f64 (sums over envs of reg, reg^2, cumreg, cumreg^2 with
    reg = max(means) - cum_means), and, if materialise, context_* [N,H,.] fp32 [+ 'noise' if dump]."""
    dev = _dev(means.device if torch.is_tensor(means) and means.is_cuda else None)
    means = _as(means, F32, dev)
    N, d = means.shape
    out = {"cum_means": torch.empty((H, N), dtype=F32, device=dev)}
    if regret:
        out["regret_sums"] = torch.zeros((H, 4), dtype=F64, device=dev)
    if materialise:
        out.update(context_states=torch.empty((N, H, 1), dtype=F32, device=dev),
                   context_actions=torch.empty((N, H, d), dtype=F32, device=dev),
                   context_next_states=torch.empty((N, H, 1), dtype=F32, device=dev),
                   context_rewards=torch.empty((N, H, 1), dtype=F32, device=dev))
    arms_t, lin_d = None, 0
    if arms is not None:
        arms_t = _as(arms, F64, dev)
        lin_d = arms_t.shape[1]
    inj_p, dump_p, keep = None, None, []
    if inject is not None:
        s = _lib.OnlineInject()
        for k, dt in (("reward_z", F32), ("ctrl_z", F32), ("first_arm", I32)):
            if inject.get(k) is not None:
                t = _as(inject[k], dt, dev)
                keep.append(t)
                setattr(s, k, ptr(t))
        inj_p = ctypes.byref(s)
    noise = None
    if dump:
        noise = {"reward_z": torch.empty((H, N), dtype=F32, device=dev)}
        if kind == "thompson":
            noise["ctrl_z"] = torch.empty((H, N, d), dtype=F32, device=dev)
        if kind == "linucb":
            noise["first_arm"] = torch.empty((N,), dtype=I32, device=dev)
        s2 = _lib.OnlineDump()
        for k, t in noise.items():
            setattr(s2, k, ptr(t))
        dump_p = ctypes.byref(s2)
    check(lib().dpt_online_loop(CTRL_KINDS[kind], p0, p1, p2, ptr(means), ptr(arms_t), lin_d, float(var), REWARD_TYPES[reward_type], seed,
                                env_id0,
                                N, H, d, ptr(out.get("context_states")), ptr(out.get("context_actions")),
                                ptr(out.get("context_next_states")), ptr(out.get("context_rewards")),
                                ptr(out["cum_means"]), ptr(out.get("regret_sums")), inj_p, dump_p, stream_ptr()),
          "dpt_online_loop")
    if noise is not None:
        out["noise"] = noise
    return out


def darkroom_policy_rollout(logits, goals, dim, horizon, sample, seed, env_id0=0, episode=0, perm_index=None,
                            inject_u=None, dump=False):
    """One darkroom episode per env from a logits table [N, dim*dim, 5] (see dpt_darkroom_policy_rollout).
    Returns dict: context rows of the episode [N,horizon,.] fp32, returns [N] [, u [horizon,N] f64]."""
    dev = _dev(logits.device)
    logits = _as(logits, F32, dev)
    goals = _as(goals, I32, dev)
    perm = None if perm_index is None else _as(perm_index, I32, dev)
    N = goals.shape[0]
    out = {"states": torch.empty((N, horizon, 2), dtype=F32, device=dev), "actions": torch.empty((N, horizon, 5), dtype=F32, device=dev),
           "next_states": torch.empty((N, horizon, 2), dtype=F32, device=dev), "rewards": torch.empty((N, horizon, 1), dtype=F32, device=dev),
           "returns": torch.empty((N,), dtype=F32, device=dev)}
    inj = None if inject_u is None else _as(inject_u, F64, dev)
    if dump:
        out["u"] = torch.zeros((horizon, N), dtype=F64, device=dev)
    check(lib().dpt_darkroom_policy_rollout(ptr(logits), ptr(goals), ptr(perm), dim, horizon, 1 if sample else 0, seed, env_id0,
                                            episode, N, ptr(out["states"]), ptr(out["actions"]), ptr(out["next_states"]),
                                            ptr(out["rewards"]), ptr(out["returns"]), ptr(inj), ptr(out.get("u")), stream_ptr()),
          "dpt_darkroom_policy_rollout")
    return out


# ------------------------------------------------------------------ offline evaluation ---------
OFFLINE_SLOTS = ("opt", "emp", "lcb", "thmp", "linreg", "lnr")   # slot order of dpt_offline_eval (DPT_OFFLINE_*)


def _rows(t, N, d):
    """(tensor, row stride in steps) of a [N, T, d] context tensor or a [:, :T] view of one, without a copy when the
    rows are laid out as [N, H_stride, d]."""
    if t.dim() == 2:
        t = t.unsqueeze(-1)
    if t.stride(-1) == 1 and t.stride(1) == d and t.stride(0) % d == 0 and t.stride(0) // d >= t.shape[1]:
        return t, t.stride(0) // d
    t = t.contiguous()
    return t, t.shape[1]


def offline_eval(means, ctx_actions, ctx_rewards, horizons, ctrls=("opt", "emp", "lcb", "thmp"), lcb_const=0.8,
                 thmp_std=0.3, thmp_prior_mean=0.5, thmp_prior_var=1 / 12.0, n_draws=100, arms=None, linreg_const=0.0,
                 learner_logits=None, seed=0, env_id0=0, per_env=True, inject=None, dump=False, sums=None):
    """Offline evaluation of every horizon in ``horizons`` in one launch (dpt_offline_eval).

    means [N,d], ctx_actions [N,H,d] one-hot and ctx_rewards [N,H(,1)] fp32 device tensors (views ``[:, :h]`` of a
    larger buffer pass without a copy); horizons: ints in [1, H], any order, duplicates allowed.  ``ctrls`` picks slots
    of OFFLINE_SLOTS: 'linreg' needs ``arms`` [d, lin_d], 'lnr' needs ``learner_logits`` [N, T >= max(horizons), d]
    (the test=False forward).  inject: {'z': f64 [K, n_draws, N, d]} Thompson normals; dump=True returns them as
    out['noise']['z'].  ``sums`` may be a caller's f64 [K, 6, 2] tensor to accumulate into (shards).
    Returns dict: sums [K, 6, 2] f64 (sum over envs of max mean - reward and its square; unselected slots stay 0),
    rewards [K, 6, N] f64 when per_env (unselected slots 0)."""
    import numpy as np
    dev = _dev(means.device if torch.is_tensor(means) and means.is_cuda else None)
    means = _as(means, F32, dev)
    N, d = means.shape
    hz = np.ascontiguousarray(np.asarray(horizons, dtype=np.int64).reshape(-1)).astype(np.int32)
    K = hz.shape[0]
    unknown = set(ctrls) - set(OFFLINE_SLOTS)
    if unknown:
        raise ValueError("offline_eval: unknown controllers %s (slots: %s)" % (sorted(unknown), OFFLINE_SLOTS))
    mask = sum(1 << OFFLINE_SLOTS.index(c) for c in ctrls)
    ca, cr, hs = None, None, 1
    if ctx_actions is not None:
        ca = ctx_actions if torch.is_tensor(ctx_actions) and ctx_actions.device == dev and ctx_actions.dtype == F32 else _as(ctx_actions, F32, dev)
        cr = ctx_rewards if torch.is_tensor(ctx_rewards) and ctx_rewards.device == dev and ctx_rewards.dtype == F32 else _as(ctx_rewards, F32, dev)
        if K and int(hz.max()) > ca.shape[1]:
            raise ValueError("offline_eval: horizon %d > context length %d" % (int(hz.max()), ca.shape[1]))
        ca, hs = _rows(ca, N, d)
        cr, hr = _rows(cr, N, 1)
        if hr != hs:
            ca, cr, hs = ca.contiguous(), cr.contiguous(), ca.shape[1]
    elif K:
        hs = int(hz.max())
    out = {"sums": sums if sums is not None else torch.zeros((K, len(OFFLINE_SLOTS), 2), dtype=F64, device=dev)}
    if per_env:
        out["rewards"] = torch.zeros((K, len(OFFLINE_SLOTS), N), dtype=F64, device=dev)
    keep = []
    prm = _lib.OfflineParams()
    prm.N, prm.d, prm.H_stride, prm.K = N, d, hs, K
    prm.horizons_host = hz.ctypes.data
    prm.ctrl_mask = mask
    prm.lcb_const = float(lcb_const)
    prm.thmp_std, prm.thmp_prior_mean, prm.thmp_prior_var = float(thmp_std), float(thmp_prior_mean), float(thmp_prior_var)
    prm.n_draws = int(n_draws)
    if arms is not None:
        arms_t = _as(arms, F64, dev)
        keep.append(arms_t)
        prm.arms, prm.lin_d = arms_t.data_ptr(), arms_t.shape[1]
    prm.linreg_const = float(linreg_const)
    if learner_logits is not None:
        lg = learner_logits.to(device=dev, dtype=F32).contiguous()
        keep.append(lg)
        prm.learner_logits, prm.logits_T = lg.data_ptr(), lg.shape[1]
    prm.seed, prm.env_id0 = int(seed), int(env_id0)
    if inject is not None and inject.get("z") is not None:
        z = _as(inject["z"], F64, dev)
        assert z.shape == (K, int(n_draws), N, d), z.shape
        keep.append(z)
        prm.inject_z = z.data_ptr()
    if dump:
        out["noise"] = {"z": torch.empty((K, int(n_draws), N, d), dtype=F64, device=dev)}
        prm.dump_z = out["noise"]["z"].data_ptr()
    check(lib().dpt_offline_eval(ctypes.byref(prm), ptr(means), ca.data_ptr() if ca is not None else None,
                                 cr.data_ptr() if cr is not None else None, ptr(out["sums"]), ptr(out.get("rewards")),
                                 stream_ptr()), "dpt_offline_eval")
    return out
