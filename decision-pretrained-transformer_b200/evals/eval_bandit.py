"""Online in-context evaluation with the reference's interface (evals/eval_bandit.py).

``deploy_online_vec(vec_env, controller, horizon, include_meta=False)`` keeps its signature and
return values (cum_means [H,N] float64, meta = four [N,H,.] float64 arrays).  When the env is this
package's ``BanditEnvVec`` and the controller exposes ``fused_spec()`` the whole loop -- controller
statistics, arm choice, env step, context rows, expected reward of the chosen arm, per-step regret
sums -- runs in ONE fused launch (dpt_online_loop / dpt_gpt2_online_loop) instead of H Python
iterations over N env objects.  Anything else takes the generic loop below, which is the reference's
loop verbatim in structure and drives ``vec_env.deploy`` one step at a time.
"""
import numpy as np
import torch

from .. import kernels, rng
from ..ctrls.ctrl_bandit import (BanditTransformerController, EmpMeanPolicy, GreedyOptPolicy, OptPolicy,  # noqa: F401
                                 PessMeanPolicy, ThompsonSamplingPolicy, UCBPolicy)
from ..envs.bandit_env import BanditEnv, BanditEnvVec


def _fusable(vec_env, controller):
    if not isinstance(vec_env, BanditEnvVec) or not callable(getattr(controller, "fused_spec", None)):
        return None
    if len({float(e.var) for e in vec_env.envs}) != 1 or len({e.type for e in vec_env.envs}) != 1:
        return None
    return controller.fused_spec()


def deploy_online_vec_device(vec_env, controller, horizon, include_meta=False, regret=True, seed=None, env_id0=0,
                             inject=None, dump=False):
    """Fused loop, results left on the device (dict of torch tensors, see kernels.online_loop)."""
    spec = _fusable(vec_env, controller)
    if spec is None:
        raise NotImplementedError("controller / env pair has no fused path")
    key = rng.next_key() if seed is None else seed
    var, rtype = float(vec_env.envs[0].var), vec_env.envs[0].type
    if spec["kind"] == "transformer":
        return controller.fused_online_loop(vec_env.means, horizon, var, key, env_id0, include_meta, regret, inject, dump,
                                            rtype)
    return kernels.online_loop(spec["kind"], vec_env.means, horizon, var, key, env_id0, spec.get("p0", 0.0),
                               spec.get("p1", 0.0), spec.get("p2", 0.0), spec.get("arms"), include_meta, regret,
                               inject, dump, rtype)


def deploy_online(env, controller, horizon):
    """evals/eval_bandit.py:24-53 (= eval_linear_bandit.py:22-51): the single-env loop with torch context
    tensors; the controller sees the first h rows through ``set_batch``.  Returns cum_means [horizon]."""
    dev = kernels._dev()
    f = lambda a: torch.as_tensor(np.asarray(a), dtype=torch.float32).to(dev)   # noqa: E731
    context_states = torch.zeros((1, horizon, env.dx), device=dev)
    context_actions = torch.zeros((1, horizon, env.du), device=dev)
    context_next_states = torch.zeros((1, horizon, env.dx), device=dev)
    context_rewards = torch.zeros((1, horizon, 1), device=dev)
    cum_means = []
    for h in range(horizon):
        controller.set_batch({"context_states": context_states[:, :h, :], "context_actions": context_actions[:, :h, :],
                              "context_next_states": context_next_states[:, :h, :],
                              "context_rewards": context_rewards[:, :h, :]})
        states_lnr, actions_lnr, next_states_lnr, rewards_lnr = env.deploy(controller)
        context_states[0, h, :] = f(states_lnr[0])
        context_actions[0, h, :] = f(actions_lnr[0])
        context_next_states[0, h, :] = f(next_states_lnr[0])
        context_rewards[0, h, :] = f(rewards_lnr[0])
        cum_means.append(env.get_arm_value(np.asarray(actions_lnr).flatten()))
    return np.array(cum_means)


def deploy_online_vec(vec_env, controller, horizon, include_meta=False):
    """evals/eval_bandit.py:56-103."""
    if _fusable(vec_env, controller) is not None:
        out = deploy_online_vec_device(vec_env, controller, horizon, include_meta, regret=False)
        cum_means = out["cum_means"].cpu().numpy().astype(np.float64)
        if not include_meta:
            return cum_means
        meta = {k: out[k].cpu().numpy().astype(np.float64) for k in
                ("context_states", "context_actions", "context_next_states", "context_rewards")}
        return cum_means, meta

    num_envs = vec_env.num_envs
    context_states = np.zeros((num_envs, horizon, vec_env.dx))
    context_actions = np.zeros((num_envs, horizon, vec_env.du))
    context_next_states = np.zeros((num_envs, horizon, vec_env.dx))
    context_rewards = np.zeros((num_envs, horizon, 1))
    cum_means = []
    for h in range(horizon):
        batch = {"context_states": context_states[:, :h, :], "context_actions": context_actions[:, :h, :],
                 "context_next_states": context_next_states[:, :h, :], "context_rewards": context_rewards[:, :h, :]}
        controller.set_batch_numpy_vec(batch)
        states_lnr, actions_lnr, next_states_lnr, rewards_lnr = vec_env.deploy(controller)
        context_states[:, h, :] = states_lnr
        context_actions[:, h, :] = actions_lnr
        context_next_states[:, h, :] = next_states_lnr
        context_rewards[:, h, :] = rewards_lnr[:, None]
        cum_means.append(vec_env.get_arm_value(actions_lnr))
    cum_means = np.array(cum_means)
    if not include_meta:
        return cum_means
    return cum_means, {"context_states": context_states, "context_actions": context_actions,
                       "context_next_states": context_next_states, "context_rewards": context_rewards}


def regret_stats(all_means):
    """evals/eval_bandit.py:169-178: dict name -> [N,H] expected reward -> per-step and cumulative
    regret mean / standard error (scipy.stats.sem, ddof=1) against all_means['opt']."""
    opt = np.asarray(all_means["opt"])
    n = opt.shape[0]
    out = {}
    for k, v in all_means.items():
        diff = opt - np.asarray(v)
        cr = np.cumsum(diff, axis=1)
        out[k] = {"mean": diff.mean(0), "sem": diff.std(0, ddof=1) / np.sqrt(n),
                  "regret_mean": cr.mean(0), "regret_sem": cr.std(0, ddof=1) / np.sqrt(n)}
    return out


def online(eval_trajs, model, n_eval, horizon, var, bandit_type="uniform"):
    """evals/eval_bandit.py:107-178 without the matplotlib part: runs Opt, the transformer (if a
    model is given), EmpMean(online), UCB(1.0) and Thompson on the same tasks and returns
    (all_means dict of [n_eval,H], regret statistics)."""
    envs = [BanditEnv(eval_trajs[i]["means"], horizon, var=var) for i in range(n_eval)]
    vec_env = BanditEnvVec(envs)
    ctrls = {"opt": OptPolicy(envs, batch_size=len(envs))}
    if model is not None:
        ctrls["Lnr"] = BanditTransformerController(model, sample=True, batch_size=len(envs))
    ctrls["Emp"] = EmpMeanPolicy(envs[0], online=True, batch_size=len(envs))
    ctrls["UCB1.0"] = UCBPolicy(envs[0], const=1.0, batch_size=len(envs))
    ctrls["Thomp"] = ThompsonSamplingPolicy(envs[0], std=var, sample=True, prior_mean=0.5, prior_var=1 / 12.0,
                                            warm_start=False, batch_size=len(envs))
    all_means = {}
    for name, c in ctrls.items():
        cm = deploy_online_vec(vec_env, c, horizon).T
        assert cm.shape[0] == n_eval
        all_means[name] = cm
    return all_means, regret_stats(all_means)


def online_population(eval_trajs, models, n_eval, horizon, var, bandit_type="uniform"):
    """``online`` for a population of same-shape models (seeds, learning rates, saved epochs): Opt, EmpMean(online),
    UCB(1.0) and Thompson run once and their arrays are shared by every member's dict; the transformer loop of all
    members runs in population launches (models.net.online_loop_population) with ONE key for the whole population, so
    every member sees the same tasks and the same noise.  Keys are drawn in ``online``'s order (opt, Lnr, Emp, UCB,
    Thomp): member i's result equals ``online(eval_trajs, models[i], ...)`` started from the same rng state, bit for bit.
    Returns (list of all_means dicts, list of regret statistics), one per member."""
    from ..models.net import online_loop_population
    envs = [BanditEnv(eval_trajs[i]["means"], horizon, var=var) for i in range(n_eval)]
    vec_env = BanditEnvVec(envs)
    models = list(models)
    ctrls = [BanditTransformerController(m, sample=True, batch_size=len(envs)) for m in models]
    if any(_fusable(vec_env, c) is None for c in ctrls):
        raise NotImplementedError("online_population: every member needs the fused transformer loop (state_dim == 1)")
    shared = {"opt": deploy_online_vec(vec_env, OptPolicy(envs, batch_size=len(envs)), horizon).T}
    lnr = online_loop_population(models, vec_env.means, horizon, float(envs[0].var), True, rng.next_key(), 0, materialise=False,
                                 regret=False, reward_type=envs[0].type)
    for name, c in (("Emp", EmpMeanPolicy(envs[0], online=True, batch_size=len(envs))),
                    ("UCB1.0", UCBPolicy(envs[0], const=1.0, batch_size=len(envs))),
                    ("Thomp", ThompsonSamplingPolicy(envs[0], std=var, sample=True, prior_mean=0.5, prior_var=1 / 12.0,
                                                     warm_start=False, batch_size=len(envs)))):
        shared[name] = deploy_online_vec(vec_env, c, horizon).T
    all_means = []
    for out in lnr:
        am = {"opt": shared["opt"], "Lnr": out["cum_means"].cpu().numpy().astype(np.float64).T}
        am.update((k, shared[k]) for k in ("Emp", "UCB1.0", "Thomp"))
        assert am["Lnr"].shape[0] == n_eval
        all_means.append(am)
    return all_means, [regret_stats(am) for am in all_means]


def offline(eval_trajs, model, n_eval, horizon, var, bandit_type="uniform", np_random_compat=False):
    """evals/eval_bandit.py:214-301 without the bar plot: every controller sees the first ``horizon``
    context rows of each eval trajectory and plays ONE noise-free pull (deploy_eval); returns the dict
    of per-env rewards {'opt','lnr','emp','thmp','lcb'} (``lnr`` only when a model is given).  Per-arm
    statistics come from dpt_arm_stats, the transformer decision from dpt_gpt2_forward."""
    num_envs = len(eval_trajs)
    tmp_env = BanditEnv(eval_trajs[0]["means"], horizon, var=var)
    context_states = np.zeros((num_envs, horizon, tmp_env.dx))
    context_actions = np.zeros((num_envs, horizon, tmp_env.du))
    context_next_states = np.zeros((num_envs, horizon, tmp_env.dx))
    context_rewards = np.zeros((num_envs, horizon, 1))
    envs = []
    for i_eval in range(n_eval):
        traj = eval_trajs[i_eval]
        envs.append(BanditEnv(traj["means"], horizon, var=var))
        context_states[i_eval] = traj["context_states"][:horizon]
        context_actions[i_eval] = traj["context_actions"][:horizon]
        context_next_states[i_eval] = traj["context_next_states"][:horizon]
        context_rewards[i_eval] = np.asarray(traj["context_rewards"])[:horizon, None]
    vec_env = BanditEnvVec(envs)
    vec_env.np_random_compat = np_random_compat     # keep np.random aligned with the reference's env draws
    batch = {"context_states": context_states, "context_actions": context_actions,
             "context_next_states": context_next_states, "context_rewards": context_rewards}
    policies = {"opt": OptPolicy(envs, batch_size=num_envs),
                "emp": EmpMeanPolicy(envs[0], online=False, batch_size=num_envs)}
    if model is not None:
        policies["lnr"] = BanditTransformerController(model, sample=False, batch_size=num_envs)
    policies["lcb"] = PessMeanPolicy(envs[0], const=.8, batch_size=len(envs))
    policies["thmp"] = ThompsonSamplingPolicy(envs[0], std=var, sample=False, prior_mean=0.5, prior_var=1 / 12.0,
                                              warm_start=False, batch_size=num_envs)
    for name in ("opt", "emp", "thmp", "lcb", "lnr"):            # set_batch order of the reference (:270-274)
        if name in policies:
            policies[name].set_batch_numpy_vec(batch)
    baselines = {}
    for name in ("opt", "emp", "lnr", "lcb", "thmp"):            # deploy order of the reference (:276-280)
        if name in policies:
            baselines[name] = np.array(vec_env.deploy_eval(policies[name])[3])
    return baselines


def _offline_context(batch_or_trajs, means, n_eval=None):
    """(means [N,d], context dict of fp32 device tensors [N,H,.]) from a device batch (e.g. collect_data.collect_bandit's
    dict, used as is) or from the reference's list of traj dicts (stacked once)."""
    dev = kernels._dev()
    if isinstance(batch_or_trajs, dict):
        ctx = {k: batch_or_trajs[k] for k in ("context_states", "context_actions", "context_next_states", "context_rewards")}
        if means is None:
            means = batch_or_trajs["means"]
    else:
        trajs = list(batch_or_trajs)[:n_eval]
        f = lambda k, tail: torch.as_tensor(np.stack([np.asarray(t[k], dtype=np.float32).reshape((-1,) + tail) for t in trajs])).to(dev)  # noqa: E731
        d = np.asarray(trajs[0]["context_actions"]).shape[-1]
        ctx = {"context_states": f("context_states", (1,)), "context_actions": f("context_actions", (d,)),
               "context_next_states": f("context_next_states", (1,)), "context_rewards": f("context_rewards", (1,))}
        if means is None:
            means = np.stack([np.asarray(t["means"], dtype=np.float64) for t in trajs])
    means = torch.as_tensor(means).to(device=dev, dtype=torch.float32) if not torch.is_tensor(means) else means.to(dev).float()
    return means, ctx


def learner_logits(model, ctx, T):
    """Logits of every context prefix 0..T-1 in one forward: row h-1 of the test=False forward over ``ctx[:, :T]``
    attends to the query token and the first h transitions at the same positions as the reference's test=True forward
    on ``ctx[:, :h]`` (models/net.py:41-60).  [N, T, d] fp32."""
    N = ctx["context_actions"].shape[0]
    dev = ctx["context_actions"].device
    was_test = model.test
    model.test = False
    try:
        x = {k: v[:, :T] for k, v in ctx.items()}
        x["query_states"] = torch.ones((N, 1), dtype=torch.float32, device=dev)   # the bandit state is the constant [1]
        return model.forward(x)
    finally:
        model.test = was_test


def offline_device(batch_or_trajs, means, horizons, model=None, var=None, seed=None, env_id0=0, per_env=True, inject=None,
                   dump=False, n_eval=None, ctrls=("opt", "emp", "lcb", "thmp")):
    """``offline`` for every horizon in ``horizons`` at once, on the device (dpt_offline_eval): one pass over the
    context gives the noise-free reward of Opt, EmpMean, LCB(0.8), Thompson(sample=False, prior 0.5 / (1/12),
    std = var) and, with a model, the transformer (one test=False forward over max(horizons) rows).

    batch_or_trajs: a dict of device tensors with context_* [N,H,.] (and ``means`` when ``means`` is None), e.g.
    collect_data.collect_bandit's output, or the reference's list of traj dicts.  inject: {'z': f64 [K,100,N,d]} the
    Thompson normals in the reference's order; dump=True returns the normals used.  Returns kernels.offline_eval's dict
    (sums [K,6,2], rewards [K,6,N] when per_env, slots kernels.OFFLINE_SLOTS) plus 'horizons', 'n_envs' and 'ctrls'
    (the slots that were computed)."""
    if var is None:
        raise ValueError("offline_device: var (the Thompson std, as in offline()) is required")
    means, ctx = _offline_context(batch_or_trajs, means, n_eval)
    hz = np.asarray(horizons, dtype=np.int64).reshape(-1)
    ctrls = tuple(ctrls)
    logits = None
    if model is not None:
        ctrls = ctrls + ("lnr",)
        logits = learner_logits(model, ctx, int(hz.max()))
    key = rng.next_key() if seed is None else seed
    out = kernels.offline_eval(means, ctx["context_actions"], ctx["context_rewards"], hz, ctrls, lcb_const=.8, thmp_std=var,
                               thmp_prior_mean=0.5, thmp_prior_var=1 / 12.0, n_draws=100, learner_logits=logits, seed=key,
                               env_id0=env_id0, per_env=per_env, inject=inject, dump=dump)
    out["horizons"], out["n_envs"] = hz, means.shape[0]
    out["ctrls"] = ("opt",) + tuple(c for c in ctrls if c != "opt")
    return out


def _names(ctrls):
    return [c for c in ("opt", "emp", "lnr", "lcb", "thmp", "linreg") if c in ctrls]   # the reference's dict order


def offline_graph_device(batch_or_trajs, means, horizon, model=None, var=None, seed=None, env_id0=0, n_eval=None):
    """``offline_graph`` from one dpt_offline_eval launch over np.linspace(1, horizon, 50, dtype=int).  Returns
    (horizons [50], {name: regret of the mean per horizon}) with sums over envs left on the device until the end."""
    horizons = np.linspace(1, horizon, 50, dtype=int)
    out = offline_device(batch_or_trajs, means, horizons, model, var, seed, env_id0, per_env=False, n_eval=n_eval)
    s = out["sums"].cpu().numpy()
    regrets = {k: s[:, kernels.OFFLINE_SLOTS.index(k), 0] / out["n_envs"] for k in _names(out["ctrls"]) if k != "opt"}
    return horizons, regrets


def offline_graph(eval_trajs, model, n_eval, horizon, var, bandit_type="uniform", fused=False):
    """evals/eval_bandit.py:304-335 without plotting: suboptimality against dataset size.  Returns
    (horizons [50], {name: regret-of-the-mean per horizon}).  fused=True computes the same curves from one
    offline_eval launch (``offline_graph_device``) instead of 50 ``offline`` calls."""
    if fused:
        return offline_graph_device(eval_trajs, None, horizon, model, var, n_eval=n_eval)
    horizons = np.linspace(1, horizon, 50, dtype=int)
    all_means = []
    for h in horizons:
        b = offline(eval_trajs, model, n_eval=n_eval, horizon=int(h), var=var, bandit_type=bandit_type)
        all_means.append({k: np.mean(v, axis=0) for k, v in b.items()})
    regrets = {k: np.array([m["opt"] - m[k] for m in all_means]) for k in all_means[0] if k != "opt"}
    return horizons, regrets
