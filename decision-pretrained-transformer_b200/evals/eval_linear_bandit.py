"""Linear-bandit evaluation (evals/eval_linear_bandit.py): same ``deploy_online`` / ``deploy_online_vec``
(:22-97 are copies of eval_bandit's) with the LinUCB / Thompson controller set of ``online`` (:101-154), and the
offline evaluation (:202-330) on the first ``horizon`` rows of each eval trajectory."""
import numpy as np

from .. import kernels, rng
from ..ctrls.ctrl_bandit import (BanditTransformerController, EmpMeanPolicy, LinUCBPolicy, OptPolicy,  # noqa: F401
                                 ThompsonSamplingPolicy)
from ..envs.bandit_env import BanditEnvVec, LinearBanditEnv
from .eval_bandit import _offline_context, deploy_online, deploy_online_vec, deploy_online_vec_device, learner_logits, regret_stats  # noqa: F401


def online(eval_trajs, model, n_eval, horizon, var):
    """evals/eval_linear_bandit.py:101-170 without plotting."""
    envs = [LinearBanditEnv(eval_trajs[i]["theta"], eval_trajs[i]["arms"], horizon, var=var) for i in range(n_eval)]
    vec_env = BanditEnvVec(envs)
    ctrls = {"opt": OptPolicy(envs, batch_size=len(envs))}
    if model is not None:
        ctrls["Lnr"] = BanditTransformerController(model, sample=True, batch_size=len(envs))
    ctrls["Thomp"] = ThompsonSamplingPolicy(envs[0], std=var, sample=True, prior_mean=0.0, prior_var=1.0,
                                            warm_start=False, batch_size=len(envs))
    ctrls["LinUCB"] = LinUCBPolicy(envs[0], const=1.0, batch_size=len(envs))
    all_means = {name: deploy_online_vec(vec_env, c, horizon).T for name, c in ctrls.items()}
    return all_means, regret_stats(all_means)


def offline(eval_trajs, model, n_eval, horizon, var):
    """evals/eval_linear_bandit.py:202-286 without the bar plot: every controller sees the first ``horizon``
    context rows of each eval trajectory and plays ONE noise-free pull (deploy_eval).  Returns the per-env
    rewards {'opt','lnr','thmp','linreg'} (``lnr`` only when a model is given)."""
    num_envs = len(eval_trajs)
    tmp_env = LinearBanditEnv(eval_trajs[0]["theta"], eval_trajs[0]["arms"], horizon, var=var)
    context_states = np.zeros((num_envs, horizon, tmp_env.dx))
    context_actions = np.zeros((num_envs, horizon, tmp_env.du))
    context_next_states = np.zeros((num_envs, horizon, tmp_env.dx))
    context_rewards = np.zeros((num_envs, horizon, 1))
    envs = []
    for i_eval in range(n_eval):
        traj = eval_trajs[i_eval]
        envs.append(LinearBanditEnv(traj["theta"], traj["arms"], horizon, var=var))
        context_states[i_eval] = traj["context_states"][:horizon]
        context_actions[i_eval] = traj["context_actions"][:horizon]
        context_next_states[i_eval] = traj["context_next_states"][:horizon]
        context_rewards[i_eval] = np.asarray(traj["context_rewards"])[:horizon, None]
    vec_env = BanditEnvVec(envs)
    batch = {"context_states": context_states, "context_actions": context_actions,
             "context_next_states": context_next_states, "context_rewards": context_rewards}
    policies = {"opt": OptPolicy(envs, batch_size=num_envs)}
    if model is not None:
        policies["lnr"] = BanditTransformerController(model, sample=False, batch_size=num_envs)
    policies["thmp"] = ThompsonSamplingPolicy(envs[0], std=var, sample=False, prior_mean=0, prior_var=1.0,
                                              warm_start=False, batch_size=num_envs)
    policies["linreg"] = LinUCBPolicy(envs[0], const=0.0, batch_size=num_envs)
    for name in ("opt", "thmp", "lnr", "linreg"):               # set_batch order of the reference (:263-266)
        if name in policies:
            policies[name].set_batch_numpy_vec(batch)
    baselines = {}
    for name in ("opt", "lnr", "thmp", "linreg"):               # deploy order of the reference (:268-271)
        if name in policies:
            baselines[name] = np.array(vec_env.deploy_eval(policies[name])[3])
    return baselines


def offline_device(batch_or_trajs, means, horizons, model=None, var=None, arms=None, seed=None, env_id0=0, per_env=True,
                   inject=None, dump=False, n_eval=None):
    """``offline`` for every horizon in ``horizons`` at once, on the device (dpt_offline_eval): Opt, Thompson
    (sample=False, prior 0 / 1, std = var), LinReg (LinUCB with const 0 on ``arms`` [d, lin_d], lin_d <= 8; taken from
    the trajs when not given) and, with a model, the transformer.  Arguments and result as eval_bandit.offline_device."""
    if var is None:
        raise ValueError("offline_device: var (the Thompson std, as in offline()) is required")
    if arms is None:
        arms = batch_or_trajs["arms"] if isinstance(batch_or_trajs, dict) else batch_or_trajs[0]["arms"]
    means, ctx = _offline_context(batch_or_trajs, means, n_eval)
    hz = np.asarray(horizons, dtype=np.int64).reshape(-1)
    ctrls = ("opt", "thmp", "linreg")
    logits = None
    if model is not None:
        ctrls = ctrls + ("lnr",)
        logits = learner_logits(model, ctx, int(hz.max()))
    key = rng.next_key() if seed is None else seed
    out = kernels.offline_eval(means, ctx["context_actions"], ctx["context_rewards"], hz, ctrls, thmp_std=var,
                               thmp_prior_mean=0.0, thmp_prior_var=1.0, n_draws=100, arms=np.asarray(arms, dtype=np.float64),
                               linreg_const=0.0, learner_logits=logits, seed=key, env_id0=env_id0, per_env=per_env,
                               inject=inject, dump=dump)
    out["horizons"], out["n_envs"], out["ctrls"] = hz, means.shape[0], ctrls
    return out


def offline_graph_device(batch_or_trajs, means, horizon, model=None, var=None, arms=None, seed=None, env_id0=0, n_eval=None):
    """``offline_graph`` from one dpt_offline_eval launch over every dataset size 1..horizon.  Returns
    (horizons, {name: (mean, sem) of opt - name per horizon}); sem is NaN for a single env, like the default path."""
    horizons = np.linspace(1, horizon, horizon, dtype=int)
    out = offline_device(batch_or_trajs, means, horizons, model, var, arms, seed, env_id0, per_env=False, n_eval=n_eval)
    s, n = out["sums"].cpu().numpy(), out["n_envs"]
    res = {}
    for k in ("lnr", "thmp", "linreg"):                          # the reference's dict order
        if k in out["ctrls"]:
            s1, s2 = s[:, kernels.OFFLINE_SLOTS.index(k), 0], s[:, kernels.OFFLINE_SLOTS.index(k), 1]
            mean = s1 / n
            sem = np.sqrt(np.maximum(s2 - s1 * mean, 0.0) / (n - 1)) / np.sqrt(n) if n > 1 else np.full(len(horizons), np.nan)
            res[k] = (mean, sem)
    return horizons, res


def offline_graph(eval_trajs, model, n_eval, horizon, var, fused=False):
    """evals/eval_linear_bandit.py:289-330 without plotting: suboptimality for every dataset size 1..horizon.
    Returns (horizons, {name: (mean, sem) of opt - name per horizon}).  fused=True computes the same from one
    offline_eval launch (``offline_graph_device``) instead of ``horizon`` ``offline`` calls."""
    if fused:
        return offline_graph_device(eval_trajs, None, horizon, model, var, n_eval=n_eval)
    horizons = np.linspace(1, horizon, horizon, dtype=int)
    sub_mean, sub_sem = {}, {}
    for h in horizons:
        b = offline(eval_trajs, model, n_eval=n_eval, horizon=int(h), var=var)
        for k, v in b.items():
            if k == "opt":
                continue
            d = b["opt"] - v
            sub_mean.setdefault(k, []).append(np.mean(d))
            sub_sem.setdefault(k, []).append(np.std(d, ddof=1) / np.sqrt(len(d)) if len(d) > 1 else np.nan)   # scipy.stats.sem
    return horizons, {k: (np.array(sub_mean[k]), np.array(sub_sem[k])) for k in sub_mean}
