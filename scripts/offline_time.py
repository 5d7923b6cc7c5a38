"""Offline bandit evaluation: offline_graph on the per-step path against the fused device path (offline_graph(fused=True)).

    python scripts/offline_time.py [--n-envs 100000] [--n-slow 200] [--reps 5] [--out FILE]

Two cases: the bandit (H = 500, d = 5, 50 horizons, 4-layer embd-32 transformer) and the linear bandit (H = 200,
d = 10, lin_d = 2, all 200 horizons, no model).  The per-step path runs at ``--n-slow`` envs (it costs O(#horizons * N)
host work) and is reported per env as well.  On the fused path the offline_eval kernel and the dense forward are timed
with CUDA events, separately from the wall time of the whole Python call.  Prints one JSON line.
"""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

import dpt_b200
from dpt_b200 import collect_data, kernels
from dpt_b200.evals import eval_bandit, eval_linear_bandit
from dpt_b200.models.net import Transformer

HBM_TBS = 7.7   # HGX B200 data sheet, per GPU


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clk = [x.strip() for x in q.split(",")]
        return {"name": name, "power_limit": power, "max_sm_clock": clk}
    except Exception as e:   # noqa: BLE001
        return {"name": torch.cuda.get_device_name(0), "error": repr(e)}


def events(fn, reps):
    """Median device time (ms) of fn() over reps passes, after one warm-up pass."""
    fn()
    ts = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b))
    return float(np.median(ts))


def wall(fn, reps):
    fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        ts.append(time.perf_counter() - t0)
    return float(np.median(ts))


def trajs_of(batch, n, arms=None, theta=None):
    ca, cr = batch["context_actions"][:n].cpu().numpy().astype(np.float64), batch["context_rewards"][:n, :, 0].cpu().numpy().astype(np.float64)
    m = batch["means"][:n].cpu().numpy().astype(np.float64)
    H = ca.shape[1]
    out = [{"means": m[i], "context_states": np.ones((H, 1)), "context_actions": ca[i], "context_next_states": np.ones((H, 1)),
            "context_rewards": cr[i]} for i in range(n)]
    if arms is not None:
        for i, t in enumerate(out):
            t["arms"], t["theta"] = arms, theta[i]
    return out


def bandit_case(N, n_slow, reps):
    H, d, var = 500, 5, 0.3
    batch = collect_data.collect_bandit(N, d, H, var, seed=1)
    torch.manual_seed(0)
    model = Transformer({"horizon": H, "state_dim": 1, "action_dim": d, "n_layer": 4, "n_embd": 32, "n_head": 1, "dropout": 0.0,
                         "test": True})
    hz = np.linspace(1, H, 50, dtype=int)
    ctx = {k: batch[k] for k in ("context_states", "context_actions", "context_next_states", "context_rewards")}
    logits = eval_bandit.learner_logits(model, ctx, H)
    ctrls = ("opt", "emp", "lcb", "thmp", "lnr")
    kern = lambda c=ctrls: kernels.offline_eval(batch["means"], batch["context_actions"], batch["context_rewards"], hz, c,  # noqa: E731
                                               thmp_std=var, learner_logits=logits, seed=3, per_env=False)
    res = {"N": N, "H": H, "d": d, "K": len(hz), "n_layer": 4, "n_embd": 32,
           "kernel_ms": events(kern, reps),
           "kernel_no_thompson_ms": events(lambda: kern(("opt", "emp", "lcb", "lnr")), reps),
           "dense_forward_ms": events(lambda: eval_bandit.learner_logits(model, ctx, H), reps),
           "fused_wall_s": wall(lambda: eval_bandit.offline_graph_device(batch, None, H, model, var, seed=3), reps)}
    trajs = trajs_of(batch, n_slow)
    t0 = time.perf_counter()
    eval_bandit.offline_graph(trajs, model, n_slow, H, var)
    res["slow_N"] = n_slow
    res["slow_wall_s"] = time.perf_counter() - t0
    t0 = time.perf_counter()
    eval_bandit.offline_graph(trajs, model, n_slow, H, var, fused=True)
    res["fused_wall_s_at_slow_N"] = time.perf_counter() - t0
    res["slow_us_per_env"] = 1e6 * res["slow_wall_s"] / n_slow
    res["fused_us_per_env"] = 1e6 * res["fused_wall_s"] / N
    return res, hz, d, H


def linear_case(N, n_slow, reps):
    H, d, lin_d, var = 200, 10, 2, 0.3
    arms = np.random.RandomState(seed=1234).normal(size=(d, lin_d)) / np.sqrt(lin_d)   # collect_data.py:230-231
    theta = torch.tensor(np.random.RandomState(5).normal(size=(N, lin_d)), dtype=torch.float64)
    means = (theta @ torch.tensor(arms).T).float().cuda()
    batch = collect_data.collect_bandit(N, d, H, var, seed=2, means=means)   # a logged context on the linear-bandit tasks
    hz = np.linspace(1, H, H, dtype=int)
    kern = lambda c=("opt", "thmp", "linreg"): kernels.offline_eval(batch["means"], batch["context_actions"],  # noqa: E731
                                                                   batch["context_rewards"], hz, c, thmp_std=var,
                                                                   thmp_prior_mean=0.0, thmp_prior_var=1.0, arms=arms,
                                                                   seed=3, per_env=False)
    res = {"N": N, "H": H, "d": d, "lin_d": lin_d, "K": len(hz),
           "kernel_ms": events(kern, reps),
           "kernel_no_thompson_ms": events(lambda: kern(("opt", "linreg")), reps),
           "fused_wall_s": wall(lambda: eval_linear_bandit.offline_graph_device(batch, None, H, None, var, arms, seed=3), reps)}
    trajs = trajs_of(batch, n_slow, arms, theta.numpy())
    t0 = time.perf_counter()
    eval_linear_bandit.offline_graph(trajs, None, n_slow, H, var)
    res["slow_N"] = n_slow
    res["slow_wall_s"] = time.perf_counter() - t0
    res["slow_us_per_env"] = 1e6 * res["slow_wall_s"] / n_slow
    res["fused_us_per_env"] = 1e6 * res["fused_wall_s"] / N
    return res, hz, d, H


def floors(res, d, H, n_draws=100):
    N, K = res["N"], res["K"]
    ctx_bytes = N * H * (d + 1) * 4
    normals = K * N * n_draws * d
    res["context_bytes"] = ctx_bytes
    res["context_floor_ms"] = ctx_bytes / (HBM_TBS * 1e12) * 1e3
    res["thompson_normals"] = normals
    res["philox_blocks"] = K * N * n_draws * ((d + 3) // 4)
    res["normals_per_s"] = normals / (res["kernel_ms"] - res["kernel_no_thompson_ms"]) * 1e3
    return res


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--n-envs", type=int, default=100000)
    ap.add_argument("--n-slow", type=int, default=200)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    kernels._dev()
    out = {"what": "offline_graph: per-step path vs fused (offline_graph(fused=True) / offline_graph_device)", "gpu": gpu_info()}
    r, hz, d, H = bandit_case(a.n_envs, a.n_slow, a.reps)
    out["bandit"] = floors(r, d, H)
    r, hz, d, H = linear_case(a.n_envs, a.n_slow, a.reps)
    out["linear_bandit"] = floors(r, d, H)
    line = json.dumps(out)
    print(line, flush=True)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")
