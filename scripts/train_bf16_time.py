"""Training step time at precision 0 (fp32, CUDA cores) and 1 (bf16 tensor cores) in the same process, alternating.

    python scripts/train_bf16_time.py [--steps 20] [--rounds 3] [--out profiles/r10_train_bf16_time.json]

Cases: bandit B = 64 x 501 tokens (H = 500, d = 5, 4 layers), darkroom B = 64 x 101 (dx = 2), bandit B = 1024 x 501, and a
k = 8 population on the bandit B = 64 shape (train_population_step).  One step is forward_train + CE-sum + backward +
AdamW.  Each round times every case at both precisions (CUDA events, `--steps` steps after warm-up); a case's figure is
the median over all rounds' steps.  A torch.profiler run of its own gives the device time per phase (forward, backward,
weight-gradient reduction, CE + AdamW + the rest).  Then one epoch of train.train on a collect_bandit dataset of 8192
envs (H = 500) at each precision, timed on the host around a device synchronise.  The card's name and power limit are
read in the same run.  Prints and writes one JSON object.
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np
import torch

import dpt_b200  # noqa: F401
from dpt_b200 import train as TR
from dpt_b200.models.net import Transformer

CASES = [("bandit_b64", 1, 5, 500, 4, 64, 1), ("darkroom_b64", 2, 5, 100, 4, 64, 1), ("bandit_b1024", 1, 5, 500, 4, 1024, 1),
         ("bandit_b64_population_k8", 1, 5, 500, 4, 64, 8)]
PHASES = {"forward": ["gpt2_train_forward", "pack_wimg"],
          "backward": ["gpt2_train_backward_kernel", "gpt2_train_rows_bf16", "gpt2_train_attn_bf16"],
          "reduction": ["weight_grad_partial_kernel", "weight_grad_reduce_kernel", "wpe_grad_kernel"]}


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    name, power, clk = [x.strip() for x in q.split(",")]
    return {"name": name, "power_limit": power, "max_sm_clock": clk}


def batch_for(dx, du, B, H, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    if dx == 1:
        cs = torch.ones(B, H, 1, device="cuda")
        q = torch.ones(B, 1, device="cuda")
        cns = cs
    else:
        cs = torch.randint(0, 10, (B, H, dx), generator=g, device="cuda").float()
        q = torch.randint(0, 10, (B, dx), generator=g, device="cuda").float()
        cns = torch.randint(0, 10, (B, H, dx), generator=g, device="cuda").float()
    return {"query_states": q, "context_states": cs, "context_next_states": cns,
            "context_actions": torch.eye(du, device="cuda")[torch.randint(0, du, (B, H), generator=g, device="cuda")],
            "context_rewards": torch.rand(B, H, 1, generator=g, device="cuda"),
            "optimal_actions": torch.eye(du, device="cuda")[torch.randint(0, du, (B,), generator=g, device="cuda")]}


def setup(case):
    name, dx, du, H, L, B, k = case
    models = []
    for i in range(k):
        torch.manual_seed(i)
        models.append(Transformer({"horizon": H, "state_dim": dx, "action_dim": du, "n_layer": L, "n_embd": 32, "n_head": 1,
                                   "dropout": 0.0, "test": False}).cuda())
    opt = torch.optim.AdamW([p for m in models for p in m.parameters()], lr=1e-3, weight_decay=1e-4)
    batches = [batch_for(dx, du, B, H, 7 + i) for i in range(k)]
    if k == 1:
        return lambda prec: TR.train_step(models[0], opt, batches[0], precision=prec)
    return lambda prec: TR.train_population_step(models, opt, batches, precision=prec)


def timed(step, prec, steps):
    ms = []
    for _ in range(steps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        step(prec)
        b.record()
        torch.cuda.synchronize()
        ms.append(a.elapsed_time(b))
    return ms


def phases(step, prec, steps=5):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(steps):
            step(prec)
        torch.cuda.synchronize()
    out = {k: 0.0 for k in list(PHASES) + ["ce_adamw_other"]}
    for e in prof.key_averages():
        t = getattr(e, "device_time_total", None)
        if t is None:
            t = e.cuda_time_total
        if t <= 0:
            continue
        key = next((k for k, names in PHASES.items() if any(n in e.key for n in names)), "ce_adamw_other")
        out[key] += t / 1000.0 / steps
    return out


def epoch_time(n_envs, H):
    from dpt_b200 import collect_data
    from dpt_b200.dataset import Dataset
    batch = collect_data.collect_bandit(n_envs, 5, H, 0.3, seed=11)
    cfg = {"horizon": H, "state_dim": 1, "action_dim": 5, "shuffle": True, "store_gpu": True}
    tr = Dataset.from_batch(batch, cfg)
    te = Dataset.from_batch({k: v[:64] for k, v in batch.items()}, cfg)
    out = {}
    for prec in (0, 1):
        torch.manual_seed(0)
        m = Transformer({"horizon": H, "state_dim": 1, "action_dim": 5, "n_layer": 4, "n_embd": 32, "n_head": 1, "dropout": 0.0,
                         "test": False}).cuda()
        TR.train(m, te, te, 1, seed=0, precision=prec)   # warm-up (module loads, allocator)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        train_loss, _, _ = TR.train(m, tr, te, 1, seed=0, precision=prec)
        torch.cuda.synchronize()
        out["precision%d" % prec] = {"epoch_s": time.perf_counter() - t0, "train_loss": train_loss[0]}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--epoch-envs", type=int, default=8192)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r10_train_bf16_time.json"))
    a = ap.parse_args()
    res = {"gpu": gpu_info(), "steps": a.steps, "rounds": a.rounds, "cases": {}}
    steps = {c[0]: setup(c) for c in CASES}
    samples = {(n, p): [] for n in steps for p in (0, 1)}
    for n, step in steps.items():   # warm-up of every shape at both precisions
        for p in (0, 1):
            timed(step, p, 3)
    for _ in range(a.rounds):
        for n, step in steps.items():
            for p in (0, 1):
                samples[(n, p)] += timed(step, p, a.steps)
    for n in steps:
        r = {"precision%d_step_ms" % p: float(np.median(samples[(n, p)])) for p in (0, 1)}
        r["speedup"] = r["precision0_step_ms"] / r["precision1_step_ms"]
        res["cases"][n] = r
    for n, step in steps.items():
        for p in (0, 1):
            res["cases"][n]["precision%d_phases_ms" % p] = phases(step, p)
    res["epoch_bandit_%d_envs_h500" % a.epoch_envs] = epoch_time(a.epoch_envs, 500)
    res["gpu_after"] = gpu_info()
    print(json.dumps(res))
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f)
        f.write("\n")


if __name__ == "__main__":
    main()
