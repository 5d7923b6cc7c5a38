"""Population training (train.train_population_step: k same-shape models in the same launches) against the two ways of
training k models without it: k sequential train_steps, and k train_steps issued on k CUDA streams from one thread.

    python scripts/population_train_time.py [--steps 20] [--reps 3] [--out FILE]

Shapes: bandit (B = 64, H = 500, d = 5, L = 4) and darkroom (B = 64, H = 100, dx = 2, du = 5, L = 4), at k = 1, 2, 4, 8, 16.
Each member has its own weights and its own batch.  The three arms are alternated `--reps` times; a step time is the
median over all timed steps of the CUDA-event time of one step of all k members (host work included, the timing ends in
a device synchronise).  The device split (forward / backward / reduction / loss + AdamW, ms per step) comes from a
torch.profiler run of its own per arm.  The same call checks that the population step leaves every member's weights
bit-identical to its own train_steps, and times one epoch of train_population against k x train on a collect_bandit
dataset of 8192 envs (host clock around work that ends in a synchronise; the weights are compared there too).  Prints
one JSON line; the GPU's name, power limit and max SM clock are read in the same call.
"""
import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))
import numpy as np
import torch

import dpt_b200  # noqa: F401
from dpt_b200 import train as TR
from dpt_b200.models.net import Transformer
from train_time import batch_for, gpu_info

SHAPES = [("bandit", 1, 5, 500, 4, 64), ("darkroom", 2, 5, 100, 4, 64)]
KS = [1, 2, 4, 8, 16]
GROUPS = {"forward": ["gpt2_train_forward_kernel"], "backward": ["gpt2_train_backward_kernel"],
          "reduction": ["weight_grad_partial_kernel", "weight_grad_reduce_kernel", "wpe_grad_kernel"]}


def models(k, dx, du, H, L, seed0=0):
    out = []
    for i in range(k):
        torch.manual_seed(seed0 + i)
        out.append(Transformer({"horizon": H, "state_dim": dx, "action_dim": du, "n_layer": L, "n_embd": 32, "n_head": 1,
                                "dropout": 0.0, "test": False}).cuda())
    return out


class Arms:
    """One step of all k members, three ways; each arm owns its models and optimizers."""

    def __init__(self, k, dx, du, H, L, bs):
        self.bs, self.k = bs, k
        self.pop = models(k, dx, du, H, L)
        self.pop_opt = torch.optim.AdamW([p for m in self.pop for p in m.parameters()], lr=1e-3, weight_decay=1e-4)
        self.seq = models(k, dx, du, H, L)
        self.seq_opt = [torch.optim.AdamW(m.parameters(), lr=1e-3, weight_decay=1e-4) for m in self.seq]
        self.str = models(k, dx, du, H, L)
        self.str_opt = [torch.optim.AdamW(m.parameters(), lr=1e-3, weight_decay=1e-4) for m in self.str]
        self.streams = [torch.cuda.Stream() for _ in range(k)]

    def population(self):
        TR.train_population_step(self.pop, self.pop_opt, self.bs)

    def sequential(self):
        for m, o, b in zip(self.seq, self.seq_opt, self.bs):
            TR.train_step(m, o, b)

    def k_streams(self):
        cur = torch.cuda.current_stream()
        for s, m, o, b in zip(self.streams, self.str, self.str_opt, self.bs):
            s.wait_stream(cur)
            with torch.cuda.stream(s):
                TR.train_step(m, o, b)
        for s in self.streams:
            cur.wait_stream(s)


def time_arm(fn, steps):
    ts = []
    for _ in range(steps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    return ts


def device_split(fn, steps=5):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(steps):
            fn()
        torch.cuda.synchronize()
    out = {k: 0.0 for k in list(GROUPS) + ["loss_adamw_other"]}
    for e in prof.key_averages():
        t = getattr(e, "device_time_total", None)
        if t is None:
            t = e.cuda_time_total
        if t <= 0:
            continue
        key = next((k for k, names in GROUPS.items() if any(n in e.key for n in names)), "loss_adamw_other")
        out[key] += t / 1000.0 / steps
    return out


def bit_identity(k, dx, du, H, L, bs, steps=2):
    """The population step against each member's own train_steps: are all weights equal after `steps` steps?"""
    a, b = models(k, dx, du, H, L, 100), models(k, dx, du, H, L, 100)
    opt = torch.optim.AdamW([p for m in a for p in m.parameters()], lr=1e-3, weight_decay=1e-4)
    opts = [torch.optim.AdamW(m.parameters(), lr=1e-3, weight_decay=1e-4) for m in b]
    for _ in range(steps):
        TR.train_population_step(a, opt, bs)
        for m, o, x in zip(b, opts, bs):
            TR.train_step(m, o, x)
    return all(torch.equal(p, q) for ma, mb in zip(a, b) for p, q in zip(ma.parameters(), mb.parameters()))


def epoch_case(k, tr, te, H):
    """One epoch of train_population (k members, one shared dataset, seeds 0..k-1) against k x train, host included."""
    d = tr.dataset["context_actions"].shape[2]
    ma, mb = models(k, 1, d, H, 4, 200), models(k, 1, d, H, 4, 200)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    TR.train_population(ma, tr, te, 1, seeds=list(range(k)))
    torch.cuda.synchronize()
    t1 = time.perf_counter()
    for i, m in enumerate(mb):
        TR.train(m, tr, te, 1, seed=i)
    torch.cuda.synchronize()
    t2 = time.perf_counter()
    same = all(torch.equal(p, q) for x, y in zip(ma, mb) for p, q in zip(x.parameters(), y.parameters()))
    return {"k": k, "train_items": len(tr), "test_items": len(te), "population_s": t1 - t0, "k_x_train_s": t2 - t1,
            "speedup": (t2 - t1) / (t1 - t0), "weights_bit_identical": same}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--ks", default=",".join(map(str, KS)))
    ap.add_argument("--epoch-ks", default="2,8")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("population_train_time.py measures on the GPU; no CUDA device")
    res = {"gpu": gpu_info(), "steps": a.steps, "reps": a.reps, "cases": [], "epoch": []}
    for name, dx, du, H, L, B in SHAPES:
        for k in [int(x) for x in a.ks.split(",")]:
            bs = [batch_for(dx, du, B, H, seed=i) for i in range(k)]
            arms = Arms(k, dx, du, H, L, bs)
            fns = {"population": arms.population, "sequential": arms.sequential, "k_streams": arms.k_streams}
            for fn in fns.values():
                time_arm(fn, 3)   # warm-up
            ts = {n: [] for n in fns}
            for _ in range(a.reps):
                for n, fn in fns.items():
                    ts[n] += time_arm(fn, a.steps)
            row = {"shape": name, "k": k, "B": B, "H": H, "dx": dx, "du": du, "L": L}
            for n, fn in fns.items():
                med = float(np.median(ts[n]))
                row[n] = {"step_ms": med, "per_member_ms": med / k, "spread_ms": [float(np.percentile(ts[n], 10)),
                                                                                  float(np.percentile(ts[n], 90))],
                          "device_ms": device_split(fn)}
            row["population_vs_k_streams"] = row["k_streams"]["step_ms"] / row["population"]["step_ms"]
            row["population_vs_sequential"] = row["sequential"]["step_ms"] / row["population"]["step_ms"]
            row["weights_bit_identical"] = bit_identity(k, dx, du, H, L, bs)
            res["cases"].append(row)
            print(json.dumps(row), file=sys.stderr)
            del arms
            torch.cuda.empty_cache()
    from dpt_b200 import collect_data
    from dpt_b200.dataset import Dataset
    H = 500
    batch = collect_data.collect_bandit(8192 + 512, 5, H, 0.3, seed=1)
    cfg = {"horizon": H, "state_dim": 1, "action_dim": 5, "shuffle": True, "store_gpu": True}
    tr = Dataset.from_batch({k: v[:8192] for k, v in batch.items()}, cfg)
    te = Dataset.from_batch({k: v[8192:] for k, v in batch.items()}, cfg)
    for k in [int(x) for x in a.epoch_ks.split(",") if x]:
        row = epoch_case(k, tr, te, H)
        res["epoch"].append(row)
        print(json.dumps(row), file=sys.stderr)
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
