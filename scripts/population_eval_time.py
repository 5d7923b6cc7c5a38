"""Population evaluation (models.net.online_loop_population: the bandit online loop of k same-shape models in shared
launches) against the two ways of evaluating k models without it: k sequential Transformer.online_loop calls, and k calls
issued on k CUDA streams from one thread.

    python scripts/population_eval_time.py [--rounds 5] [--ks 1,2,4,8,16] [--ns 100,1000,10000] [--out FILE]

(default --out: profiles/r09_population_eval_time.json)

Cases: k members x N envs x H = 500, fp32 and bf16 K/V (precision 0 and 1), 4 layers, d = 5, sampling, regret sums on and
contexts off (what evals.eval_bandit evaluates).  Every member has its own weights; all see the same means and seed.  Every
shape is warmed up first, then the three arms are alternated `--rounds` times (at N = 10 000: at most 3 rounds); a time is
the median over the rounds of the CUDA-event time of all k members, including the host work of the calls.  The same run
checks that every member's cum_means from the population call equal its sequential call's bit for bit.  Then one
`eval_bandit.online_population` is timed against k x `eval_bandit.online` at n_eval = 100, H = 500 (host clock around
work that ends in a device synchronise, baselines and regret statistics included).  Prints one JSON line; the GPU's name,
power limit and max SM clock are read in the same call.
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

import dpt_b200
from dpt_b200.evals import eval_bandit
from dpt_b200.models.net import Transformer, online_loop_population
from train_time import gpu_info

H, D, L, VAR = 500, 5, 4, 0.3


def members(k, precision, seed0=0):
    out = []
    for i in range(k):
        torch.manual_seed(seed0 + i)
        m = Transformer({"horizon": H, "state_dim": 1, "action_dim": D, "n_layer": L, "n_embd": 32, "n_head": 1, "dropout": 0.0,
                         "test": True}).cuda()
        m.precision = precision
        out.append(m)
    return out


class Arms:
    def __init__(self, ms, means):
        self.ms, self.means = ms, means
        self.streams = [torch.cuda.Stream() for _ in ms]
        self.last = {}

    def _one(self, m):
        return m.online_loop(self.means, H, VAR, True, 7, 0, materialise=False, regret=True)

    def population(self):
        self.last["population"] = online_loop_population(self.ms, self.means, H, VAR, True, 7, 0, materialise=False, regret=True)

    def sequential(self):
        self.last["sequential"] = [self._one(m) for m in self.ms]

    def k_streams(self):
        cur, outs = torch.cuda.current_stream(), []
        for s, m in zip(self.streams, self.ms):
            s.wait_stream(cur)
            with torch.cuda.stream(s):
                outs.append(self._one(m))
        for s in self.streams:
            cur.wait_stream(s)
        self.last["k_streams"] = outs


def time_once(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1)


def eval_case(k, n_eval=100):
    """One online_population against k x online (n_eval envs, H = 500, fp32), host included; all_means compared."""
    ms = members(k, 0, 300)
    rs = np.random.RandomState(0)
    trajs = [{"means": rs.uniform(0, 1, D)} for _ in range(n_eval)]
    for _ in range(2):   # warm-up of both forms
        dpt_b200.rng.seed(1)
        eval_bandit.online_population(trajs, ms, n_eval, H, VAR)
        dpt_b200.rng.seed(1)
        eval_bandit.online(trajs, ms[0], n_eval, H, VAR)
    torch.cuda.synchronize()
    tp, tk = [], []
    for _ in range(3):
        dpt_b200.rng.seed(1)
        t0 = time.perf_counter()
        pop, _ = eval_bandit.online_population(trajs, ms, n_eval, H, VAR)
        torch.cuda.synchronize()
        t1 = time.perf_counter()
        ref = []
        for m in ms:
            dpt_b200.rng.seed(1)
            ref.append(eval_bandit.online(trajs, m, n_eval, H, VAR)[0])
        torch.cuda.synchronize()
        t2 = time.perf_counter()
        tp.append(t1 - t0)
        tk.append(t2 - t1)
    same = all(np.array_equal(p[c], r[c]) for p, r in zip(pop, ref) for c in r)
    return {"k": k, "n_eval": n_eval, "H": H, "online_population_s": float(np.median(tp)), "k_x_online_s": float(np.median(tk)),
            "speedup": float(np.median(tk) / np.median(tp)), "all_means_bit_identical": same}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--ks", default="1,2,4,8,16")
    ap.add_argument("--ns", default="100,1000,10000")
    ap.add_argument("--eval-ks", default="4,16")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r09_population_eval_time.json"))
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("population_eval_time.py measures on the GPU; no CUDA device")
    res = {"gpu": gpu_info(), "sms": torch.cuda.get_device_properties(0).multi_processor_count, "H": H, "d": D, "n_layer": L,
           "rounds": a.rounds, "population_max": dpt_b200.models.net.ONLINE_POPULATION_MAX, "cases": [], "eval": []}
    for precision in (0, 1):
        for N in [int(x) for x in a.ns.split(",")]:
            means, _, _ = dpt_b200.kernels.bandit_sample_means(N, D, 3, 0)
            for k in [int(x) for x in a.ks.split(",")]:
                arms = Arms(members(k, precision), means)
                fns = {"population": arms.population, "sequential": arms.sequential, "k_streams": arms.k_streams}
                for fn in fns.values():
                    time_once(fn)   # warm-up: every shape, every arm
                ts = {n: [] for n in fns}
                for _ in range(min(a.rounds, 3) if N >= 10000 else a.rounds):
                    for n, fn in fns.items():
                        ts[n].append(time_once(fn))
                row = {"precision": ["fp32", "bf16"][precision], "N": N, "k": k,
                       "env_warps_per_sm": -(-k * N // res["sms"])}
                for n in fns:
                    med = float(np.median(ts[n]))
                    row[n] = {"ms": med, "per_member_ms": med / k, "min_max_ms": [float(min(ts[n])), float(max(ts[n]))]}
                row["sequential_over_population"] = row["sequential"]["ms"] / row["population"]["ms"]
                row["k_streams_over_population"] = row["k_streams"]["ms"] / row["population"]["ms"]
                row["cum_means_bit_identical"] = all(torch.equal(p["cum_means"], s["cum_means"])
                                                     for p, s in zip(arms.last["population"], arms.last["sequential"]))
                res["cases"].append(row)
                print(json.dumps(row), file=sys.stderr)
                del arms, fns
                torch.cuda.empty_cache()
    for k in [int(x) for x in a.eval_ks.split(",") if x]:
        row = eval_case(k)
        res["eval"].append(row)
        print(json.dumps(row), file=sys.stderr)
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
