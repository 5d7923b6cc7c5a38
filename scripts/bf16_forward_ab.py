"""A/B of the bf16 (precision 1) dense forward between two builds of libdpt_b200.so with the same ABI, in one process.

    git worktree add /tmp/base <commit> && make -C /tmp/base/decision-pretrained-transformer_b200/csrc -j8
    python scripts/bf16_forward_ab.py --base /tmp/base/decision-pretrained-transformer_b200/libdpt_b200.so [--out FILE]

--new defaults to this tree's library.  Each build creates its own model handles (dpt_gpt2_create), so the weight images
it packs are part of what is compared.

Bits: every result must be torch.equal between the builds.
- Transformer.forward at precision 1 for L in {1, 4, 8}, dx in {1, 2}, T in {10, 127, 128, 200, 511}, test in {0, 1}
  (B = 24 sequences, one model per (L, dx)), and one ctx_share = 4 call;
- one bf16 training step (forward_train_population(..., precision=1), CE-sum, backward, AdamW) for one model at
  T = 100, 300 and 500 and for a k = 3 population at T = 100 and 500: logits, every gradient and the updated weights.
Time: dense forward (4 layers, d = 5) at B = 100 and 4096 x 101 tokens (gpt2_dense_kernel), B = 1024 x 201 and x 501 tokens
(gpt2_dense_long_kernel<2> / <4>), all inputs L2-resident after the first call, and a bf16 train_step at bandit
B = 64 x 501 and darkroom B = 64 x 101 tokens.  Each round runs every case on both builds, the order alternating per
round; CUDA events around a fixed number of back-to-back calls after a warm-up call.  A case's figure is the median of
the rounds, and the min / max of a build's rounds is its spread.  The card's name, power limit and max SM clock are read
in the same run.  Prints one JSON object and writes it to --out.
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np
import torch

import dpt_b200  # noqa: F401
from dpt_b200 import _lib
from dpt_b200 import train as TR
from dpt_b200.models.net import Transformer, forward_train_population

DU = 5


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    name, power, clk = [x.strip() for x in q.split(",")]
    return {"name": name, "power_limit": power, "max_sm_clock": clk}


class Builds:
    """Both libraries loaded at once; use(name, models) makes `name` the one every entry point calls."""

    def __init__(self, paths):
        self.libs = {}
        for name, path in paths.items():
            _lib.LIB_PATH, _lib._lib = path, None
            self.libs[name] = _lib.lib()

    def use(self, name, models=()):
        for m in models:
            m._free()   # a handle is destroyed by the library that created it
        _lib._lib = self.libs[name]


def model(dx, L, H, seed, test=False):
    torch.manual_seed(seed)
    m = Transformer({"horizon": H, "state_dim": dx, "action_dim": DU, "n_layer": L, "n_embd": 32, "n_head": 1,
                     "dropout": 0.0, "test": test}).cuda()
    with torch.no_grad():
        for k, p in m.named_parameters():
            if "wte" not in k:
                p.add_(0.15 * torch.randn_like(p))
    return m


def batch(dx, B, T, seed, n_query=None):
    g = torch.Generator(device="cuda").manual_seed(seed)
    n_query = B if n_query is None else n_query
    if dx == 1:
        cs, q = torch.ones(B, T, 1, device="cuda"), torch.ones(n_query, 1, device="cuda")
        cns = cs
    else:
        cs = torch.randint(0, 10, (B, T, dx), generator=g, device="cuda").float()
        q = torch.randint(0, 10, (n_query, dx), generator=g, device="cuda").float()
        cns = torch.randint(0, 10, (B, T, dx), generator=g, device="cuda").float()
    return {"query_states": q, "context_states": cs, "context_next_states": cns,
            "context_actions": torch.eye(DU, device="cuda")[torch.randint(0, DU, (B, T), generator=g, device="cuda")],
            "context_rewards": torch.rand(B, T, 1, generator=g, device="cuda"),
            "optimal_actions": torch.eye(DU, device="cuda")[torch.randint(0, DU, (n_query,), generator=g, device="cuda")]}


def forward_results(builds, name):
    out = {}
    for L in (1, 4, 8):
        for dx in (1, 2):
            m = model(dx, L, 511, seed=100 * L + dx)
            m.precision = 1
            builds.use(name)
            for T in (10, 127, 128, 200, 511):
                b = batch(dx, 24, T, seed=T)
                for test in (0, 1):
                    m.test = bool(test)
                    out["forward L=%d dx=%d T=%d test=%d" % (L, dx, T, test)] = m(b)
            builds.use(name, [m])
    m = model(1, 4, 511, seed=7, test=True)
    m.precision = 1
    builds.use(name)
    out["forward ctx_share=4 L=4 T=200"] = m(batch(1, 16, 200, seed=3, n_query=64), ctx_share=4)
    builds.use(name, [m])
    return out


def train_results(builds, name):
    out = {}
    builds.use(name)
    for k, T in ((1, 100), (1, 300), (1, 500), (3, 100), (3, 500)):
        ms = [model(1, 4, 500, seed=20 + i) for i in range(k)]
        bs = [batch(1, 16, T, seed=30 + i) for i in range(k)]
        opt = torch.optim.AdamW([p for m in ms for p in m.parameters()], lr=1e-3, weight_decay=1e-4)
        preds = forward_train_population(ms, bs, precision=1)
        sum(TR.ce_sum_loss(p, b) for p, b in zip(preds, bs)).backward()
        opt.step()
        tag = "train k=%d T=%d" % (k, T)
        for i, (m, p) in enumerate(zip(ms, preds)):
            out["%s member %d logits" % (tag, i)] = p.detach()
            for j, q in enumerate(m._train_params()):
                out["%s member %d grad %d" % (tag, i, j)] = q.grad
            for pn, q in m.named_parameters():
                out["%s member %d weight %s" % (tag, i, pn)] = q.detach()
    return out


def bits(builds):
    res = {n: {**forward_results(builds, n), **train_results(builds, n)} for n in builds.libs}
    a, b = res["base"], res["new"]
    assert a.keys() == b.keys()
    diff = [k for k in a if not torch.equal(a[k], b[k])]
    return {"compared": len(a), "forward_cases": sum(k.startswith("forward") for k in a),
            "train_tensors": sum(k.startswith("train") for k in a), "not_equal": diff}


def timing(builds, rounds):
    fwd = [("forward B=100 x 101 tokens", 100, 100, 1000), ("forward B=4096 x 101 tokens", 4096, 100, 60),
           ("forward B=1024 x 201 tokens", 1024, 200, 100), ("forward B=1024 x 501 tokens", 1024, 500, 40)]
    cases = []
    for tag, B, T, iters in fwd:
        m = model(1, 4, 500, seed=1)
        m.precision = 1
        b = batch(1, B, T, seed=2)
        cases.append((tag, [m], lambda m=m, b=b: m(b), iters))
    for tag, dx, H in (("train_step bandit B=64 x 501 tokens", 1, 500), ("train_step darkroom B=64 x 101 tokens", 2, 100)):
        m = model(dx, 4, H, seed=3)
        opt = torch.optim.AdamW(m.parameters(), lr=1e-3, weight_decay=1e-4)
        b = batch(dx, 64, H, seed=4)
        cases.append((tag, [], lambda m=m, opt=opt, b=b: TR.train_step(m, opt, b, precision=1), 100))
    ms = {tag: {n: [] for n in builds.libs} for tag, _, _, _ in cases}
    names = list(builds.libs)
    for r in range(rounds):
        for n in (names if r % 2 == 0 else names[::-1]):
            for tag, models, fn, iters in cases:
                builds.use(n, models)
                fn()
                torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(iters):
                    fn()
                e1.record()
                torch.cuda.synchronize()
                ms[tag][n].append(e0.elapsed_time(e1) / iters)
    out = {}
    for tag, per in ms.items():
        med = {n: float(np.median(v)) for n, v in per.items()}
        spread = {n: [min(v), max(v)] for n, v in per.items()}
        within = any(spread[o][0] <= med[n] <= spread[o][1] for n in per for o in per if o != n)
        out[tag] = {"ms_median": med, "ms_min_max": spread, "rounds_ms": per, "new_over_base": med["new"] / med["base"],
                    "median_within_other_build_spread": within}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--base", required=True, help="libdpt_b200.so of the base build")
    ap.add_argument("--new", default=_lib.LIB_PATH, help="libdpt_b200.so of the new build (default: this tree's)")
    ap.add_argument("--rounds", type=int, default=6)
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    builds = Builds({"base": a.base, "new": a.new})
    rel = lambda p: os.path.relpath(p, ROOT) if os.path.abspath(p).startswith(ROOT + os.sep) else p   # noqa: E731
    res = {"gpu": gpu_info(), "base": rel(a.base), "new": rel(a.new), "bits": bits(builds), "time": timing(builds, a.rounds)}
    s = json.dumps(res, indent=1)
    print(s)
    if a.out:
        with open(a.out, "w") as f:
            f.write(s + "\n")
    if res["bits"]["not_equal"]:
        sys.exit("results differ between the builds: %s" % res["bits"]["not_equal"][:8])


if __name__ == "__main__":
    main()
