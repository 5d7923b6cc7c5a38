"""One training step of the GPT-2 (forward_train + CE-sum + backward + AdamW) on the fused CUDA path against the same step
of the fp32 eager torch restatement (tests/train_oracle.py with F.scaled_dot_product_attention, autograd, the same
AdamW) and, when `transformers` is installed, the HF GPT2Model.

    python scripts/train_time.py [--steps 20] [--out FILE]

Cases: bandit B = 64 (H = 500, d = 5, L = 4), darkroom B = 64 (H = 100, dx = 2, du = 5, L = 4), bandit B = 1024.
Step times are medians of CUDA-event timings after warm-up, with the phases separated by events: forward_train, CE +
backward (the backward kernel and the weight-gradient reduction), AdamW.  A separate torch.profiler pass gives the
device time per kernel (forward, backward, reduction).  FLOPs are computed from the shapes.  Prints one JSON line.
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np
import torch
import torch.nn.functional as F

import dpt_b200  # noqa: F401
from dpt_b200 import train as TR
from dpt_b200.models.net import Transformer
import train_oracle as TO

CASES = [("bandit_b64", 1, 5, 500, 4, 64), ("darkroom_b64", 2, 5, 100, 4, 64), ("bandit_b1024", 1, 5, 500, 4, 1024)]


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clk = [x.strip() for x in q.split(",")]
        return {"name": name, "power_limit": power, "max_sm_clock": clk}
    except Exception as e:   # noqa: BLE001
        return {"name": torch.cuda.get_device_name(0), "error": repr(e)}


def flops(B, T, dx, du, L):
    """Forward FLOPs of one batch (2 per multiply-add): the row matmuls, causal attention (QK^T and PV over keys <= i),
    embedding and head; a training step counts the backward as twice the forward."""
    S = T + 1
    din = 2 * dx + du + 1
    per_row_layer = 2 * (32 * 96 + 32 * 32 + 32 * 128 + 128 * 32)
    attn = 2 * 2 * 32 * S * (S + 1) // 2
    fwd = B * (L * (S * per_row_layer + attn) + S * 2 * din * 32 + T * 2 * 32 * du)
    return fwd, 3 * fwd


def batch_for(dx, du, B, H, seed=0):
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


def timed_steps(fwd, opt, b, steps, warmup=3):
    """Median (total, forward, loss + backward, AdamW) in ms over `steps` steps."""
    for _ in range(warmup):
        opt.zero_grad()
        TR.ce_sum_loss(fwd(b), b).backward()
        opt.step()
    torch.cuda.synchronize()
    rows = []
    for _ in range(steps):
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
        opt.zero_grad()
        ev[0].record()
        pred = fwd(b)
        ev[1].record()
        TR.ce_sum_loss(pred, b).backward()
        ev[2].record()
        opt.step()
        ev[3].record()
        torch.cuda.synchronize()
        rows.append([ev[0].elapsed_time(ev[3]), ev[0].elapsed_time(ev[1]), ev[1].elapsed_time(ev[2]), ev[2].elapsed_time(ev[3])])
    med = np.median(np.array(rows), axis=0)
    return {"step_ms": float(med[0]), "forward_ms": float(med[1]), "loss_backward_ms": float(med[2]), "adamw_ms": float(med[3])}


def kernel_split(fwd, opt, b, steps=5):
    """Device time per step (ms) of the fused path's kernels, from torch.profiler (a run of its own)."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(steps):
            opt.zero_grad()
            TR.ce_sum_loss(fwd(b), b).backward()
            opt.step()
        torch.cuda.synchronize()
    groups = {"forward": ["gpt2_train_forward_kernel"], "backward": ["gpt2_train_backward_kernel"],
              "reduction": ["weight_grad_partial_kernel", "weight_grad_reduce_kernel", "wpe_grad_kernel"]}
    out = {k: 0.0 for k in list(groups) + ["other"]}
    for e in prof.key_averages():
        t = getattr(e, "device_time_total", None)
        if t is None:
            t = e.cuda_time_total
        if t <= 0:
            continue
        key = next((k for k, names in groups.items() if any(n in e.key for n in names)), "other")
        out[key] += t / 1000.0 / steps
    return out


def eager_model(m):
    P = {k: p.detach().clone().float().requires_grad_(True) for k, p in m.named_parameters() if "wte" not in k}
    L = m.n_layer

    def fwd(b):
        return TO.forward(P, L, b["query_states"], b["context_states"], b["context_actions"], b["context_next_states"],
                          b["context_rewards"], False, sdpa=True)
    return fwd, torch.optim.AdamW(list(P.values()), lr=1e-3, weight_decay=1e-4)


def hf_model(m, dx, du):
    try:
        import transformers
    except ImportError:
        return None
    cfg = transformers.GPT2Config(n_positions=m.transformer.wpe.weight.shape[0], n_embd=32, n_layer=m.n_layer, n_head=1,
                                  resid_pdrop=0.0, embd_pdrop=0.0, attn_pdrop=0.0, use_cache=False)
    hf = transformers.GPT2Model(cfg).cuda()
    emb, head = torch.nn.Linear(2 * dx + du + 1, 32).cuda(), torch.nn.Linear(32, du).cuda()
    mods = torch.nn.ModuleList([hf, emb, head])

    def fwd(b):
        return head(hf(inputs_embeds=emb(TO.tokens(b["query_states"], b["context_states"], b["context_actions"],
                                                   b["context_next_states"], b["context_rewards"]))).last_hidden_state)[:, 1:, :]
    return fwd, torch.optim.AdamW(mods.parameters(), lr=1e-3, weight_decay=1e-4)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("train_time.py measures on the GPU; no CUDA device")
    res = {"gpu": gpu_info(), "steps": a.steps, "cases": []}
    for name, dx, du, H, L, B in CASES:
        torch.manual_seed(0)
        m = Transformer({"horizon": H, "state_dim": dx, "action_dim": du, "n_layer": L, "n_embd": 32, "n_head": 1,
                         "dropout": 0.0, "test": False}).cuda()
        b = batch_for(dx, du, B, H)
        fl_fwd, fl_step = flops(B, H, dx, du, L)
        row = {"case": name, "B": B, "H": H, "dx": dx, "du": du, "L": L, "fwd_gflop": fl_fwd / 1e9, "step_gflop": fl_step / 1e9}
        opt = torch.optim.AdamW(m.parameters(), lr=1e-3, weight_decay=1e-4)
        row["fused"] = timed_steps(m.forward_train, opt, b, a.steps)
        row["fused"]["tflops"] = fl_step / row["fused"]["step_ms"] / 1e9
        row["fused"]["kernels_ms"] = kernel_split(m.forward_train, opt, b)
        fwd, opt2 = eager_model(m)
        row["torch_eager"] = timed_steps(fwd, opt2, b, a.steps)
        h = hf_model(m, dx, du)
        if h is not None:
            row["hf_gpt2"] = timed_steps(h[0], h[1], b, a.steps)
        row["speedup_vs_eager"] = row["torch_eager"]["step_ms"] / row["fused"]["step_ms"]
        res["cases"].append(row)
        print(json.dumps(row), file=sys.stderr)
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
