#!/usr/bin/env python
"""Cost of one training-state save (checkpoint.save_state) against one training epoch, at the reference's scale:
100 000 bandit envs, H = 500, d = 5, an 80 / 20 split (1250 steps of batch 64 per epoch), 4-layer GPT-2 (embd 32), for
one model and for a k = 16 population (train_population at k = 1, the path train takes, and k = 16).  The epoch is timed
without a save (host clock around train_population with num_epochs = 1, after a warm-up epoch on 640 items); the save is the median of 5 calls
that write the state the epoch ended with to a temporary directory (torch.save of the weights, AdamW state and
generators, fsync, rename).  Prints one JSON line, and writes it to --out when given.

    python scripts/checkpoint_save_time.py [--out FILE]
"""
import argparse
import json
import os
import shutil
import statistics
import subprocess
import sys
import tempfile
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import dpt_b200  # noqa: E402,F401
from dpt_b200 import checkpoint as C, collect_data, train as TR  # noqa: E402
from dpt_b200.dataset import Dataset  # noqa: E402
from dpt_b200.models.net import Transformer  # noqa: E402

N_ENVS, H, D, L = 100000, 500, 5, 4


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i",
                        str(torch.cuda.current_device())], capture_output=True, text=True)
    return q.stdout.strip() or torch.cuda.get_device_name()


def model(seed):
    torch.manual_seed(seed)
    return Transformer({"horizon": H, "state_dim": 1, "action_dim": D, "n_layer": L, "n_embd": 32, "n_head": 1, "dropout": 0.0,
                        "test": False}).cuda()


def run(k, tr, te, warm_tr, warm_te, tmp):
    models = [model(i) for i in range(k)]
    seeds = list(range(k))
    TR.train_population(models, warm_tr, warm_te, 1, seeds=seeds)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    _, _, opt = TR.train_population(models, tr, te, 1, seeds=seeds)
    torch.cuda.synchronize()
    epoch = time.perf_counter() - t0
    gens = [torch.Generator(device="cuda").manual_seed(s) for s in seeds]
    args = C.train_args(64, [1e-3] * k, [1e-4] * k, seeds, [tr] * k, [te] * k, "cuda")
    path = os.path.join(tmp, "state_k%d.pt" % k)
    saves = []
    for _ in range(5):
        t0 = time.perf_counter()
        C.save_state(path, C.training_state("population", models, opt, args, 1, {"train_loss": [[0.0]] * k,
                                                                               "test_loss": [[0.0]] * k}, gens))
        saves.append(time.perf_counter() - t0)
    save = statistics.median(saves)
    return {"k": k, "epoch_s": epoch, "save_ms": save * 1e3, "save_ms_all": [s * 1e3 for s in saves],
            "state_bytes": os.path.getsize(path), "save_over_epoch": save / epoch}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out")
    a = ap.parse_args()
    batch = collect_data.collect_bandit(N_ENVS, D, H, 0.3, seed=0)
    cfg = {"horizon": H, "state_dim": 1, "action_dim": D, "shuffle": True, "store_gpu": True}
    n_tr = N_ENVS * 4 // 5
    tr = Dataset.from_batch({k: v[:n_tr] for k, v in batch.items()}, cfg)
    te = Dataset.from_batch({k: v[n_tr:] for k, v in batch.items()}, cfg)
    warm_tr = Dataset.from_batch({k: v[:640] for k, v in batch.items()}, cfg)
    warm_te = Dataset.from_batch({k: v[640:800] for k, v in batch.items()}, cfg)
    tmp = tempfile.mkdtemp(prefix="dpt_ckpt_time_")
    try:
        rows = [run(k, tr, te, warm_tr, warm_te, tmp) for k in (1, 16)]
    finally:
        shutil.rmtree(tmp)
    out = {"card": card(), "workload": "bandit %d envs (80/20), H=%d, d=%d, %d layers, batch 64" % (N_ENVS, H, D, L),
           "rows": rows}
    line = json.dumps(out)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
