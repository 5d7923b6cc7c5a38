#!/usr/bin/env python
"""Multi-GPU check of the data-parallel interactive trainer, run under torchrun on the GPU box:
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port 29512 \\
        scripts/interactive_train_check.py [--precision 0|1]
Every rank trains the same model for 3 iterations with dist.train_interactive_sharded; the weights and losses of all
ranks must be bit-identical, and rank 0 checks them against train.train_interactive (world size 1) of the same problem on
its own GPU, both at the training precision ``--precision`` (default 0 = fp32, 1 = bf16).  Cases: N divisible by
mb * world, a ragged last micro-batch, ranks that own no micro-batch, and N = 6000 (one GPU runs the register-staged decode kernel in the rollout, the shards the bulk-copy one).
With more ranks than GPUs the ranks share the GPUs round-robin and the host collectives go over gloo (NCCL takes one
rank per GPU); the slots are still exchanged through CUDA IPC mappings, of the same device."""
import argparse
import os
import sys

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import dpt_b200  # noqa: E402,F401
from dpt_b200 import dist as D, train as TR  # noqa: E402
from dpt_b200.models.net import Transformer  # noqa: E402

D_ARMS, L, ITERS, SEED, VAR = 5, 2, 3, 17, 0.3


def model(K):
    torch.manual_seed(0)
    m = Transformer({"horizon": K, "state_dim": 1, "action_dim": D_ARMS, "n_layer": L, "n_embd": 32, "n_head": 1, "dropout": 0.0,
                     "test": True}).cuda()
    with torch.no_grad():
        for k, p in m.named_parameters():
            if "wte" not in k:
                p.add_(0.15 * torch.randn_like(p))
    return m


def flat(m):
    return torch.cat([p.detach().reshape(-1) for p in m.parameters()])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--precision", type=int, default=0, choices=(0, 1))
    precision = ap.parse_args().precision
    rank, ws, lr = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    n_gpus = torch.cuda.device_count()
    torch.cuda.set_device(lr % n_gpus)
    if ws <= n_gpus:
        dist.init_process_group("nccl", device_id=torch.device("cuda", lr))
    else:
        dist.init_process_group("gloo")
    mb = 256
    cases = {"divisible": (2 * mb * ws, mb, 24), "ragged": (2 * mb * ws - 100, mb, 24),
             "idle ranks": (mb * (ws - 1) - 7, mb, 24), "bulk-copy shards": (6000, 1024, 24)}
    ok, report = True, []
    for name, (N, b, K) in cases.items():
        m = model(K)
        losses, _ = D.train_interactive_sharded(m, D_ARMS, N, K, ITERS, mb=b, var=VAR, seed=SEED, precision=precision)
        w = flat(m).cpu()
        allw = [None] * ws
        dist.all_gather_object(allw, (w, losses))
        same_ranks = all(torch.equal(allw[0][0], x) and x_l == allw[0][1] for x, x_l in allw)
        same_one = True
        if rank == 0:
            m1 = model(K)
            losses1, _ = TR.train_interactive(m1, D_ARMS, N, K, ITERS, mb=b, var=VAR, seed=SEED, precision=precision)
            same_one = torch.equal(flat(m1).cpu(), w) and losses1 == losses
            report.append("%s (N=%d, mb=%d): ranks %s, one GPU %s, losses %s" % (
                name, N, b, "same" if same_ranks else "DIFFER", "same" if same_one else "DIFFER",
                ["%.6f" % x for x in losses]))
        ok &= same_ranks and same_one
        dist.barrier()
    if rank == 0:
        print("\n".join(report))
        print("training precision %d" % precision)
        print("interactive_train_check world=%d gpus=%d: %s" % (ws, min(ws, n_gpus), "OK" if ok else "MISMATCH"))
    dist.barrier()
    dist.destroy_process_group()
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
