#!/usr/bin/env python
"""Multi-GPU check of resuming the interactive trainer across world sizes, run under torchrun on the GPU box:
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port 29513 \\
        scripts/checkpoint_resume_check.py
Rank 0 trains 3 of 5 iterations with train.train_interactive (world size 1) and saves the training state; every rank
resumes it with dist.train_interactive_sharded to 5 iterations.  Then every rank trains 3 iterations sharded (rank 0
saves) and rank 0 resumes that state at world size 1.  Every result, weights and losses, must be bit-identical to the
uninterrupted one-GPU run of 5 iterations.  The resumed runs start from other initial weights than the saved ones, so
everything they end with comes from the file.  Cases: a ragged last micro-batch, and ranks that own no micro-batch.
With more ranks than GPUs the ranks share the GPUs round-robin and the host collectives go over gloo."""
import os
import shutil
import sys
import tempfile

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import dpt_b200  # noqa: E402,F401
from dpt_b200 import dist as D, train as TR  # noqa: E402
from dpt_b200.models.net import Transformer  # noqa: E402

D_ARMS, L, K, SEED, VAR, ITERS, CUT = 5, 2, 24, 17, 0.3, 5, 3


def model(init):
    torch.manual_seed(init)
    m = Transformer({"horizon": K, "state_dim": 1, "action_dim": D_ARMS, "n_layer": L, "n_embd": 32, "n_head": 1, "dropout": 0.0,
                     "test": True}).cuda()
    with torch.no_grad():
        for k, p in m.named_parameters():
            if "wte" not in k:
                p.add_(0.15 * torch.randn_like(p))
    return m


def flat(m, opt):
    """Every weight and every AdamW state tensor (step included), on the host."""
    ts = [p.detach().reshape(-1) for p in m.parameters()]
    ts += [opt.state[p][n].reshape(-1).to(ts[0].device, torch.float32) for p in m.parameters() if p in opt.state
           for n in ("step", "exp_avg", "exp_avg_sq")]
    return torch.cat(ts).cpu()


def main():
    rank, ws, lr = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    n_gpus = torch.cuda.device_count()
    torch.cuda.set_device(lr % n_gpus)
    if ws <= n_gpus:
        dist.init_process_group("nccl", device_id=torch.device("cuda", lr))
    else:
        dist.init_process_group("gloo")
    box = [tempfile.mkdtemp(prefix="dpt_ckpt_") if rank == 0 else None]
    dist.broadcast_object_list(box, src=0)
    mb = 256
    cases = {"ragged": (2 * mb * ws - 100, mb), "idle ranks": (mb * (ws - 1) - 7, mb)}
    ok, report = True, []
    for c, (name, (N, b)) in enumerate(cases.items()):
        kw = dict(mb=b, var=VAR, seed=SEED)
        one, sharded = os.path.join(box[0], "one_%d.pt" % c), os.path.join(box[0], "sharded_%d.pt" % c)
        if rank == 0:
            ref = model(0)
            ref_losses, ref_opt = TR.train_interactive(ref, D_ARMS, N, K, ITERS, **kw)
            ref = (flat(ref, ref_opt), ref_losses)
            TR.train_interactive(model(0), D_ARMS, N, K, CUT, state_path=one, **kw)
        dist.barrier()
        m = model(1)                       # world size 1 -> sharded
        losses, opt = D.train_interactive_sharded(m, D_ARMS, N, K, ITERS, state_path=one, resume=True, **kw)
        got = [None] * ws
        dist.all_gather_object(got, (flat(m, opt), losses))
        D.train_interactive_sharded(model(0), D_ARMS, N, K, CUT, state_path=sharded, **kw)
        dist.barrier()
        if rank == 0:                      # sharded -> world size 1
            m = model(2)
            losses, opt = TR.train_interactive(m, D_ARMS, N, K, ITERS, state_path=sharded, resume=True, **kw)
            same_up = all(torch.equal(w, ref[0]) and l == ref[1] for w, l in got)
            same_down = torch.equal(flat(m, opt), ref[0]) and losses == ref[1]
            report.append("%s (N=%d, mb=%d): one GPU -> %d ranks %s, %d ranks -> one GPU %s, losses %s" % (
                name, N, b, ws, "same" if same_up else "DIFFER", ws, "same" if same_down else "DIFFER",
                ["%.6f" % x for x in ref[1]]))
            ok &= same_up and same_down
        dist.barrier()
    flag = [ok]
    dist.broadcast_object_list(flag, src=0)
    if rank == 0:
        shutil.rmtree(box[0])
        print("\n".join(report))
        print("checkpoint_resume_check world=%d gpus=%d: %s" % (ws, min(ws, n_gpus), "OK" if flag[0] else "MISMATCH"))
    dist.barrier()
    dist.destroy_process_group()
    sys.exit(0 if flag[0] else 1)


if __name__ == "__main__":
    main()
