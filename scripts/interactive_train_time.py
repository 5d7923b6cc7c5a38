"""One iteration of the interactive trainer (train.train_interactive / dist.train_interactive_sharded) at the fork's
scale, on 1, 2, 4 and 8 GPUs (as many as the box has), each world size under torch.distributed.run:

    python scripts/interactive_train_time.py [--out FILE] [--iters 5] [--warmup 2] [--precision 0 1]
                                             [--rollout-precision 0 1] [--rounds 3]

Problem: d = 5 arms, 4 layers, n_embd 32, N = 100 000 envs per iteration, micro-batches of 1024 envs, K = 100 and
K = 500.  Per world size, K, rollout precision (``model.precision``, ``--rollout-precision``) and training precision
(the ``precision`` argument, ``--precision``): the median over ``--iters`` iterations (after ``--warmup``) of every round
of the CUDA-event phases the trainer records (rollout, forward + backward of all micro-batches, exchange = host barrier to
the end of the ordered sum, AdamW, whole iteration), per rank and the slowest rank.  The training precisions alternate
within each of ``--rounds`` rounds, in one process, so that they see the same card state; with two of them the ratio of
their phase times is recorded too.  Comparison arm, one GPU, N = 8192: the same iteration composed
from the step-by-step pieces (``Transformer.decoder`` + ``GPUBanditEnv.step`` per step, then one whole-batch
``forward_train``) against ``train_interactive`` at that N.  The card's name and power limit are read in the same run.
Writes one JSON file (default: profiles/r06_interactive_train_time.json) and prints it.
"""
import argparse
import json
import os
import socket
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import torch  # noqa: E402

D_ARMS, L, VAR, SEED, N, MB, KS = 5, 4, 0.3, 2024, 100_000, 1024, (100, 500)
N_COMPOSED = 8192
PHASES = ("rollout", "fwd_bwd", "exchange", "optimizer", "total")


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        rows = [[x.strip() for x in r.split(",")] for r in q]
        return {"name": rows[0][0], "power_limit": sorted({r[1] for r in rows}), "max_sm_clock": rows[0][2], "gpus": len(rows)}
    except Exception as e:   # noqa: BLE001
        return {"name": torch.cuda.get_device_name(0), "error": repr(e)}


def model(K):
    from dpt_b200.models.net import Transformer
    torch.manual_seed(0)
    return Transformer({"horizon": K, "state_dim": 1, "action_dim": D_ARMS, "n_layer": L, "n_embd": 32, "n_head": 1,
                        "dropout": 0.0, "test": True}).cuda()


def med(rows):
    return {k: float(np.median([r[k] for r in rows])) for k in PHASES}


def case(args, K, rollout_precision):
    """The timed runs of one K and rollout precision on this rank: {training precision: (timings, losses of round 0)}."""
    from dpt_b200 import dist as D
    runs = {p: ([], None) for p in args.precision}
    for _ in range(args.rounds):
        for p in args.precision:
            m, tm = model(K), []
            m.precision = rollout_precision
            losses, _ = D.train_interactive_sharded(m, D_ARMS, N, K, args.warmup + args.iters, mb=MB, var=VAR, seed=SEED,
                                                    timings=tm, precision=p)
            runs[p] = (runs[p][0] + tm[args.warmup:], runs[p][1] or losses)
            del m
            torch.cuda.empty_cache()
    return runs


def worker(args):
    """One rank of one world size (under torch.distributed.run): rank 0 writes the gathered timings to args.worker."""
    import torch.distributed as dist
    import dpt_b200  # noqa: F401
    from dpt_b200 import dist as D
    rank, ws, lr = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(lr)
    dist.init_process_group("nccl", device_id=torch.device("cuda", lr))
    out = {"world": ws}
    _, _, lo, hi = D.microbatch_shard(N, MB, rank, ws)
    envs = [None] * ws
    dist.all_gather_object(envs, hi - lo)
    for K in KS:
        res = out["K%d" % K] = {"envs_per_rank": envs}
        for rp in args.rollout_precision:
            t0 = time.perf_counter()
            runs = case(args, K, rp)
            wall = time.perf_counter() - t0
            r = res["rollout_precision_%d" % rp] = {"wall_s_all_runs_rank0": wall}
            for p, (tm, losses) in runs.items():
                per_rank = [None] * ws
                dist.all_gather_object(per_rank, tm)
                meds = [med(x) for x in per_rank]
                r["precision_%d" % p] = {"median_ms_rank0": meds[0],
                                         "median_ms_slowest_rank": {k: max(x[k] for x in meds) for k in PHASES},
                                         "exchange_share_rank0": meds[0]["exchange"] / meds[0]["total"], "losses": losses,
                                         "iterations_ms_rank0": per_rank[0]}
            if set(args.precision) == {0, 1}:
                a, b = r["precision_1"]["median_ms_rank0"], r["precision_0"]["median_ms_rank0"]
                r["precision_1_over_0_rank0"] = {k: a[k] / b[k] for k in PHASES}
    if rank == 0:
        with open(args.worker, "w") as f:
            json.dump(out, f)
    dist.barrier()
    dist.destroy_process_group()


def composed_iteration(m, opt, n, K, it):
    """train_interactive's iteration from the step-by-step pieces (the reference's loop, train_interactive.py:97-139)."""
    from dpt_b200 import rng, train as TR
    from dpt_b200.envs.gpu_bandit_env import GPUBanditEnv
    env = GPUBanditEnv(D_ARMS, n, K, VAR, "uniform", seed=rng.key_for(SEED, it))
    dec = m.decoder(n, K)
    ctx = {k: torch.zeros((n, K, w), device="cuda") for k, w in (("context_states", 1), ("context_actions", D_ARMS),
                                                                 ("context_next_states", 1), ("context_rewards", 1))}
    state = env.reset()
    for t in range(K):
        logits = dec.query(state) if t == 0 else dec.append(*(ctx[k][:, t - 1] for k in ctx))
        action = torch.nn.functional.one_hot(torch.distributions.Categorical(logits=logits).sample(), D_ARMS).float()
        next_state, reward, _, _ = env.step(action)
        ctx["context_states"][:, t] = state
        ctx["context_actions"][:, t] = action
        ctx["context_next_states"][:, t] = next_state
        ctx["context_rewards"][:, t, 0] = reward
        state = next_state
    b = {k: v[:, :K - 1] for k, v in ctx.items()}
    b["query_states"] = torch.ones((n, 1), device="cuda")
    opt.zero_grad()
    loss = TR.interactive_loss(m.forward_train(b), env.opt_a_index, n)
    loss.backward()
    opt.step()
    return loss.detach()


def composed_arm(args):
    import dpt_b200  # noqa: F401
    from dpt_b200 import train as TR
    res = {"N": N_COMPOSED, "mb_fused": MB}
    for K in KS:
        m = model(K)
        opt = torch.optim.AdamW(m.parameters(), lr=1e-3, weight_decay=1e-4)
        ts = []
        for it in range(args.warmup + args.iters):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            composed_iteration(m, opt, N_COMPOSED, K, it)
            b.record()
            b.synchronize()
            ts.append(a.elapsed_time(b))
        del m, opt
        torch.cuda.empty_cache()
        m, tm = model(K), []
        TR.train_interactive(m, D_ARMS, N_COMPOSED, K, args.warmup + args.iters, mb=MB, var=VAR, seed=SEED, timings=tm)
        fused = med(tm[args.warmup:])
        res["K%d" % K] = {"composed_ms": float(np.median(ts[args.warmup:])), "fused_median_ms": fused,
                          "speedup": float(np.median(ts[args.warmup:])) / fused["total"]}
        del m
        torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r06_interactive_train_time.json"))
    ap.add_argument("--iters", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--precision", type=int, nargs="+", default=[0], choices=(0, 1),
                    help="training precisions, alternated within each round")
    ap.add_argument("--rollout-precision", type=int, nargs="+", default=[0], choices=(0, 1),
                    help="model.precision values, the precision of the rollout")
    ap.add_argument("--rounds", type=int, default=1)
    ap.add_argument("--worker", default=None, help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.worker:
        return worker(args)
    if not torch.cuda.is_available():
        raise SystemExit("interactive_train_time.py measures on the GPU; no CUDA device found")
    n_gpus = torch.cuda.device_count()
    res = {"gpu": gpu_info(), "config": {"d": D_ARMS, "n_layer": L, "n_embd": 32, "N": N, "mb": MB, "K": list(KS), "var": VAR,
                                         "iters": args.iters, "warmup": args.warmup, "rounds": args.rounds,
                                         "precision": args.precision, "rollout_precision": args.rollout_precision},
           "worlds": {}}
    with tempfile.TemporaryDirectory() as tmp:
        for ws in (1, 2, 4, 8):
            if ws > n_gpus:
                res["worlds"][str(ws)] = "not measured: %d GPUs on this box" % n_gpus
                continue
            with socket.socket() as s:
                s.bind(("127.0.0.1", 0))
                port = s.getsockname()[1]
            path = os.path.join(tmp, "w%d.json" % ws)
            cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(ws), "--master-addr",
                   "127.0.0.1", "--master-port", str(port), os.path.abspath(__file__), "--worker", path,
                   "--iters", str(args.iters), "--warmup", str(args.warmup), "--rounds", str(args.rounds),
                   "--precision", *map(str, args.precision), "--rollout-precision", *map(str, args.rollout_precision)]
            r = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True, timeout=3000)
            if r.returncode != 0:
                raise SystemExit("world %d failed:\n%s\n%s" % (ws, r.stdout[-3000:], r.stderr[-3000:]))
            with open(path) as f:
                res["worlds"][str(ws)] = json.load(f)
    res["composed_vs_fused_one_gpu"] = composed_arm(args)
    res["gpu_after"] = gpu_info()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
