#!/usr/bin/env python
"""bench.py -- both halves of BASELINE.json's metric for the DPT rollout hot path on B200.

Headline (``metric`` / ``value``): rollout-collection env-steps/s.  Workload = BASELINE.json configs[4]'s
per-GPU shard, the configuration the env-steps/s target is quoted on: bandit rollin_bandit collection,
H=500, dim=5, var=0.3, 125 000 envs per GPU (weak scaling: 1M envs on 8 GPUs), Philox noise, outputs in
the reference consumer's fp32 layout (32 B per env-step, 2 GB per step per GPU -- larger than the 126 MB
L2, so no flush is needed between steps).  A "step" is one pass of the fused kernel over the GPU's env shard.

Second half (``online_eval`` block, measured at EVERY N): online in-context evaluation trajectories/s --
BASELINE.json configs[3]: deploy_online_vec with the GPT-2 (embd 32, 4 layers, 1 head) transformer
controller, H=500, sample=True, K/V-cached fused loop, fp32 and bf16 K/V, weak-scaled (10 000 envs per GPU)
and strong-scaled (10 000 envs in total), the [H,4] regret-sum all-reduce inside the timed region, with a
roofline block (K/V bytes / event time / measured HBM peak), an end-to-end figure through
``dist.online_eval_sharded`` (host means in, host regret curves out) and the reference's own
deploy_online_vec + BanditTransformerController timed on the host cores at reduced N.

    python bench.py [--gpus N --steps K --warmup W] [--impl reference] [--workload collect|online_eval] [--dump-outputs DIR]

Prints ONE JSON line (rank 0).  See DESIGN.md "Measurement" for every field.  --dump-outputs DIR writes what the
collection's last timed step returned as DIR/<name>.npy (see dump_outputs), so that two builds can be compared
output for output: with the same arguments the inputs are identical from run to run.
"""
import argparse
import json
import os
import statistics
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

H, DIM, VAR = 500, 5, 0.3
ENVS_PER_GPU = int(os.environ.get("DPT_BENCH_ENVS", 125000))
BYTES_PER_STEP = 4 * (2 * 1 + DIM + 1)          # SURVEY.md §8d: four fp32 context rows per env-step
METRIC = "env-steps/sec (bandit rollout collect, H=500 dim=5)"
UNIT = "env-steps/s"
OE_ENVS = int(os.environ.get("DPT_BENCH_OE_ENVS", 10000))    # BASELINE configs[3]: 10k envs
OE_LAYERS, OE_EMBD = 4, 32
OE_METRIC = "online-eval trajs/sec (deploy_online_vec, GPT-2 embd=32 layer=4 head=1 controller, H=500 dim=5)"
DUMP_ENVS = 2048     # envs in the --dump-outputs sample: 2048 x H=500 x 32 B = 31 MiB of the 2 GB a step writes


def workload_name(n_gpus):
    return ("bandit rollin_bandit collection H=%d dim=%d var=%.1f, %d envs/GPU x %d GPU (BASELINE configs[4] shard), "
            "outputs %.2f GB/step/GPU > L2 (no flush needed)" % (H, DIM, VAR, ENVS_PER_GPU, n_gpus,
                                                                  ENVS_PER_GPU * H * BYTES_PER_STEP / 1e9))


def load_peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:   # noqa: BLE001
        return {}


# ----------------------------------------------------------------------------- clocks ---------
class ClockSampler:
    """Samples SM clock and throttle reasons of one GPU via NVML while the timed region runs."""
    BITS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap",
            0x80: "hw_power_brake_slowdown", 0x2: "applications_clocks_setting", 0x10: "sync_boost"}

    def __init__(self, uuid):
        self.samples, self.reasons, self.max_mhz, self._stop, self.ok = [], set(), None, threading.Event(), False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            try:
                self.h = pynvml.nvmlDeviceGetHandleByUUID(uuid.encode() if isinstance(uuid, str) else uuid)
            except Exception:
                self.h = pynvml.nvmlDeviceGetHandleByIndex(0)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.ok = True
        except Exception as e:   # noqa: BLE001
            self.err = repr(e)

    def _once(self):
        nv = self.nv
        self.samples.append(float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
        try:
            m = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
        except Exception:
            m = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
        for bit, name in self.BITS.items():
            if m & bit:
                self.reasons.add(name)

    def _loop(self):
        while not self._stop.is_set():
            self._once()
            time.sleep(0.002)

    def start(self):
        if self.ok:
            self._once()
            self.t = threading.Thread(target=self._loop, daemon=True)
            self.t.start()
        return self

    def stop(self):
        if self.ok:
            self._stop.set()
            self.t.join()
            self._once()

    def summary(self):
        if not self.ok or not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [], "note": "nvml unavailable"}
        return {"sm_mhz": statistics.median(self.samples), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(self.samples)}


# ----------------------------------------------------------------------------- CPU legs -------
def _rate(r, per="env_steps"):
    return r[per] / r["wall"]


def cpu_collect_leg(pool, seconds):
    """Headline CPU figure: the reference's own generate_bandit_histories on every host core (kind 'reference'
    when baseline/_ref is staged, else the oracle port), sized for ~`seconds` of wall time; plus the port."""
    probe = pool.run("bandit", 20, H, dim=DIM, var=VAR)
    epc = max(20, int(20 * seconds / max(probe["worker_s"], 1e-3)))
    r = pool.run("bandit", epc, H, seed0=100, dim=DIM, var=VAR)
    what = ("collect_data.generate_bandit_histories of the unmodified reference (baseline/_ref)" if r["kind"] == "reference"
            else "oracle port of collect_data.generate_bandit_histories")
    out = {"value": _rate(r), "unit": UNIT, "cores": r["cores"], "kind": r["kind"],
           "sample": "%d cores x %d envs x H=%d, %s, one process per core (%.2f s wall, %.2f s mean per worker)" % (
               r["cores"], epc, H, what, r["wall"], r["worker_s"])}
    if r["kind"] == "reference":
        p = pool.run("bandit", 1500, H, seed0=200, kind="port", dim=DIM, var=VAR)
        out["port_value"] = _rate(p)
        out["port_note"] = ("oracle port (numpy restatement, bit-identical outputs): %.1fx the reference per core -- it builds the "
                            "categorical cdf once per env instead of np.random.choice re-validating p at every draw" % (
                                _rate(p) / max(out["value"], 1e-9)))
    return out


def cpu_online_leg(pool, n_per_core=None):
    """The reference's deploy_online_vec + BanditTransformerController (full recompute, no K/V cache) at reduced N."""
    if pool.kind != "reference":
        return None
    n = max(2, n_per_core or int(os.environ.get("DPT_CPU_OE_ENVS_PER_CORE", 2)))   # the reference controller needs batch_size >= 2
    r = pool.run("gpt2_online", n, H, seed0=300, dim=DIM, var=VAR)
    return {"value": _rate(r, "trajs"), "unit": "trajs/s", "env_steps_per_s": _rate(r), "cores": r["cores"], "kind": "reference",
            "sample": "%d cores x %d envs x H=%d, evals/eval_bandit.deploy_online_vec + ctrls.BanditTransformerController(sample=True) of "
                      "the unmodified reference, GPT-2 embd=32 layer=4 random init, one process per core, torch threads=1 "
                      "(%.2f s wall)" % (r["cores"], n, H, r["wall"])}


def cpu_other_legs(pool):
    """Reference CPU timings of configs 2, 3a, 3b and config 4's classical controllers at reduced N (SURVEY.md §8d)."""
    if pool.kind != "reference":
        return None
    out = {}
    for name, wl, n, hh, extra in (
            ("config2_darkroom_rollin_H100", "darkroom", 400, 100, dict(dim=10)),
            ("config3_linear_thompson_collect_H200_d10", "lin_thomp", 60, 200, dict(dim=10, lin_d=2, var=VAR)),
            ("config3_linucb_online_H200_d10", "lin_ucb", 60, 200, dict(dim=10, lin_d=2, var=VAR)),
            ("config4_emp_online_H500_d5", "emp", 40, H, dict(dim=DIM, var=VAR)),
            ("config4_thompson_online_H500_d5", "thompson", 20, H, dict(dim=DIM, var=VAR)),
            ("darkroom_online_eval_dim10_H100_Heps4", "darkroom_online", 4, 100, dict(dim=10, horizon=100, Heps=4))):
        r = pool.run(wl, n, hh, seed0=400, **extra)
        out[name] = {"env_steps_per_s": _rate(r), "trajs_per_s": _rate(r, "trajs"), "cores": r["cores"], "kind": "reference",
                     "sample": "%d cores x %d envs x H=%d (%.2f s wall)" % (r["cores"], n, hh, r["wall"])}
    return out


def run_reference(args, rank):
    """--impl reference: the reference's own CPU implementation of the path on all host cores (one process per
    core).  Live reference from baseline/_ref when staged (kind 'reference'), else its oracle port."""
    if rank != 0:
        return
    from oracle import cpu_bench
    pool = cpu_bench.CpuPool()
    epc = int(os.environ.get("DPT_REF_ENVS_PER_CORE", 40 if pool.kind == "reference" else 400))
    for _ in range(min(args.warmup, 2)):
        pool.run("bandit", 4, H, dim=DIM, var=VAR)
    tot_steps, t0 = 0, time.perf_counter()
    for i in range(args.steps):
        r = pool.run("bandit", epc, H, seed0=1000 * (i + 1), dim=DIM, var=VAR)
        tot_steps += r["env_steps"]
    wall = time.perf_counter() - t0
    v = tot_steps / wall
    what = "collect_data.generate_bandit_histories of the unmodified reference (baseline/_ref)" if pool.kind == "reference" \
        else "oracle port of collect_data.generate_bandit_histories"
    sample = "%d cores x %d envs x H=%d per step, %s" % (pool.cores, epc, H, what)
    line = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * wall / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": workload_name(args.gpus), "sample": sample},
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": pool.cores, "kind": pool.kind, "sample": sample},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    oe = cpu_online_leg(pool)
    if oe is not None:
        line["online_eval"] = {"metric": OE_METRIC, "value": oe["value"], "unit": "trajs/s", "cpu_baseline": oe,
                               "e2e": {"value": oe["value"], "unit": "trajs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    pool.close()
    print(json.dumps(line))


# ----------------------------------------------------------------------------- GPU helpers ----
def time_events(torch, fn, reps, warm):
    for i in range(warm):
        fn(i)
    torch.cuda.synchronize()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(reps + 1)]
    ev[0].record()
    for i in range(reps):
        fn(warm + i)
        ev[i + 1].record()
    torch.cuda.synchronize()
    return [ev[i].elapsed_time(ev[i + 1]) for i in range(reps)], ev[0].elapsed_time(ev[reps])


def dump_outputs(path, out, stats):
    """Writes what one bandit_rollin step returned as path/<name>.npy: the four fp32 context arrays [n, H, *] at a fixed
    sample of DUMP_ENVS envs of this rank's shard (np.random.RandomState(0), in ascending env order; every env when the
    shard is smaller) and, when the step accumulated them, its float64 return statistics [3]."""
    import numpy as np
    import torch
    os.makedirs(path, exist_ok=True)
    first = next(iter(out.values()))
    n = first.shape[0]
    idx = np.sort(np.random.RandomState(0).choice(n, min(n, DUMP_ENVS), replace=False))
    rows = torch.as_tensor(idx, device=first.device)
    arrays = {name: t.index_select(0, rows) for name, t in out.items()}
    if stats is not None:
        arrays["return_stats"] = stats
    for name, t in arrays.items():
        np.save(os.path.join(path, name + ".npy"), t.cpu().numpy())


def other_workloads(kernels, torch):
    """The other BASELINE.json configs on one GPU (informational; CUDA events, 3 warm-up + 5 timed runs each)."""
    import numpy as np

    def t(fn, reps=5, warm=3):
        per, _ = time_events(torch, lambda i: fn(), reps, warm)
        return statistics.mean(per)
    peak = float(load_peaks().get("hbm_gbs", 6650.0))
    out = {}
    goals = torch.tensor(np.repeat(np.stack(np.meshgrid(np.arange(10), np.arange(10), indexing="ij"), -1).reshape(-1, 2), 1000, 0),
                         dtype=torch.int32, device="cuda")
    ms = t(lambda: kernels.darkroom_rollin(goals, 10, 100, "uniform", 1, 0, None, 1))
    out["config2_darkroom_rollin_100k_envs_H100"] = {"ms": ms, "env_steps_per_s": 1e7 / (ms * 1e-3), "gbs": 4e8 / (ms * 1e-3) / 1e9,
                                                     "frac_of_hbm_peak": 4e8 / (ms * 1e-3) / 1e9 / peak}
    means10, _, _ = kernels.bandit_sample_means(100000, 10, 0, 0)
    arms = torch.tensor(np.random.RandomState(1234).normal(size=(10, 2)) / np.sqrt(2), dtype=torch.float64, device="cuda")
    ms = t(lambda: kernels.online_loop("thompson", means10, 200, 0.3, 1, 0, p0=0.3, p1=0.0, p2=1.0))
    out["config3_linear_thompson_collect_100k_envs_H200_d10"] = {"ms": ms, "env_steps_per_s": 2e7 / (ms * 1e-3), "trajs_per_s": 1e5 / (ms * 1e-3),
                                                                 "frac_of_hbm_peak": 2e7 * 56 / (ms * 1e-3) / 1e9 / peak}
    ms = t(lambda: kernels.online_loop("linucb", means10, 200, 0.3, 1, 0, p0=1.0, arms=arms))
    out["config3_linucb_online_100k_envs_H200_d10"] = {"ms": ms, "env_steps_per_s": 2e7 / (ms * 1e-3), "trajs_per_s": 1e5 / (ms * 1e-3),
                                                       "frac_of_hbm_peak": 2e7 * 56 / (ms * 1e-3) / 1e9 / peak}
    means5, _, _ = kernels.bandit_sample_means(100000, 5, 0, 0)
    for kind, kw in (("emp", dict(p0=1.0)), ("ucb", dict(p0=1.0)), ("thompson", dict(p0=0.3, p1=0.5, p2=1 / 12.0))):
        ms = t(lambda: kernels.online_loop(kind, means5, 500, 0.3, 1, 0, **kw))
        out["config4_%s_online_100k_envs_H500_d5" % kind] = {"ms": ms, "env_steps_per_s": 5e7 / (ms * 1e-3), "trajs_per_s": 1e5 / (ms * 1e-3),
                                                             "frac_of_hbm_peak": 5e7 * 36 / (ms * 1e-3) / 1e9 / peak}
    # SURVEY.md §8 (f)4: the no-grad half of an explorer / exploiter episode (train_explorer_exploiter.py:110-166), 2 000 envs x K = 100
    # steps, two GPT-2 (embd 32, 4 layers) models: ONE fused launch against the step-by-step form (2 decode launches + torch ops per step)
    try:
        from dpt_b200.envs.gpu_bandit_env import GPUBanditEnv
        from dpt_b200.models.net import Transformer
        torch.manual_seed(1)
        cfg = {"horizon": 100, "state_dim": 1, "action_dim": 5, "n_layer": 4, "n_embd": 32, "n_head": 1, "dropout": 0.0, "test": True}
        ex, xp = Transformer(cfg), Transformer(cfg)
        genv = GPUBanditEnv(5, 2000, 100, var=0.3, seed=3)
        for fused, name in ((True, "fused"), (False, "step_by_step")):
            genv.rollout_explorer_exploiter(ex, xp, fused=fused)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(3):
                genv.rollout_explorer_exploiter(ex, xp, fused=fused)
            torch.cuda.synchronize()
            ms = (time.perf_counter() - t0) * 1e3 / 3
            out["explorer_exploiter_rollout_2000_envs_K100_%s" % name] = {"ms": ms, "env_steps_per_s": 2e5 / (ms * 1e-3),
                                                                          "timing": "wall clock around GPUBanditEnv.rollout_explorer_exploiter"}
    except Exception as e:   # noqa: BLE001
        out["explorer_exploiter_rollout"] = {"error": repr(e)}
    # SURVEY.md §8 (f)1: darkroom online evaluation (evals/eval_darkroom.py:20-84), the reference's shape: 100 envs x 40 episodes
    # of 100 steps on a 10 x 10 grid, context H = 100, GPT-2 embd 32 / 4 layers: per episode ONE dense forward over the 100
    # query states of every env (fp32 CUDA-core kernel, or tcgen05 with precision 1) + ONE rollout launch
    try:
        from dpt_b200.ctrls.ctrl_darkroom import DarkroomTransformerController
        from dpt_b200.envs.darkroom_env import DarkroomEnv, DarkroomEnvVec
        from dpt_b200.evals import eval_darkroom
        from dpt_b200.models.net import Transformer
        torch.manual_seed(0)
        dm = Transformer({"horizon": 100, "state_dim": 2, "action_dim": 5, "n_layer": 4, "n_embd": 32, "n_head": 1, "dropout": 0.0, "test": True})
        vec = DarkroomEnvVec([DarkroomEnv(10, (i % 10, (3 * i + 1) % 10), 100) for i in range(100)])
        for prec, name in ((0, "fp32"), (1, "tcgen05_bf16")):
            dm.precision = prec
            ctrl = DarkroomTransformerController(dm, batch_size=100, sample=True)
            eval_darkroom.deploy_online_vec(vec, ctrl, 2, 100, 100)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            eval_darkroom.deploy_online_vec(vec, ctrl, 40, 100, 100)
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            out["darkroom_online_eval_100_envs_40_episodes_" + name] = {"ms": 1e3 * dt, "env_steps_per_s": 100 * 40 * 100 / dt, "trajs_per_s": 100 / dt,
                                                                        "timing": "wall clock around evals.eval_darkroom.deploy_online_vec (returns on the host)"}
    except Exception as e:   # noqa: BLE001
        out["darkroom_online_eval"] = "failed: %s" % str(e)[:120]
    return out


def oe_bytes(n_envs, esz):
    """Algorithmic HBM bytes of one online-eval pass over n_envs envs (SURVEY.md §8d): K/V rows read by every
    token-forward (token h reads h cached rows per layer, K and V, 32 channels), K/V rows appended, and the 36 B of
    outputs (context row + cum_means) per env-step."""
    kv_read = n_envs * OE_LAYERS * 2 * OE_EMBD * esz * (H * (H - 1) // 2)
    kv_write = n_envs * OE_LAYERS * 2 * OE_EMBD * esz * H
    return kv_read + kv_write + n_envs * H * 36


def online_eval_block(args, torch, dist, rank, world, dev, pool):
    """Online-eval trajs/s at this N: config 4 weak- and strong-scaled, fp32 and bf16 K/V."""
    import dpt_b200
    from dpt_b200 import dist as ddist
    from dpt_b200 import kernels
    from dpt_b200.models.net import Transformer
    torch.manual_seed(0)
    model = Transformer({"horizon": H, "state_dim": 1, "action_dim": DIM, "n_layer": OE_LAYERS, "n_embd": OE_EMBD, "n_head": 1,
                         "dropout": 0.0, "test": True})
    peak = float(load_peaks().get("hbm_gbs", 6650.0))
    # --steps sets the timed passes when this block is the line's headline; as the secondary block it keeps its own count
    reps = args.steps if args.workload == "online_eval" else int(os.environ.get("DPT_BENCH_OE_STEPS", 3))
    block = {"metric": OE_METRIC, "unit": "trajs/s", "H": H, "dim": DIM, "var": VAR, "sample": True, "steps": reps, "warmup": 3,
             "model": "GPT-2 trunk embd=32 layer=4 head=1, random init (torch.manual_seed(0)), one token-forward per env-step on a per-env K/V cache",
             "l2": "K/V caches of a pass (%.2f GB fp32 / %.2f GB bf16 per 10k envs) exceed the 126 MB L2; no flush" % (
                 OE_ENVS * OE_LAYERS * 2 * OE_EMBD * 4 * 512 / 1e9, OE_ENVS * OE_LAYERS * 2 * OE_EMBD * 2 * 512 / 1e9),
             "exchange": "all-reduce (NCCL) of the [H,4] float64 regret sums inside the timed region" if world > 1 else "none (1 GPU)",
             "runs": {}}
    sampler = ClockSampler("GPU-" + str(torch.cuda.get_device_properties(dev).uuid)).start() if rank == 0 else None
    for scaling, total in (("weak", OE_ENVS * world), ("strong", OE_ENVS)):
        if scaling == "strong" and world == 1:
            block["runs"]["strong"] = "same as weak at 1 GPU"
            continue
        lo, hi = ddist.shard_range(total, rank, world)
        n_loc = hi - lo
        means, _, _ = kernels.bandit_sample_means(n_loc, DIM, 0, lo)
        for prec, pname, esz in ((0, "fp32", 4), (1, "bf16_kv", 2)):
            model.precision = prec
            sums_keep = []

            def step(i):
                out = model.online_loop(means, H, VAR, True, 1 + i, lo, True, True)
                sums_keep.append(ddist.all_reduce_sums(out["regret_sums"]))
            if world > 1:
                dist.barrier()
            per, tot_ms = time_events(torch, step, reps, 3)
            t = torch.tensor([tot_ms, statistics.mean(per)], dtype=torch.float64, device=dev)
            tmax = t.clone()
            if world > 1:
                dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
            tot_ms, ms_mean = float(tmax[0]), float(tmax[1])
            nbytes = oe_bytes(n_loc, esz)
            achieved = nbytes / (statistics.mean(per) * 1e-3) / 1e9
            curves = ddist.regret_stats_from_sums(sums_keep[-1].cpu().numpy(), total)
            block["runs"].setdefault(scaling, {})[pname] = {
                "value": total * reps / (tot_ms * 1e-3), "unit": "trajs/s", "env_steps_per_s": total * H * reps / (tot_ms * 1e-3),
                "envs_total": total, "envs_per_gpu": n_loc, "ms_per_pass": tot_ms / reps,
                "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                             "kernel": "gpt2_online_kernel<%s>" % pname, "algorithmic_bytes_per_launch": nbytes,
                             "launch_ms_mean": statistics.mean(per), "launch_ms_min": min(per), "traffic": None,
                             "note": "rank 0's launch (kernel + all-reduce of 16 KB); bytes = K/V rows read + appended + 36 B outputs per env-step"},
                "final_cumulative_regret_mean": float(curves["regret_mean"][-1])}
            del sums_keep[:]
    # end to end through the public sharded API: host means in (pinned), host regret curves out, every pass
    model.precision = 0
    total = OE_ENVS * world
    lo, hi = ddist.shard_range(total, rank, world)
    means_host = kernels.bandit_sample_means(hi - lo, DIM, 0, lo)[0].cpu().pin_memory()
    for i in range(2):
        ddist.online_eval_sharded("transformer", total, DIM, H, VAR, 50 + i, model=model, means_local=means_host)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for i in range(reps):
        _, curves = ddist.online_eval_sharded("transformer", total, DIM, H, VAR, 60 + i, model=model, means_local=means_host)
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    t = torch.tensor([wall], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    wall = float(t[0])
    block["e2e"] = {"value": total * reps / wall, "unit": "trajs/s", "h2d_bytes_per_step": (hi - lo) * DIM * 4,
                    "d2h_bytes_per_step": H * 4 * 8, "steps": reps, "ms_per_step": 1e3 * wall / reps, "precision": "fp32",
                    "api": "dist.online_eval_sharded('transformer', ...): pinned host means -> device, fused loop, all-reduce, [H,4] sums -> host curves"}
    if sampler:
        sampler.stop()
        block["clocks"] = sampler.summary()
    block["value"] = block["runs"]["weak"]["fp32"]["value"]
    block["scaling"] = "weak (10k envs/GPU) and strong (10k envs total) both reported; `value` = weak, fp32 (the reference's precision)"
    block["gpu_launches"] = reps * 2 * (2 if world > 1 else 1) + reps
    if rank == 0 and pool is not None:
        cb = cpu_online_leg(pool)
        if cb is not None:
            block["cpu_baseline"] = cb
    return block


# ----------------------------------------------------------------------------- our arm --------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="collect", choices=["collect", "online_eval"],
                    help="which half of the metric is the line's headline `value` (both are always measured)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--e2e-steps", type=int, default=None)
    ap.add_argument("--no-other", action="store_true", help="skip the secondary workloads (configs 2-4)")
    ap.add_argument("--no-online-eval", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the outputs of the collection's last timed step (rank 0's shard) "
                         "as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the GPU collection's outputs; it does not apply to --impl reference")
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    if args.impl == "reference":
        run_reference(args, rank)
        return
    args.warmup = max(args.warmup, 3)   # timing rule: at least 3 warm-up steps (the JSON line reports the value used)

    # CPU legs first (rank 0, N=1 only), before the GPU is busy: bounded samples on all host cores
    cpu_baseline, cpu_other, pool = None, None, None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        from oracle import cpu_bench
        pool = cpu_bench.CpuPool()
        cpu_baseline = cpu_collect_leg(pool, float(os.environ.get("DPT_CPU_SECONDS", 10)))
        if not args.no_other:
            cpu_other = cpu_other_legs(pool)

    import torch
    import torch.distributed as dist
    import dpt_b200
    from dpt_b200 import kernels
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    N = ENVS_PER_GPU
    env_id0 = rank * N                        # contiguous global env ranges (SURVEY.md §8e)
    seed = 0
    means, _, _ = kernels.bandit_sample_means(N, DIM, seed, env_id0)
    out = {"context_states": torch.empty((N, H, 1), device=dev), "context_actions": torch.empty((N, H, DIM), device=dev),
           "context_next_states": torch.empty((N, H, 1), device=dev), "context_rewards": torch.empty((N, H, 1), device=dev)}
    # per-step return statistics: one pre-zeroed slot per step, so the timed loop launches nothing but the
    # fused kernel (and, multi-GPU, the async NCCL gather of that step's [3] statistics, which overlaps the
    # next step's kernel)
    n_slots = args.steps + args.warmup
    stats = torch.zeros((n_slots, 3), dtype=torch.float64, device=dev)
    gathered = torch.zeros((n_slots, 3 * world), dtype=torch.float64, device=dev)
    pending = []
    peer, gather_how = None, "none"
    gather_mode = os.environ.get("DPT_BENCH_GATHER", "p2p")     # p2p | nccl | none (statistics off: attribution runs)
    if world > 1 and gather_mode != "none":
        from dpt_b200 import dist as ddist
        try:      # all-gather fused into the kernel: the last CTA stores the totals into every rank's buffer over NVLink
            if gather_mode != "p2p":
                raise RuntimeError("NCCL gather requested")
            peer = ddist.PeerGather(n_slots)
            gather_how = "all-gather of return stats over NVLink peer memory (CUDA IPC): a one-warp kernel behind each rollin launch stores the totals into every rank's buffer; no collective launch, no host sync"
        except Exception as e:   # noqa: BLE001
            peer = None
            gather_how = "NCCL all-gather of return stats every step (async) [p2p unavailable: %s]" % str(e)[:80]
    elif world > 1:
        gather_how = "DPT_BENCH_GATHER=none: return statistics and their exchange switched off (attribution run)"

    def step(i):
        if gather_mode == "none":
            kernels.bandit_rollin(means, H, VAR, seed + i, env_id0, out=out)
        elif peer is not None:
            kernels.bandit_rollin(means, H, VAR, seed + i, env_id0, out=out, stats=stats[i], peer=peer, peer_slot=i)
        else:
            kernels.bandit_rollin(means, H, VAR, seed + i, env_id0, out=out, stats=stats[i])
            if world > 1:   # every pass's statistics are gathered; the call is asynchronous (overlaps the next pass)
                pending.append(dist.all_gather_into_tensor(gathered[i], stats[i], async_op=True))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for i in range(args.warmup):
        step(i)
    barrier()
    sampler = ClockSampler("GPU-" + str(torch.cuda.get_device_properties(dev).uuid)) if rank == 0 else None
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
    if sampler:
        sampler.start()
    ev[0].record()
    for i in range(args.steps):
        step(args.warmup + i)
        ev[i + 1].record()
    for w_ in pending:      # the statistics exchange belongs to the timed region
        w_.wait()
    end_ev = torch.cuda.Event(enable_timing=True)
    end_ev.record()
    barrier()
    if sampler:
        sampler.stop()
    if args.dump_outputs and rank == 0:   # `out` still holds the last timed step's outputs
        dump_outputs(args.dump_outputs, out, stats[args.warmup + args.steps - 1] if gather_mode != "none" else None)
    total_ms = ev[0].elapsed_time(end_ev)
    per = [ev[i].elapsed_time(ev[i + 1]) for i in range(args.steps)]
    t = torch.tensor([total_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms = float(t[0])
    value = world * N * H * args.steps / (total_ms * 1e-3)
    # every rank's own mean launch time (attribution of multi-GPU efficiency: which rank is slow, by how much)
    mine = torch.tensor([statistics.mean(per)], dtype=torch.float64, device=dev)
    per_rank = [mine.clone() for _ in range(world)]
    if world > 1:
        dist.all_gather(per_rank, mine)
    per_rank = [float(x[0]) for x in per_rank]

    # roofline of the dominant kernel (bandit_rollin_fast<5>): algorithmic bytes / mean launch duration.
    # A step IS one launch of it, so the per-step event deltas are its launch durations.
    kern_ms = statistics.mean(per)
    peaks = load_peaks()
    peak = float(peaks.get("hbm_gbs", 6650.0))
    achieved = N * H * BYTES_PER_STEP / (kern_ms * 1e-3) / 1e9
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": None, "kernel": "bandit_rollin_fast<5,PHILOX>", "algorithmic_bytes_per_launch": N * H * BYTES_PER_STEP,
                "peak_source": "MEASURED_PEAKS.json hbm_gbs (of measured)" if peaks else "fallback 6650 GB/s (of fallback)",
                "launch_ms_mean": kern_ms, "launch_ms_min": min(per),
                "launch_ms_mean_per_rank": per_rank, "launch_ms_rank_min_max": [min(per_rank), max(per_rank)]}
    tfile = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tfile) and N == 125000:
        try:
            tj = json.load(open(tfile))
            roofline["traffic"] = tj.get("bandit_rollin_fast_dram_bytes_per_launch")
            roofline["traffic_source"] = ("NOT measured in this run: dram__bytes_read.sum + dram__bytes_write.sum of one `ncu --set full` "
                                          "capture of this kernel at this shape, committed as " + str(tj.get("source", "profiles/traffic.json")))
        except Exception:   # noqa: BLE001
            pass

    # e2e: the same collection through the host-buffer C-ABI call (means in pinned host memory,
    # contexts returned to pinned host memory), copies inside the timed region.
    e2e_steps = args.e2e_steps or max(3, min(args.steps, 10))
    means_host = means.cpu().pin_memory()
    host_out, scratch = kernels.bandit_rollin_host(means_host, H, VAR, seed, env_id0)
    for i in range(2):
        kernels.bandit_rollin_host(means_host, H, VAR, seed + i, env_id0, out=host_out, scratch=scratch)
    barrier()
    t0 = time.perf_counter()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    d2h_sum = 0
    for i in range(e2e_steps):
        kernels.bandit_rollin_host(means_host, H, VAR, seed + 100 + i, env_id0, out=host_out, scratch=scratch)
        d2h_sum += int(dpt_b200._lib.lib().dpt_bandit_rollin_host_last_d2h_bytes())
    e1.record()
    barrier()
    e2e_ms = max(e0.elapsed_time(e1), 1e3 * (time.perf_counter() - t0))
    t = torch.tensor([e2e_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_ms = float(t[0])
    e2e = {"value": world * N * H * e2e_steps / (e2e_ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": N * DIM * 4,
           # what crossed PCIe per timed call (mean over the timed calls of this rank): chunks returned by DMA carry
           # actions + rewards (4*(d+1) B per step), chunks returned in compact form 5 B per step (expanded by host
           # threads); the constant state columns are always written on the host
           "d2h_bytes_per_step": d2h_sum // e2e_steps, "steps": e2e_steps, "ms_per_step": e2e_ms / e2e_steps,
           "host_bytes_written_per_step": N * H * BYTES_PER_STEP,
           "api": "dpt_bandit_rollin_host (pinned host buffers, chunked H2D/kernel/D2H pipeline, hybrid DMA / host expansion)"}
    try:    # the host side of the e2e path is a pure memory-write stream: report it against the box's measured store peak
        # (non-temporal stores of this rank's share of the host cores into the SAME pinned output array, all ranks at once)
        n_thr = max(1, len(os.sched_getaffinity(0)) // max(1, int(os.environ.get("LOCAL_WORLD_SIZE", world))))
        hps = []
        for _ in range(3):      # three barrier-synchronised measurements (all ranks write at once); median of the sums
            barrier()
            t = torch.tensor([kernels.host_write_peak(buf=host_out["context_actions"], n_threads=n_thr)], dtype=torch.float64, device=dev)
            if world > 1:
                dist.all_reduce(t)
            hps.append(float(t[0]))
        hp = statistics.median(hps)
        e2e["host_write_peak_samples_gbs"] = hps
        e2e["host_write_peak_gbs"] = hp
        e2e["host_write_peak_note"] = "sum over ranks of dpt_host_write_peak into the pinned actions array, %d threads per rank, all ranks concurrently" % n_thr
        e2e["frac_of_host_peak"] = world * N * H * BYTES_PER_STEP * e2e_steps / (e2e_ms * 1e-3) / 1e9 / hp
    except Exception as e:   # noqa: BLE001
        e2e["host_write_peak_gbs"] = None
        e2e["host_write_peak_note"] = str(e)[:100]

    for w_ in pending:
        w_.wait()
    torch.cuda.synchronize()
    if gather_mode == "none":
        totals = None
    elif peer is not None:
        barrier()
        totals = torch.tensor(peer.read().sum((0, 1)))
        barrier()
        peer.close()
    elif world > 1:
        totals = gathered.view(-1, 3).sum(0)
    else:
        totals = stats.sum(0)
    del out, host_out, scratch
    torch.cuda.empty_cache()

    online = None
    if not args.no_online_eval:
        online = online_eval_block(args, torch, dist, rank, world, dev, pool)
    other = None
    if rank == 0 and world == 1 and not args.no_other:
        other = other_workloads(kernels, torch)
        if cpu_other:
            other["reference_cpu"] = cpu_other
    if pool is not None:
        pool.close()
    if rank == 0:
        n_tot = world * N * H * (args.steps + args.warmup)
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_name(world), "envs_per_gpu": N, "H": H, "dim": DIM, "var": VAR,
                       "noise": "philox4x32-10", "l2": "outputs larger than L2, no flush",
                       "parallelism": "env-sharded x%d%s" % (world, ", " + gather_how if world > 1 else "")},
            "roofline": roofline, "e2e": e2e, "gpu_launches": args.steps,
            "clocks": sampler.summary() if sampler else None,
        }
        if totals is not None:
            line["return_stats"] = {"mean_reward": float(totals[0]) / n_tot, "frac_optimal_arm": float(totals[2]) / n_tot}
        if cpu_baseline is not None:
            line["cpu_baseline"] = cpu_baseline
        if online is not None:
            line["online_eval"] = online
        if other is not None:
            line["other_workloads"] = other
        if args.workload == "online_eval" and online is not None:
            # same line, other half as the headline: the collection numbers move under "collect"
            w = online["runs"]["weak"]["fp32"]
            line["collect"] = {k: line[k] for k in ("metric", "value", "unit", "ms_per_step", "roofline", "e2e", "gpu_launches")}
            line.update(metric=OE_METRIC, value=w["value"], unit="trajs/s", ms_per_step=w["ms_per_pass"], roofline=w["roofline"],
                        e2e=online["e2e"], gpu_launches=online["gpu_launches"], steps=online["steps"], warmup=online["warmup"],
                        config={"workload": "deploy_online_vec + GPT-2 transformer controller, H=500 dim=5, %d envs/GPU x %d GPU "
                                            "(BASELINE configs[3], weak-scaled), fp32 K/V" % (OE_ENVS, world)})
            if "cpu_baseline" in online:
                line["cpu_baseline"] = online["cpu_baseline"]
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
