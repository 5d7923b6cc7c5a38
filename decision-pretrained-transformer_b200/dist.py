"""Multi-GPU layer: one process per GPU (torchrun), contiguous env-range sharding, no data-path
collective.

Envs are independent (SURVEY.md §8e), so rank r of R owns the global env ids
``[r*N/R, (r+1)*N/R)``; Philox counters use the GLOBAL env id, hence every rank's output is
bit-identical to the corresponding slice of a single-GPU run.  The only exchange is the small
statistics block -- ``[3]`` return statistics for collection, ``[H,4]`` regret sums for the online
loop -- all-gathered / all-reduced over NCCL (NVLink 5 / NVSwitch on the B200 box; gloo in the CPU
tests).  Context tensors and K/V caches never leave the GPU that produced them.
"""
import numpy as np
import torch
import torch.distributed as dist


def world():
    if dist.is_available() and dist.is_initialized():
        return dist.get_rank(), dist.get_world_size()
    return 0, 1


def shard_range(n_total, rank, world_size):
    """Contiguous, balanced split of ``range(n_total)``: returns (lo, hi) of ``rank``."""
    base, rem = divmod(n_total, world_size)
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


def microbatch_shard(n_total, mb, rank, world_size):
    """Micro-batch m covers the global items ``[m*mb, min(n_total, (m+1)*mb))``; rank r owns the contiguous micro-batch
    range ``shard_range(M, r, world_size)`` of the M = ceil(n_total / mb).  Returns (m_lo, m_hi, lo, hi): its micro-batches
    and the global item range they cover (empty, lo == hi, when the rank owns none)."""
    if mb < 1:
        raise ValueError("micro-batch size must be >= 1 (got %d)" % mb)
    m_lo, m_hi = shard_range(-(-n_total // mb), rank, world_size)
    return m_lo, m_hi, min(n_total, m_lo * mb), min(n_total, m_hi * mb)


def all_gather_stats(local, group=None):
    """All-gather a small per-rank statistics tensor -> [world, ...] (same on every rank)."""
    rank, ws = world()
    if ws == 1:
        return local[None]
    out = torch.empty((ws,) + tuple(local.shape), dtype=local.dtype, device=local.device)
    dist.all_gather_into_tensor(out.view(-1), local.contiguous().view(-1), group=group)
    return out


def all_reduce_sums(local, group=None):
    """Sum a per-rank block of additive statistics over all ranks (in place, returns it)."""
    _, ws = world()
    if ws > 1:
        dist.all_reduce(local, op=dist.ReduceOp.SUM, group=group)
    return local


def merge_return_stats(per_rank, steps_per_rank):
    """[world,3] (sum r, sum r^2, #optimal pulls) + env-steps per rank -> dict of global statistics."""
    per_rank = np.asarray(per_rank, dtype=np.float64)
    n = float(np.sum(steps_per_rank))
    s = per_rank.sum(0)
    mean = s[0] / n
    return {"env_steps": n, "mean_reward": mean, "var_reward": max(s[1] / n - mean * mean, 0.0),
            "frac_optimal_arm": s[2] / n}


def regret_stats_from_sums(sums, n_envs):
    """[H,4] regret sums over ``n_envs`` envs -> the four curves of evals/eval_bandit.py:169-178:
    per-step regret mean / sem and cumulative regret mean / sem (scipy.stats.sem, ddof = 1)."""
    s = np.asarray(sums, dtype=np.float64)
    n = float(n_envs)

    def mean_sem(s1, s2):
        mean = s1 / n
        var = np.maximum(s2 - s1 * s1 / n, 0.0) / max(n - 1.0, 1.0)
        return mean, np.sqrt(var / n)
    m, se = mean_sem(s[:, 0], s[:, 1])
    cm, cse = mean_sem(s[:, 2], s[:, 3])
    return {"mean": m, "sem": se, "regret_mean": cm, "regret_sem": cse}


class PeerBuffer:
    """One device buffer per rank (``nbytes`` of it on this rank, zero-filled; the size may differ between ranks), mapped
    into every rank's address space over CUDA IPC: ``peer_ptrs[r]`` is rank r's buffer as seen from this rank (its own
    buffer at r == rank).  Kernels read or store through these pointers over NVLink; ordering against the other ranks is
    the caller's job (stream synchronise + barrier).  ``rank_world``: (rank, world size) to use instead of ``world()``;
    (0, 1) is a buffer of this process alone, with no exchange, even inside a process group."""

    def __init__(self, nbytes, rank_world=None):
        import ctypes
        from ._lib import check, lib
        self.rank, self.world = world() if rank_world is None else rank_world
        self.ptr = ctypes.c_void_p()
        self.peer_ptrs, self._opened = [], []
        self._ctypes = ctypes
        handle = (ctypes.c_ubyte * 64)()
        # every step is followed by an exchange of success flags, so that all ranks agree on failure
        # (a rank that raised on its own would leave the others blocked in the next collective)
        err = None
        try:
            check(lib().dpt_peer_buffer_create(nbytes, ctypes.byref(self.ptr), handle), "dpt_peer_buffer_create")
        except Exception as e:   # noqa: BLE001
            err = str(e)
        handles = [bytes(handle) if err is None else None]
        if self.world > 1:
            handles = [None] * self.world
            dist.all_gather_object(handles, bytes(handle) if err is None else None)
        if any(h is None for h in handles):
            self.close()
            raise RuntimeError("peer buffer allocation failed on some rank: %s" % err)
        for r in range(self.world):
            if r == self.rank:
                self.peer_ptrs.append(self.ptr.value)
                continue
            try:
                h = (ctypes.c_ubyte * 64).from_buffer_copy(handles[r])
                pp = ctypes.c_void_p()
                check(lib().dpt_peer_buffer_open(h, ctypes.byref(pp)), "dpt_peer_buffer_open")
                self.peer_ptrs.append(pp.value)
                self._opened.append(pp)
            except Exception as e:   # noqa: BLE001
                err = str(e)
                break
        if self.world > 1:
            oks = [None] * self.world
            dist.all_gather_object(oks, err is None)
            if not all(oks):
                self.close()
                raise RuntimeError("CUDA IPC peer mapping failed on some rank: %s" % err)

    def local_f32(self, n):
        """The first ``n`` floats of this rank's own buffer as a float32 torch tensor (a view: no copy, no ownership; valid
        until ``close``)."""
        class _View:
            __cuda_array_interface__ = {"shape": (n,), "typestr": "<f4", "data": (self.ptr.value, False), "version": 3,
                                        "strides": None}
        return torch.as_tensor(_View(), device=torch.device("cuda", torch.cuda.current_device()))

    def close(self):
        from ._lib import lib
        for pp in self._opened:
            lib().dpt_peer_buffer_close(pp)
        self._opened = []
        if self.ptr is not None and self.ptr.value:
            lib().dpt_peer_buffer_destroy(self.ptr)
        self.ptr = None


class PeerGather(PeerBuffer):
    """Per-rank gather buffers [slots, world, width] float64, mutually mapped over CUDA IPC.

    Rank r's kernels store their statistics for slot s straight into element [s, r, :] of EVERY rank's
    buffer over NVLink (dpt_bandit_rollin_p2p): an all-gather with no collective launch.  Readers must
    order themselves after all ranks' launches (stream synchronise + barrier), then ``read()``."""

    def __init__(self, slots, width=3):
        self.slots, self.width = slots, width
        self.data_bytes = slots * world()[1] * width * 8
        super().__init__(self.data_bytes + 256)
        self.counter_ptr = self.ptr.value + self.data_bytes          # uint32 done-counter of this rank's launches

    def dst_array(self, slot):
        """Host array of device pointers: element [slot, my rank, 0] of every rank's buffer."""
        ct = self._ctypes
        off = ((slot * self.world + self.rank) * self.width) * 8
        return (ct.c_void_p * self.world)(*[p + off for p in self.peer_ptrs])

    def publish_zeros(self, slot):
        """What a rank with an EMPTY env shard does instead of launching: zero element [slot, my rank, :] of every
        rank's buffer (cudaMemsetAsync on the current stream through the peer mappings)."""
        from ._lib import check, lib, stream_ptr
        off = ((slot * self.world + self.rank) * self.width) * 8
        for p in self.peer_ptrs:
            check(lib().dpt_peer_buffer_zero(self._ctypes.c_void_p(p + off), self.width * 8, stream_ptr()), "dpt_peer_buffer_zero")

    def read(self):
        """This rank's buffer as a numpy array [slots, world, width] (synchronises the current stream)."""
        from ._lib import check, lib, stream_ptr
        out = np.empty((self.slots, self.world, self.width), dtype=np.float64)
        check(lib().dpt_peer_buffer_read(self.ptr, out.ctypes.data, self.data_bytes, stream_ptr()), "dpt_peer_buffer_read")
        return out


# ------------------------------------------------------------------ sharded entry points -------
def collect_bandit_sharded(n_envs_total, dim, horizon, var, seed, device=None, peer=None, peer_slot=0):
    """BASELINE config 5: bandit collection over all ranks.  Returns (local batch dict, global
    statistics dict).  The local batch holds this rank's env slice only (possibly empty when
    ``n_envs_total < world``: such a rank launches nothing and contributes zeros)."""
    from . import kernels
    rank, ws = world()
    lo, hi = shard_range(n_envs_total, rank, ws)
    means, opt_idx, opt_a = kernels.bandit_sample_means(hi - lo, dim, seed, lo, device)
    stats = torch.zeros(3, dtype=torch.float64, device=means.device)
    if peer is not None:   # fused all-gather over NVLink peer memory, no collective launch
        if hi > lo:
            batch = kernels.bandit_rollin(means, horizon, float(var), seed, lo, stats=stats, peer=peer, peer_slot=peer_slot)
        else:              # empty shard: no launch; publish zeros so that every rank's slot row is defined
            batch = kernels.bandit_rollin(means, horizon, float(var), seed, lo)
            peer.publish_zeros(peer_slot)
        torch.cuda.synchronize()
        if ws > 1:
            dist.barrier()           # every rank's launch (and its NVLink stores) has completed
        gathered = peer.read()[peer_slot].copy()
        if ws > 1:
            dist.barrier()           # nobody re-uses `peer_slot` before every rank has read it (ADVICE r1: a fast
                                     # rank's next launch could otherwise overwrite a slow rank's unread slot)
    else:
        batch = kernels.bandit_rollin(means, horizon, float(var), seed, lo, stats=stats)
        gathered = all_gather_stats(stats).cpu().numpy()
    batch.update(means=means, opt_a_index=opt_idx, optimal_actions=opt_a, env_range=(lo, hi))
    steps = [(shard_range(n_envs_total, r, ws)[1] - shard_range(n_envs_total, r, ws)[0]) * horizon for r in range(ws)]
    return batch, merge_return_stats(gathered, steps)


def online_eval_sharded(kind, n_envs_total, dim, horizon, var, seed, model=None, materialise=False, means_local=None, **ctrl):
    """Online in-context evaluation over all ranks: each rank draws (or receives) and evaluates its env slice with
    the fused loop, then the [H,4] regret sums are all-reduced.  ``kind``: 'opt' | 'emp' | 'ucb' |
    'thompson' | 'linucb' | 'transformer'.  ``means_local``: optional [hi-lo, dim] fp32 task means of THIS rank's slice
    (host -- ideally pinned -- or device tensor); default: drawn on the device from Philox(seed, global env id).
    Returns (local result dict, global regret curves)."""
    from . import kernels
    rank, ws = world()
    lo, hi = shard_range(n_envs_total, rank, ws)
    if means_local is not None:
        assert tuple(means_local.shape) == (hi - lo, dim), "means_local must be this rank's [%d, %d] slice" % (hi - lo, dim)
        means = means_local.to(device=kernels._dev(), dtype=torch.float32, non_blocking=True)
    else:
        means, _, _ = kernels.bandit_sample_means(hi - lo, dim, seed, lo)
    if kind == "transformer":
        out = model.online_loop(means, horizon, var, ctrl.get("sample", True), seed, lo, materialise, True)
    else:
        out = kernels.online_loop(kind, means, horizon, var, seed, lo, materialise=materialise, regret=True, **ctrl)
    sums = all_reduce_sums(out["regret_sums"].clone())
    return out, regret_stats_from_sums(sums.cpu().numpy(), n_envs_total)


def collect_darkroom_sharded(goals_total, dim, horizon, seed, rollin_type="uniform", perm_index_total=None, n_samples=1):
    """BASELINE config 2 over all ranks: rank r runs ``rollin_mdp`` + query states for the env slice
    ``shard_range(len(goals_total), r, world)`` (global env ids in the Philox counters, so the shards are slices of
    the single-GPU result).  The exchange is one all-reduce of two integers: total reward and number of env-steps.
    Returns (local batch dict, {'mean_reward', 'env_steps'})."""
    from . import kernels
    rank, ws = world()
    goals_total = np.asarray(goals_total)
    lo, hi = shard_range(len(goals_total), rank, ws)
    perm = None if perm_index_total is None else np.asarray(perm_index_total)[lo:hi]
    batch = kernels.darkroom_rollin(goals_total[lo:hi], dim, horizon, rollin_type, seed, lo, perm, n_samples)
    local = torch.stack((batch["context_rewards"].double().sum(), torch.tensor(float((hi - lo) * horizon), dtype=torch.float64,
                                                                             device=batch["context_rewards"].device)))
    tot = all_reduce_sums(local).cpu().numpy()
    batch["env_range"] = (lo, hi)
    return batch, {"mean_reward": float(tot[0] / max(tot[1], 1.0)), "env_steps": int(tot[1])}


def train_interactive_sharded(model, dim, n_envs_total, K, n_iters, mb=1024, **kw):
    """``train.train_interactive`` over all ranks (one process per GPU): rank r rolls out and differentiates its contiguous
    range of micro-batches (``microbatch_shard``; Philox counters use global env ids, so its contexts are slices of the
    one-GPU rollout), keeps their gradient slots in a ``PeerBuffer``, and every rank sums all slots in micro-batch order
    (``dpt_ordered_sum_f32`` over the peer mappings) before its AdamW step.  The weights after every iteration are
    bit-identical on every rank and to the one-GPU run, for any world size and at either training ``precision`` (0 = fp32,
    1 = bf16; the rollout runs at ``model.precision``).  Same arguments and return value; with
    ``state_path``, rank 0 writes the training state after the iteration's AdamW step (a failed write makes every rank
    raise), and on ``resume`` every rank reads the same file, which may come from any world size."""
    from . import train
    rank, ws = world()
    return train._interactive(model, dim, n_envs_total, K, n_iters, mb, rank, ws, **kw)
