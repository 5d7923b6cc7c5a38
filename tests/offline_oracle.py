"""numpy restatement of the offline bandit evaluation -- TEST INFRASTRUCTURE (used by test_offline_eval_*.py).

``offline_eval`` is evals/eval_bandit.py:214-335 (``offline`` once per horizon, as ``offline_graph`` calls it) driven
with the oracle's controllers: each controller sees the first h context rows and plays one noise-free pull, whose
reward is means[a] (BanditEnvVec.deploy_eval, envs/bandit_env.py:115-123).  Thompson(sample=False) draws through the
noise source, so ``ReplayNoise({'thompson_z': z.reshape(K * n_draws, N, d)})`` replays the device's normals.
"""
import numpy as np

from oracle import dpt_oracle as O

STREAM_OFFLINE = 7   # csrc/philox.cuh: Philox stream tag of the offline evaluation's Thompson normals


class PessMeanCtrl:
    """ctrls/ctrl_bandit.py:255-314: lower confidence bound b/max(1,n) - const/max(1,sqrt(n)), no untried-arm override."""
    def __init__(self, d, const=.8):
        self.d, self.const = d, const

    def act(self, ctx_a, ctx_r, noise, h):
        N = ctx_a.shape[0]
        b, counts = O._arm_stats(ctx_a, ctx_r, self.d)
        bounds = b / np.maximum(1, counts) - self.const / np.maximum(1, np.sqrt(counts))
        a = np.zeros((N, self.d))
        a[np.arange(N), np.argmax(bounds, axis=-1)] = 1.0
        return a


def offline_eval(means, ctx_a, ctx_r, horizons, ctrls, noise):
    """means [N,d], ctx_a [N,H,d] one-hot, ctx_r [N,H]; ctrls: {name: oracle controller}.  Horizons are visited in
    list order, controllers in dict order.  Returns ({name: rewards [K,N]}, {name: sums [K,2]}) with sums over envs of
    (max mean - reward, its square)."""
    means = np.asarray(means, dtype=np.float64)
    ctx_a, ctx_r = np.asarray(ctx_a, dtype=np.float64), np.asarray(ctx_r, dtype=np.float64).reshape(ctx_a.shape[:2])
    N = means.shape[0]
    rew = {name: np.zeros((len(horizons), N)) for name in ctrls}
    for k, h in enumerate(horizons):
        for name, c in ctrls.items():
            hot = c.act(ctx_a[:, :h], ctx_r[:, :h], noise, h)
            rew[name][k] = means[np.arange(N), np.argmax(hot, axis=-1)]
    best = means.max(1)
    sums = {name: np.stack([(best - r).sum(1), ((best - r) ** 2).sum(1)], 1) for name, r in rew.items()}
    return rew, sums
