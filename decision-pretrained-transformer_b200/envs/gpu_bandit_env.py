"""GPUBanditEnv with the reference's interface (envs/gpu_bandit_env.py:8-82).

The reference's step is ~6 small ATen launches plus a host sync on ``current_step.max()`` (:67);
here the constructor is one launch (means + argmax + one-hot) and a step is ONE launch
(argmax -> gather -> Philox normal / Bernoulli) with the step counter kept on the host, so there is
no device->host synchronisation on the step path.
"""
import torch

from .. import kernels, rng
from .base_env import BaseEnv

_TYPES = {"uniform": 0, "bernoulli": 1}


class GPUBanditEnv(BaseEnv):
    def __init__(self, dims, n_envs, H, var=0.0, type="uniform", device=None, seed=None, env_id0=0):
        if type not in _TYPES:
            raise NotImplementedError
        self.dims = dims
        self.dim = dims
        self.n_envs = n_envs
        self._device = kernels._dev(device)
        self._key = rng.next_key() if seed is None else seed
        self._env_id0 = env_id0
        with torch.cuda.device(self._device):
            # uniform: U[0,1) like torch.rand (:19); bernoulli: Beta(1,1) == U(0,1) (:21)
            self.means, self.opt_a_index, self.opt_a = kernels.bandit_sample_means(n_envs, dims, self._key, env_id0,
                                                                                   self._device)
        self.opt_a_index = self.opt_a_index.long()
        self.H_context = H
        self.H = H
        self.var = var
        self.dx = 1
        self.du = dims
        self.topk = False
        self.type = type
        self.state = torch.ones((n_envs, 1), device=self._device)
        self.current_step = torch.zeros(n_envs, device=self._device)
        self._step = 0        # host mirror of current_step (all envs advance together)
        self._draws = 0
        self._rollouts = 0    # fused rollouts so far: each gets its own Philox key (a re-used env object must not replay noise)

    def get_arm_value(self, actions):
        return torch.sum(self.means * actions, dim=1)

    def reset(self):
        self.current_step = torch.zeros(self.n_envs, device=self._device)
        self._step = 0
        return self.state.detach()

    def transit(self, x, us, inject=None):
        us = us.to(self._device) if us.device != self._device else us
        with torch.cuda.device(self._device):
            r = kernels.gpu_bandit_step(self.means, us, float(self.var), _TYPES[self.type], self._key ^ 0x5DEECE66D,
                                        self._env_id0, self._draws, inject=inject)
        self._draws += 1
        return self.state.detach(), r

    def set_means(self, means):
        """Replace the drawn tasks (tests / callers that bring their own tasks): means [n_envs, dims]."""
        self.means = kernels._as(means, torch.float32, self._device)
        assert tuple(self.means.shape) == (self.n_envs, self.dims)
        with torch.cuda.device(self._device):
            idx, self.opt_a = kernels.bandit_opt_action(self.means)
        self.opt_a_index = idx.long()

    def step(self, actions, inject=None):
        """``inject``: optional [n_envs] noise to consume instead of the Philox draw (parity runs): the standard
        normals of type 'uniform' / the uniforms of type 'bernoulli'."""
        if self._step >= self.H:
            raise ValueError("Episode has already ended")
        _, r = self.transit(self.state, actions, inject=inject)
        self._step += 1
        self.current_step += 1
        done = self.current_step >= self.H
        return self.state.detach(), r, done, {}

    def deploy_eval(self, ctrl):
        tmp = self.var
        self.var = 0.0
        res = self.deploy(ctrl)
        self.var = tmp
        return res

    # ---- interactive rollouts (train_interactive.py:97-134, rollout half) ----------------------------
    def rollout(self, model, K=None, sample=True, logits=True):
        """The K-step interactive rollout of the reference's on-policy trainers in ONE fused launch: at each
        step the transformer sees the context so far (K/V-cached), an action is drawn from its logits, the env
        steps, the row is appended.  Returns the four context tensors [n_envs,K,.] (device, fp32), the logits
        the model produced at every step [K,n_envs,du] (not written with ``logits=False``; the rollout is the same)
        and ``target = opt_a_index`` (:134).  The gradient half (train_interactive.py:134-139) re-runs the model on
        ``context[:, :K-1]`` with a gradient: ``train.train_interactive`` does both halves."""
        K = self.H if K is None else K
        with torch.cuda.device(self._device):
            key = (self._key ^ 0x2545F4914F6CDD1D) + 0x9E3779B97F4A7C15 * self._rollouts & 0xFFFFFFFFFFFFFFFF
            out = model.online_loop(self.means, K, float(self.var), sample, key, self._env_id0,
                                    materialise=True, regret=False, dump=logits, reward_type=self.type)
        self._draws += K
        self._rollouts += 1
        res = {"context_states": out["context_states"], "context_actions": out["context_actions"],
               "context_next_states": out["context_next_states"], "context_rewards": out["context_rewards"]}
        if logits:
            res["logits"] = out["noise"]["logits"]
        res["target"] = self.opt_a_index
        return res

    @torch.no_grad()
    def rollout_explorer_exploiter(self, explorer, exploiter, K=None, fused=True, inject=None, dump=False):
        """The replay-buffer fill of train_explorer_exploiter.py:110-166 (the no-grad half of an episode): at every step
        both models score the context so far (K/V-cached), the explorer's sampled arm is what gets RECORDED in the
        context while the env is stepped with a uniformly random arm (:141-152, as in the reference), and the advantage
        of step t-1 is the change of the exploiter's cross-entropy against the optimal arm (:160-164).  Returns the
        context tensors [n_envs,K,.], ``advantages`` [n_envs,K-1,1], both models' logits per step [K,n_envs,du] and
        ``target``.

        ``fused=True`` (default): ONE launch for all K steps (``dpt_gpt2_explore_exploit_rollout``; Philox draws addressed
        by (env, step); ``inject`` / ``dump``: ctrl_u f64 [K,n], random_arm int32 [K,n], reward_z fp32 [K,n]).
        ``fused=False``: the step-by-step form over ``Transformer.decoder`` + ``step`` with torch's device generator, as the
        reference samples."""
        if fused:
            return self._rollout_explorer_exploiter_fused(explorer, exploiter, self.H if K is None else K, inject, dump)
        K = self.H if K is None else K
        n, du, dev = self.n_envs, self.du, self._device
        dec_e, dec_x = explorer.decoder(n, K), exploiter.decoder(n, K)
        ctx = {"context_states": torch.zeros((n, K, self.dx), device=dev), "context_actions": torch.zeros((n, K, du), device=dev),
               "context_next_states": torch.zeros((n, K, self.dx), device=dev), "context_rewards": torch.zeros((n, K, 1), device=dev)}
        advantages = torch.zeros((n, max(K - 1, 0), 1), device=dev)
        logits_e, logits_x = [], []
        target = self.opt_a_index.to(dev)
        state, prev_loss = self.reset(), None
        for t in range(K):
            if t == 0:
                le, lx = dec_e.query(state), dec_x.query(state)
            else:
                row = [ctx[k][:, t - 1] for k in ("context_states", "context_actions", "context_next_states", "context_rewards")]
                le, lx = dec_e.append(*row), dec_x.append(*row)
            logits_e.append(le), logits_x.append(lx)
            action = torch.nn.functional.one_hot(torch.distributions.Categorical(logits=le).sample(), num_classes=du).float()
            random_action = torch.nn.functional.one_hot(torch.randint(0, du, (n,), device=dev), num_classes=du).float()
            next_state, reward, _, _ = self.step(random_action)
            ctx["context_states"][:, t] = state.float()
            ctx["context_actions"][:, t] = action
            ctx["context_next_states"][:, t] = next_state.float()
            ctx["context_rewards"][:, t, 0] = reward.float()
            state = next_state
            loss = torch.nn.functional.cross_entropy(lx, target, reduction="none")
            if t > 0:
                advantages[:, t - 1] = (loss - prev_loss).unsqueeze(-1)
            prev_loss = loss
        return dict(ctx, advantages=advantages, explorer_logits=torch.stack(logits_e), exploiter_logits=torch.stack(logits_x),
                    target=target)

    def _rollout_explorer_exploiter_fused(self, explorer, exploiter, K, inject, dump):
        import ctypes
        from .. import _lib
        n, du, dev = self.n_envs, self.du, self._device
        assert explorer.precision == 0 and exploiter.precision == 0, "the fused explorer / exploiter rollout is fp32"
        with torch.cuda.device(dev):
            he, hx = explorer.handle(), exploiter.handle()
            lib = _lib.lib()
            out = {"context_states": torch.empty((n, K, self.dx), device=dev), "context_actions": torch.empty((n, K, du), device=dev),
                   "context_next_states": torch.empty((n, K, self.dx), device=dev), "context_rewards": torch.empty((n, K, 1), device=dev),
                   "advantages": torch.zeros((n, max(K - 1, 0), 1), device=dev)}
            kv_bytes = max(lib.dpt_gpt2_online_kv_bytes(he, n, K, 0), lib.dpt_gpt2_online_kv_bytes(hx, n, K, 0))
            kv_e = torch.empty((max(int(kv_bytes), 1),), dtype=torch.uint8, device=dev)
            kv_x = torch.empty((max(int(kv_bytes), 1),), dtype=torch.uint8, device=dev)
            inj_p, keep = None, []
            if inject is not None:
                si = _lib.ExploreInject()
                for k, dt in (("ctrl_u", torch.float64), ("random_arm", torch.int32), ("reward_z", torch.float32)):
                    if inject.get(k) is not None:
                        t = kernels._as(inject[k], dt, dev)
                        keep.append(t)
                        setattr(si, k, kernels.ptr(t))
                inj_p = ctypes.byref(si)
            sd = _lib.ExploreDump()
            out["explorer_logits"] = torch.empty((K, n, du), device=dev)
            out["exploiter_logits"] = torch.empty((K, n, du), device=dev)
            sd.logits_explorer, sd.logits_exploiter = kernels.ptr(out["explorer_logits"]), kernels.ptr(out["exploiter_logits"])
            if dump:
                out["noise"] = {"ctrl_u": torch.empty((K, n), dtype=torch.float64, device=dev),
                                "random_arm": torch.empty((K, n), dtype=torch.int32, device=dev),
                                "reward_z": torch.empty((K, n), dtype=torch.float32, device=dev)}
                for k, t in out["noise"].items():
                    setattr(sd, k, kernels.ptr(t))
            key = (self._key ^ 0x6A09E667F3BCC909) + 0x9E3779B97F4A7C15 * self._rollouts & 0xFFFFFFFFFFFFFFFF
            kernels.check(lib.dpt_gpt2_explore_exploit_rollout(
                he, hx, kernels.ptr(self.means), float(self.var), kernels.REWARD_TYPES[self.type], key, self._env_id0, n, K,
                kernels.ptr(kv_e), kernels.ptr(kv_x), kv_e.numel(), kernels.ptr(out["context_states"]),
                kernels.ptr(out["context_actions"]), kernels.ptr(out["context_next_states"]), kernels.ptr(out["context_rewards"]),
                kernels.ptr(out["advantages"]), inj_p, ctypes.byref(sd), kernels.stream_ptr()), "dpt_gpt2_explore_exploit_rollout")
        self._draws += K
        self._rollouts += 1
        self.reset()
        self._step = K                     # the episode of K steps is over (envs/gpu_bandit_env.py:59-61)
        self.current_step = self.current_step + K
        out["target"] = self.opt_a_index.to(dev)
        return out
