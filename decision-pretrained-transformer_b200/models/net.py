"""Transformer with the reference's interface (models/net.py:9-60), inference on the CUDA path.

``Transformer(config)`` takes the reference's config dict (horizon, state_dim, action_dim, n_layer,
n_embd, n_head, dropout, test); ``forward(x)`` takes the reference's batch dict and returns
``preds[:, -1, :]`` (test) or ``preds[:, 1:, :]``.  The module's ``state_dict`` uses the reference's
key layout (HuggingFace GPT2Model under ``transformer.``, ``embed_transition.*``, ``pred_actions.*``),
so checkpoints written by the reference's train.py load unchanged.  As in the reference, ``n_head``
from the config is ignored: the trunk always has ONE head (models/net.py:29), head_dim = n_embd.

``forward`` is dpt_gpt2_forward (hand-written CUDA, fp32) under ``torch.no_grad()``.  ``forward_train`` is the
same computation with a gradient: dpt_gpt2_train_forward / dpt_gpt2_train_backward (hand-written CUDA, fp32) read
the parameter tensors in place, and autograd receives a gradient for every parameter except ``transformer.wte``
(which the model never reads, as in the reference).  ``forward_train(x, precision=1)`` is bf16 mixed-precision
training (the same entry points at precision 1): the tcgen05 forward of ``forward`` at ``model.precision = 1`` and a
tensor-core attention backward, with fp32 master weights and gradient sums.  The class holds no HuggingFace dependency.
"""
import ctypes

import torch
import torch.nn as nn

from .. import _lib, kernels
from .._lib import check, lib, ptr, stream_ptr


class _Conv1D(nn.Module):
    """transformers.pytorch_utils.Conv1D parameter layout: weight [in, out], y = x @ W + b."""

    def __init__(self, nf, nx):
        super().__init__()
        self.weight = nn.Parameter(torch.empty(nx, nf).normal_(std=0.02))
        self.bias = nn.Parameter(torch.zeros(nf))


class _Attn(nn.Module):
    def __init__(self, E):
        super().__init__()
        self.c_attn = _Conv1D(3 * E, E)
        self.c_proj = _Conv1D(E, E)


class _MLP(nn.Module):
    def __init__(self, E):
        super().__init__()
        self.c_fc = _Conv1D(4 * E, E)
        self.c_proj = _Conv1D(E, 4 * E)


class _Block(nn.Module):
    def __init__(self, E):
        super().__init__()
        self.ln_1 = nn.LayerNorm(E, eps=1e-5)
        self.attn = _Attn(E)
        self.ln_2 = nn.LayerNorm(E, eps=1e-5)
        self.mlp = _MLP(E)


class _GPT2Trunk(nn.Module):
    def __init__(self, n_positions, E, n_layer, vocab=50257):
        super().__init__()
        self.wte = nn.Embedding(vocab, E)       # unused by inputs_embeds, kept for checkpoint compatibility
        self.wpe = nn.Embedding(n_positions, E)
        self.h = nn.ModuleList([_Block(E) for _ in range(n_layer)])
        self.ln_f = nn.LayerNorm(E, eps=1e-5)
        nn.init.normal_(self.wte.weight, std=0.02)
        nn.init.normal_(self.wpe.weight, std=0.02)


class Transformer(nn.Module):
    """Transformer class (models/net.py:9)."""

    def __init__(self, config):
        super().__init__()
        self.config = config
        self.test = config["test"]
        self.horizon = config["horizon"]
        self.n_embd = config["n_embd"]
        self.n_layer = config["n_layer"]
        self.n_head = config["n_head"]
        self.state_dim = config["state_dim"]
        self.action_dim = config["action_dim"]
        self.dropout = config["dropout"]
        self.transformer = _GPT2Trunk(4 * (1 + self.horizon), self.n_embd, self.n_layer)
        self.embed_transition = nn.Linear(2 * self.state_dim + self.action_dim + 1, self.n_embd)
        self.pred_actions = nn.Linear(self.n_embd, self.action_dim)
        self._handle = None
        self._handle_version = None
        self._workspace = None
        self.precision = 0      # 0 = fp32 (reference parity 1e-5); 1 = bf16 K/V cache, fp32 arithmetic (2e-2)

    # ---- checkpoint compatibility --------------------------------------------------------
    def load_state_dict(self, state_dict, strict=True, **kw):
        # transformers 4.5.1 (the reference's pin) stores the causal mask buffers in the state dict
        sd = {k: v for k, v in state_dict.items() if not (k.endswith(".attn.bias") or k.endswith(".attn.masked_bias"))}
        res = super().load_state_dict(sd, strict=strict, **kw)
        self._handle_version = None
        return res

    # ---- device handle -------------------------------------------------------------------
    def _version(self):
        return tuple((p.data_ptr(), p._version) for p in self.parameters())

    def handle(self):
        """Opaque dpt_gpt2_t* for the current weights (repacked once per weight update)."""
        dev = kernels._dev()
        if next(self.parameters()).device != dev:
            self.to(dev)
        ver = self._version()
        if self._handle is not None and ver == self._handle_version:
            return self._handle
        self._free()
        ps, keep = [p.detach().float().contiguous() for p in self._train_params()], []
        w = _weights_struct(self, ps, keep)
        h = ctypes.c_void_p()
        check(lib().dpt_gpt2_create(ctypes.byref(w), ctypes.byref(h), stream_ptr()), "dpt_gpt2_create")
        torch.cuda.current_stream().synchronize()      # the D2D repack read `ps`
        self._handle, self._handle_version = h, ver
        return h

    def _free(self):
        if self._handle is not None:
            lib().dpt_gpt2_destroy(self._handle)
            self._handle = None

    def __del__(self):
        try:
            self._free()
        except Exception:   # noqa: BLE001
            pass

    def _scratch(self, nbytes):
        if self._workspace is None or self._workspace.numel() < nbytes:
            self._workspace = torch.empty((max(int(nbytes), 1),), dtype=torch.uint8, device=kernels._dev())
        return self._workspace

    # ---- models/net.py:41-60 --------------------------------------------------------------
    @torch.no_grad()
    def forward(self, x, ctx_share=1):
        """``ctx_share`` > 1: ``query_states`` has ctx_share rows per context row (see dpt_gpt2_forward)."""
        dev = kernels._dev()
        h = self.handle()
        q, cs, ca, cns, cr, B, T, stride = _batch_inputs(x, dev, ctx_share)
        out = torch.empty((B, self.action_dim) if self.test else (B, T, self.action_dim), dtype=torch.float32, device=dev)
        nbytes = lib().dpt_gpt2_forward_workspace_bytes(h, B, T, self.precision)
        ws = self._scratch(nbytes)
        check(lib().dpt_gpt2_forward(h, q.data_ptr(), cs.data_ptr() if T else None, ca.data_ptr() if T else None,
                                     cns.data_ptr() if T else None, cr.data_ptr() if T else None, B, T, stride, ctx_share,
                                     1 if self.test else 0, self.precision, ptr(out), ptr(ws), ws.numel(), stream_ptr()),
              "dpt_gpt2_forward")
        return out

    # ---- training: models/net.py:41-60 with a gradient ----------------------------------------
    def _train_params(self):
        """The parameters forward_train differentiates, in the order of dpt_gpt2_weights_t (transformer.wte excluded)."""
        t = self.transformer
        ps = [t.wpe.weight, self.embed_transition.weight, self.embed_transition.bias, self.pred_actions.weight,
              self.pred_actions.bias, t.ln_f.weight, t.ln_f.bias]
        for f in _LAYER_FIELDS:
            ps += [f(b) for b in t.h]
        return ps

    def forward_train(self, x, precision=0):
        """``forward(x)`` with an autograd graph: returns ``preds[:, -1, :]`` (test) or ``preds[:, 1:, :]`` with a
        ``grad_fn``; ``backward`` fills ``.grad`` of every parameter except ``transformer.wte``.  The context inputs get
        no gradient.  Sequences of <= 512 tokens.  This is the one-member case of ``forward_train_population``.

        ``precision`` is the precision of this training step, independent of ``self.precision`` (the precision of
        ``forward``, of the online loop and of rollouts):

        - 0 (default): fp32 on the CUDA cores; the logits are bit-identical to ``forward(x)`` at ``self.precision = 0``.
        - 1: bf16 mixed precision.  bf16 operands at the tensor-core inputs, fp32 accumulation, LayerNorm, softmax
          statistics, residual stream and gradient sums; the parameters (master weights) stay fp32.  The logits are
          bit-identical to ``forward(x)`` at ``self.precision = 1`` (within 2e-2 of fp32); the gradients are
          deterministic."""
        return forward_train_population([self], [x], precision)[0]

    # ---- step-by-step K/V-cached decode (callers that choose the pulled arm themselves) -------------
    def decoder(self, n_seqs, max_transitions=None):
        """A K/V-cached incremental view of ``forward(...)[:, -1]`` for loops that are driven from outside (the rollout
        half of train_interactive.py:97-132 / train_explorer_exploiter.py:110-166): ``dec.query(states)`` appends the
        query token (position 0) and returns the logits on an empty context; each ``dec.append(states, actions,
        next_states, rewards)`` appends one transition and returns the logits given everything appended so far --
        O(context) work per step instead of a dense forward over the whole context."""
        return _Decoder(self, n_seqs, self.horizon if max_transitions is None else max_transitions)

    # ---- fused in-context evaluation loop ---------------------------------------------------
    def online_loop(self, means, horizon, var, sample, seed, env_id0=0, materialise=True, regret=True, inject=None,
                    dump=False, reward_type="uniform"):
        """deploy_online_vec with BanditTransformerController in one launch (KV-cached decode +
        sampling + env step).  Returns the same dict as kernels.online_loop.  This is the one-member case of
        ``online_loop_population``."""
        return online_loop_population([self], means, horizon, var, sample, seed, env_id0, materialise, regret, inject, dump,
                                      reward_type)[0]


_LAYER_FIELDS = (lambda b: b.ln_1.weight, lambda b: b.ln_1.bias, lambda b: b.attn.c_attn.weight, lambda b: b.attn.c_attn.bias,
                 lambda b: b.attn.c_proj.weight, lambda b: b.attn.c_proj.bias, lambda b: b.ln_2.weight, lambda b: b.ln_2.bias,
                 lambda b: b.mlp.c_fc.weight, lambda b: b.mlp.c_fc.bias, lambda b: b.mlp.c_proj.weight, lambda b: b.mlp.c_proj.bias)
_LAYER_NAMES = ("ln1_w", "ln1_b", "attn_w", "attn_b", "proj_w", "proj_b", "ln2_w", "ln2_b", "fc_w", "fc_b", "fc2_w", "fc2_b")
_TOP_NAMES = ("wpe", "embed_w", "embed_b", "pred_w", "pred_b", "lnf_w", "lnf_b")


def _pointer_struct(cls, model, tensors, keep, **extra):
    """dpt_gpt2_weights_t / dpt_gpt2_grads_t over `tensors` (ordered as Transformer._train_params); the per-layer pointer
    arrays go to `keep`."""
    L = model.n_layer
    for t in tensors:
        if t.dtype != torch.float32 or not t.is_contiguous() or not t.is_cuda:
            raise ValueError("forward_train needs contiguous fp32 CUDA parameters")
    kw = {n: t.data_ptr() for n, t in zip(_TOP_NAMES, tensors)}
    for i, n in enumerate(_LAYER_NAMES):
        a = (ctypes.c_void_p * L)(*[t.data_ptr() for t in tensors[7 + i * L:7 + (i + 1) * L]])
        keep.append(a)
        kw[n] = ctypes.cast(a, ctypes.POINTER(ctypes.c_void_p))
    kw.update(extra)
    return cls(**kw)


def _weights_struct(model, params, keep):
    return _pointer_struct(_lib.Gpt2Weights, model, params, keep, horizon=model.horizon, state_dim=model.state_dim,
                           action_dim=model.action_dim, n_layer=model.n_layer, n_embd=model.n_embd,
                           n_positions=model.transformer.wpe.weight.shape[0])


def _batch_inputs(x, dev, ctx_share=1):
    """(q, cs, ca, cns, cr, B, T, stride) of a batch dict, B = ctx_share * context rows (see dpt_gpt2_forward); context
    views [:, :h] of a [B,H,.] buffer keep their row stride, other layouts are made contiguous."""
    f = lambda t: t.to(device=dev, dtype=torch.float32)   # noqa: E731
    q = f(x["query_states"]).contiguous()
    cs, ca, cns, cr = f(x["context_states"]), f(x["context_actions"]), f(x["context_next_states"]), f(x["context_rewards"])
    Bc, T = ca.shape[0], ca.shape[1]
    B = Bc * ctx_share
    assert q.shape[0] == B, "query_states and the context disagree on the batch size"
    stride = ca.stride(0) // max(1, ca.shape[2]) if T > 0 else 0
    ok = T > 0 and stride >= T and all(t.stride(-1) == 1 and t.stride(1) == t.shape[2] and t.stride(0) == stride * t.shape[2]
                                       for t in (cs, ca, cns, cr.reshape(Bc, T, 1) if cr.dim() == 2 else cr))
    if not ok:
        cs, ca, cns, cr = cs.contiguous(), ca.contiguous(), cns.contiguous(), cr.contiguous()
        stride = T
    return [q, cs, ca, cns, cr, B, T, stride]


_MEMBER_FIELDS = ("n_layer", "state_dim", "action_dim", "horizon", "test")


def forward_train_population(models, batches, precision=0):
    """``[m.forward_train(x, precision) for m, x in zip(models, batches)]`` in the same kernel launches: member i's logits, and
    after ``backward`` the ``.grad`` of its parameters, are bit-identical to training it alone.  The members are
    same-shape Transformers (``n_layer``, ``state_dim``, ``action_dim``, ``horizon`` and ``test`` agree, else
    ``ValueError``) on one device, and the batches share B and T.  All members' parameters go through ONE autograd
    Function; a member whose logits get no gradient keeps ``.grad`` as it was, as if it had not been trained.  At most
    ``POPULATION_MAX`` members per call are launched together; larger populations are cut into such calls."""
    models, batches = list(models), list(batches)
    if precision not in (0, 1):
        raise ValueError("forward_train: precision=%r, training supports 0 (fp32) and 1 (bf16)" % (precision,))
    if len(models) != len(batches):
        raise ValueError("forward_train_population: %d models and %d batches" % (len(models), len(batches)))
    if not models:
        return []
    m0 = models[0]
    devs = [next(m.parameters()).device for m in models]
    for i, m in enumerate(models):
        if m.dropout > 0:
            raise NotImplementedError("forward_train: dropout=%g, the fused training path has no dropout" % m.dropout)
        for f in _MEMBER_FIELDS:
            if getattr(m, f) != getattr(m0, f):
                raise ValueError("forward_train_population: member %d has %s=%r, member 0 has %r"
                                 % (i, f, getattr(m, f), getattr(m0, f)))
        if devs[i] != devs[0]:
            raise ValueError("forward_train_population: member %d is on %s, member 0 on %s" % (i, devs[i], devs[0]))
    dev = kernels._dev()
    if devs[0] != dev:
        for m in models:
            m.to(dev)
    ins = [_batch_inputs(x, dev) for x in batches]
    for i, x in enumerate(ins):
        if x[5:7] != ins[0][5:7]:
            raise ValueError("forward_train_population: batch %d has B, T = %d, %d, batch 0 has %d, %d"
                             % (i, x[5], x[6], ins[0][5], ins[0][6]))
    if len({x[7] for x in ins}) > 1:   # one context row stride per call
        for x in ins:
            x[1:5] = [t.contiguous() for t in x[1:5]]
            x[7] = x[6]
    out = []
    for a in range(0, len(models), POPULATION_MAX):
        ms = models[a:a + POPULATION_MAX]
        params = [p for m in ms for p in m._train_params()]
        out += list(_PopulationTrainFn.apply(ms, ins[a:a + POPULATION_MAX], precision, *params))
    return out


POPULATION_MAX = 32   # DPT_GPT2_POPULATION_MAX: members per population launch


class _TrainCall:
    """The arguments of dpt_gpt2_train_forward / dpt_gpt2_train_backward for k same-shape members: the weights array over
    the members' parameter tensors, the HOST arrays of k device pointers (refilled by every call, never reallocated) and
    the workspace that holds the saved activations from a forward to its backward."""

    def __init__(self, models, params, precision):
        k = len(models)
        n = len(params) // k
        self.models, self.k, self.precision, self._keep = models, k, precision, []
        self.w = (_lib.Gpt2Weights * k)(*[_weights_struct(m, params[i * n:(i + 1) * n], self._keep)
                                          for i, m in enumerate(models)])
        self._arrays = [(ctypes.c_void_p * k)() for _ in range(6)]   # query, the four context inputs, out / dout
        self.ws = None

    def reserve(self, B, T, dev):
        """Allocate the workspace for calls of up to B sequences of T transitions."""
        nbytes = lib().dpt_gpt2_train_workspace_bytes(self.w, self.k, B, T, self.precision)
        self.ws = torch.empty((max(int(nbytes), 16),), dtype=torch.uint8, device=dev)

    def _fill(self, j, ptrs):
        a = self._arrays[j]
        a[:] = ptrs
        return a

    def grads(self, tensors):
        """dpt_gpt2_grads_t of every member over ``tensors[i]`` (ordered as Transformer._train_params)."""
        return (_lib.Gpt2Grads * self.k)(*[_pointer_struct(_lib.Gpt2Grads, m, ts, self._keep)
                                           for m, ts in zip(self.models, tensors)])

    def forward(self, inputs, outs, B, T, stride, test):
        """``inputs[i]``: member i's query states and four context tensors; ``outs[i]``: its logits."""
        ins = [self._fill(j, [x[j].data_ptr() if j == 0 or T else None for x in inputs]) for j in range(5)]
        check(lib().dpt_gpt2_train_forward(self.w, self.k, *ins, B, T, stride, 1 if test else 0, self.precision,
                                           self._fill(5, [o.data_ptr() for o in outs]), self.ws.data_ptr(), self.ws.numel(),
                                           stream_ptr()), "dpt_gpt2_train_forward")

    def backward(self, douts, grads, B, T, test):
        """``douts[i]``: the gradient of member i's logits; ``grads``: from ``self.grads``."""
        check(lib().dpt_gpt2_train_backward(self.w, self.k, self._fill(5, [d.data_ptr() for d in douts]), B, T, 1 if test else 0,
                                            self.precision, grads, self.ws.data_ptr(), self.ws.numel(), stream_ptr()),
              "dpt_gpt2_train_backward")


class _PopulationTrainFn(torch.autograd.Function):
    """dpt_gpt2_train_forward / dpt_gpt2_train_backward over k members.  One workspace holds every member's saved
    activations between the two."""

    @staticmethod
    def forward(ctx, models, inputs, precision, *params):
        ctx.set_materialize_grads(False)
        k, m0 = len(models), models[0]
        B, T, stride = inputs[0][5:8]
        dev = inputs[0][0].device
        call = _TrainCall(models, params, precision)
        call.reserve(B, T, dev)
        outs = [torch.empty((B, m0.action_dim) if m0.test else (B, T, m0.action_dim), dtype=torch.float32, device=dev)
                for _ in range(k)]
        call.forward([x[:5] for x in inputs], outs, B, T, stride, m0.test)
        ctx.call, ctx.B, ctx.T, ctx.test, ctx.out_shape = call, B, T, m0.test, outs[0].shape
        ctx.save_for_backward(*params)
        return tuple(outs)

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, *douts):
        params = ctx.saved_tensors
        call, k = ctx.call, ctx.call.k
        n = len(params) // k
        dev = params[0].device
        grads = []
        for i in range(k):   # one buffer per member, a view per parameter
            ps = params[i * n:(i + 1) * n]
            flat = torch.empty(sum(p.numel() for p in ps), dtype=torch.float32, device=dev)
            o = 0
            for p in ps:
                grads.append(flat[o:o + p.numel()].view_as(p))
                o += p.numel()
        if ctx.B == 0:
            for g in grads:
                g.zero_()
        else:
            # a member whose logits got no gradient runs on a zero dout; its gradients are dropped below
            ds = [torch.zeros(ctx.out_shape, dtype=torch.float32, device=dev) if d is None else d.to(torch.float32).contiguous()
                  for d in douts]
            call.backward(ds, call.grads([grads[i * n:(i + 1) * n] for i in range(k)]), ctx.B, ctx.T, ctx.test)
        ctx.call = None
        return (None, None, None, *[None if douts[i // n] is None else g for i, g in enumerate(grads)])


ONLINE_POPULATION_MAX = 16              # DPT_GPT2_ONLINE_POPULATION_MAX: members per population launch of the online loop
ONLINE_KV_LAUNCH_BYTES = 8 * 1024 ** 3   # K/V scratch one population launch may take (one member may take more on its own)
_ONLINE_FIELDS = ("horizon", "state_dim", "action_dim", "n_layer", "precision")


def online_launch_groups(k, kv_bytes_per_member):
    """[(first, stop)] member ranges of the population launches for ``k`` members of ``kv_bytes_per_member`` bytes of K/V
    scratch each: at most ONLINE_POPULATION_MAX members and ONLINE_KV_LAUNCH_BYTES of scratch per launch, at least one
    member.  At 100 envs x H = 500 fp32 a member takes 52 MB and a launch holds 16; at 10 000 envs it takes 5.2 GB and
    runs alone -- where one member fills the GPU, grouping gains nothing, and a population must never need more memory
    than k one-model calls."""
    per = max(1, min(ONLINE_POPULATION_MAX, ONLINE_KV_LAUNCH_BYTES // max(1, int(kv_bytes_per_member))))
    return [(a, min(k, a + per)) for a in range(0, k, per)]


@torch.no_grad()
def online_loop_population(models, means, horizon, var, sample, seed, env_id0=0, materialise=True, regret=True, inject=None,
                           dump=False, reward_type="uniform"):
    """``[m.online_loop(means, horizon, ...) for m in models]`` in shared launches: the bandit online loop of several
    same-shape Transformers on the same tasks and the same noise (same means, seed, env ids, inject).  Member i's dict is
    bit for bit what ``models[i].online_loop`` returns alone (``regret_sums`` are float64 atomics: equal up to their order
    of addition).  Members must agree on ``horizon``, ``state_dim``, ``action_dim``, ``n_layer``, ``precision`` and the
    device, else ``ValueError`` naming the member and the field.  Populations are cut into launches by
    ``online_launch_groups``."""
    models = list(models)
    if not models:
        return []
    m0 = models[0]
    devs = [next(m.parameters()).device for m in models]
    for i, m in enumerate(models):
        for f in _ONLINE_FIELDS:
            if getattr(m, f) != getattr(m0, f):
                raise ValueError("online_loop_population: member %d has %s=%r, member 0 has %r"
                                 % (i, f, getattr(m, f), getattr(m0, f)))
        if devs[i] != devs[0]:
            raise ValueError("online_loop_population: member %d is on %s, member 0 on %s" % (i, devs[i], devs[0]))
    dev = kernels._dev()
    hs = [m.handle() for m in models]
    means = kernels._as(means, torch.float32, dev)
    N, d = means.shape
    assert d == m0.action_dim
    H, k = horizon, len(models)
    outs = []
    for _ in models:
        out = {"cum_means": torch.empty((H, N), dtype=torch.float32, device=dev)}
        if regret:
            out["regret_sums"] = torch.zeros((H, 4), dtype=torch.float64, device=dev)
        if materialise:
            out.update(context_states=torch.empty((N, H, 1), dtype=torch.float32, device=dev),
                       context_actions=torch.empty((N, H, d), dtype=torch.float32, device=dev),
                       context_next_states=torch.empty((N, H, 1), dtype=torch.float32, device=dev),
                       context_rewards=torch.empty((N, H, 1), dtype=torch.float32, device=dev))
        if dump:
            out["noise"] = {"reward_z": torch.empty((H, N), dtype=torch.float32, device=dev),
                            "ctrl_u": torch.zeros((H, N), dtype=torch.float64, device=dev),
                            "logits": torch.empty((H, N, d), dtype=torch.float32, device=dev)}
        outs.append(out)
    inj_p, keep = None, []
    if inject is not None:
        s = _lib.Gpt2OnlineInject()
        for key, dt in (("reward_z", torch.float32), ("ctrl_u", torch.float64)):
            if inject.get(key) is not None:
                t = kernels._as(inject[key], dt, dev)
                keep.append(t)
                setattr(s, key, ptr(t))
        inj_p = ctypes.byref(s)
    kv_bytes = lib().dpt_gpt2_online_kv_bytes(hs[0], N, H, m0.precision)
    for a, b in online_launch_groups(k, kv_bytes):
        n, os_ = b - a, outs[a:b]
        # one member reuses its model's scratch, as the one-model call always has; a group takes a buffer of its own
        kv = models[a]._scratch(kv_bytes) if n == 1 else torch.empty((max(n * int(kv_bytes), 1),), dtype=torch.uint8, device=dev)
        arr = lambda vals: (ctypes.c_void_p * n)(*vals)   # noqa: E731
        col = lambda key: arr([ptr(o.get(key)) for o in os_])   # noqa: E731
        dump_p = None
        if dump:
            dump_p = (_lib.Gpt2OnlineDump * n)(*[_lib.Gpt2OnlineDump(**{key: ptr(t) for key, t in o["noise"].items()}) for o in os_])
        check(lib().dpt_gpt2_online_loop(arr(hs[a:b]), n, ptr(means), float(var), kernels.REWARD_TYPES[reward_type],
                                         1 if sample else 0, seed, env_id0, N, H, m0.precision, ptr(kv), kv.numel(),
                                         col("context_states"), col("context_actions"), col("context_next_states"),
                                         col("context_rewards"), col("cum_means"), col("regret_sums"), inj_p, dump_p,
                                         stream_ptr()), "dpt_gpt2_online_loop")
    return outs


class _Decoder:
    """See ``Transformer.decoder``.  Owns its K/V cache (per sequence [L][2][Tpad][32], fp32 or bf16 with
    ``model.precision``); valid while the query state of a sequence does not change (bandits: the constant [1])."""

    def __init__(self, model, n_seqs, max_transitions):
        self.model, self.n, self.t_max, self.pos = model, n_seqs, max_transitions + 1, 0
        self.precision = model.precision
        dev = kernels._dev()
        self._h = model.handle()
        nbytes = lib().dpt_gpt2_online_kv_bytes(self._h, n_seqs, self.t_max, self.precision)
        self.kv = torch.empty((max(int(nbytes), 1),), dtype=torch.uint8, device=dev)
        self.din = 2 * model.state_dim + model.action_dim + 1
        self._tok = torch.zeros((n_seqs, self.din), dtype=torch.float32, device=dev)

    def _step(self):
        # the handle is owned by the model and destroyed when its weights change (handle() repacks): a decoder must
        # never launch on a freed blob, and its K/V cache belongs to the old weights anyway
        if self.model.handle() is not self._h:
            raise RuntimeError("the model's weights changed since this decoder was created: build a new decoder")
        out = torch.empty((self.n, self.model.action_dim), dtype=torch.float32, device=self._tok.device)
        check(lib().dpt_gpt2_decode_step(self._h, ptr(self._tok), self.n, self.pos, self.t_max, self.precision, ptr(self.kv),
                                         self.kv.numel(), ptr(out), stream_ptr()), "dpt_gpt2_decode_step")
        self.pos += 1
        return out

    @torch.no_grad()
    def query(self, query_states):
        assert self.pos == 0, "the query token is position 0"
        dx = self.model.state_dim
        self._tok.zero_()
        self._tok[:, :dx] = torch.as_tensor(query_states, dtype=torch.float32).to(self._tok.device).reshape(self.n, dx)
        return self._step()

    @torch.no_grad()
    def append(self, states, actions, next_states, rewards):
        assert 0 < self.pos < self.t_max, "query() first; at most max_transitions appends"
        dx, du, dev = self.model.state_dim, self.model.action_dim, self._tok.device
        f = lambda a, w: torch.as_tensor(a, dtype=torch.float32).to(dev).reshape(self.n, w)   # noqa: E731
        self._tok[:, :dx] = f(states, dx)
        self._tok[:, dx:dx + du] = f(actions, du)
        self._tok[:, dx + du:2 * dx + du] = f(next_states, dx)
        self._tok[:, 2 * dx + du:] = f(rewards, 1)
        return self._step()
