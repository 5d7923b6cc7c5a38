"""Pretraining loop of the reference's train.py (SURVEY §2.1) on device-resident datasets.

``train(model, train_dataset, test_dataset, num_epochs)`` runs the reference's epochs: the test loss under
``no_grad`` through ``model.forward`` first, then one pass over the training set with ``torch.optim.AdamW(lr,
weight_decay)``, batch 64, and the sum-reduced cross-entropy of the logits of every context row against the
optimal action.  Both epoch losses are reported as the reference reports them: sum of the batch losses / horizon /
len(dataset).  The forward of training is ``model.forward_train`` (hand-written CUDA forward and backward).
``train_population`` trains k same-shape models at once, each bit-identical to ``train`` on it alone.

Unlike the reference's DataLoader, batches are gathered on the device from ``Dataset.dataset`` with a seeded
permutation (and, with ``Dataset.shuffle``, a seeded per-item context permutation), and the losses stay on the
device until one host read per epoch.  There is no argparse or plotting.

Every trainer can write a training-state file at epoch (iteration) boundaries and resume from it (``state_path``,
``save_every``, ``resume``); a resumed run ends bit-identical to the run that was never interrupted (``checkpoint``).
``train`` and ``train_population`` also write the reference's weight files (``weights_dir``, ``stems``).

``train_interactive`` is the on-policy trainer of the reference's train_interactive.py (:97-139): every iteration rolls
out a fresh ``GPUBanditEnv`` with the current model and takes one AdamW step on the cross-entropy of the last logits
against the optimal arm.  ``dist.train_interactive_sharded`` runs the same code over a box's GPUs.
"""
import os

import torch
import torch.nn.functional as F

from . import checkpoint as C

_CTX = ("context_states", "context_actions", "context_next_states", "context_rewards")
_KEYS = _CTX + ("query_states", "optimal_actions")


def ce_sum_loss(pred, batch):
    """train.py's loss: CrossEntropyLoss(reduction='sum') of every row's logits against the optimal action (one-hot
    probability targets) repeated over the rows."""
    du = pred.shape[-1]
    target = batch["optimal_actions"]
    if pred.dim() == 3:
        target = target.unsqueeze(1).expand(-1, pred.shape[1], -1)
    return F.cross_entropy(pred.reshape(-1, du), target.reshape(-1, du), reduction="sum")


def train_step(model, optimizer, batch, loss_fn=ce_sum_loss, precision=0):
    """One optimizer step: ``model.forward_train(batch, precision)``, ``loss_fn(pred, batch)``, backward,
    ``optimizer.step()``.  Returns the loss as a device tensor (no host synchronisation)."""
    optimizer.zero_grad()
    pred = model.forward_train(batch, precision)
    loss = loss_fn(pred, batch)
    loss.backward()
    optimizer.step()
    return loss.detach()


def batches(dataset, batch_size, generator, shuffle_items=None):
    """The dataset's items in a seeded random order, ``batch_size`` at a time (the last batch may be smaller), gathered
    on the device.  ``shuffle_items`` (default: ``dataset.shuffle``) permutes each item's context rows."""
    data = dataset.dataset
    dev = data["context_actions"].device
    n = data["context_actions"].shape[0]
    shuffle_items = dataset.shuffle if shuffle_items is None else shuffle_items
    order = torch.randperm(n, generator=generator, device=generator.device).to(dev)
    for i in range(0, n, batch_size):
        idx = order[i:i + batch_size]
        b = {k: data[k][idx] for k in _KEYS}
        if shuffle_items:
            H = b["context_actions"].shape[1]
            perm = torch.argsort(torch.rand((idx.shape[0], H), generator=generator, device=generator.device).to(dev), dim=1)
            for k in _CTX:
                b[k] = torch.gather(b[k], 1, perm.unsqueeze(-1).expand(-1, -1, b[k].shape[-1]))
        yield b


def train(model, train_dataset, test_dataset, num_epochs, batch_size=64, lr=1e-3, weight_decay=1e-4, seed=None,
          optimizer=None, *, state_path=None, save_every=50, resume=False, weights_dir=None, stems=None, precision=0):
    """The reference's epoch loop.  Returns ``(train_loss, test_loss, optimizer)``: per-epoch lists of floats and the
    AdamW optimizer (its ``state_dict`` is the reference's).  This is the one-member case of ``train_population``, whose
    docstring describes the checkpoint arguments and ``precision``; ``stems`` is one stem here."""
    tr, te, optimizer = _population("train", [model], train_dataset, test_dataset, num_epochs, batch_size, lr, weight_decay,
                                    [seed], optimizer, state_path, save_every, resume, weights_dir,
                                    None if stems is None else [stems], precision)
    return tr[0], te[0], optimizer


def train_population_step(models, optimizer, batches, loss_fn=ce_sum_loss, precision=0):
    """One optimizer step of every member: ``forward_train_population``, the loss of each member on its own batch, one
    backward and ``optimizer.step()``.  Member i's gradient is the one ``train_step(models[i], ..., batches[i])`` computes,
    bit for bit.  With the default loss the cross-entropy runs once on the stacked logits (per-row reduction, then a sum
    per member), so a member's loss value can differ from ``train_step``'s in the last bits (within 1e-6 relative); with
    one member, or another ``loss_fn``, each member's loss is ``loss_fn(pred, batch)`` as in ``train_step``.  Returns the
    losses as one device tensor [k] (no host synchronisation).  ``precision``: that of ``forward_train_population``."""
    from .models.net import forward_train_population
    optimizer.zero_grad()
    preds = forward_train_population(models, batches, precision)
    if loss_fn is ce_sum_loss and len(preds) > 1:
        pred = torch.stack(preds)
        du, k = pred.shape[-1], pred.shape[0]
        target = torch.stack([b["optimal_actions"] for b in batches])
        if pred.dim() == 4:
            target = target.unsqueeze(2).expand(-1, -1, pred.shape[2], -1)
        losses = F.cross_entropy(pred.reshape(-1, du), target.reshape(-1, du), reduction="none").view(k, -1).sum(1)
    else:
        losses = torch.stack([loss_fn(p, b) for p, b in zip(preds, batches)])
    losses.sum().backward()
    optimizer.step()
    return losses.detach()


def _per_member(v, k, name):
    v = list(v) if isinstance(v, (list, tuple)) else [v] * k
    if len(v) != k:
        raise ValueError("train_population: %d values of %s for %d models" % (len(v), name, k))
    return v


def _population_batches(datasets, batch_size, gens):
    """``batches(datasets[i], batch_size, gens[i])`` of every member, step by step: yields a list of k batch dicts.  Each
    member draws from its own generator in the order ``batches`` does, so its batches are the ones ``train`` gathers.
    Members that share a dataset are gathered with one index per key (and one context permutation gather)."""
    k = len(datasets)
    groups = {}
    for i, d in enumerate(datasets):
        groups.setdefault(id(d), []).append(i)
    data0 = datasets[0].dataset
    n = data0["context_actions"].shape[0]
    dev = data0["context_actions"].device
    orders = [torch.randperm(n, generator=g, device=g.device).to(dev) for g in gens]
    for a in range(0, n, batch_size):
        out = [None] * k
        for members in groups.values():
            ds = datasets[members[0]]
            data = ds.dataset
            idx = [orders[i][a:a + batch_size] for i in members]
            nb = idx[0].shape[0]
            cat = torch.cat(idx) if len(idx) > 1 else idx[0]
            b = {key: data[key][cat] for key in _KEYS}
            if ds.shuffle:
                H = b["context_actions"].shape[1]
                perm = [torch.argsort(torch.rand((nb, H), generator=gens[i], device=gens[i].device).to(dev), dim=1) for i in members]
                perm = torch.cat(perm) if len(perm) > 1 else perm[0]
                for key in _CTX:
                    b[key] = torch.gather(b[key], 1, perm.unsqueeze(-1).expand(-1, -1, b[key].shape[-1]))
            for j, i in enumerate(members):
                out[i] = {key: v[j * nb:(j + 1) * nb] for key, v in b.items()} if len(members) > 1 else b
        yield out


def train_population(models, train_datasets, test_datasets, num_epochs, batch_size=64, lr=1e-3, weight_decay=1e-4, seeds=None,
                     optimizer=None, *, state_path=None, save_every=50, resume=False, weights_dir=None, stems=None,
                     precision=0):
    """``train`` of k same-shape models at once (``forward_train_population``): the members' forward and backward run in
    the same kernel launches, their batches are gathered together and their AdamW updates go through one optimizer.

    ``train_datasets`` / ``test_datasets``: one ``Dataset`` shared by every member or a list of k; all datasets of one
    split have the same length, so that the members' steps line up.  ``lr``, ``weight_decay`` and ``seeds``: a scalar or
    a list of k.  The default optimizer is one ``torch.optim.AdamW`` with a parameter group per distinct (lr,
    weight_decay); AdamW's update is elementwise, so the grouping does not change any weight.

    Member i ends bit-identical to ``train(models[i], train_i, test_i, num_epochs, batch_size, lr_i, weight_decay_i,
    seed=seeds[i])``: the same weights and the same AdamW state of its parameters.  Its test losses are bit for bit
    ``train``'s (the same per-member computation); its train losses are summed from the stacked cross-entropy of
    ``train_population_step`` and match ``train``'s within 1e-6 relative (bit for bit when k = 1).  Returns
    ``(train_loss, test_loss, optimizer)``: ``train_loss[i][e]`` and ``test_loss[i][e]`` are floats.

    Checkpoints (all off by default):

    - ``state_path``: the training state (``checkpoint``) is written there after every epoch e with
      ``(e + 1) % save_every == 0`` and after the last epoch (``save_every=10`` is the reference's linear-bandit cadence).
    - ``resume=True``: if ``state_path`` exists, the models, the optimizer (built as without it, then
      ``load_state_dict``) and the batch generators are restored from it and training continues at its next epoch;
      otherwise training starts from scratch.  ``num_epochs`` stays the total, and the loss lists returned are the full
      ones.  The result is bit-identical to the call that was never interrupted.  A state that does not match the call
      (model configs, member count, ``batch_size``, lr, weight_decay, seeds, dataset lengths, shuffle flags and sharing,
      optimizer groups) raises ``ValueError`` before anything is modified.
    - ``weights_dir`` with ``stems`` (k distinct stems, e.g. from ``utils.build_bandit_model_filename``): member i's
      ``state_dict`` goes to ``{weights_dir}/{stems[i]}_epoch{e + 1}.pt`` at the same epochs and to
      ``{weights_dir}/{stems[i]}.pt`` at the end (``checkpoint.save_weights``), as the reference's train.py writes them.

    ``precision``: the precision of the training steps (``forward_train``): 0 = fp32 (default), 1 = bf16 mixed precision
    with fp32 master weights and AdamW state.  The test loss is ``model.forward`` at ``model.precision`` either way.  A
    resume must repeat it (a state saved at one precision and resumed at the other raises ``ValueError``); states written
    before this argument existed were fp32 and resume at 0.  The weight files do not depend on it."""
    return _population("population", models, train_datasets, test_datasets, num_epochs, batch_size, lr, weight_decay, seeds,
                       optimizer, state_path, save_every, resume, weights_dir, stems, precision)


def _population(kind, models, train_datasets, test_datasets, num_epochs, batch_size, lr, weight_decay, seeds, optimizer,
                state_path, save_every, resume, weights_dir, stems, precision):
    models = list(models)
    k = len(models)
    if k == 0:
        return [], [], optimizer
    trs, tes = _per_member(train_datasets, k, "train_datasets"), _per_member(test_datasets, k, "test_datasets")
    lrs, wds = _per_member(lr, k, "lr"), _per_member(weight_decay, k, "weight_decay")
    seeds = _per_member(seeds, k, "seeds")
    _check_saving(state_path, save_every, resume)
    if precision not in (0, 1):
        raise ValueError("train_population: precision=%r, training supports 0 (fp32) and 1 (bf16)" % (precision,))
    if weights_dir is not None:
        stems = _per_member(stems, k, "stems")
        if None in stems or len(set(stems)) != k:
            raise ValueError("train_population: weights_dir needs %d distinct stems, got %r" % (k, stems))
    for split, ds in (("train", trs), ("test", tes)):
        for i, d in enumerate(ds):
            if len(d) != len(ds[0]):
                raise ValueError("train_population: %s dataset of member %d has %d items, member 0's has %d"
                                 % (split, i, len(d), len(ds[0])))
    dev = trs[0].dataset["context_actions"].device
    for m in models:
        if next(m.parameters()).device != dev:
            m.to(dev)
    if optimizer is None:
        groups = {}
        for m, a, b in zip(models, lrs, wds):
            groups.setdefault((a, b), []).extend(m.parameters())
        optimizer = torch.optim.AdamW([{"params": ps, "lr": a, "weight_decay": b} for (a, b), ps in groups.items()])
    gens = []
    for s in seeds:
        g = torch.Generator(device=dev)
        if s is None:
            g.seed()
        else:
            g.manual_seed(s)
        gens.append(g)
    horizon = models[0].horizon
    train_loss, test_loss = [[] for _ in range(k)], [[] for _ in range(k)]
    args = C.train_args(batch_size, lrs, wds, seeds, trs, tes, dev, precision)
    e0 = 0
    if resume and os.path.exists(state_path):
        e0, hist = C.load_state(state_path, kind, models, optimizer, args, num_epochs, gens)
        train_loss, test_loss = hist["train_loss"], hist["test_loss"]
    for e in range(e0, num_epochs):
        with torch.no_grad():
            te = [torch.zeros((), dtype=torch.float32, device=dev) for _ in range(k)]
            for bs in _population_batches(tes, batch_size, gens):
                for i, (m, b) in enumerate(zip(models, bs)):
                    te[i] += ce_sum_loss(m(b), b)
        tr = torch.zeros((k,), dtype=torch.float32, device=dev)
        for bs in _population_batches(trs, batch_size, gens):
            if k == 1:
                tr[0] += train_step(models[0], optimizer, bs[0], precision=precision)
            else:
                tr += train_population_step(models, optimizer, bs, precision=precision)
        losses = torch.stack([torch.stack(te) / horizon / len(tes[0]), tr / horizon / len(trs[0])]).tolist()   # one host read
        for i in range(k):
            test_loss[i].append(losses[0][i])
            train_loss[i].append(losses[1][i])
        # weight files first: a state written after them means they are on disk, and a resume rewrites them otherwise
        if weights_dir is not None and (e + 1) % save_every == 0:
            for m, stem in zip(models, stems):
                C.save_weights(m, weights_dir, stem, e + 1)
        if state_path is not None and ((e + 1) % save_every == 0 or e + 1 == num_epochs):
            C.save_state(state_path, C.training_state(kind, models, optimizer, args, e + 1,
                                                      {"train_loss": train_loss, "test_loss": test_loss}, gens))
    if weights_dir is not None:
        for m, stem in zip(models, stems):
            C.save_weights(m, weights_dir, stem)
    return train_loss, test_loss, optimizer


def _check_saving(state_path, save_every, resume):
    if save_every < 1:
        raise ValueError("save_every=%r, it must be >= 1" % (save_every,))
    if resume and state_path is None:
        raise ValueError("resume=True needs a state_path")



def interactive_loss(last_logits, target, n_envs):
    """train_interactive.py's loss: the mean over the iteration's ``n_envs`` envs of the cross-entropy of the last logits
    against the optimal arm index.  It is written as the sum over the rows given divided by ``n_envs``, so that the losses
    (and gradients) of the micro-batches add up to those of the whole batch."""
    return F.cross_entropy(last_logits, target, reduction="sum") / n_envs


def train_interactive(model, dim, n_envs, K, n_iters, mb=1024, var=0.0, env_type="uniform", seed=0, lr=1e-3,
                      weight_decay=1e-4, optimizer=None, timings=None, *, state_path=None, save_every=50, resume=False,
                      precision=0):
    """On-policy training (train_interactive.py:97-139) on one GPU.  Iteration ``it``:

    1. ``env = GPUBanditEnv(dim, n_envs, K, var, env_type, seed=rng.key_for(seed, it))``;
    2. ``env.rollout(model, K, sample=True)``: the fused K-step rollout with the current weights (``model.precision``);
    3. the last logits on ``context[:, :K-1]`` with a gradient (``dpt_gpt2_train_population_forward_ex`` with one member,
       last position, whatever ``model.test`` says), ``interactive_loss`` against ``env.opt_a_index`` and
       ``dpt_gpt2_train_population_backward_ex``, one micro-batch of ``mb`` envs at a time (micro-batch m is envs
       ``[m*mb, min(n_envs, (m+1)*mb))``), each into its own gradient slot;
    4. the slots summed in micro-batch order into the parameters' ``.grad`` (one flat buffer; ``transformer.wte`` gets
       none), then ``optimizer.step()`` (default ``torch.optim.AdamW(lr, weight_decay)``).

    ``precision``: the precision of step 3 only, as in ``train``: 0 = fp32 (default), 1 = bf16 mixed precision with fp32
    master weights, gradient slots, gradient sum and AdamW state.  The rollout of step 2 runs at ``model.precision``
    whatever ``precision`` is.  Values other than 0 and 1 raise ``ValueError`` before anything else is checked.

    With ``mb >= n_envs`` an iteration is exactly ``env.rollout`` + ``forward_train(b, precision)`` + ``interactive_loss``
    + ``backward`` + ``step``.  The result does not depend on how the micro-batches are spread over GPUs
    (``dist.train_interactive_sharded``), only on ``mb``.  ``dropout == 0`` and K <= 512 (the limits of ``forward_train``),
    checked before the first rollout.  ``n_envs == 0`` runs nothing.  ``timings``: a list that receives, per iteration,
    the CUDA-event milliseconds of the rollout, the forward and backward of all micro-batches, the exchange (host barrier
    to the end of the sum), the optimizer and the whole iteration.  Returns ``(losses, optimizer)``: the per-iteration
    losses (one host read at the end) and the optimizer.

    ``state_path``, ``save_every`` and ``resume`` work as in ``train_population``, per iteration: the state is written
    after every iteration it with ``(it + 1) % save_every == 0`` and after the last one, and a resumed call continues at
    the saved iteration with its keys ``rng.key_for(seed, it)``; ``n_iters`` stays the total.  The arguments a resume must
    repeat are ``dim``, ``n_envs``, ``K``, ``mb``, ``var``, ``env_type``, ``seed``, ``lr``, ``weight_decay`` and
    ``precision`` (states written before ``precision`` existed were fp32 and resume at 0), not the world size: a state
    saved by ``dist.train_interactive_sharded`` at one world size resumes at any other."""
    return _interactive(model, dim, n_envs, K, n_iters, mb, 0, 1, var=var, env_type=env_type, seed=seed, lr=lr,
                        weight_decay=weight_decay, optimizer=optimizer, timings=timings, state_path=state_path,
                        save_every=save_every, resume=resume, precision=precision)


def _agree(err, ws):
    """Every rank learns whether any rank failed (so that no rank is left blocked in a collective); raises if one did."""
    bad = []
    if ws > 1:
        import torch.distributed as tdist
        msgs = [None] * ws
        tdist.all_gather_object(msgs, None if err is None else "%s: %s" % (type(err).__name__, err))
        bad = [(r, m) for r, m in enumerate(msgs) if m is not None]
    if err is not None:
        raise err
    if bad:
        raise RuntimeError("train_interactive failed on rank %d: %s" % bad[0])


def _interactive(model, dim, n_envs, K, n_iters, mb, rank, ws, var=0.0, env_type="uniform", seed=0, lr=1e-3,
                 weight_decay=1e-4, optimizer=None, timings=None, state_path=None, save_every=50, resume=False, precision=0):
    """train_interactive on rank ``rank`` of ``ws`` (ws == 1: the one-GPU trainer; see dist.train_interactive_sharded)."""
    if precision not in (0, 1):
        raise ValueError("train_interactive: precision=%r, training supports 0 (fp32) and 1 (bf16)" % (precision,))
    import ctypes
    from . import _lib, dist as D, kernels, rng
    from ._lib import check, lib, stream_ptr
    from .envs.gpu_bandit_env import GPUBanditEnv
    from .models import net
    if model.dropout > 0:
        raise NotImplementedError("train_interactive: dropout=%g, the fused training path has no dropout" % model.dropout)
    if K < 1:
        raise ValueError("train_interactive: K=%d, the rollout needs at least one step" % K)
    _check_saving(state_path, save_every, resume)
    dev = kernels._dev()
    if next(model.parameters()).device != dev:
        model.to(dev)
    if optimizer is None:
        optimizer = torch.optim.AdamW(model.parameters(), lr=lr, weight_decay=weight_decay)
    m_lo, m_hi, lo, hi = D.microbatch_shard(n_envs, mb, rank, ws)
    M = -(-n_envs // mb)
    if M == 0:
        return [], optimizer
    params = model._train_params()
    sizes = [p.numel() for p in params]
    offs = [sum(sizes[:i]) for i in range(len(sizes))]
    P = sum(sizes) + 1                 # a slot: every trained parameter (_train_params order), then the micro-batch's loss
    Ps = (P + 3) & ~3                  # slot stride: 16 B aligned slots
    T, du, st = K - 1, model.action_dim, stream_ptr()
    fwd, bwd = "dpt_gpt2_train_population_forward_ex", "dpt_gpt2_train_population_backward_ex"
    one = lambda *ps: (ctypes.c_void_p * 1)(*ps)   # noqa: E731  (the one-member pointer arrays of the population calls)
    w = (_lib.Gpt2Weights * 1)(net._weights_struct(model, params, []))
    # the train kernels' shape and precision checks (n_embd, n_layer, sequence length) before any rollout: a B = 0 call
    # only validates
    check(lib().dpt_gpt2_train_population_forward_ex(w, 1, None, None, None, None, None, 0, T, K, 1, precision, None, None, 0,
                                                     st), fwd)
    args = C.interactive_args(dim, n_envs, K, mb, var, env_type, seed, lr, weight_decay, precision)
    it0, done = 0, []
    if resume:   # every rank reads the same file; all raise if one fails to
        err = None
        try:
            if os.path.exists(state_path):
                it0, hist = C.load_state(state_path, "interactive", [model], optimizer, args, n_iters)
                done = hist["losses"]
        except Exception as e:   # noqa: BLE001
            err = e
        _agree(err, ws)
    n_local, n_mb = hi - lo, m_hi - m_lo
    peer = D.PeerBuffer(max(n_mb, 1) * Ps * 4, (rank, ws))
    try:
        slots = peer.local_f32(max(n_mb, 1) * Ps).view(-1, Ps)
        grad_slots = [[slots[j, o:o + n].view_as(p) for p, o, n in zip(params, offs, sizes)] for j in range(n_mb)]
        owner_lo = [D.microbatch_shard(n_envs, mb, r, ws)[:2] for r in range(ws)]
        src = (ctypes.c_void_p * M)(*[peer.peer_ptrs[r] + (m - a) * Ps * 4 for r, (a, b) in enumerate(owner_lo)
                                      for m in range(a, b)])
        flat = torch.zeros(Ps, dtype=torch.float32, device=dev)
        for p, o, n in zip(params, offs, sizes):
            p.grad = flat[o:o + n].view_as(p)
        losses = torch.zeros(n_iters, dtype=torch.float32, device=dev)
        losses[:it0] = torch.tensor(done, dtype=torch.float32)
        if n_local:
            q = torch.ones((min(mb, n_local), model.state_dim), dtype=torch.float32, device=dev)
            wbytes = int(lib().dpt_gpt2_train_population_workspace_bytes_ex(w, 1, min(mb, n_local), T, precision))
            work = torch.empty((max(wbytes, 16),), dtype=torch.uint8, device=dev)
        for it in range(it0, n_iters):
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(5)] if timings is not None else []
            mark = lambda i: ev and ev[i].record()   # noqa: E731
            err = None
            try:
                mark(0)
                if n_local:
                    env = GPUBanditEnv(dim, n_local, K, var, env_type, device=dev, seed=rng.key_for(seed, it), env_id0=lo)
                    ro = env.rollout(model, K, sample=True, logits=False)
                    mark(1)
                    keep = []
                    w = (_lib.Gpt2Weights * 1)(net._weights_struct(model, params, keep))
                    ctx = [ro[k] for k in _CTX]
                    for j in range(n_mb):
                        a, b = j * mb, min(n_local, (j + 1) * mb)
                        out = torch.empty((b - a, du), dtype=torch.float32, device=dev)
                        cp = [one(c[a:b].data_ptr() if T else None) for c in ctx]
                        check(lib().dpt_gpt2_train_population_forward_ex(w, 1, one(q.data_ptr()), *cp, b - a, T, K, 1, precision,
                                                                         one(out.data_ptr()), work.data_ptr(), work.numel(), st),
                              fwd)
                        lg = out.requires_grad_()
                        with torch.enable_grad():
                            loss = interactive_loss(lg, ro["target"][a:b], n_envs)
                            dout, = torch.autograd.grad(loss, lg)
                        dout = dout.contiguous()
                        g = net._pointer_struct(_lib.Gpt2Grads, model, grad_slots[j], keep)
                        check(lib().dpt_gpt2_train_population_backward_ex(w, 1, one(dout.data_ptr()), b - a, T, 1, precision,
                                                                          ctypes.byref(g), work.data_ptr(), work.numel(), st),
                              bwd)
                        slots[j, P - 1].copy_(loss.detach())
                else:
                    mark(1)
                mark(2)
                torch.cuda.current_stream().synchronize()   # this rank's slots are written ...
            except Exception as e:   # noqa: BLE001
                err = e
            _agree(err, ws)                                 # ... and so are every rank's (the exchange is a barrier)
            try:
                check(lib().dpt_ordered_sum_f32(src, M, Ps, flat.data_ptr(), st), "dpt_ordered_sum_f32")
                mark(3)
                losses[it].copy_(flat[P - 1])
                optimizer.step()
                mark(4)
                torch.cuda.current_stream().synchronize()
                # every rank holds the same weights and AdamW state; a failed write makes every rank raise
                if state_path is not None and rank == 0 and ((it + 1) % save_every == 0 or it + 1 == n_iters):
                    C.save_state(state_path, C.training_state("interactive", [model], optimizer, args, it + 1,
                                                              {"losses": losses[:it + 1].tolist()}))
            except Exception as e:   # noqa: BLE001
                err = e
            _agree(err, ws)                                 # no rank rewrites its slots before every rank has summed them
            if ev:
                timings.append({"rollout": ev[0].elapsed_time(ev[1]), "fwd_bwd": ev[1].elapsed_time(ev[2]),
                                "exchange": ev[2].elapsed_time(ev[3]), "optimizer": ev[3].elapsed_time(ev[4]),
                                "total": ev[0].elapsed_time(ev[4])})
        return losses.tolist(), optimizer
    finally:
        torch.cuda.current_stream().synchronize()           # nothing in flight uses the slots when they are freed
        peer.close()
