"""Training checkpoints: the training-state file that a run resumes from, and the reference's per-epoch weight files.

A training-state file (``save_state`` / ``load_state``) is one ``torch.save`` dict holding everything a resume needs:

- ``version`` (``VERSION``) and ``kind``: ``"train"``, ``"population"`` or ``"interactive"``;
- ``members``: per model its config (``MODEL_FIELDS``), ``state_dict()`` and, for the epoch trainers, the state of its
  batch generator (``Generator.get_state()``, so that runs seeded with ``None`` resume exactly too);
- ``optimizer``: ``optimizer.state_dict()`` (AdamW's ``exp_avg``, ``exp_avg_sq`` and ``step``);
- ``next``: the next epoch (or iteration), and ``history``: the per-epoch (per-iteration) losses so far;
- ``args``: the arguments that must be the same for the resumed run to be the uninterrupted one (``train_args``,
  ``interactive_args``).  The world size of the interactive trainer is not among them: its results do not depend on it.

The trainers only ever stand at an epoch (iteration) boundary when they save, and every source of randomness they use
is in the file (the batch generators) or keyed by the iteration (``rng.key_for(seed, it)``), with deterministic
kernels: a resumed run ends bit-identical to the run that was never interrupted.

Writes are atomic (a temporary file in the same directory, flushed to disk, then ``os.replace``): a process killed
mid-save leaves the previous file intact.  ``load_state`` checks the whole file against the call before it modifies
any model, optimizer or generator, and raises ``ValueError`` naming the first field that differs and both values.

``save_weights`` writes the reference's weight files, ``{stem}_epoch{epoch}.pt`` and ``{stem}.pt`` (train.py:313-315,331),
which the reference's eval.py loads by epoch (eval.py:141-152).
"""
import os
from collections import OrderedDict

import torch

VERSION = 1
KINDS = ("train", "population", "interactive")
# what a member's results depend on: the reference's config keys, and the inference precision that the test loss of
# the epoch trainers and the rollout of the interactive trainer run at
MODEL_FIELDS = ("horizon", "state_dim", "action_dim", "n_layer", "n_embd", "n_head", "dropout", "test", "precision")
# transformers 4.5.1 (the reference's pin) registers the causal mask of every attention layer as a persistent buffer of
# GPT2Config.n_ctx rows, whose default is 1024; the reference's GPT2Config sets n_positions only (DESIGN §1, row T1)
N_CTX = 1024


def model_config(model):
    return {f: getattr(model, f) for f in MODEL_FIELDS}


def weights(model):
    """``model.state_dict()`` as a plain ordered dict of tensors.  It leaves out ``state_dict()``'s ``_metadata``, where
    ``Transformer``'s own ``_version`` method (the weight-version key of its device handle) lands in place of torch's
    integer: pickled, it names this package's class, which ``torch.load(weights_only=True)`` refuses and the reference
    cannot import."""
    return OrderedDict(model.state_dict())


def train_args(batch_size, lrs, wds, seeds, train_datasets, test_datasets, device, precision=0):
    """The arguments of ``train`` / ``train_population`` that a resume must repeat: the batch size, the device the batches
    are drawn on, the training precision (``forward_train``'s), and per member its lr, weight_decay and seed, the length
    and shuffle flag of its train and test datasets and which members share them (``train_set`` / ``test_set``: the first
    member with the same dataset)."""
    def first(ds, i):
        return next(j for j in range(i + 1) if ds[j] is ds[i])
    members = []
    for i in range(len(lrs)):
        a = {"lr": float(lrs[i]), "weight_decay": float(wds[i]), "seed": None if seeds[i] is None else int(seeds[i])}
        for split, ds in (("train", train_datasets), ("test", test_datasets)):
            a.update({split + "_items": len(ds[i]), split + "_shuffle": bool(ds[i].shuffle), split + "_set": first(ds, i)})
        members.append(a)
    return {"batch_size": int(batch_size), "device": torch.device(device).type, "precision": int(precision), "members": members}


def interactive_args(dim, n_envs, K, mb, var, env_type, seed, lr, weight_decay, precision=0):
    """The arguments of ``train_interactive`` / ``dist.train_interactive_sharded`` that a resume must repeat, the training
    precision of the gradient half among them."""
    return {"dim": int(dim), "n_envs": int(n_envs), "K": int(K), "mb": int(mb), "var": float(var), "env_type": str(env_type),
            "seed": int(seed), "lr": float(lr), "weight_decay": float(weight_decay), "precision": int(precision)}


def training_state(kind, models, optimizer, args, next_index, history, generators=None):
    """The training-state dict of ``models`` and ``optimizer`` (see the module docstring).  The tensors are the live
    ones: save the dict before the next step."""
    if kind not in KINDS:
        raise ValueError("unknown training-state kind %r (known: %s)" % (kind, ", ".join(KINDS)))
    members = [{"config": model_config(m), "model": weights(m),
                "generator": None if generators is None else generators[i].get_state()} for i, m in enumerate(models)]
    return {"version": VERSION, "kind": kind, "args": args, "members": members, "optimizer": optimizer.state_dict(),
            "next": int(next_index), "history": history}


def _atomic_save(obj, path):
    path = os.fspath(path)
    tmp = "%s.%d.tmp" % (path, os.getpid())
    try:
        with open(tmp, "wb") as f:
            torch.save(obj, f)
            f.flush()
            os.fsync(f.fileno())
        os.replace(tmp, path)
    except BaseException:
        if os.path.exists(tmp):
            os.unlink(tmp)
        raise
    d = os.open(os.path.dirname(os.path.abspath(path)), os.O_RDONLY)   # the rename survives a crash once the
    try:                                                                 # directory is on disk too
        os.fsync(d)
    finally:
        os.close(d)


def save_state(path, state):
    """Writes the training-state dict ``state`` to ``path`` atomically."""
    _atomic_save(state, path)


def _differ(name, ours, theirs, who=""):
    return ValueError("%s%s=%r, the checkpoint %r" % (who, name, ours, theirs))


def _compare(ours, theirs, who=""):
    for key in list(ours) + [k for k in theirs if k not in ours]:
        if key not in ours or key not in theirs or ours[key] != theirs[key]:
            raise _differ(key, ours.get(key), theirs.get(key), who)


def check_state(state, kind, models, optimizer, args, total):
    """Raises ``ValueError`` unless ``state`` is a training state of ``kind`` that ``models``, ``optimizer`` and ``args``
    can resume exactly, within ``total`` epochs (iterations).  Modifies nothing."""
    if not isinstance(state, dict) or state.get("version") != VERSION:
        raise ValueError("training state of format version %r; this package reads version %d"
                         % (state.get("version") if isinstance(state, dict) else None, VERSION))
    if state.get("kind") not in KINDS:
        raise ValueError("training state of unknown kind %r (known: %s)" % (state.get("kind"), ", ".join(KINDS)))
    if state["kind"] != kind:
        raise _differ("kind", kind, state["kind"])
    if state["next"] > total:
        name, unit = ("n_iters", "iteration") if kind == "interactive" else ("num_epochs", "epoch")
        raise ValueError("%s=%d, the checkpoint is past it, at %s %d" % (name, total, unit, state["next"]))
    saved = state["members"]
    if len(models) != len(saved):
        raise ValueError("%d members, the checkpoint %d" % (len(models), len(saved)))
    for i, (m, s) in enumerate(zip(models, saved)):
        _compare(model_config(m), s["config"], "member %d has " % i)
    ours, theirs = dict(args), dict(state["args"])
    theirs.setdefault("precision", 0)   # states written before the training precision was an argument were fp32
    om, tm = ours.pop("members", None), theirs.pop("members", None)
    _compare(ours, theirs)
    for i, (a, b) in enumerate(zip(om or [], tm or [])):
        _compare(a, b, "member %d has " % i)
    groups = state["optimizer"]["param_groups"]
    if len(groups) != len(optimizer.param_groups):
        raise ValueError("the optimizer has %d parameter groups, the checkpoint %d" % (len(optimizer.param_groups), len(groups)))
    for j, (a, b) in enumerate(zip(optimizer.param_groups, groups)):
        if len(a["params"]) != len(b["params"]):
            raise ValueError("optimizer group %d has %d parameters, the checkpoint %d" % (j, len(a["params"]), len(b["params"])))


def load_state(path, kind, models, optimizer, args, total, generators=None):
    """Reads the training state at ``path``, checks it (``check_state``), then restores every model's weights, the
    optimizer's state and, when given, every batch generator's state.  Returns ``(next_index, history)``."""
    state = torch.load(path, map_location="cpu", weights_only=True)
    check_state(state, kind, models, optimizer, args, total)
    for m, s in zip(models, state["members"]):
        m.load_state_dict(s["model"])
    optimizer.load_state_dict(state["optimizer"])
    for g, s in zip(generators or [], state["members"]):
        g.set_state(s["generator"])
    return state["next"], state["history"]


def weights_path(directory, stem, epoch=None):
    """``{directory}/{stem}_epoch{epoch}.pt``, or ``{directory}/{stem}.pt`` without an epoch: the names of train.py, with
    ``stem`` from ``utils.build_bandit_model_filename`` and its linear-bandit and darkroom siblings."""
    return os.path.join(directory, stem + ".pt" if epoch is None else "%s_epoch%d.pt" % (stem, epoch))


def save_weights(model, directory, stem, epoch=None):
    """Writes ``model.state_dict()`` (the reference's HF key layout) to ``weights_path(directory, stem, epoch)``
    atomically, creating ``directory`` if needed, and returns the path.  Every attention layer also gets the two buffers
    a transformers 4.5.1 model holds, ``attn.bias`` (the causal ``tril`` mask, uint8 [1, 1, N_CTX, N_CTX]) and
    ``attn.masked_bias`` (-1e4), so that the reference's strict ``load_state_dict`` finds every key it expects;
    ``Transformer.load_state_dict`` drops them."""
    os.makedirs(directory, exist_ok=True)
    mask = torch.tril(torch.ones((N_CTX, N_CTX), dtype=torch.uint8)).view(1, 1, N_CTX, N_CTX)
    sd = OrderedDict()
    for k, v in weights(model).items():
        if k.endswith(".attn.c_attn.weight"):   # where 4.5.1's state_dict has them: the attention module's own buffers
            p = k[:-len("c_attn.weight")]
            sd[p + "bias"], sd[p + "masked_bias"] = mask, torch.tensor(-1e4)
        sd[k] = v
    path = weights_path(directory, stem, epoch)
    _atomic_save(sd, path)
    return path
