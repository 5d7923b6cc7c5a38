"""Pretraining loop of the reference's train.py (SURVEY §2.1) on device-resident datasets.

``train(model, train_dataset, test_dataset, num_epochs)`` runs the reference's epochs: the test loss under
``no_grad`` through ``model.forward`` first, then one pass over the training set with ``torch.optim.AdamW(lr,
weight_decay)``, batch 64, and the sum-reduced cross-entropy of the logits of every context row against the
optimal action.  Both epoch losses are reported as the reference reports them: sum of the batch losses / horizon /
len(dataset).  The forward of training is ``model.forward_train`` (hand-written CUDA forward and backward).

Unlike the reference's DataLoader, batches are gathered on the device from ``Dataset.dataset`` with a seeded
permutation (and, with ``Dataset.shuffle``, a seeded per-item context permutation), and the losses stay on the
device until one host read per epoch.  There is no argparse, plotting or checkpoint naming.
"""
import torch
import torch.nn.functional as F

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


def train_step(model, optimizer, batch, loss_fn=ce_sum_loss):
    """One optimizer step: ``model.forward_train(batch)``, ``loss_fn(pred, batch)``, backward, ``optimizer.step()``.
    Returns the loss as a device tensor (no host synchronisation)."""
    optimizer.zero_grad()
    pred = model.forward_train(batch)
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
          optimizer=None):
    """The reference's epoch loop.  Returns ``(train_loss, test_loss, optimizer)``: per-epoch lists of floats and the
    AdamW optimizer (its ``state_dict`` is the reference's)."""
    dev = train_dataset.dataset["context_actions"].device
    if next(model.parameters()).device != dev:
        model.to(dev)
    if optimizer is None:
        optimizer = torch.optim.AdamW(model.parameters(), lr=lr, weight_decay=weight_decay)
    gen = torch.Generator(device=dev)
    if seed is None:
        gen.seed()
    else:
        gen.manual_seed(seed)
    horizon = model.horizon
    train_loss, test_loss = [], []
    for _ in range(num_epochs):
        with torch.no_grad():
            te = torch.zeros((), dtype=torch.float32, device=dev)
            for b in batches(test_dataset, batch_size, gen):
                te += ce_sum_loss(model(b), b)
        tr = torch.zeros((), dtype=torch.float32, device=dev)
        for b in batches(train_dataset, batch_size, gen):
            tr += train_step(model, optimizer, b)
        losses = torch.stack([te / horizon / len(test_dataset), tr / horizon / len(train_dataset)]).tolist()   # one host read
        test_loss.append(losses[0])
        train_loss.append(losses[1])
    return train_loss, test_loss, optimizer
