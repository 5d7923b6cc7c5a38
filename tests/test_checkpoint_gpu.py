"""GPU tier of training checkpoints: a run interrupted at an epoch (iteration) boundary and resumed with fresh models and
optimizers ends bit-identical to the run that was never interrupted (every parameter, every AdamW state tensor with its
step, every loss) for train, train_population and train_interactive; the reference's weight files appear at the right
epochs and reproduce the trained model's logits; a mismatched resume raises before any weight changes."""
import os
import shutil

import pytest
import torch

pytestmark = pytest.mark.gpu

H = 40


def _model(seed, L=2, test=False, scale=0.02):
    from dpt_b200.models.net import Transformer
    torch.manual_seed(seed)
    m = Transformer({"horizon": H, "state_dim": 1, "action_dim": 5, "n_layer": L, "n_embd": 32, "n_head": 1, "dropout": 0.0,
                     "test": test}).cuda()
    with torch.no_grad():
        for k, p in m.named_parameters():
            if "wte" not in k:
                p.add_(scale * torch.randn_like(p))
    return m


def _datasets(seed, shuffle=True, n_items=424):
    """424 bandit items split 318 / 106: ragged last batches of 62 and 42 at batch 64."""
    from dpt_b200 import collect_data
    from dpt_b200.dataset import Dataset
    batch = collect_data.collect_bandit(n_items, 5, H, 0.3, seed=seed)
    cfg = {"horizon": H, "state_dim": 1, "action_dim": 5, "shuffle": shuffle, "store_gpu": True}
    n_tr = n_items * 3 // 4
    return (Dataset.from_batch({k: v[:n_tr] for k, v in batch.items()}, cfg),
            Dataset.from_batch({k: v[n_tr:] for k, v in batch.items()}, cfg))


def _adam_state(opt, models):
    return [opt.state[p] for m in models for p in m.parameters() if p in opt.state]


def _assert_same(models_a, opt_a, losses_a, models_b, opt_b, losses_b):
    for a, b in zip(models_a, models_b):
        for (k, p), q in zip(a.state_dict().items(), b.state_dict().values()):
            assert torch.equal(p, q), k
    sa, sb = _adam_state(opt_a, models_a), _adam_state(opt_b, models_b)
    assert len(sa) == len(sb) == sum(len(m._train_params()) for m in models_a)
    for s, t in zip(sa, sb):
        assert s.keys() == t.keys() == {"step", "exp_avg", "exp_avg_sq"}
        assert all(torch.equal(s[n], t[n]) for n in s)
    assert losses_a == losses_b


@pytest.fixture
def snapshots(monkeypatch):
    """Keeps a copy of every training state a trainer writes: {next epoch or iteration: path}."""
    from dpt_b200 import checkpoint as C
    kept, save = {}, C.save_state

    def keep(path, state):
        save(path, state)
        kept[state["next"]] = "%s.at%d" % (path, state["next"])
        shutil.copyfile(path, kept[state["next"]])
    monkeypatch.setattr(C, "save_state", keep)
    return kept


@pytest.mark.parametrize("shuffle,seed", [(True, 7), (False, 7), (True, None)])
def test_train_resumed_is_the_uninterrupted_run(dpt, tmp_path, monkeypatch, snapshots, shuffle, seed):
    from dpt_b200 import train as TR
    tr, te = _datasets(5, shuffle)
    full = _model(1)
    tl, vl, opt = TR.train(full, tr, te, 4, seed=seed, state_path=str(tmp_path / "full.pt"), save_every=2)
    assert sorted(snapshots) == [2, 4] and len(tl) == len(vl) == 4
    path = str(tmp_path / "cut.pt")
    if seed is None:             # the batch order was drawn from a fresh seed: resume the uninterrupted run's own state
        shutil.copyfile(snapshots[2], path)
    else:
        tl2, vl2, _ = TR.train(_model(1), tr, te, 2, seed=seed, state_path=path)
        assert tl2 == tl[:2] and vl2 == vl[:2]
        monkeypatch.chdir(tmp_path)   # without the new arguments nothing is written, and the results are the same
        files = sorted(os.listdir(tmp_path))
        plain = _model(1)
        tlp, vlp, optp = TR.train(plain, tr, te, 4, seed=seed)
        assert sorted(os.listdir(tmp_path)) == files
        _assert_same([full], opt, (tl, vl), [plain], optp, (tlp, vlp))
    res = _model(3)                 # other initial weights: everything comes from the file
    tlr, vlr, optr = TR.train(res, tr, te, 4, seed=seed, state_path=path, resume=True)
    _assert_same([full], opt, (tl, vl), [res], optr, (tlr, vlr))


def test_train_resumes_from_every_saved_epoch(dpt, tmp_path, snapshots):
    from dpt_b200 import train as TR
    tr, te = _datasets(6)
    full = _model(1)
    tl, vl, opt = TR.train(full, tr, te, 4, seed=9, state_path=str(tmp_path / "s.pt"), save_every=1)
    assert sorted(snapshots) == [1, 2, 3, 4]
    for e, path in sorted(snapshots.items()):
        res = _model(10 + e)
        tlr, vlr, optr = TR.train(res, tr, te, 4, seed=9, state_path=path, resume=True)
        _assert_same([full], opt, (tl, vl), [res], optr, (tlr, vlr))
    # resume=True without a state file starts from scratch
    scratch = _model(1)
    tls, vls, opts = TR.train(scratch, tr, te, 4, seed=9, state_path=str(tmp_path / "none.pt"), save_every=3, resume=True)
    _assert_same([full], opt, (tl, vl), [scratch], opts, (tls, vls))


@pytest.mark.parametrize("k", [3, 1])
def test_population_resumed_is_the_uninterrupted_run(dpt, tmp_path, k):
    from dpt_b200 import train as TR
    tr_a, te_a = _datasets(5)
    tr_b, te_b = _datasets(6, shuffle=False)
    trs, tes = [tr_a, tr_a, tr_b][:k], [te_a, te_a, te_b][:k]     # members 0 and 1 share their datasets
    lrs, wds, seeds = [1e-3, 3e-3, 1e-3][:k], [1e-4, 1e-4, 1e-4][:k], [11, 12, 13][:k]   # two (lr, wd) groups at k = 3

    def run(init, n, **kw):
        ms = [_model(init + i) for i in range(k)]
        return ms, TR.train_population(ms, trs, tes, n, lr=lrs, weight_decay=wds, seeds=seeds, **kw)
    full, (tl, vl, opt) = run(1, 4)
    assert len(opt.param_groups) == (2 if k == 3 else 1)
    path = str(tmp_path / "pop.pt")
    run(1, 2, state_path=path)
    res, (tlr, vlr, optr) = run(40, 4, state_path=path, resume=True)
    _assert_same(full, opt, (tl, vl), res, optr, (tlr, vlr))


def test_interactive_resumed_is_the_uninterrupted_run(dpt, tmp_path, snapshots):
    from dpt_b200 import train as TR
    d, N, K, mb, var, seed = 5, 1000, 24, 256, 0.3, 4      # micro-batches of 256, 256, 256 and 232 envs
    full = _model(1, test=True, scale=0.15)
    losses, opt = TR.train_interactive(full, d, N, K, 5, mb=mb, var=var, seed=seed)
    path = str(tmp_path / "it.pt")
    cut = _model(1, test=True, scale=0.15)
    first, _ = TR.train_interactive(cut, d, N, K, 3, mb=mb, var=var, seed=seed, state_path=path, save_every=2)
    assert sorted(snapshots) == [2, 3] and first == losses[:3]
    res = _model(3, test=True, scale=0.15)
    lr_, optr = TR.train_interactive(res, d, N, K, 5, mb=mb, var=var, seed=seed, state_path=path, resume=True)
    _assert_same([full], opt, losses, [res], optr, lr_)
    assert sorted(snapshots) == [2, 3, 5]


def test_weight_files_at_the_right_epochs(dpt, tmp_path):
    from dpt_b200 import train as TR, utils as U
    from dpt_b200.models.net import Transformer
    tr, te = _datasets(5)
    cfg = {"n_hists": 1, "n_samples": 1, "horizon": H, "dim": 5, "var": 0.3, "cov": 0.0, "shuffle": True, "lr": 0.001,
           "dropout": 0.0, "n_embd": 32, "n_layer": 2, "n_head": 1, "n_envs": 424}
    stems = [U.build_bandit_model_filename("bandit", dict(cfg, seed=s)) for s in (0, 1)]
    out = str(tmp_path / "models")
    ms = [_model(1), _model(2)]
    TR.train_population(ms, tr, te, 5, seeds=[0, 1], weights_dir=out, stems=stems, save_every=2)
    at2 = [_model(1), _model(2)]
    TR.train_population(at2, tr, te, 2, seeds=[0, 1])
    at4 = [_model(1), _model(2)]
    TR.train_population(at4, tr, te, 4, seeds=[0, 1])
    assert sorted(os.listdir(out)) == sorted(s + e for s in stems for e in ("_epoch2.pt", "_epoch4.pt", ".pt"))
    b = {k: v[:16] for k, v in te.dataset.items()}
    for i, stem in enumerate(stems):
        for name, trained in (("_epoch2.pt", at2[i]), ("_epoch4.pt", at4[i]), (".pt", ms[i])):
            fresh = Transformer(dict(ms[i].config)).cuda()
            fresh.load_state_dict(torch.load(os.path.join(out, stem + name), weights_only=True), strict=True)
            assert torch.equal(fresh(b), trained(b)), stem + name
            assert all(torch.equal(p, q) for p, q in zip(fresh.parameters(), trained.parameters())), stem + name
    # train: one stem
    one = _model(1)
    TR.train(one, tr, te, 1, seed=0, weights_dir=out, stems="single", save_every=1)
    assert os.path.exists(os.path.join(out, "single_epoch1.pt")) and os.path.exists(os.path.join(out, "single.pt"))


def test_mismatched_resume_raises_before_any_weight_changes(dpt, tmp_path):
    from dpt_b200 import train as TR
    tr, te = _datasets(5)
    path = str(tmp_path / "s.pt")
    TR.train(_model(1), tr, te, 2, seed=3, state_path=path)
    for model, kw, message in ((_model(2), {"lr": 3e-3}, "member 0 has lr=0.003, the checkpoint 0.001"),
                               (_model(2), {"seed": 4}, "member 0 has seed=4, the checkpoint 3"),
                               (_model(2, L=3), {}, "member 0 has n_layer=3, the checkpoint 2"),
                               (_model(2), {"batch_size": 32}, "batch_size=32, the checkpoint 64")):
        before = [p.detach().clone() for p in model.parameters()]
        with pytest.raises(ValueError) as e:
            TR.train(model, tr, te, 4, **dict({"seed": 3}, **kw), state_path=path, resume=True)
        assert str(e.value) == message
        assert all(torch.equal(a, p) for a, p in zip(before, model.parameters()))
    with pytest.raises(ValueError, match="kind='population', the checkpoint 'train'"):
        TR.train_population([_model(2)], tr, te, 4, seeds=[3], state_path=path, resume=True)
    m = _model(1, test=True, scale=0.15)
    TR.train_interactive(m, 5, 300, 12, 2, mb=128, seed=1, state_path=path)
    m = _model(2, test=True, scale=0.15)
    before = [p.detach().clone() for p in m.parameters()]
    with pytest.raises(ValueError, match="^mb=256, the checkpoint 128$"):
        TR.train_interactive(m, 5, 300, 12, 4, mb=256, seed=1, state_path=path, resume=True)
    assert all(torch.equal(a, p) for a, p in zip(before, m.parameters()))
