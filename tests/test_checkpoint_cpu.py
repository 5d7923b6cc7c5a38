"""CPU tier of training checkpoints (checkpoint.py): the training state round-trips through save and load, every field a
resume must repeat is checked before anything is modified, a failed save leaves the previous file as it was, and the
weight files carry the reference's names and keys."""
import os

import pytest
import torch

CFG = {"horizon": 6, "state_dim": 1, "action_dim": 5, "n_layer": 2, "n_embd": 32, "n_head": 1, "dropout": 0.0, "test": False}


def _model(seed, **over):
    from dpt_b200.models.net import Transformer
    torch.manual_seed(seed)
    return Transformer(dict(CFG, **over))


class _Data:
    """What the checkpoint arguments read of a dataset.Dataset: its length and shuffle flag."""

    def __init__(self, n, shuffle=True):
        self.n, self.shuffle = n, shuffle

    def __len__(self):
        return self.n


def _optimizer(models, lrs=(1e-3, 3e-3, 1e-3), wds=(1e-4, 1e-4, 1e-4)):
    """train_population's default optimizer: one AdamW group per distinct (lr, weight_decay), in member order."""
    groups = {}
    for m, a, b in zip(models, lrs, wds):
        groups.setdefault((a, b), []).extend(m.parameters())
    return torch.optim.AdamW([{"params": ps, "lr": a, "weight_decay": b} for (a, b), ps in groups.items()])


def _step(models, opt, seed):
    g = torch.Generator().manual_seed(seed)
    for m in models:
        for p in m._train_params():
            p.grad = torch.randn(p.shape, generator=g)
    opt.step()


def _gens(seeds):
    gs = []
    for s in seeds:
        g = torch.Generator()
        g.seed() if s is None else g.manual_seed(s)
        torch.randperm(100, generator=g)       # advanced past its seed, as after an epoch
        gs.append(g)
    return gs


def _population(k=3, seeds=(11, 12, 13), lrs=(1e-3, 3e-3, 1e-3), wds=(1e-4, 1e-4, 1e-4), batch_size=64, train_sets=None,
                test_sets=None, init=0, **over):
    """(models, optimizer, generators, args) of a population of k whose members 0 and 1 share their datasets."""
    from dpt_b200 import checkpoint as C
    a, b, t = _Data(318), _Data(318), _Data(106, shuffle=False)
    train = [a, a, b][:k] if train_sets is None else train_sets
    test = [t, t, t][:k] if test_sets is None else test_sets
    models = [_model(init + i, **(over if i == 2 else {})) for i in range(k)]
    opt = _optimizer(models, lrs[:k], wds[:k])
    args = C.train_args(batch_size, lrs[:k], wds[:k], list(seeds[:k]), train, test, "cpu")
    return models, opt, _gens(seeds[:k]), args


def _snapshot(models, opt, gens):
    return ([p.detach().clone() for m in models for p in m.state_dict().values()],
            {i: {n: v.clone() for n, v in s.items()} for i, s in enumerate(opt.state.values())}, [g.get_state() for g in gens])


def test_state_round_trips(dpt, tmp_path):
    from dpt_b200 import checkpoint as C
    models, opt, gens, args = _population()
    _step(models, opt, 0)
    _step(models, opt, 1)
    hist = {"train_loss": [[0.5, 0.25]] * 3, "test_loss": [[0.75, 0.5]] * 3}
    path = tmp_path / "state.pt"
    C.save_state(path, C.training_state("population", models, opt, args, 2, hist, gens))
    assert os.listdir(tmp_path) == ["state.pt"]                     # no temporary file left behind
    state = torch.load(path, weights_only=True)
    assert state["version"] == C.VERSION and state["kind"] == "population" and state["next"] == 2
    assert [s["config"]["n_layer"] for s in state["members"]] == [2, 2, 2]
    # a fresh population (other initial weights, empty optimizer, other generator states) takes all of it
    fresh, fopt, fgens, fargs = _population(init=50, seeds=(11, 12, 13))
    for g in fgens:
        torch.rand(7, generator=g)
    nxt, h = C.load_state(path, "population", fresh, fopt, fargs, 4, fgens)
    assert nxt == 2 and h == hist
    want, got = _snapshot(models, opt, gens), _snapshot(fresh, fopt, fgens)
    assert all(torch.equal(a, b) for a, b in zip(want[0], got[0]))
    assert want[1].keys() == got[1].keys()
    for i in want[1]:
        assert want[1][i].keys() == {"step", "exp_avg", "exp_avg_sq"} == got[1][i].keys()
        assert all(torch.equal(want[1][i][n], got[1][i][n]) for n in want[1][i])
    assert all(torch.equal(a, b) for a, b in zip(want[2], got[2]))
    assert [g["lr"] for g in fopt.param_groups] == [1e-3, 3e-3]
    # and the restored generators draw what the saved ones draw next
    assert all(torch.equal(torch.randperm(50, generator=a), torch.randperm(50, generator=b)) for a, b in zip(gens, fgens))


def _interactive_args(**over):
    from dpt_b200 import checkpoint as C
    kw = dict(dim=5, n_envs=1000, K=40, mb=256, var=0.3, env_type="uniform", seed=3, lr=1e-3, weight_decay=1e-4)
    kw.update(over)
    return C.interactive_args(**kw)


# (what the resuming call changes, the message it must raise)
POPULATION_MISMATCHES = [
    ({"n_layer": 3}, "member 2 has n_layer=3, the checkpoint 2"),
    ({"horizon": 7}, "member 2 has horizon=7, the checkpoint 6"),
    ({"test": True}, "member 2 has test=True, the checkpoint False"),
    ({"k": 2}, "2 members, the checkpoint 3"),
    ({"batch_size": 32}, "batch_size=32, the checkpoint 64"),
    ({"lrs": (1e-3, 1e-3, 1e-3)}, "member 1 has lr=0.001, the checkpoint 0.003"),
    ({"wds": (1e-4, 1e-4, 0.0)}, "member 2 has weight_decay=0.0, the checkpoint 0.0001"),
    ({"seeds": (11, 12, 14)}, "member 2 has seed=14, the checkpoint 13"),
    ({"seeds": (11, None, 13)}, "member 1 has seed=None, the checkpoint 12"),
    ({"train_sets": [_Data(300), _Data(300), _Data(300)]}, "member 0 has train_items=300, the checkpoint 318"),
    ({"train_sets": [_Data(318, shuffle=False)] * 2 + [_Data(318)]}, "member 0 has train_shuffle=False, the checkpoint True"),
    ({"test_sets": [_Data(106, shuffle=False)] * 2 + [_Data(107, shuffle=False)]}, "member 2 has test_items=107, the checkpoint 106"),
    ({"train_sets": [_Data(318), _Data(318), _Data(318)]}, "member 1 has train_set=1, the checkpoint 0"),   # no longer shared
]


@pytest.mark.parametrize("change,message", POPULATION_MISMATCHES)
def test_mismatched_resume_names_the_field_and_changes_nothing(dpt, tmp_path, change, message):
    from dpt_b200 import checkpoint as C
    models, opt, gens, args = _population()
    _step(models, opt, 0)
    path = tmp_path / "state.pt"
    C.save_state(path, C.training_state("population", models, opt, args, 1, {}, gens))
    over = {k: v for k, v in change.items() if k in CFG}
    kw = {k: v for k, v in change.items() if k not in CFG}
    fresh, fopt, fgens, fargs = _population(init=50, **kw, **over)
    before = _snapshot(fresh, fopt, fgens)
    with pytest.raises(ValueError) as e:
        C.load_state(path, "population", fresh, fopt, fargs, 4, fgens)
    assert str(e.value) == message
    after = _snapshot(fresh, fopt, fgens)
    assert all(torch.equal(a, b) for a, b in zip(before[0], after[0])) and not after[1]
    assert all(torch.equal(a, b) for a, b in zip(before[2], after[2]))


def test_interactive_and_format_mismatches(dpt, tmp_path):
    from dpt_b200 import checkpoint as C
    m = _model(0)
    opt = torch.optim.AdamW(m.parameters())
    _step([m], opt, 0)
    path = tmp_path / "state.pt"
    args = _interactive_args()
    C.save_state(path, C.training_state("interactive", [m], opt, args, 3, {"losses": [1.0, 0.5, 0.25]}))

    def load(args=args, kind="interactive", total=5, opt=None):
        """The message of the ValueError a fresh model's resume raises; the model and optimizer stay as they were."""
        fresh = _model(9)
        before = [p.detach().clone() for p in fresh.parameters()]
        fo = torch.optim.AdamW(fresh.parameters()) if opt is None else opt(fresh)
        with pytest.raises(ValueError) as e:
            C.load_state(path, kind, [fresh], fo, args, total)
        assert all(torch.equal(a, p) for a, p in zip(before, fresh.parameters())) and not fo.state
        return str(e.value)
    for field, value, message in (("mb", 512, "mb=512, the checkpoint 256"), ("n_envs", 999, "n_envs=999, the checkpoint 1000"),
                                  ("K", 41, "K=41, the checkpoint 40"), ("dim", 4, "dim=4, the checkpoint 5"),
                                  ("var", 0.0, "var=0.0, the checkpoint 0.3"), ("seed", 4, "seed=4, the checkpoint 3"),
                                  ("env_type", "bernoulli", "env_type='bernoulli', the checkpoint 'uniform'"),
                                  ("lr", 3e-3, "lr=0.003, the checkpoint 0.001")):
        assert load(_interactive_args(**{field: value})) == message, field
    assert load(total=2) == "n_iters=2, the checkpoint is past it, at iteration 3"
    assert load(kind="train") == "kind='train', the checkpoint 'interactive'"
    assert load(opt=lambda f: torch.optim.AdamW([{"params": list(f.parameters())[:3]}, {"params": list(f.parameters())[3:]}])) \
        == "the optimizer has 2 parameter groups, the checkpoint 1"
    fresh = _model(9)
    assert C.load_state(path, "interactive", [fresh], torch.optim.AdamW(fresh.parameters()), args, 3) == \
        (3, {"losses": [1.0, 0.5, 0.25]})   # the unchanged call resumes, up to a total of exactly the saved iterations
    assert all(torch.equal(a, b) for a, b in zip(fresh.state_dict().values(), m.state_dict().values()))
    good = torch.load(path, weights_only=True)
    for key, value, message in (("version", 2, "training state of format version 2; this package reads version 1"),
                                ("kind", "explorer", "training state of unknown kind 'explorer' (known: train, population, interactive)")):
        state = dict(good)
        state[key] = value
        torch.save(state, path)
        assert load() == message


def test_failed_save_leaves_the_previous_file(dpt, tmp_path, monkeypatch):
    from dpt_b200 import checkpoint as C
    m = _model(0)
    opt = torch.optim.AdamW(m.parameters())
    path = tmp_path / "state.pt"
    C.save_state(path, C.training_state("interactive", [m], opt, _interactive_args(), 1, {"losses": [1.0]}))
    good = path.read_bytes()
    _step([m], opt, 0)

    def dies_midway(obj, f, *a, **kw):
        f.write(b"\0" * 4096)
        raise OSError("disk full")
    monkeypatch.setattr(torch, "save", dies_midway)
    with pytest.raises(OSError, match="disk full"):
        C.save_state(path, C.training_state("interactive", [m], opt, _interactive_args(), 2, {"losses": [1.0, 0.5]}))
    assert path.read_bytes() == good
    assert os.listdir(tmp_path) == ["state.pt"]


def test_weight_files_have_the_reference_names(dpt, tmp_path):
    from dpt_b200 import checkpoint as C, utils as U
    cfg = {"n_hists": 1, "n_samples": 1, "horizon": 6, "dim": 5, "var": 0.3, "cov": 0.0, "lin_d": 2, "shuffle": True,
           "lr": 0.001, "dropout": 0.0, "n_embd": 32, "n_layer": 2, "n_head": 1, "n_envs": 100000, "seed": 1}
    stems = [U.build_bandit_model_filename("bandit", cfg), U.build_linear_bandit_model_filename("linear_bandit", cfg),
             U.build_darkroom_model_filename("darkroom_heldout", cfg)]
    assert stems[0] == "bandit_shufTrue_lr0.001_do0.0_embd32_layer2_head1_envs100000_hists1_samples1_var0.3_cov0.0_H6_d5_seed1"
    m = _model(0)
    written = []
    for s in stems:
        for e in (10, 50, None):
            written.append(C.save_weights(m, str(tmp_path / "models"), s, e))
    names = [s + "_epoch10.pt" for s in stems] + [s + "_epoch50.pt" for s in stems] + [s + ".pt" for s in stems]
    assert sorted(os.listdir(tmp_path / "models")) == sorted(names)
    assert written[:3] == [str(tmp_path / "models" / n) for n in (stems[0] + "_epoch10.pt", stems[0] + "_epoch50.pt",
                                                                   stems[0] + ".pt")]
    sd = torch.load(written[0], weights_only=True)
    own = m.state_dict()
    assert set(sd) == set(own) | {"transformer.h.%d.attn.%s" % (i, b) for i in range(2) for b in ("bias", "masked_bias")}
    assert all(torch.equal(sd[k], v) for k, v in own.items())
    assert sd["transformer.h.1.attn.bias"].shape == (1, 1, C.N_CTX, C.N_CTX)
    assert torch.equal(sd["transformer.h.1.attn.bias"][0, 0], torch.tril(torch.ones(C.N_CTX, C.N_CTX, dtype=torch.uint8)))
    assert sd["transformer.h.0.attn.masked_bias"].item() == -1e4
    fresh = _model(7)
    fresh.load_state_dict(sd, strict=True)
    assert all(torch.equal(a, b) for a, b in zip(fresh.state_dict().values(), own.values()))


def test_trainer_checkpoint_arguments_are_checked_first(dpt):
    from dpt_b200 import train as TR
    ms = [_model(0), _model(1)]
    d = _Data(8)
    with pytest.raises(ValueError, match="save_every=0"):
        TR.train_population(ms, d, d, 1, state_path="s.pt", save_every=0)
    with pytest.raises(ValueError, match="resume=True needs a state_path"):
        TR.train(ms[0], d, d, 1, resume=True)
    with pytest.raises(ValueError, match="weights_dir needs 2 distinct stems"):
        TR.train_population(ms, d, d, 1, weights_dir="models", stems="bandit")
    with pytest.raises(ValueError, match="weights_dir needs 1 distinct stems"):
        TR.train(ms[0], d, d, 1, weights_dir="models")
    with pytest.raises(ValueError, match="resume=True needs a state_path"):
        TR.train_interactive(ms[0], 5, 64, 6, 1, resume=True)
