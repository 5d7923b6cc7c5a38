"""CPU tier of bf16 interactive training (train_interactive(..., precision=1)): the training precision in the resume
arguments of checkpoint.interactive_args, including interactive states written before it was recorded, and the
precision check that train_interactive runs before it touches a device."""
import pytest
import torch


def _model(seed):
    from dpt_b200.models.net import Transformer
    torch.manual_seed(seed)
    return Transformer({"horizon": 4, "state_dim": 1, "action_dim": 5, "n_layer": 1, "n_embd": 32, "n_head": 1, "dropout": 0.0,
                        "test": True})


def _args(precision=None):
    from dpt_b200 import checkpoint as C
    kw = {} if precision is None else {"precision": precision}
    return C.interactive_args(5, 1000, 40, 256, 0.3, "uniform", 3, 1e-3, 1e-4, **kw)


def test_interactive_args_record_the_precision(dpt):
    assert _args(0)["precision"] == 0 and _args(1)["precision"] == 1
    assert _args() == _args(0)


def test_interactive_state_without_precision_is_fp32(dpt):
    from dpt_b200 import checkpoint as C
    m = _model(0)
    opt = torch.optim.AdamW(m.parameters())
    old = C.training_state("interactive", [m], opt, {k: v for k, v in _args(0).items() if k != "precision"}, 1,
                           {"losses": [1.0]})
    C.check_state(old, "interactive", [m], opt, _args(0), 2)
    with pytest.raises(ValueError, match=r"precision=1, the checkpoint 0"):
        C.check_state(old, "interactive", [m], opt, _args(1), 2)


@pytest.mark.parametrize("saved,resumed", [(1, 0), (0, 1)])
def test_resume_at_the_other_precision_raises(dpt, tmp_path, saved, resumed):
    from dpt_b200 import checkpoint as C
    m = _model(0)
    opt = torch.optim.AdamW(m.parameters())
    path = tmp_path / "state.pt"
    C.save_state(path, C.training_state("interactive", [m], opt, _args(saved), 2, {"losses": [1.0, 0.5]}))
    fresh = _model(1)
    fopt = torch.optim.AdamW(fresh.parameters())
    before = [p.detach().clone() for p in fresh.parameters()]
    with pytest.raises(ValueError, match=r"precision=%d, the checkpoint %d" % (resumed, saved)):
        C.load_state(path, "interactive", [fresh], fopt, _args(resumed), 4)
    assert all(torch.equal(a, p) for a, p in zip(before, fresh.parameters())) and not fopt.state
    assert C.load_state(path, "interactive", [fresh], fopt, _args(saved), 4) == (2, {"losses": [1.0, 0.5]})


@pytest.mark.parametrize("precision", [2, -1, "1"])
def test_unknown_precision_raises_before_the_device(dpt, precision):
    from dpt_b200 import train as TR
    m = _model(0)   # on the CPU: the check comes before anything needs a GPU
    with pytest.raises(ValueError, match=r"train_interactive: precision=%r" % (precision,)):
        TR.train_interactive(m, 5, 64, 10, 1, precision=precision)
    assert next(m.parameters()).device.type == "cpu"
