"""CPU tier of population training: argument checks of dpt_gpt2_train_forward / _backward over several members at
precision 0 (they run before any launch, so no GPU is needed) and the ValueErrors of forward_train_population /
train_population for members or datasets that do not line up."""
import ctypes

import pytest
import torch

E_ARG, E_UNSUP = -1, -3


def _weights(dpt, keep, n_layer=2, state_dim=1, action_dim=5, n_embd=32, n_positions=2004):
    """A dpt_gpt2_weights_t with non-null (never dereferenced) fake device pointers."""
    fake = 4096
    arr = lambda: ctypes.cast((ctypes.c_void_p * n_layer)(*[fake] * n_layer), ctypes.POINTER(ctypes.c_void_p))   # noqa: E731
    kw = {n: arr() for n in ("ln1_w", "ln1_b", "attn_w", "attn_b", "proj_w", "proj_b", "ln2_w", "ln2_b", "fc_w", "fc_b",
                             "fc2_w", "fc2_b")}
    keep.append(kw)
    return dpt._lib.Gpt2Weights(horizon=500, state_dim=state_dim, action_dim=action_dim, n_layer=n_layer, n_embd=n_embd,
                                n_positions=n_positions, wpe=fake, embed_w=fake, embed_b=fake, pred_w=fake, pred_b=fake,
                                lnf_w=fake, lnf_b=fake, **kw)


def _fwd(lib, w, n, ptrs=None, B=4, T=10):
    p = ptrs if ptrs is not None else (ctypes.c_void_p * max(n, 1))(*[4096] * max(n, 1))
    return lib.dpt_gpt2_train_forward(w, n, p, p, p, p, p, B, T, T, 0, 0, p, None, 0, None)


def test_population_entry_points_reject_bad_arguments(dpt):
    lib = dpt._lib.lib()
    err = lambda: lib.dpt_last_error().decode()   # noqa: E731
    keep = []
    two = (dpt._lib.Gpt2Weights * 2)(_weights(dpt, keep), _weights(dpt, keep))
    limit = dpt.models.net.POPULATION_MAX
    assert limit >= 16
    # member count
    for n in (-1, limit + 1):
        assert _fwd(lib, two, n) == E_ARG and ("n_models=%d" % n) in err()
        assert lib.dpt_gpt2_train_backward(two, n, None, 4, 10, 0, 0, None, None, 0, None) == E_ARG
    assert lib.dpt_gpt2_train_workspace_bytes(two, limit + 1, 4, 10, 0) == 0
    # null pointers
    assert _fwd(lib, None, 2) == E_ARG and "null weights" in err()
    assert lib.dpt_gpt2_train_forward(two, 2, None, None, None, None, None, 4, 10, 10, 0, 0, None, None, 0, None) == E_ARG
    assert "null input or output pointer array" in err()
    nulls = (ctypes.c_void_p * 2)(4096, None)
    assert _fwd(lib, two, 2, nulls) == E_ARG and "member 1: null input or output pointer" in err()
    assert lib.dpt_gpt2_train_backward(two, 2, None, 4, 10, 0, 0, None, None, 0, None) == E_ARG and "null dout" in err()
    ws_needed = lib.dpt_gpt2_train_workspace_bytes(two, 2, 4, 10, 0)
    assert ws_needed == 2 * lib.dpt_gpt2_train_workspace_bytes(two, 1, 4, 10, 0) > 0
    assert _fwd(lib, two, 2) == E_ARG and "workspace" in err()
    # a member of another shape: the message names the member and the field
    for field, kw in (("n_layer", {"n_layer": 3}), ("state_dim", {"state_dim": 2}), ("action_dim", {"action_dim": 4}),
                      ("n_positions", {"n_positions": 404})):
        odd = (dpt._lib.Gpt2Weights * 3)(_weights(dpt, keep), _weights(dpt, keep), _weights(dpt, keep, **kw))
        assert _fwd(lib, odd, 3) == E_ARG and ("member 2 has %s" % field) in err(), field
        assert lib.dpt_gpt2_train_backward(odd, 3, None, 4, 10, 0, 0, None, None, 0, None) == E_ARG
    # the one-model limits, per member
    wide = (dpt._lib.Gpt2Weights * 2)(_weights(dpt, keep), _weights(dpt, keep, n_embd=64))
    assert _fwd(lib, wide, 2) == E_UNSUP and "member 1: n_embd=64" in err()
    assert _fwd(lib, two, 2, T=512) == E_UNSUP and "512 tokens" in err()
    deep = (dpt._lib.Gpt2Weights * 1)(_weights(dpt, keep, n_layer=9))
    assert _fwd(lib, deep, 1) == E_UNSUP
    # no-ops: no member, or an empty batch
    assert _fwd(lib, None, 0) == 0
    assert lib.dpt_gpt2_train_backward(None, 0, None, 4, 10, 0, 0, None, None, 0, None) == 0
    assert _fwd(lib, two, 2, B=0) == 0
    assert lib.dpt_gpt2_train_backward(two, 2, None, 0, 10, 0, 0, None, None, 0, None) == 0
    with pytest.raises(ValueError, match="dpt_gpt2_train_forward"):
        dpt._lib.check(_fwd(lib, two, -1), "dpt_gpt2_train_forward")


def _model(**over):
    from dpt_b200.models.net import Transformer
    cfg = {"horizon": 20, "state_dim": 1, "action_dim": 5, "n_layer": 2, "n_embd": 32, "n_head": 1, "dropout": 0.0, "test": False}
    cfg.update(over)
    return Transformer(cfg)


def test_forward_train_population_rejects_mismatched_members(dpt):
    from dpt_b200.models.net import forward_train_population
    assert forward_train_population([], []) == []
    with pytest.raises(ValueError, match="2 models and 1 batches"):
        forward_train_population([_model(), _model()], [{}])
    for field, kw in (("n_layer", {"n_layer": 3}), ("state_dim", {"state_dim": 2}), ("action_dim", {"action_dim": 4}),
                      ("horizon", {"horizon": 30}), ("test", {"test": True})):
        with pytest.raises(ValueError, match="member 1 has %s" % field):
            forward_train_population([_model(), _model(**kw)], [{}, {}])
    with pytest.raises(NotImplementedError, match="dropout"):
        forward_train_population([_model(), _model(dropout=0.1)], [{}, {}])


class _Data:
    """The part of dataset.Dataset that train_population reads before it touches the data."""

    def __init__(self, n):
        self.dataset = {"context_actions": torch.zeros(n, 20, 5)}
        self.shuffle = False

    def __len__(self):
        return self.dataset["context_actions"].shape[0]


def test_train_population_rejects_unequal_datasets(dpt):
    from dpt_b200 import train as TR
    ms = [_model(), _model()]
    with pytest.raises(ValueError, match="train dataset of member 1 has 9 items, member 0's has 8"):
        TR.train_population(ms, [_Data(8), _Data(9)], _Data(4), 1)
    with pytest.raises(ValueError, match="test dataset of member 1 has 5 items"):
        TR.train_population(ms, _Data(8), [_Data(4), _Data(5)], 1)
    with pytest.raises(ValueError, match="3 values of lr for 2 models"):
        TR.train_population(ms, _Data(8), _Data(4), 1, lr=[1e-3, 1e-3, 1e-3])
    assert TR.train_population([], _Data(8), _Data(4), 1) == ([], [], None)
