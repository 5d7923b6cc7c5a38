"""CPU tier of bf16 training (precision = 1): the ABI version, the precision argument of dpt_gpt2_train_workspace_bytes /
_forward / _backward (a B = 0 call only validates, so no GPU is needed), and the training precision in the resume
arguments of checkpoint.train_args, including states written before it was recorded."""
import ctypes

import pytest
import torch

E_UNSUP = -3


def _weights(dpt, keep, n_layer=2, n_embd=32, n_positions=2004):
    """A dpt_gpt2_weights_t with non-null (never dereferenced) fake device pointers."""
    fake = 4096
    arr = lambda: ctypes.cast((ctypes.c_void_p * n_layer)(*[fake] * n_layer), ctypes.POINTER(ctypes.c_void_p))   # noqa: E731
    kw = {n: arr() for n in ("ln1_w", "ln1_b", "attn_w", "attn_b", "proj_w", "proj_b", "ln2_w", "ln2_b", "fc_w", "fc_b",
                             "fc2_w", "fc2_b")}
    keep.append(kw)
    return dpt._lib.Gpt2Weights(horizon=500, state_dim=1, action_dim=5, n_layer=n_layer, n_embd=n_embd,
                                n_positions=n_positions, wpe=fake, embed_w=fake, embed_b=fake, pred_w=fake, pred_b=fake,
                                lnf_w=fake, lnf_b=fake, **kw)


def test_abi_version(dpt):
    assert dpt._lib.ABI_VERSION == 10 == dpt._lib.lib().dpt_version()


@pytest.mark.parametrize("case,kw,T,precision,msg", [
    ("n_embd", {"n_embd": 64}, 10, 1, "n_embd=64"),
    ("n_layer", {"n_layer": 9}, 10, 1, "n_layer=9"),
    ("tokens", {}, 512, 1, "512 tokens"),
    ("precision", {}, 10, 2, "precision=2"),
])
def test_precision_entry_points_validate_at_b0(dpt, case, kw, T, precision, msg):
    lib = dpt._lib.lib()
    keep = []
    w = (dpt._lib.Gpt2Weights * 1)(_weights(dpt, keep, **kw))
    p = (ctypes.c_void_p * 1)(4096)
    assert lib.dpt_gpt2_train_forward(w, 1, p, p, p, p, p, 0, T, T, 0, precision, p, None, 0, None) == E_UNSUP
    assert msg in lib.dpt_last_error().decode()
    assert lib.dpt_gpt2_train_backward(w, 1, p, 0, T, 0, precision, None, None, 0, None) == E_UNSUP
    assert msg in lib.dpt_last_error().decode()


def test_precision_workspace_and_valid_b0_calls(dpt):
    lib = dpt._lib.lib()
    keep = []
    w = (dpt._lib.Gpt2Weights * 2)(_weights(dpt, keep), _weights(dpt, keep))
    p = (ctypes.c_void_p * 2)(4096, 4096)
    fp32 = lib.dpt_gpt2_train_workspace_bytes(w, 2, 64, 500, 0)
    assert fp32 > 0
    # precision 1 also holds the packed weight images (40 KB per layer) and one layer's attention-output gradients
    bf16 = lib.dpt_gpt2_train_workspace_bytes(w, 2, 64, 500, 1)
    assert bf16 == fp32 + 2 * (2 * 40960 + 64 * 501 * 36 * 4)
    assert lib.dpt_gpt2_train_workspace_bytes(w, 2, 64, 500, 2) == 0
    for prec in (0, 1):   # a valid shape at B = 0: nothing to do
        assert lib.dpt_gpt2_train_forward(w, 2, p, p, p, p, p, 0, 10, 10, 0, prec, p, None, 0, None) == 0
        assert lib.dpt_gpt2_train_backward(w, 2, p, 0, 10, 0, prec, None, None, 0, None) == 0


def test_python_rejects_unknown_precision(dpt):
    from dpt_b200.models.net import forward_train_population
    from dpt_b200 import train as TR
    with pytest.raises(ValueError, match="precision=2"):
        forward_train_population([object()], [{}], precision=2)
    with pytest.raises(ValueError, match="precision=3"):
        TR.train_population([_model(0)], [_Ds(8)], [_Ds(8)], 1, precision=3)


class _Ds:
    def __init__(self, n, shuffle=False):
        self.n, self.shuffle = n, shuffle
        self.dataset = {"context_actions": torch.zeros(n, 4, 5)}

    def __len__(self):
        return self.n


def _model(seed):
    from dpt_b200.models.net import Transformer
    torch.manual_seed(seed)
    return Transformer({"horizon": 4, "state_dim": 1, "action_dim": 5, "n_layer": 1, "n_embd": 32, "n_head": 1, "dropout": 0.0,
                        "test": False})


def test_checkpoint_records_the_training_precision(dpt):
    from dpt_b200 import checkpoint as C
    m = _model(0)
    opt = torch.optim.AdamW(m.parameters())
    ds = [_Ds(8)]
    args = {p: C.train_args(64, [1e-3], [1e-4], [0], ds, ds, "cpu", p) for p in (0, 1)}
    assert args[0]["precision"] == 0 and args[1]["precision"] == 1
    assert C.train_args(64, [1e-3], [1e-4], [0], ds, ds, "cpu") == args[0]
    state = C.training_state("train", [m], opt, args[1], 1, {"train_loss": [[1.0]], "test_loss": [[1.0]]})
    C.check_state(state, "train", [m], opt, args[1], 2)
    with pytest.raises(ValueError, match=r"precision=0, the checkpoint 1"):
        C.check_state(state, "train", [m], opt, args[0], 2)
    # a state written before the precision was recorded is an fp32 state
    old = dict(state, args={k: v for k, v in args[1].items() if k != "precision"})
    C.check_state(old, "train", [m], opt, args[0], 2)
    with pytest.raises(ValueError, match=r"precision=1, the checkpoint 0"):
        C.check_state(old, "train", [m], opt, args[1], 2)
