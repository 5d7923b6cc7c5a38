"""CPU tier of training: the float64 torch restatement of the forward (tests/train_oracle.py), which is the yardstick of
the training kernels' gradients, against the reference's golden logits, the numpy oracle and (when installed) the
HuggingFace GPT2Model's autograd."""
import numpy as np
import pytest
import torch

from conftest import golden
from oracle import dpt_oracle as O
import train_oracle as TO


def _golden_params(g):
    return {k[3:]: torch.tensor(g[k], dtype=torch.float64, requires_grad=True) for k in g.files
            if k.startswith("sd/") and "wte" not in k and not k.endswith(".attn.bias") and not k.endswith(".attn.masked_bias")}


def _golden_batch(g, t):
    d = int(g["d"])
    acts, rew = g["fwd_actions"].astype(np.int64), g["fwd_rewards"]
    B = acts.shape[0]
    f = lambda a: torch.tensor(a, dtype=torch.float64)   # noqa: E731
    return (f(np.ones((B, 1))), f(np.ones((B, t, 1))), f(np.eye(d)[acts[:, :t]]), f(np.ones((B, t, 1))), f(rew[:, :t]))


@pytest.mark.parametrize("name", ["transformer_l2", "transformer_l4"])
def test_restatement_matches_reference_logits(name):
    g = golden(name)
    P, L = _golden_params(g), int(g["n_layer"])
    n = 0
    for k in g.files:
        if not k.startswith("logits_"):
            continue
        t = int(k.rsplit("_t", 1)[1])
        test = not k.startswith("logits_all")
        with torch.no_grad():
            out = TO.forward(P, L, *_golden_batch(g, t), test=test).numpy()
        ref = g[k]
        assert out.shape == ref.shape
        assert np.abs(out - ref).max() <= 1e-5 * max(1.0, np.abs(ref).max()), k
        n += 1
    assert n >= 7


def test_restatement_matches_numpy_oracle():
    from dpt_b200.models.net import Transformer   # noqa: F401  (import only: no GPU needed to build the module)
    torch.manual_seed(1)
    m = Transformer({"horizon": 30, "state_dim": 2, "action_dim": 5, "n_layer": 3, "n_embd": 32, "n_head": 1, "dropout": 0.0,
                     "test": True})
    with torch.no_grad():
        for k, p in m.named_parameters():
            p.add_(0.2 * torch.randn_like(p))
    P = TO.params64(m)
    sd = {k: v.detach().numpy() for k, v in P.items()}
    rng = np.random.RandomState(0)
    B, T = 4, 17
    q, cs, ns = rng.randint(0, 5, (B, 2)), rng.randint(0, 5, (B, T, 2)), rng.randint(0, 5, (B, T, 2))
    ca, cr = np.eye(5)[rng.randint(0, 5, (B, T))], rng.rand(B, T, 1)
    args = [torch.tensor(a, dtype=torch.float64) for a in (q, cs, ca, ns, cr)]
    for test in (True, False):
        with torch.no_grad():
            out = TO.forward(P, 3, *args, test=test).numpy()
        ref = O.transformer_forward(sd, q, cs, ca, ns, cr, 3, test=test)
        assert np.abs(out - ref).max() <= 1e-12 * max(1.0, np.abs(ref).max())


def test_restatement_gradients_match_hf_gpt2():
    transformers = pytest.importorskip("transformers")
    g = golden("transformer_l2")
    P, L = _golden_params(g), int(g["n_layer"])
    d = int(g["d"])
    cfg = transformers.GPT2Config(n_positions=P["transformer.wpe.weight"].shape[0], n_embd=32, n_layer=L, n_head=1,
                                  resid_pdrop=0.0, embd_pdrop=0.0, attn_pdrop=0.0, use_cache=False)
    hf = transformers.GPT2Model(cfg).double()
    hf.load_state_dict({k[len("transformer."):]: v.detach() for k, v in P.items() if k.startswith("transformer.")}, strict=False)
    emb, head = torch.nn.Linear(1 + d + 1 + 1, 32).double(), torch.nn.Linear(32, d).double()
    with torch.no_grad():
        emb.weight.copy_(P["embed_transition.weight"]), emb.bias.copy_(P["embed_transition.bias"])
        head.weight.copy_(P["pred_actions.weight"]), head.bias.copy_(P["pred_actions.bias"])
    batch = _golden_batch(g, 12)
    target = torch.eye(d, dtype=torch.float64)[torch.tensor([0, 1, 2, 3, 4, 0])]
    ours = TO.forward(P, L, *batch, test=False)
    loss = torch.nn.functional.cross_entropy(ours.reshape(-1, d), target[:, None].expand(-1, 12, -1).reshape(-1, d), reduction="sum")
    loss.backward()
    x = hf(inputs_embeds=emb(TO.tokens(*batch))).last_hidden_state
    theirs = head(x)[:, 1:, :]
    loss2 = torch.nn.functional.cross_entropy(theirs.reshape(-1, d), target[:, None].expand(-1, 12, -1).reshape(-1, d), reduction="sum")
    loss2.backward()
    hp = dict(hf.named_parameters())
    for k, p in P.items():
        if k.startswith("transformer."):
            ref = hp[k[len("transformer."):]].grad
        else:
            ref = (emb if k.startswith("embed") else head).state_dict(keep_vars=True)[k.split(".", 1)[1]].grad
        assert torch.allclose(p.grad, ref, rtol=1e-9, atol=1e-12), k
