"""Float64 torch restatement of models/net.py's forward (the reference's GPT-2 trunk with one head, embed_transition,
pred_actions) in plain ops, for autograd: the yardstick of the training kernels' gradients.  Like offline_oracle.py it
lives outside the pinned oracle/ package."""
import math

import torch


def params64(model, device="cpu"):
    """The model's parameters except transformer.wte (unused by the forward) as float64 leaf tensors that require grad,
    keyed by the reference state_dict names."""
    return {k: p.detach().to(device=device, dtype=torch.float64).clone().requires_grad_(True)
            for k, p in model.named_parameters() if "wte" not in k}


def _ln(x, w, b):
    mu = x.mean(-1, keepdim=True)
    var = ((x - mu) ** 2).mean(-1, keepdim=True)
    return (x - mu) / torch.sqrt(var + 1e-5) * w + b


def _gelu_new(x):
    return 0.5 * x * (1.0 + torch.tanh(math.sqrt(2.0 / math.pi) * (x + 0.044715 * x ** 3)))


def tokens(q, cs, ca, cns, cr):
    """[B, T+1, 2dx+du+1]: query token at position 0 (zero action / next state / reward), then the transitions."""
    B, T, dx = ca.shape[0], ca.shape[1], q.shape[-1]
    first = torch.cat([q.reshape(B, 1, dx), torch.zeros(B, 1, ca.shape[-1] + dx + 1, dtype=q.dtype, device=q.device)], -1)
    rest = torch.cat([cs, ca, cns, cr.reshape(B, T, 1)], -1)
    return torch.cat([first, rest], 1)


def forward(P, n_layer, q, cs, ca, cns, cr, test, sdpa=False):
    """Transformer.forward in the dtype of P (float64 for the yardstick; float32 with sdpa=True is the eager torch
    training step that scripts/train_time.py times)."""
    dt = P["embed_transition.weight"].dtype
    seq = tokens(*(t.to(dt) for t in (q, cs, ca, cns, cr)))
    S = seq.shape[1]
    x = seq @ P["embed_transition.weight"].T + P["embed_transition.bias"] + P["transformer.wpe.weight"][:S]
    E = x.shape[-1]
    mask = torch.ones(S, S, dtype=torch.bool, device=x.device).tril()
    for l in range(n_layer):
        p = "transformer.h.%d." % l
        h = _ln(x, P[p + "ln_1.weight"], P[p + "ln_1.bias"])
        qkv = h @ P[p + "attn.c_attn.weight"] + P[p + "attn.c_attn.bias"]
        qq, k, v = qkv[..., :E], qkv[..., E:2 * E], qkv[..., 2 * E:]
        if sdpa:
            a = torch.nn.functional.scaled_dot_product_attention(qq, k, v, is_causal=True)
        else:
            s = (qq @ k.transpose(-1, -2)) / math.sqrt(E)
            a = torch.softmax(s.masked_fill(~mask, float("-inf")), -1) @ v
        x = x + a @ P[p + "attn.c_proj.weight"] + P[p + "attn.c_proj.bias"]
        h = _ln(x, P[p + "ln_2.weight"], P[p + "ln_2.bias"])
        x = x + _gelu_new(h @ P[p + "mlp.c_fc.weight"] + P[p + "mlp.c_fc.bias"]) @ P[p + "mlp.c_proj.weight"] + P[p + "mlp.c_proj.bias"]
    x = _ln(x, P["transformer.ln_f.weight"], P["transformer.ln_f.bias"])
    preds = x @ P["pred_actions.weight"].T + P["pred_actions.bias"]
    return preds[:, -1, :] if test else preds[:, 1:, :]
