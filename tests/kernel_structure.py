"""Helpers of the structural kernel tests (test_kernel_structure_cpu.py, test_kernel_structure_gpu.py): the model they
use, a batch whose sequences differ from a base sequence in exactly one token each, the check that an output row
depends on a token exactly when causality says it must, and the online-loop cases (one per kernel variant) that
test_sharp_attention_gpu.py shares.

Token convention (the reference's models/net.py): token 0 is the query, token t >= 1 is context row t - 1.  With
``test=False`` output row r is token r + 1; with ``test=True`` the only output is token T."""
import torch

SHAPES = [(1, 5, 1), (1, 5, 4), (2, 5, 1), (2, 5, 4)]   # (dx, du, L): bandit and darkroom token layouts


def model(dx, du, L, horizon, test, seed=0, scale=0.15):
    """A Transformer with n_embd = 32 and ``scale * randn`` added to every parameter except wte, as the other tests."""
    from dpt_b200.models.net import Transformer
    torch.manual_seed(seed)
    m = Transformer({"horizon": horizon, "state_dim": dx, "action_dim": du, "n_layer": L, "n_embd": 32, "n_head": 1,
                     "dropout": 0.0, "test": test})
    with torch.no_grad():
        for k, p in m.named_parameters():
            if "wte" not in k:
                p.add_(scale * torch.randn_like(p))
    return m


def probes(S, edges=(0, 1, 63, 64, 126, 127, 128, 129, 255, 256, 383, 384)):
    """Token positions at the 64- and 128-row tile edges, and the last two tokens, of a sequence of S tokens."""
    return sorted({j for j in edges + (S - 2, S - 1) if 0 <= j < S})


def base_batch(dx, du, B, T, seed, dtype=torch.float32, device="cpu"):
    """B random sequences of T transitions: bandit (dx = 1) constant states, darkroom (dx = 2) integer states 0..9,
    one-hot actions, rewards in [0, 1); ``optimal_actions`` one-hot targets."""
    g = torch.Generator().manual_seed(seed)
    if dx == 1:
        q, cs, cns = torch.ones(B, 1), torch.ones(B, T, 1), torch.ones(B, T, 1)
    else:
        q = torch.randint(0, 10, (B, dx), generator=g).float()
        cs = torch.randint(0, 10, (B, T, dx), generator=g).float()
        cns = torch.randint(0, 10, (B, T, dx), generator=g).float()
    ca = torch.eye(du)[torch.randint(0, du, (B, T), generator=g)]
    cr = torch.rand(B, T, 1, generator=g)
    opt = torch.eye(du)[torch.randint(0, du, (B,), generator=g)]
    b = {"query_states": q, "context_states": cs, "context_actions": ca, "context_next_states": cns, "context_rewards": cr,
         "optimal_actions": opt}
    return {k: v.to(device=device, dtype=dtype) for k, v in b.items()}


def perturbed_batch(dx, du, S, js, seed, dtype=torch.float32, device="cpu"):
    """1 + len(js) sequences of S tokens: sequence 0 is the base, sequence k (k >= 1) equals it except token js[k - 1].
    Token 0 gets another query state; a context token another one-hot action, reward + 3 and, for dx = 2, other states."""
    T = S - 1
    b = base_batch(dx, du, 1, T, seed)
    b = {k: v.repeat(1 + len(js), *([1] * (v.dim() - 1))) for k, v in b.items()}
    for k, j in enumerate(js, 1):
        if j == 0:
            b["query_states"][k] += 3.0 if dx == 2 else -3.0
            continue
        t = j - 1
        a = int(b["context_actions"][k, t].argmax())
        b["context_actions"][k, t] = torch.eye(du)[(a + 1 + (k - 1) % (du - 1)) % du]
        b["context_rewards"][k, t] += 3.0
        if dx == 2:
            b["context_states"][k, t] += 3.0
            b["context_next_states"][k, t] -= 3.0
    return {k: v.to(device=device, dtype=dtype) for k, v in b.items()}


def dependency_violations(out, js, first_token=1, test=False, coverage=True):
    """Where ``out`` (sequence 0 = base, sequence k differs in token js[k - 1]) breaks causality or coverage.

    ``test=False``: out is [B, R, du] and row r holds the output of token r + first_token; a row must be bitwise equal to
    the base row when its token comes before j, and differ from it (in some logit) when its token is j or later.
    ``test=True``: out is [B, du], the output of the last token, which comes at or after every j: it must differ.
    ``coverage=False`` checks causality alone.  Returns a list of readable violations (empty when the properties hold)."""
    out = out.detach().cpu()
    bad = []
    if not bool(torch.isfinite(out).all()):
        bad.append("non-finite logits")
    if test:
        for k, j in enumerate(js, 1):
            if coverage and torch.equal(out[k], out[0]):
                bad.append("j=%d: last-token logits unchanged" % j)
        return bad
    differs = (out[1:] != out[:1]).any(-1)                         # [B - 1, R]
    tok = torch.arange(out.shape[1]) + first_token
    for k, j in enumerate(js):
        must = tok >= j
        leak = (differs[k] & ~must).nonzero().flatten()
        miss = (~differs[k] & must).nonzero().flatten()
        if len(leak):
            bad.append("j=%d: tokens %s changed although they come before j" % (j, (leak + first_token).tolist()[:8]))
        if coverage and len(miss):
            bad.append("j=%d: tokens %s unchanged although they come at or after j" % (j, (miss + first_token).tolist()[:8]))
    return bad


def row_weighted_ce(pred, target, r):
    """Cross-entropy of output row r only: the per-row losses times a one-hot row weight (as ce_weighted in
    test_train_gpu.py, with all weight on one row)."""
    B, R, du = pred.shape
    w = torch.zeros(R, dtype=pred.dtype, device=pred.device)
    w[r] = 1.0
    t = target[:, None].expand(-1, R, -1).to(pred.dtype)
    ce = torch.nn.functional.cross_entropy(pred.reshape(-1, du), t.reshape(-1, du), reduction="none").reshape(B, R)
    return (ce * w).sum()


def wpe_grad_violations(g, r):
    """wpe.grad after a loss on output row r (token r + 1): rows j <= r + 1 must be nonzero, rows j > r + 1 exactly 0."""
    nz = (g.detach().cpu() != 0).any(-1)
    pos = torch.arange(len(nz))
    bad = []
    zero = ((pos <= r + 1) & ~nz).nonzero().flatten()
    leak = ((pos > r + 1) & nz).nonzero().flatten()
    if len(zero):
        bad.append("r=%d: wpe.grad rows %s are zero" % (r, zero.tolist()[:8]))
    if len(leak):
        bad.append("r=%d: wpe.grad rows %s are nonzero past r + 1" % (r, leak.tolist()[:8]))
    return bad


def online_cases():
    """(precision, L, N, H, variant) of the online loop, one per instantiation of gpt2_online_kernel: gpt2.cu
    online_launch picks the variant from the env-warps per SM (one env per warp) at precision 0 and from the shared
    memory the weight fragments need at precision 1.  test_kernel_structure_gpu.py checks with the profiler that each
    case launches the variant it is named after."""
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    return [(0, 2, 37, 100, "fp32 bulk-copy ring, 1-warp CTAs"),
            (0, 2, 16 * sms, 100, "fp32 bulk-copy ring, 2-warp CTAs"),
            (0, 2, 24 * sms, 100, "fp32 bulk-copy ring, 4-warp CTAs"),
            (0, 2, 24 * sms + 1, 100, "fp32 register-staged"),
            (1, 2, 37, 100, "bf16 warp-specialised"),
            (1, 4, 6, 1300, "bf16 fallback")]


# (BF16, WS, TMA) template arguments of gpt2_online_kernel per variant of online_cases
ONLINE_VARIANT_ARGS = {"fp32 bulk-copy ring": ("false", "false", "true"),
                       "fp32 register-staged": ("false", "false", "false"),
                       "bf16 warp-specialised": ("true", "true", "false"), "bf16 fallback": ("true", "false", "false")}
