"""GPU tier of the structural kernel tests: properties that a correct GPT-2 kernel satisfies bit for bit, at the 64- and
128-row tile edges where a mask or a tile range is most easily off by one key.

- Causality: changing token j leaves the logits of every earlier token bitwise unchanged (a masked score gets P = 0
  exactly, and 0 * v adds nothing).
- Coverage: changing token j changes the logits of token j and of every later token.
- Gradients: with the loss on output row r only, every wpe.grad row past r + 1 is exactly zero and every row up to
  r + 1 is nonzero.
- Scratch: outputs, dumps and gradients do not depend on what the workspace, K/V cache and output buffers held before
  the call (every torch.empty filled with NaN / 0xFF against filled with zeros).

These catch a key missing or leaking at a tile edge, which moves bf16 logits by less than the bf16 noise floor and so
passes the 2e-2 tolerance tests.  Value-level errors below that floor (a dropped LayerNorm epsilon, a rounding change)
are out of scope here: the tolerance tests against the float64 oracle stay responsible for those.  The token / row
convention and the checks themselves are exercised on the float64 restatement in test_kernel_structure_cpu.py."""
import re

import pytest
import torch

import kernel_structure as KS

pytestmark = pytest.mark.gpu

HORIZON = 540     # n_positions = 4 * (1 + horizon) covers every length below
S_DENSE = [2, 64, 65, 127, 128, 129, 255, 256, 257, 383, 384, 385, 511, 512]   # dense kernels (fp32 and tcgen05)
S_SEQ = [513, 540]                                                                  # token-sequential kernel


def _model(dx, du, L, test=False, seed=0):
    return KS.model(dx, du, L, HORIZON, test, seed=seed).cuda()


def _check(out, js, what, test=False, first_token=1, coverage=True):
    bad = KS.dependency_violations(out, js, first_token, test, coverage)
    assert not bad, "%s: %s" % (what, "; ".join(bad[:6]))


def _entries(m, m2, S, precision):
    """(name, test flag, fn(batch) -> logits per member) of every forward entry point that takes S tokens."""
    from dpt_b200.models.net import forward_train_population

    def fwd(x):
        m.precision = precision
        return [m(x)]
    es = [("forward", fwd)]
    if S <= 512:
        es.append(("forward_train", lambda x: [m.forward_train(x, precision).detach()]))
        if precision == 1:   # k > 1 runs the population (NM = 32) instances of the training kernels
            es.append(("forward_train_population", lambda x: [o.detach() for o in forward_train_population([m, m2], [x, x], 1)]))
    return [(name, test, fn) for name, fn in es for test in (False, True)]


@pytest.mark.parametrize("precision", [0, 1])
@pytest.mark.parametrize("dx,du,L", KS.SHAPES)
def test_forward_dependency(dpt, dx, du, L, precision):
    """Every forward entry point at lengths around the tile edges: causality and coverage of every output row, and the
    base sequence's logits independent of the other sequences in its batch.

    Coverage is not a bitwise property of the bf16 dense kernels at L = 1: they round the attention output to bf16 before
    c_proj, and with one layer that output is the only path from token j to a later row.  A token that gets ~1/S of the
    attention moves a far row's attention output by less than one bf16 step (float64 restatement, darkroom, query
    perturbed: 0.04 of a step at S = 511, token 478), so the logits can stay bitwise equal on a correct kernel (seen:
    S = 127, token 121).  The token-sequential kernel (S > 512) keeps that output in fp32.  At L = 4 the change also reaches the row through every intermediate row's keys and values; there,
    and at L = 1 in fp32, coverage is asserted."""
    m, m2 = _model(dx, du, L), _model(dx, du, L, seed=1)
    for S in S_DENSE + S_SEQ:
        js = KS.probes(S)
        x = KS.perturbed_batch(dx, du, S, js, seed=S, device="cuda")
        x1 = {k: v[:1] for k, v in x.items()}
        for name, test, fn in _entries(m, m2, S, precision):
            m.test = m2.test = test
            outs, alone = fn(x), fn(x1)
            for i, (o, a) in enumerate(zip(outs, alone)):
                what = "%s member %d precision %d S=%d test=%s" % (name, i, precision, S, test)
                _check(o, js, what, test, coverage=not (precision == 1 and L == 1 and S <= 512))
                assert torch.equal(o[:1], a), "%s: the base sequence depends on its batch" % what


ROWS = (0, 62, 63, 64, 65, 127, 128, 191, 192, 255, 256, 447, 448)


@pytest.mark.parametrize("precision", [0, 1])
@pytest.mark.parametrize("dx,du,L", KS.SHAPES)
def test_backward_dependency(dpt, dx, du, L, precision):
    """Loss on one output row r: the gradient reaches the position embedding of every token up to r + 1 and of no later
    one.  Covers the bf16 attention backward's dq range (key tiles 0..t) and dk/dv range (query tiles t..nt-1), the bf16
    row kernels and the fp32 backward."""
    m = _model(dx, du, L)
    for T in (65, 200, 511):
        x = KS.base_batch(dx, du, 2, T, seed=T, device="cuda")
        bad = []
        for r in sorted(set(ROWS + (T - 1,)) & set(range(T))):
            m.zero_grad(set_to_none=True)
            KS.row_weighted_ce(m.forward_train(x, precision), x["optimal_actions"], r).backward()
            bad += KS.wpe_grad_violations(m.transformer.wpe.weight.grad, r)
        assert not bad, "precision %d T=%d: %s" % (precision, T, "; ".join(bad[:6]))


def _decode(m, x, H):
    """Logits of every position 0..H of a decoder fed the batch token by token: [B, H + 1, du]."""
    dec = m.decoder(x["query_states"].shape[0], H)
    out = [dec.query(x["query_states"])]
    for t in range(H):
        out.append(dec.append(*(x[k][:, t] for k in ("context_states", "context_actions", "context_next_states",
                                                      "context_rewards"))))
    return torch.stack(out, 1)


DECODE_PROBES = (0, 7, 8, 15, 16, 31, 32, 63, 64, 65, 127, 128)   # 16-key V blocks, 64-key K tiles, the trimmed last tile


@pytest.mark.parametrize("precision", [0, 1])
@pytest.mark.parametrize("dx,du,L", KS.SHAPES)
def test_decode_dependency(dpt, dx, du, L, precision):
    """Transformer.decoder: the logits at position h are bitwise the base's for h < j and differ for h >= j, where the
    sequence differs from the base in the token at position j."""
    H = 200
    m = _model(dx, du, L, test=True)
    m.precision = precision
    js = list(DECODE_PROBES) + [H - 1, H]
    x = KS.perturbed_batch(dx, du, H + 1, js, seed=H, device="cuda")
    out = _decode(m, x, H)
    _check(out, js, "decoder precision %d" % precision, first_token=0)
    assert torch.equal(out[:1], _decode(m, {k: v[:1] for k, v in x.items()}, H)), "the base sequence depends on its batch"


def test_decode_dependency_long(dpt):
    """The bf16 decode past 1024 cached keys: probes at the 512- and 1024-key edges."""
    H = 1100
    m = _model(1, 5, 4, test=True)
    m.precision = 1
    js = [0, 64, 511, 512, 1023, 1024, H]
    x = KS.perturbed_batch(1, 5, H + 1, js, seed=H, device="cuda")
    _check(_decode(m, x, H), js, "decoder precision 1 H=%d" % H, first_token=0)


# ---- scratch independence ----------------------------------------------------------------------------------------

def _poison(t):
    if t.dtype == torch.uint8:
        return t.fill_(0xFF)
    return t.fill_(float("nan")) if t.is_floating_point() else t.fill_(-1)


@pytest.fixture
def filled_runs(monkeypatch):
    """run(fn, models) -> (out_poisoned, out_zeroed): fn() once with every torch.empty filled with NaN (floats), 0xFF
    (uint8) or -1 (integers), and once with every torch.empty zero-filled; the models' cached workspaces are dropped
    before each run so that they are allocated under the fill."""
    def run(fn, models=()):
        outs = []
        for fill in (_poison, torch.Tensor.zero_):
            with monkeypatch.context() as mp:
                empty = torch.empty
                mp.setattr(torch, "empty", lambda *a, **k: fill(empty(*a, **k)))
                for m in models:
                    m._workspace = None
                outs.append(fn())
                torch.cuda.synchronize()
        for m in models:
            m._workspace = None
        return outs
    return run


def _tensors(o, key=""):
    if isinstance(o, torch.Tensor):
        yield key, o
    elif isinstance(o, dict):
        for k in sorted(o):
            yield from _tensors(o[k], key + "/" + str(k))
    elif isinstance(o, (list, tuple)):
        for i, v in enumerate(o):
            yield from _tensors(v, key + "/" + str(i))


def _same(a, b, what):
    ta, tb = list(_tensors(a)), list(_tensors(b))
    assert [k for k, _ in ta] == [k for k, _ in tb]
    for (k, x), (_, y) in zip(ta, tb):
        if x.is_floating_point():
            assert bool(torch.isfinite(x).all()) and bool(torch.isfinite(y).all()), "%s %s: not finite" % (what, k)
        if k.endswith("regret_sums"):   # float64 atomics: equal up to their order of addition
            assert torch.allclose(x, y, rtol=1e-12, atol=0), "%s %s" % (what, k)
        else:
            assert torch.equal(x, y), "%s %s: depends on what the buffers held" % (what, k)


@pytest.mark.parametrize("precision", [0, 1])
def test_forward_scratch_independent(dpt, filled_runs, precision):
    for dx in (1, 2):
        m = _model(dx, 5, 4)
        m.precision = precision
        for S in (100, 300, 540):   # one-tile, multi-tile and token-sequential (K/V workspace) kernels
            x = KS.base_batch(dx, 5, 9, S - 1, seed=S, device="cuda")
            for test in (False, True):
                m.test = test
                _same(*filled_runs(lambda: m(x), [m]), "forward dx=%d S=%d test=%s" % (dx, S, test))


@pytest.mark.parametrize("precision", [0, 1])
def test_train_scratch_independent(dpt, filled_runs, precision):
    """forward_train + backward, one model and a two-member population: logits and every gradient."""
    from dpt_b200.models.net import forward_train_population
    ms = [_model(2, 5, 4, seed=i) for i in range(2)]
    for T in (100, 300):
        x = KS.base_batch(2, 5, 6, T, seed=T, device="cuda")

        def step(members):
            for mm in members:
                mm.zero_grad(set_to_none=True)
            outs = forward_train_population(members, [x] * len(members), precision)
            sum(KS.row_weighted_ce(o, x["optimal_actions"], slice(None)) for o in outs).backward()
            return [o.detach() for o in outs], [[p.grad.clone() for p in mm._train_params()] for mm in members]
        _same(*filled_runs(lambda: step(ms[:1])), "forward_train T=%d" % T)
        _same(*filled_runs(lambda: step(ms)), "forward_train_population T=%d" % T)


@pytest.mark.parametrize("precision", [0, 1])
def test_decoder_scratch_independent(dpt, filled_runs, precision):
    m = _model(1, 5, 4, test=True)
    m.precision = precision
    x = KS.base_batch(1, 5, 11, 130, seed=3, device="cuda")
    _same(*filled_runs(lambda: _decode(m, x, 130)), "decoder")


def _bf16_ws_fits(L, H):
    """The online loop's choice at precision 1 (gpt2.cu online_launch): the warp-specialised kernel when L layers of
    weight fragments (24 KB each) and 24 warps of score scratch ((32 + 128 + Tpad) floats, Tpad = H rounded up to 64)
    fit the 227 KB of one SM's shared memory, else the 4-warp fallback."""
    return L * 24576 + 24 * (32 + 128 + (H + 63) // 64 * 64) * 4 <= 227 * 1024


def test_online_loop_cases_reach_their_variants(dpt):
    """The N / H of the scratch cases launch the kernel variant they are named after (kernel names from the profiler),
    with the one-model parameter block (member capacity NM = 1).  At L = 4 a horizon of 1210 (Tpad 1216) still fits the
    warp-specialised kernel; 1300 is past it."""
    for precision, L, N, H, variant in KS.online_cases() + [(1, 4, 6, 1210, "bf16 warp-specialised")]:
        assert _bf16_ws_fits(L, H) == (variant == "bf16 warp-specialised") or precision == 0
        m = KS.model(1, 5, L, H, True).cuda()
        m.precision = precision
        means, _, _ = dpt.kernels.bandit_sample_means(N, 5, 1, 0)
        m.online_loop(means, 2, 0.3, True, 1, 0)     # module load and handle outside the profile
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            m.online_loop(means, H, 0.3, True, 1, 0)
            torch.cuda.synchronize()
        names = [e.name for e in prof.events() if "gpt2_online_kernel" in e.name]
        args = {re.search(r"gpt2_online_kernel<(\w+), ?(\w+), ?(\w+), ?(\w+)", n).groups() for n in names}
        assert args == {KS.ONLINE_VARIANT_ARGS[variant.split(",")[0]] + ("1",)}, (variant, names)


# the training kernels, each templated on the member capacity NM of its launch (its last template argument)
TRAIN_KERNELS = {0: {"gpt2_train_forward_kernel", "gpt2_train_backward_kernel", "weight_grad_reduce_kernel", "wpe_grad_kernel"},
                 1: {"pack_wimg_kernel", "gpt2_train_forward_bf16_kernel", "gpt2_train_rows_bf16_kernel",
                     "gpt2_train_attn_bf16_kernel", "weight_grad_reduce_kernel", "wpe_grad_kernel"}}


@pytest.mark.parametrize("precision", [0, 1])
def test_training_launches_reach_their_member_capacity(dpt, precision):
    """A one-model forward_train + backward launches the NM = 1 instances of the training kernels (small parameter
    blocks), a two-member population the NM = 32 ones (kernel names from the profiler)."""
    from dpt_b200.models.net import POPULATION_MAX, forward_train_population
    ms = [_model(1, 5, 2, seed=i) for i in range(2)]
    x = KS.base_batch(1, 5, 4, 100, seed=1, device="cuda")
    pat = re.compile(r"(%s)<([^<>]*)>" % "|".join(TRAIN_KERNELS[precision]))
    for members, nm in ((ms[:1], "1"), (ms, str(POPULATION_MAX))):
        def step():
            outs = forward_train_population(members, [x] * len(members), precision)
            sum(KS.row_weighted_ce(o, x["optimal_actions"], slice(None)) for o in outs).backward()
        step()   # module load outside the profile
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            step()
            torch.cuda.synchronize()
        found = {(m.group(1), m.group(2).split(",")[-1].strip()) for m in map(pat.search, (e.name for e in prof.events())) if m}
        assert found == {(k, nm) for k in TRAIN_KERNELS[precision]}, (len(members), sorted(found))


@pytest.mark.parametrize("case", range(6))
def test_online_loop_scratch_independent(dpt, filled_runs, case):
    """online_loop with dump=True in every kernel variant, and a two-member online_loop_population: context, cumulative
    means, regret sums, reward noise, uniforms and logits."""
    from dpt_b200.models.net import online_loop_population
    precision, L, N, H, variant = KS.online_cases()[case]
    ms = [KS.model(1, 5, L, H, True, seed=i).cuda() for i in range(2)]
    for mm in ms:
        mm.precision = precision
    means, _, _ = dpt.kernels.bandit_sample_means(N, 5, 2, 0)
    _same(*filled_runs(lambda: ms[0].online_loop(means, H, 0.3, True, 5, 0, dump=True), ms), "online_loop " + variant)
    if N < 1000 and H <= 100:
        _same(*filled_runs(lambda: online_loop_population(ms, means, H, 0.3, True, 5, 0, dump=True), ms),
              "online_loop_population " + variant)


@pytest.mark.parametrize("precision", [0, 1])
def test_rollout_scratch_independent(dpt, filled_runs, precision):
    from dpt_b200.envs.gpu_bandit_env import GPUBanditEnv
    m = KS.model(1, 5, 3, 40, True).cuda()
    m.precision = precision
    _same(*filled_runs(lambda: GPUBanditEnv(5, 300, 40, var=0.3, seed=4).rollout(m, K=40), [m]), "GPUBanditEnv.rollout")
