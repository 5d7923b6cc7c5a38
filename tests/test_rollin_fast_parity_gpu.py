"""GPU tier: the fast bandit rollin kernel (lane = step quad, 128-step warp tasks) against the generic kernel (lane = step) at
the same shape.  The generic path is forced with output views that are not 16 B aligned.  Both draw the same Philox words per
(env, step), so the four context tensors are bit-identical; the return statistics group their fp32 partial sums differently,
so the optimal-pull count is exact and the two sums agree to 1e-6 relative.

The grid covers what the fast kernel's structure introduces: a single quad (H = 4), ragged last 128-step ranges (124, 132,
500), 64-bit quad bit strings (d = 10, 16), a single env and fewer envs than warps per CTA."""
import pytest
import torch

pytestmark = pytest.mark.gpu

KEYS = ("context_states", "context_actions", "context_next_states", "context_rewards")


def _unaligned_like(out):
    return {n: torch.empty(t.numel() + 1, device=t.device, dtype=t.dtype)[1:].view_as(t) for n, t in out.items()}


def _run(k, means, H, seed, generic, **kw):
    N, d = means.shape
    out = {"context_states": torch.empty((N, H, 1), device="cuda"), "context_actions": torch.empty((N, H, d), device="cuda"),
           "context_next_states": torch.empty((N, H, 1), device="cuda"), "context_rewards": torch.empty((N, H, 1), device="cuda")}
    if generic:
        out = _unaligned_like(out)
        assert all(t.data_ptr() % 16 for t in out.values())
    stats = torch.zeros(3, dtype=torch.float64, device="cuda")
    res = k.bandit_rollin(means, H, 0.3, seed, 11, out=out, stats=stats, **kw)
    torch.cuda.synchronize()
    return res, stats.cpu()


def _check_stats(fast, gen):
    assert fast[2].item() == gen[2].item()
    for i in (0, 1):
        assert abs(fast[i].item() - gen[i].item()) <= 1e-6 * max(abs(gen[i].item()), 1e-30), (i, fast[i].item(), gen[i].item())


@pytest.mark.parametrize("N", [1, 33, 1000])
@pytest.mark.parametrize("H", [4, 124, 128, 132, 500])
@pytest.mark.parametrize("d", [2, 3, 4, 5, 6, 8, 10, 16])
def test_bandit_rollin_fast_matches_generic(dpt, d, H, N):
    k = dpt.kernels
    means, _, _ = k.bandit_sample_means(N, d, 5 + d, 11)
    fast, sf = _run(k, means, H, 321, False)
    gen, sg = _run(k, means, H, 321, True)
    for n in KEYS:
        assert torch.equal(fast[n], gen[n]), n
    _check_stats(sf, sg)


@pytest.mark.parametrize("d,H,N", [(5, 500, 40), (10, 132, 33), (3, 4, 1)])
def test_bandit_rollin_fast_matches_generic_bernoulli(dpt, d, H, N):
    k = dpt.kernels
    means, _, _ = k.bandit_sample_means(N, d, 3, 0)
    fast, sf = _run(k, means, H, 77, False, reward_type="bernoulli")
    gen, sg = _run(k, means, H, 77, True, reward_type="bernoulli")
    for n in KEYS:
        assert torch.equal(fast[n], gen[n]), n
    _check_stats(sf, sg)


@pytest.mark.parametrize("d,H,N", [(5, 500, 40), (16, 260, 9), (2, 4, 3)])
def test_bandit_rollin_fast_dump_and_inject_match_generic(dpt, d, H, N):
    """Dump mode writes the same u, z and actions per step from both kernels; injecting them back reproduces the run."""
    k = dpt.kernels
    means, _, _ = k.bandit_sample_means(N, d, 9, 0)
    fast, _ = _run(k, means, H, 5, False, dump=True)
    gen, _ = _run(k, means, H, 5, True, dump=True)
    for n in KEYS:
        assert torch.equal(fast[n], gen[n]), n
    for n in fast["noise"]:
        assert torch.equal(fast["noise"][n], gen["noise"][n]), n
    nz = fast["noise"]
    inj = {"cov_idx": nz["cov_idx"], "dir_probs": nz["dir_probs"], "rand_idx": nz["rand_idx"], "u": nz["u"], "z": nz["z"]}
    for kw in ({"inject": inj}, {"inject": {"actions": nz["actions"], "z": nz["z"]}}):
        again, _ = _run(k, means, H, 0, False, **kw)
        for n in KEYS:
            assert torch.equal(again[n], fast[n]), n
