"""CPU tier of the sharp-attention tests: the inputs of test_sharp_attention_gpu.py are in the regime they claim, and the
float64 reference is well enough conditioned there for the fp32 and bf16 bars.

- Regime (layer 0, every case and length of the GPU file): median score range >= 10 nats and median largest
  probability >= 0.3; past 128 tokens, at least a quarter of the rows past token 128 have their argmax key past the
  first 128-key tile, and the batch has a row whose argmax key is in the last tile, except at the darkroom lengths
  listed in UNCOVERED.
- Conditioning: the float32 restatement at ALPHA_FP32 is within 4e-6 of float64 (2.5x under 1e-5); a restatement that
  rounds q, k, v, P and the projection operands to bf16 at ALPHA_BF16 is within 1e-2 of float64, normwise (half the 2e-2
  bar).  That bf16 estimate is not an emulation of the kernels' rounding, only a measure of how much the regime amplifies
  it."""
import functools

import pytest
import torch

import sharp_attention as SA


@functools.lru_cache(maxsize=None)
def _stats(dx, seed, alpha, T):
    m = SA.model(dx, SA.DU, SA.L, False, alpha, seed=seed)
    s = SA.layer_stats(m, SA.L, SA.batch(dx, SA.DU, 4, T, seed=T))[0]
    return s["range"], s["top"], s["moved"], tuple(s["last_tile"])


# (dx, T) where the tile-crossing statistics do not hold, and what is missing.  In the darkroom layout the integer states
# weigh more in a token than the landmark rewards, and at these lengths no landmark takes a row maximum past the first
# tile (T = 128, 129) or into a last tile of a single key (T = 256, 384: the only row that can reach it is the last).
UNCOVERED = {(2, 128): "moved, last tile", (2, 129): "moved, last tile", (2, 256): "moved, last tile",
             (2, 384): "last tile"}


@pytest.mark.parametrize("dx,seed", SA.CASES)
def test_regime_is_sharp(dx, seed):
    """Per length: median score range >= 10 nats and median largest probability >= 0.3; past 128 tokens, at least a
    quarter of the rows past token 128 have their argmax key past the first 128-key tile, and the batch has a row
    whose argmax key is in the last tile, except at the lengths listed in UNCOVERED."""
    for T in SA.TS:
        rng, top, moved, last = _stats(dx, seed, SA.ALPHA_FP32, T)
        what = "dx=%d T=%d: range %.1f top %.2f moved %.2f last tile %s" % (dx, T, rng, top, moved, last)
        print(what)
        assert rng >= 10 and top >= 0.3, what
        gap = UNCOVERED.get((dx, T), "")
        if T >= 128:
            assert "moved" in gap or moved >= 0.25, what
            assert "last tile" in gap or any(last), what


def test_restatement_unchanged_without_hooks():
    """train_oracle.forward without record / rnd computes the same products as with an identity rnd."""
    m = SA.model(2, SA.DU, 2, False, SA.ALPHA_FP32)
    x = {k: v.double() for k, v in SA.batch(2, SA.DU, 2, 70, seed=1).items()}
    P = SA.params(m)
    for test in (False, True):
        assert torch.equal(SA.forward(P, 2, x, test), SA.forward(P, 2, x, test, record=[], rnd=lambda t: t))


@pytest.mark.parametrize("dx,seed", SA.CASES)
def test_bf16_regime_is_sharper_than_init(dx, seed):
    """At ALPHA_BF16 the rows are still far from uniform: median score range >= 4 nats at every length."""
    for T in SA.TS:
        rng, top, moved, last = _stats(dx, seed, SA.ALPHA_BF16, T)
        print("bf16 dx=%d T=%d: range %.1f top %.2f moved %.2f" % (dx, T, rng, top, moved))
        assert rng >= 4, (T, rng)


def _errors(dx, seed, T):
    x = SA.batch(dx, SA.DU, 4, T, seed=T)
    x64 = {k: v.double() for k, v in x.items()}
    m = SA.model(dx, SA.DU, SA.L, False, SA.ALPHA_FP32, seed=seed)
    with torch.no_grad():
        o32 = SA.forward(SA.params(m, torch.float32), SA.L, x, False)
        e32 = SA.rel_err(o32, SA.forward(SA.params(m), SA.L, x64, False))
        m = SA.model(dx, SA.DU, SA.L, False, SA.ALPHA_BF16, seed=seed)
        P = SA.params(m)
        o64 = SA.forward(P, SA.L, x64, False)
        ob = SA.forward(P, SA.L, x64, False, rnd=SA.bf16)
    return e32, ((ob - o64).abs().max() / o64.abs().max().clamp_min(1.0)).item()


@pytest.mark.parametrize("dx,seed", SA.CASES)
def test_reference_conditioning(dx, seed):
    for T in SA.TS:
        e32, eb = _errors(dx, seed, T)
        print("dx=%d T=%d: float32 restatement %.2e, bf16 estimate %.2e" % (dx, T, e32, eb))
        assert e32 <= 4e-6, (T, e32)
        assert eb <= 1e-2, (T, eb)
