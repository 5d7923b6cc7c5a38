"""CPU tier of the offline evaluation: argument validation of dpt_offline_eval without a GPU, and the numpy restatement
(tests/offline_oracle.py) against the reference's own offline() run in tests/golden/offline_bandit.npz."""
import ctypes

import numpy as np
import pytest

from conftest import golden
from oracle import dpt_oracle as O
from oracle import philox as P
import offline_oracle as OO

EMP, LCB, THMP, LINREG = 1 << 1, 1 << 2, 1 << 3, 1 << 4


def _params(dpt, horizons, N=4, d=5, H_stride=8, mask=1 | EMP | LCB | THMP, lin_d=0, n_draws=100):
    hz = np.asarray(horizons, dtype=np.int32)
    p = dpt._lib.OfflineParams()
    p.N, p.d, p.H_stride, p.K = N, d, H_stride, len(hz)
    p.horizons_host = hz.ctypes.data
    p.ctrl_mask, p.lcb_const = mask, 0.8
    p.thmp_std, p.thmp_prior_mean, p.thmp_prior_var, p.n_draws = 0.3, 0.5, 1 / 12.0, n_draws
    p.lin_d = lin_d
    return p, hz


def _call(dpt, p):
    return dpt._lib.lib().dpt_offline_eval(ctypes.byref(p), None, None, None, None, None, None)


@pytest.mark.parametrize("case,horizons,kw,word", [
    ("horizon0", [3, 0, 2], {}, b"horizon 0"),
    ("horizon_gt_stride", [9], {}, b"horizon 9"),
    ("d33", [1], dict(d=33), b"d=33"),
    ("lin_d9", [1], dict(mask=1 | LINREG, lin_d=9), b"lin_d=9"),
    ("n_draws0", [1], dict(n_draws=0), b"n_draws=0"),
])
def test_offline_eval_rejects_bad_args(dpt, case, horizons, kw, word):
    p, hz = _params(dpt, horizons, **kw)
    lib = dpt._lib.lib()
    assert _call(dpt, p) == dpt._lib.ERR_INVALID_ARG
    assert word in lib.dpt_last_error(), lib.dpt_last_error()


def test_offline_eval_empty_batch_is_noop(dpt):
    p, hz = _params(dpt, [1, 8, 4], N=0)
    assert _call(dpt, p) == 0
    p, hz = _params(dpt, [], N=4)
    assert _call(dpt, p) == 0
    p, hz = _params(dpt, [1], N=4)
    assert _call(dpt, p) == dpt._lib.ERR_INVALID_ARG and b"null" in dpt._lib.lib().dpt_last_error()   # N > 0 needs buffers


def test_stream_tag_is_new():
    tags = [getattr(P, n) for n in dir(P) if n.startswith("STREAM_")]
    assert OO.STREAM_OFFLINE not in tags and OO.STREAM_OFFLINE == max(tags) + 1


def _golden_ctx():
    g = golden("offline_bandit")
    d = int(g["d"])
    return g, d, np.eye(d)[g["context_actions"]], np.asarray(g["context_rewards"], dtype=np.float64)


def test_oracle_driver_matches_reference_golden():
    """The restated driver with PessMeanCtrl and the 100-draw Thompson mode reproduces the reference's offline()
    rewards for opt / emp / lcb / thmp when fed the reference's normals (np.random.seed(seed + h), 4N env draws first)."""
    g, d, ca, cr = _golden_ctx()
    N, H, var, seed = g["means"].shape[0], int(g["H"]), float(g["var"]), int(g["seed"])
    horizons = [H, H // 2, 1]
    zs = []
    for h in horizons:
        np.random.seed(seed + h)
        np.random.standard_normal(4 * N)
        zs.append(np.random.standard_normal((100, N, d)))
    ctrls = {"opt": O.OptCtrl(g["means"]), "emp": O.EmpMeanCtrl(d, online=False), "lcb": OO.PessMeanCtrl(d, .8),
             "thmp": O.ThompsonCtrl(d, std=var, sample=False, prior_mean=.5, prior_var=1 / 12.0)}
    rew, sums = OO.offline_eval(g["means"], ca, cr, horizons, ctrls, O.ReplayNoise({"thompson_z": np.concatenate(zs)}))
    for k, h in enumerate(horizons):
        for name in ctrls:
            assert np.allclose(rew[name][k], g["h%d_%s" % (h, name)], rtol=0, atol=1e-6), (h, name)
    best = g["means"].max(1)
    assert np.allclose(sums["emp"][:, 0], (best[None] - rew["emp"]).sum(1)) and np.all(sums["opt"] == 0)
