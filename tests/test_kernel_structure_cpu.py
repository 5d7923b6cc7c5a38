"""CPU tier of the structural kernel tests: the perturbed batches, the token / output-row convention and the dependency
checks of test_kernel_structure_gpu.py, run against the float64 restatement in train_oracle.py.  Where the GPU file finds
a violation, this file shows that the harness itself expects the right pattern."""
import pytest
import torch

import kernel_structure as KS
import train_oracle as TO


def _forward(P, L, x, test):
    return TO.forward(P, L, x["query_states"], x["context_states"], x["context_actions"], x["context_next_states"],
                      x["context_rewards"], test)


@pytest.mark.parametrize("dx,du,L", KS.SHAPES)
def test_forward_dependency_float64(dx, du, L):
    m = KS.model(dx, du, L, 140, False)
    P = TO.params64(m)
    for S in (2, 64, 65, 129, 257):
        js = KS.probes(S)
        x = KS.perturbed_batch(dx, du, S, js, seed=S, dtype=torch.float64)
        assert x["context_actions"].shape == (1 + len(js), S - 1, du)
        # the perturbed token is the only difference from the base
        for k, j in enumerate(js, 1):
            if j == 0:
                assert not torch.equal(x["query_states"][k], x["query_states"][0])
                assert all(torch.equal(x[n][k], x[n][0]) for n in ("context_actions", "context_rewards"))
            else:
                assert torch.equal(x["query_states"][k], x["query_states"][0])
                rows = (x["context_actions"][k] != x["context_actions"][0]).any(-1).nonzero().flatten().tolist()
                assert rows == [j - 1] and x["context_rewards"][k, j - 1, 0] > x["context_rewards"][0, j - 1, 0] + 2.5
        with torch.no_grad():
            rows = _forward(P, L, x, False)
            last = _forward(P, L, x, True)
        assert rows.shape == (1 + len(js), S - 1, du) and last.shape == (1 + len(js), du)
        # test=True is the last row of test=False: the only output is token T
        assert torch.equal(last, rows[:, -1])
        assert KS.dependency_violations(rows, js) == [], S
        assert KS.dependency_violations(last, js, test=True) == [], S


def test_dependency_check_flags_leaks_and_misses():
    """The check itself: a row that changes before j, and a row that does not change at or after j, are reported."""
    out = torch.zeros(3, 6, 2)
    out[1, 2:] = 1.0                 # token j = 3 (row r = 2) onwards differs: correct
    out[2, 3:] = 1.0                 # j = 3, but row 2 (token 3) unchanged: a miss
    assert KS.dependency_violations(out[:2], [3]) == []
    assert KS.dependency_violations(out[[0, 2]], [3]) == ["j=3: tokens [3] unchanged although they come at or after j"]
    out[2, 0] = 1.0
    assert "j=3: tokens [1] changed although they come before j" in KS.dependency_violations(out[[0, 2]], [3])
    assert KS.dependency_violations(out[:2, 0], [1], test=True) == ["j=1: last-token logits unchanged"]
    g = torch.zeros(10, 4)
    g[:4] = 1.0
    assert KS.wpe_grad_violations(g, 2) == []
    assert KS.wpe_grad_violations(g, 1) == ["r=1: wpe.grad rows [3] are nonzero past r + 1"]
    assert KS.wpe_grad_violations(g, 3) == ["r=3: wpe.grad rows [4] are zero"]


@pytest.mark.parametrize("dx,du,L", KS.SHAPES)
def test_wpe_gradient_pattern_float64(dx, du, L):
    m = KS.model(dx, du, L, 140, False)
    for T in (65, 130):
        x = KS.base_batch(dx, du, 2, T, seed=T, dtype=torch.float64)
        for r in sorted({0, 63, 64, 127, 128, T - 1} & set(range(T))):
            P = TO.params64(m)
            KS.row_weighted_ce(_forward(P, L, x, False), x["optimal_actions"], r).backward()
            g = P["transformer.wpe.weight"].grad
            assert g.shape[0] == 4 * 141
            assert KS.wpe_grad_violations(g, r) == [], (T, r)
