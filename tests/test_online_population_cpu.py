"""CPU tier of population evaluation: argument checks of dpt_gpt2_online_loop_population that run before any launch (no
GPU needed), the ValueErrors of online_loop_population for members that do not line up, and how a population is cut into
launches by member capacity and by the K/V scratch bound."""
import ctypes
import os
import re

import pytest

E_ARG = -1
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _call(lib, models, n, N=100, H=50, kv=None, kv_bytes=0):
    return lib.dpt_gpt2_online_loop_population(models, n, None, 0.3, 0, 1, 7, 0, N, H, 0, kv, kv_bytes, None, None, None,
                                               None, None, None, None, None, None)


def test_population_online_entry_point_rejects_bad_arguments(dpt):
    lib = dpt._lib.lib()
    err = lambda: lib.dpt_last_error().decode()   # noqa: E731
    limit = dpt.models.net.ONLINE_POPULATION_MAX
    header = open(os.path.join(ROOT, "include", "dpt_b200.h")).read()
    assert int(re.search(r"#define DPT_GPT2_ONLINE_POPULATION_MAX (\d+)", header).group(1)) == limit
    nulls = (ctypes.c_void_p * (limit + 1))()
    for n in (-1, limit + 1):
        assert _call(lib, nulls, n) == E_ARG and ("n_models=%d" % n) in err()
    assert _call(lib, None, 2) == E_ARG and "null models array" in err()
    assert _call(lib, nulls, 3) == E_ARG and "member 0 is a null model" in err()
    # no member: nothing to check, nothing to launch
    assert _call(lib, None, 0) == 0
    assert _call(lib, nulls, 0, N=0, H=0) == 0
    with pytest.raises(ValueError, match="dpt_gpt2_online_loop_population"):
        dpt._lib.check(_call(lib, nulls, -1), "dpt_gpt2_online_loop_population")


def _model(**over):
    from dpt_b200.models.net import Transformer
    cfg = {"horizon": 20, "state_dim": 1, "action_dim": 5, "n_layer": 2, "n_embd": 32, "n_head": 1, "dropout": 0.0, "test": True}
    cfg.update(over)
    return Transformer(cfg)


@pytest.mark.parametrize("field,over", [("action_dim", {"action_dim": 4}), ("n_layer", {"n_layer": 3}),
                                        ("horizon", {"horizon": 30}), ("state_dim", {"state_dim": 2})])
def test_online_loop_population_rejects_mismatched_members(dpt, field, over):
    from dpt_b200.models.net import online_loop_population
    models = [_model(), _model(), _model(**over)]
    with pytest.raises(ValueError, match="member 2 has %s" % field):
        online_loop_population(models, [[0.1] * 5] * 4, 10, 0.3, True, 1)
    assert all(m._handle is None for m in models)   # raised before any handle was built


def test_online_loop_population_rejects_mixed_precision_and_devices(dpt):
    from dpt_b200.models.net import online_loop_population
    odd = _model()
    odd.precision = 1
    with pytest.raises(ValueError, match="member 1 has precision=1, member 0 has 0"):
        online_loop_population([_model(), odd], [[0.1] * 5] * 4, 10, 0.3, True, 1)
    with pytest.raises(ValueError, match="member 1 is on meta"):
        online_loop_population([_model(), _model().to("meta")], [[0.1] * 5] * 4, 10, 0.3, True, 1)
    assert online_loop_population([], [[0.1] * 5] * 4, 10, 0.3, True, 1) == []


def test_online_launch_groups_cut_by_capacity_and_kv_bound(dpt):
    from dpt_b200.models import net
    cap, bound = net.ONLINE_POPULATION_MAX, net.ONLINE_KV_LAUNCH_BYTES
    small = 100 * 4 * 2 * 32 * 512 * 4           # 100 envs x H = 500, fp32, 4 layers: 52 MB per member
    big = 10000 * 4 * 2 * 32 * 512 * 4           # 10 000 envs: 5.2 GB per member
    assert net.online_launch_groups(0, small) == []
    assert net.online_launch_groups(1, small) == [(0, 1)]
    assert net.online_launch_groups(cap, small) == [(0, cap)]
    assert net.online_launch_groups(2 * cap + 3, small) == [(0, cap), (cap, 2 * cap), (2 * cap, 2 * cap + 3)]
    assert net.online_launch_groups(3, big) == [(0, 1), (1, 2), (2, 3)]          # one member fills the bound
    assert net.online_launch_groups(2, 2 * bound) == [(0, 1), (1, 2)]            # a member above the bound still runs, alone
    third = bound // 3
    assert net.online_launch_groups(7, third) == [(0, 3), (3, 6), (6, 7)]
    assert net.online_launch_groups(7, third + 1) == [(0, 2), (2, 4), (4, 6), (6, 7)]
    for k, per in ((5, small), (40, small), (9, bound // 4 + 7), (3, 0)):
        groups = net.online_launch_groups(k, per)
        assert [g[0] for g in groups[1:]] == [g[1] for g in groups[:-1]] and groups[0][0] == 0 and groups[-1][1] == k
        assert all(1 <= b - a <= cap and ((b - a) * per <= bound or b - a == 1) for a, b in groups)
