"""CPU tier of the interactive trainer: the micro-batch partition over ranks (dist.microbatch_shard) and the argument
checks of dpt_ordered_sum_f32, the sum that joins the micro-batches' gradients (no GPU needed for either)."""
import ctypes

import pytest


@pytest.mark.parametrize("n,mb", [(0, 4), (1, 4), (3, 1), (10, 4), (4096, 1024), (4097, 1024), (100000, 1024), (6000, 1024),
                                  (5, 64)])
def test_microbatch_partition(dpt, n, mb):
    from dpt_b200.dist import microbatch_shard
    M = -(-n // mb)
    for ws in (1, 2, 3, 8):
        parts = [microbatch_shard(n, mb, r, ws) for r in range(ws)]
        # the ranks' micro-batch ranges tile [0, M) in rank order, balanced to within one micro-batch
        assert parts[0][0] == 0 and parts[-1][1] == M
        assert all(parts[r][1] == parts[r + 1][0] for r in range(ws - 1))
        counts = [b - a for a, b, _, _ in parts]
        assert max(counts) - min(counts) <= 1
        for m_lo, m_hi, lo, hi in parts:
            # a rank's env range is exactly the union of its micro-batches [m*mb, min(n, (m+1)*mb)): the same
            # micro-batches whatever the world size
            assert (lo, hi) == (min(n, m_lo * mb), min(n, m_hi * mb))
            if m_lo == m_hi:
                assert lo == hi
        assert parts[0][2] == 0 and parts[-1][3] == n
        if M < ws:      # fewer micro-batches than ranks: the last ranks own none
            assert [b - a for a, b, _, _ in parts] == [1] * M + [0] * (ws - M)
    if mb > n > 0:      # one micro-batch: rank 0 takes every env
        assert microbatch_shard(n, mb, 0, 8) == (0, 1, 0, n)


def test_microbatch_size_must_be_positive(dpt):
    from dpt_b200.dist import microbatch_shard
    with pytest.raises(ValueError, match="micro-batch"):
        microbatch_shard(10, 0, 0, 1)


def test_ordered_sum_rejects_bad_arguments(dpt):
    lib, E = dpt._lib.lib(), dpt._lib.ERR_INVALID_ARG
    assert lib.dpt_ordered_sum_f32(None, -1, 10, None, None) == E and b"M=-1" in lib.dpt_last_error()
    assert lib.dpt_ordered_sum_f32(None, 2, -3, None, None) == E and b"n=-3" in lib.dpt_last_error()
    assert lib.dpt_ordered_sum_f32(None, 2, 10, None, None) == E and b"null src" in lib.dpt_last_error()
    src = (ctypes.c_void_p * 2)(256, None)
    assert lib.dpt_ordered_sum_f32(src, 2, 10, None, None) == E and b"null dst" in lib.dpt_last_error()
    assert lib.dpt_ordered_sum_f32(src, 2, 10, 512, None) == E and b"src[1] is null" in lib.dpt_last_error()
    src = (ctypes.c_void_p * 2)(256, 512)
    assert lib.dpt_ordered_sum_f32(src, 2, 10, 512, None) == E and b"aliases dst" in lib.dpt_last_error()
    with pytest.raises(ValueError, match="dpt_ordered_sum_f32"):
        dpt._lib.check(lib.dpt_ordered_sum_f32(src, -2, 10, 1024, None), "dpt_ordered_sum_f32")
    # nothing to sum: no launch, no device needed
    assert lib.dpt_ordered_sum_f32(None, 0, 10, None, None) == 0
    assert lib.dpt_ordered_sum_f32(src, 2, 0, 1024, None) == 0
