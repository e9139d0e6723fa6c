"""The shape lists of tests/sv_lag_edge_shapes.py reach the corners of each kernel's accepted (lag, n_obs) region."""
import pytest

import sv_lag_edge_shapes as sh

KERNELS = sorted(sh.RULES)


def _lag_range(kernel):
    return [lag for lag in range(sh.MIN_LAG, sh.MAX_LAG + 1) if sh.RULES[kernel](lag, 2 * lag + 1)]


@pytest.mark.parametrize("kernel", KERNELS)
def test_every_shape_is_accepted(kernel):
    for lag, nobs in sh.shapes(kernel):
        assert sh.RULES[kernel](lag, nobs), (lag, nobs)
        assert sh.entry_accepts(lag, nobs)


@pytest.mark.parametrize("kernel", KERNELS)
def test_shapes_reach_the_corners(kernel):
    """the smallest and the largest lag the kernel takes, each at its shortest accepted series; the shortest series
    overall; and, where the kernel takes such series, the last one whose tail drops terms (2 lag - 2) next to the first
    that drops none (2 lag - 1)"""
    got = set(sh.shapes(kernel))
    lags = _lag_range(kernel)
    lo, hi = lags[0], lags[-1]
    assert (lo, sh.min_nobs(kernel, lo)) in got
    assert (hi, sh.min_nobs(kernel, hi)) in got
    assert min(m - lag for lag, m in got) == min(sh.min_nobs(kernel, lag) - lag for lag in lags)
    short = [lag for lag in lags if sh.RULES[kernel](lag, 2 * lag - 2) and 2 * lag - 2 >= lag + 1]
    if short:
        assert any((lag, 2 * lag - 2) in got and (lag, 2 * lag - 1) in got for lag in sh.LAGS[kernel])
        assert (max(short), 2 * max(short) - 2) in got
        assert any(sh.drops_terms(lag, m) for lag, m in got)
    else:
        assert not any(sh.drops_terms(lag, m) for lag, m in got)
    for lag in sh.LAGS[kernel]:
        m0 = sh.min_nobs(kernel, lag)
        assert (lag, m0) in got and (lag, m0 + 1) in got


def test_region_rules():
    """the rules restate the C ones: the entry takes 2 <= lag <= 63, n_obs >= lag + 1; the chain and grid kernels stop
    at lag 10; the grid and streaming kernels need n_obs >= 2 lag"""
    assert sh.entry_accepts(2, 3) and sh.entry_accepts(63, 64)
    assert not sh.entry_accepts(1, 10) and not sh.entry_accepts(64, 200) and not sh.entry_accepts(10, 10)
    assert sh.RULES["chain"](10, 11) and not sh.RULES["chain"](11, 12)
    assert sh.RULES["grid"](10, 20) and not sh.RULES["grid"](10, 19) and not sh.RULES["grid"](11, 22)
    assert sh.RULES["streaming"](63, 126) and not sh.RULES["streaming"](63, 125)
    assert sh.min_nobs("general", 63) == 64 and sh.min_nobs("streaming", 63) == 126


def test_streaming_lags_cover_every_jump_table_size():
    """every Q from 0 to Q(63) = 5, each q >= 1 at lag - 2 = 2^q and at a neighbour 2^q +- 1"""
    lags = sh.LAGS["streaming"]
    qmax = sh.jump_levels(sh.MAX_LAG)
    assert qmax == 5
    assert {sh.jump_levels(lag) for lag in lags} == set(range(qmax + 1))
    assert sh.MAX_LAG in lags
    for q in range(1, qmax + 1):
        assert 2 ** q + 2 in lags, q
        assert (2 ** q + 1 in lags) or (2 ** q + 3 in lags), q
    assert [sh.jump_levels(lag) for lag in (3, 4, 5, 6, 9, 10, 18, 34, 63)] == [0, 1, 1, 2, 2, 3, 4, 5, 5]
