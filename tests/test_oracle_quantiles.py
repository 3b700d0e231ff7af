"""The quantile oracle (oracle/quantiles_np.py) on cases small enough to work by hand, and against
np.quantile(method="linear") on finite data."""
import math

import numpy as np
import pytest

from oracle import quantiles_np as qn


def _q(values, probs):
    return qn.quantiles(np.asarray(values, dtype=np.float64).reshape(-1, 1, 1), probs)[0]


def test_interpolation_by_hand():
    x = [3.0, 1.0, 4.0, 2.0]                     # sorted 1 2 3 4, N - 1 = 3
    got = _q(x, [0.0, 0.25, 0.5, 1 / 3, 0.9, 1.0])
    np.testing.assert_array_equal(got, [1.0, 1.75, 2.5, 2.0, 3.7, 4.0])
    assert got[4] == 3.0 + (3.0 * 0.9 - 2.0) * (4.0 - 3.0)


def test_order_statistics_by_hand():
    blk = np.array([[[5.0, -1.0]], [[2.0, 7.0]]])   # n = 2, F = 1, C = 2: pool 5 -1 2 7
    np.testing.assert_array_equal(qn.order_statistics(blk, [0, 1, 2, 3]), [[-1.0, 2.0, 5.0, 7.0]])


def test_infinities_next_to_finite_values():
    x = [-np.inf, 0.0, 1.0, np.inf]
    got = _q(x, [0.0, 0.1, 1 / 3, 0.5, 0.9, 1.0])
    assert got[0] == -np.inf and got[1] == -np.inf      # a = -inf, b = 0
    assert got[2] == 0.0                                # g = 0
    assert got[3] == 0.5
    assert got[4] == np.inf and got[5] == np.inf        # b = +inf


def test_minus_inf_next_to_plus_inf():
    got = _q([np.inf, -np.inf], [0.0, 0.5, 1.0])
    assert got[0] == -np.inf and math.isnan(got[1]) and got[2] == np.inf
    assert _q([np.inf, np.inf], [0.5])[0] == np.inf     # a = b
    assert _q([-np.inf, -np.inf], [0.5])[0] == -np.inf


def test_negative_zero_is_zero_and_returned_positive():
    got = _q([-0.0, 0.0, -0.0], [0.0, 0.5, 1.0])
    np.testing.assert_array_equal(got, [0.0, 0.0, 0.0])
    assert not np.signbit(got).any()
    k = qn.ordered_keys([-0.0, 0.0])
    assert k[0] == k[1]
    o = qn.order_statistics(np.array([[[-0.0]], [[-1.0]]]), [1])
    assert o[0, 0] == 0.0 and not np.signbit(o[0, 0])


def test_nan_poisons_its_field_only():
    blk = np.arange(12.0).reshape(3, 2, 2)
    blk[1, 0, 1] = np.nan
    got = qn.quantiles(blk, [0.0, 0.5, 1.0])
    assert np.isnan(got[0]).all()
    np.testing.assert_array_equal(got[1], [2.0, 6.5, 11.0])   # pool 2 3 6 7 10 11


def test_single_value():
    np.testing.assert_array_equal(_q([2.5], [0.0, 0.3, 1.0]), [2.5, 2.5, 2.5])
    np.testing.assert_array_equal(qn.order_statistics(np.full((1, 1, 1), -7.0), [0]), [[-7.0]])


def test_ordered_keys_round_trip_and_order():
    x = np.array([-np.inf, -1e308, -1.0, -5e-324, 0.0, 5e-324, 1.0, 1e308, np.inf])
    k = qn.ordered_keys(x)
    assert (np.diff(k.astype(object)) > 0).all()
    np.testing.assert_array_equal(qn.from_keys(k), x)


@pytest.mark.parametrize("seed", range(6))
def test_agrees_with_numpy_linear_within_one_ulp(seed):
    """numpy evaluates b - (b - a)(1 - g) when g >= 0.5; the two roundings differ by at most one ulp of the largest
    of |a|, |b| and |b - a| (the last exceeds the first two only when a and b have opposite signs)"""
    rng = np.random.default_rng(seed)
    for _ in range(100):
        N = int(rng.integers(1, 60))
        scale = 10.0 ** rng.integers(-5, 6)
        x = rng.standard_normal(N) * scale + rng.choice([0.0, 1e8])
        p = rng.random(10)
        got = _q(x, p)
        want = np.quantile(x, p, method="linear")
        s = np.sort(x)
        for pi, g, w in zip(p, got, want):
            lo = int(np.floor((N - 1) * pi))
            a, b = s[lo], s[min(lo + 1, N - 1)]
            mag = max(abs(a), abs(b), abs(b - a))
            assert abs(g - w) <= np.spacing(mag), (N, pi, g, w)
