"""The numpy transcription of the ensemble diagnostics (oracle/diagnostics_np.py) against hand-computed values and
known answers: AR(1) integrated autocorrelation times, split-Rhat of offset chain groups, Geyer's monotone step and the
NaN / inf rules.  CPU only."""
import math

import numpy as np
import pytest

from oracle import diagnostics_np as dg


def test_hand_computed_two_chains_six_steps():
    # chain 0: 1..6, chain 1: 2 0 1 3 1 2; split: N = 3, M = 4, L = 2
    x = np.array([[1, 2], [2, 0], [3, 1], [4, 3], [5, 1], [6, 2]], dtype=np.float64)[:, None, :]
    r = dg.chain_diagnostics(x, 2, split=True, per_sequence=True)
    # sequences [1 2 3], [2 0 1], [4 5 6], [3 1 2]: means 2, 1, 5, 2
    # deviations (-1 0 1), (1 -1 0), (-1 0 1), (1 -1 0): gamma(0) = 2/3 each, gamma(1) = 0, -1/3, 0, -1/3
    # s2 = 3/2 * 2/3 = 1 each -> W = 1; grand mean 2.5, sum of squared offsets 9 -> B = 3/3 * 9 = 9
    assert r.W[0] == pytest.approx(1.0, rel=1e-15)
    assert r.B[0] == pytest.approx(9.0, rel=1e-15)
    # var+ = 2/3 * 1 + 9/3 = 11/3, Rhat = sqrt(11/3)
    assert r.var_plus[0] == pytest.approx(11 / 3, rel=1e-15)
    assert r.rhat[0] == pytest.approx(math.sqrt(11 / 3), rel=1e-15)
    # mean gamma(1) = -1/6 -> rho_1 = 1 - (1 + 1/6) / (11/3) = 15/22
    np.testing.assert_allclose(r.rho[0], [1.0, 15 / 22], rtol=1e-15)
    # one pair P_0 = 37/22 > 0: the window does not close, tau = -1 + 2 * 37/22 = 26/11, ESS = 12 / tau
    assert r.window_closed[0] == 0
    assert r.tau[0] == pytest.approx(26 / 11, rel=1e-15)
    assert r.ess[0] == pytest.approx(12 * 11 / 26, rel=1e-15)
    # per sequence: rho_m(1) = 0, -1/2, 0, -1/2 -> tau_m = 1, 0, 1, 0
    np.testing.assert_allclose(r.seq_tau[0], [1.0, 0.0, 1.0, 0.0], atol=1e-15)


def test_split_drops_the_middle_row_of_an_odd_block():
    x = np.arange(7.0)[:, None, None] * np.ones((1, 1, 3))
    seq, N = dg.sequences(x, True)
    assert N == 3 and seq.shape == (1, 6, 3)
    np.testing.assert_array_equal(seq[0, 0], [0, 1, 2])
    np.testing.assert_array_equal(seq[0, 3], [4, 5, 6])


def test_geyer_monotone_step_and_window():
    rho = [1.0, 0.5, 0.1, 0.0, 0.3, 0.2, -0.4, 0.1]
    # pairs 1.5, 0.1, 0.5, -0.3: K = 3, closed; monotone 1.5, 0.1, 0.1 -> tau = -1 + 2 * 1.7
    tau, closed, P = dg.geyer(rho)
    np.testing.assert_allclose(P, [1.5, 0.1, 0.5, -0.3])
    assert closed == 1 and tau == pytest.approx(2.4, rel=1e-15)
    # no non-positive pair: the whole window counts and window_closed = 0
    tau, closed, _ = dg.geyer([1.0, 0.9, 0.8, 0.7])
    assert closed == 0 and tau == pytest.approx(-1 + 2 * (1.9 + 1.5))
    # a non-positive first pair: tau = -1 (antithetic limit), no cap
    tau, closed, _ = dg.geyer([1.0, -1.0, 0.5, 0.5])
    assert closed == 1 and tau == -1.0
    # an odd window ignores its last lag
    assert dg.geyer([1.0, 0.2, 0.1])[0] == dg.geyer([1.0, 0.2])[0]


def test_exact_and_fast_sums_agree():
    x = dg.ar1_block(301, 3, 5, [0.3, 0.8, -0.2], seed=3) + 1e3
    a = dg.chain_diagnostics(x, 40, per_sequence=True, exact=True)
    b = dg.chain_diagnostics(x, 40, per_sequence=True, exact=False)
    for k in ("rhat", "ess", "tau", "rho", "seq_tau"):
        np.testing.assert_allclose(getattr(a, k), getattr(b, k), rtol=1e-9, atol=1e-12, err_msg=k)
    np.testing.assert_array_equal(a.window_closed, b.window_closed)


def test_ar1_integrated_autocorrelation_time():
    phis = np.array([0.0, 0.5, 0.9, -0.5])
    x = dg.ar1_block(5000, 4, 1000, phis, seed=11)           # M N = 2000 * 2500 = 5e6 per field, split
    r = dg.chain_diagnostics(x, 64, exact=False)
    want = (1 + phis) / (1 - phis)
    np.testing.assert_allclose(r.tau, want, rtol=0.04)
    np.testing.assert_allclose(r.ess, 2000 * 2500 / want, rtol=0.04)
    np.testing.assert_allclose(r.rhat, 1.0, atol=1e-2)       # finite-N excess ~ tau / (2N)
    np.testing.assert_array_equal(r.window_closed[[0, 1, 3]], [1, 1, 1])   # phi = 0.9: rho_64 ~ 1e-3, still open
    np.testing.assert_allclose(r.rho[1, :5], 0.5 ** np.arange(5), atol=3e-3)


def test_rhat_of_two_offset_groups():
    # half the chains shifted by delta = sigma: Rhat -> sqrt(1 + delta^2 / (4 sigma^2)) = 1.118
    C, n = 2000, 5000
    off = np.zeros((1, C))
    off[0, C // 2:] = 1.0
    x = dg.ar1_block(n, 1, C, 0.0, seed=5, offset=off)
    r = dg.chain_diagnostics(x, 8, split=False, exact=False)
    assert r.rhat[0] == pytest.approx(math.sqrt(1.25), rel=2e-3)


def test_single_sequence_has_no_rhat():
    x = dg.ar1_block(400, 1, 1, 0.5, seed=2)
    r = dg.chain_diagnostics(x, 20, split=False)
    assert np.isnan(r.rhat[0]) and r.B[0] == 0.0
    assert r.var_plus[0] == pytest.approx(399 / 400 * r.W[0])
    assert np.isfinite(r.tau[0]) and np.isfinite(r.ess[0])


def test_constant_field_is_nan_and_other_fields_are_not():
    x = dg.ar1_block(200, 3, 4, 0.5, seed=1)
    x[:, 1, :] = -7.25                                        # e.g. log_prior under a flat prior
    r = dg.chain_diagnostics(x, 10, per_sequence=True)
    for k in ("rhat", "ess", "tau"):
        v = getattr(r, k)
        assert np.isnan(v[1]) and np.isfinite(v[[0, 2]]).all(), k
    assert np.isnan(r.rho[1]).all() and np.isfinite(r.rho[[0, 2]]).all()
    assert np.isnan(r.seq_tau[1]).all() and np.isfinite(r.seq_tau[[0, 2]]).all()


def test_stuck_chains_give_infinite_rhat():
    x = np.broadcast_to(np.arange(5.0)[None, None, :], (50, 1, 5)).copy()   # every chain stuck at its own value
    r = dg.chain_diagnostics(x, 4, per_sequence=True)
    assert r.rhat[0] == np.inf
    assert np.isnan(r.seq_tau[0]).all()


@pytest.mark.parametrize("bad", [np.nan, np.inf, -np.inf])
def test_non_finite_value_poisons_its_field_only(bad):
    x = dg.ar1_block(120, 3, 6, 0.3, seed=4)
    x[17, 2, 4] = bad
    r = dg.chain_diagnostics(x, 8, per_sequence=True)
    for k in ("rhat", "ess", "tau"):
        v = getattr(r, k)
        assert np.isnan(v[2]) and np.isfinite(v[:2]).all(), k
    assert np.isnan(r.rho[2]).all()
    assert np.isnan(r.seq_tau[2, 4]) and np.isfinite(r.seq_tau[:2]).all()


@pytest.mark.parametrize("n,L,split", [(3, 2, True), (10, 1, True), (10, 5, True), (10, 10, False)])
def test_invalid_configurations(n, L, split):
    with pytest.raises(ValueError):
        dg.chain_diagnostics(np.zeros((n, 1, 2)), L, split=split)
