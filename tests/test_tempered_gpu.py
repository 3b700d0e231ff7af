"""mg_evidence_tempered on the GPU: parity with the oracle (tests/_parity.py rule for the MH and swap tests), the same
draws as mg_mcmc_array without swaps, independence from how ladders are split over calls, the accuracy of the
stepping-stone estimate on config 3's 20-D model, argument errors, an NVRTC user plugin, and the one-rank communicator."""
import ctypes as C

import numpy as np
import pytest
from scipy.stats import norm

from mcmc_ocaml_b200 import InvalidArgument, _abi, evidence, mcmc, plugins as P
from mcmc_ocaml_b200.comm import Comm
from oracle import tempered as ot
from tests._parity import NEAR_TIE
from tests.test_misc_gpu import GAUSS_BODY
from tests.test_oracle_tempered import box_model, box_props, exact_mean_ll

pytestmark = pytest.mark.gpu


def _props(kind, betas, D, sigma):
    if kind == "box":
        return box_props(betas, D, sigma)
    if kind == "left_biased":          # 1-D, asymmetric
        return [P.left_biased_proposal(0.5 if b == 0 else min(0.5, 2.4 * sigma / np.sqrt(b))) for b in betas]
    # mixture of a box and an independent Gaussian (asymmetric log_q)
    return [P.combine_jump_proposals([(0.7, p), (0.3, P.indep_gauss_proposal(np.full(D, 0.5), np.full(D, 0.3)))])
            for p in box_props(betas, D, sigma)]


def _compare(got, want, what):
    """final states and counts identical, except ladders that left the oracle after a near-tie; per-ladder means to
    1e-13, pooled outputs to 1e-12"""
    M = want["final"].shape[0]
    bad = [m for m in range(M) if not np.array_equal(got.final[m], want["final"][m])]
    for m in bad:
        assert want["margins"][m].min() <= NEAR_TIE, f"{what}: ladder {m} diverges without a near-tie"
    print(f"[parity] {what}: {len(bad)} of {M} ladders diverge (all at near-ties)")
    ok = np.setdiff1d(np.arange(M), bad)
    np.testing.assert_allclose(got.ladder_mean_ll[ok], want["ladder_mean_ll"][ok], rtol=1e-13, atol=1e-13)
    if bad:
        return
    for key in ("accept", "swaps_accepted", "swaps_tried"):
        assert np.array_equal(getattr(got, key), want[key]), key
    for key in ("mean_ll", "mean_ll_err"):
        np.testing.assert_allclose(getattr(got, key), want[key], rtol=1e-12, atol=1e-12, err_msg=key)
    for key in ("log_z_ss", "log_z_ss_err", "log_z_ti", "log_z_ti_err"):
        np.testing.assert_allclose(getattr(got, key), want[key], rtol=1e-12, atol=1e-12, err_msg=key)


@pytest.mark.parametrize("T,D,every,kind", [(2, 1, 0, "left_biased"), (5, 3, 1, "mixture"), (8, 10, 7, "box"),
                                            (32, 20, 1, "box"), (5, 3, 7, "box"), (8, 1, 1, "left_biased")])
def test_parity_with_the_oracle(ctx, T, D, every, kind):
    M, sigma, nbin, nsteps = 64, 0.1, 30, 150
    like, prior = box_model(D, sigma)
    betas = (np.arange(T) / (T - 1.0)) ** 3
    props = _props(kind, betas, D, sigma)
    x0 = np.random.default_rng(T * 100 + D).uniform(0.3, 0.7, (M, D))
    ctx.set_seed(77)
    got = evidence.evidence_tempered(like, prior, props, betas, x0, nladders=M, nbin=nbin, nsteps=nsteps,
                                     swap_every=every, ctx=ctx)
    want = ot.evidence_tempered(77, 0, like, prior, props, betas, x0, nladders=M, nbin=nbin, nsteps=nsteps,
                                swap_every=every, nthreads=8)
    _compare(got, want, f"T={T} D={D} every={every} {kind}")
    if every:
        assert got.swaps_accepted.sum() > 0


def test_user_plugin_gives_the_builtin_run(ctx):
    """a likelihood registered as source (NVRTC) with the built-in's arithmetic gives the built-in's run bit for bit"""
    D, T, M = 3, 6, 40
    mu, sig = np.full(D, 0.5), np.full(D, 0.1)
    user = P.register_source("tempered_gaussian", GAUSS_BODY, D, np.concatenate([mu, sig]), ctx=ctx)
    _, prior = box_model(D, 0.1)
    betas = np.linspace(0.0, 1.0, T) ** 2
    props = box_props(betas, D, 0.1)
    runs = []
    for like in (user, P.gauss_diag(mu, sig)):
        ctx.set_seed(91)
        runs.append(evidence.evidence_tempered(like, prior, props, betas, np.full(D, 0.5), nladders=M, nbin=20,
                                               nsteps=200, swap_every=3, ctx=ctx))
    a, b = runs
    assert np.array_equal(a.final, b.final) and np.array_equal(a.ladder_mean_ll, b.ladder_mean_ll)
    assert a.log_z_ss == b.log_z_ss and a.log_z_ti == b.log_z_ti and np.array_equal(a.swaps_accepted, b.swaps_accepted)


def test_beta_one_rungs_are_the_plain_sampler(ctx):
    """swap_every = 0: the beta = 1 rung of ladder m is chain m T + T - 1 of mg_mcmc_array, same seed and epoch"""
    D, T, M, nbin, nsteps = 10, 4, 96, 25, 300
    like, prior = box_model(D, 0.1)
    betas = np.array([0.0, 0.2, 0.6, 1.0])
    prop = P.combine_jump_proposals([(0.8, P.box_proposal(np.full(D, 0.05))),
                                     (0.2, P.indep_gauss_proposal(np.full(D, 0.5), np.full(D, 0.2)))])
    x0 = np.random.default_rng(5).uniform(0.4, 0.6, (M, D))
    ctx.set_seed(123)
    r = evidence.evidence_tempered(like, prior, prop, betas, x0, nladders=M, nbin=nbin, nsteps=nsteps, swap_every=0,
                                   ctx=ctx)
    ctx.set_seed(123)
    s = mcmc.mcmc_array(1, like, prior, prop, np.repeat(x0, T, axis=0), nbin=nbin + nsteps, ctx=ctx)
    plain = s.block[0].T.reshape(M, T, D + 2)
    assert np.array_equal(r.final[:, T - 1], plain[:, T - 1])


def test_ladders_do_not_depend_on_the_split(ctx):
    """two calls over the halves (ladder_offset 0 and M/2) give the per-ladder outputs of one call over all M"""
    D, T, M = 4, 7, 50
    like, prior = box_model(D, 0.1)
    betas = np.linspace(0.0, 1.0, T) ** 3
    props = box_props(betas, D, 0.1)
    x0 = np.random.default_rng(8).uniform(0.3, 0.7, (M, D))
    kw = dict(nbin=10, nsteps=120, swap_every=2, ctx=ctx)
    ctx.set_seed(31)
    full = evidence.evidence_tempered(like, prior, props, betas, x0, nladders=M, **kw)
    h = M // 2
    parts = []
    for off, n in ((0, h), (h, M - h)):
        ctx.set_seed(31)
        parts.append(evidence.evidence_tempered(like, prior, props, betas, x0[off:off + n], nladders=n,
                                                ladder_offset=off, **kw))
    assert np.array_equal(np.concatenate([p.final for p in parts]), full.final)
    assert np.array_equal(np.concatenate([p.ladder_mean_ll for p in parts]), full.ladder_mean_ll)
    assert np.array_equal(parts[0].swaps_accepted + parts[1].swaps_accepted, full.swaps_accepted)
    assert np.array_equal(parts[0].accept + parts[1].accept, full.accept)


def test_stepping_stones_on_config3_model(ctx):
    """Config 3's model (20-D, sigma = 0.05, unit box, analytic log Z = 0 to 1e-20), where the kd-tree estimators fail:
    log_z_ss within 4 errors of the truth, and the TI integrand mean_ll[k] within 4 errors of E_beta[ll]"""
    D, sigma, T, M = 20, 0.05, 32, 512
    like, prior = box_model(D, sigma)
    betas = (np.arange(T) / (T - 1.0)) ** 3
    x0 = np.random.default_rng(1).uniform(0.0, 1.0, (M, D))
    ctx.set_seed(2024)
    r = evidence.evidence_tempered(like, prior, box_props(betas, D, sigma), betas, x0, nladders=M, nbin=2000,
                                   nsteps=10000, swap_every=1, ctx=ctx)
    log_z = D * np.log(2.0 * norm.cdf(0.5 / sigma) - 1.0)
    print(f"config 3 model: log_z_ss = {r.log_z_ss:.5f} +- {r.log_z_ss_err:.5f}, log_z_ti = {r.log_z_ti:.5f} "
          f"+- {r.log_z_ti_err:.5f}, exact {log_z:.3g}; swap acceptance {np.round(r.swaps_accepted / r.swaps_tried, 2)}")
    assert abs(r.log_z_ss - log_z) < 4.0 * r.log_z_ss_err
    want = np.array([exact_mean_ll(b, D, sigma) for b in betas])
    z = (r.mean_ll - want) / r.mean_ll_err
    print("mean_ll z-scores", np.round(z, 2))
    assert np.all(np.abs(z) < 4.0)


def _raw_call(ctx, like, prior, props, betas, cfg, x0, out):
    pa = (_abi.mg_proposal * len(props))(*[p.spec() for p in props]) if props is not None else None
    ls, ps = like.spec(), prior.spec()
    b = _abi.as_f64(betas) if betas is not None else None
    x = _abi.as_f64(x0) if x0 is not None else None
    return ctx.lib.mg_evidence_tempered(ctx.h, C.byref(ls), C.byref(ps), pa, _abi.ptr(b), C.byref(cfg), _abi.ptr(x),
                                        C.byref(out) if out is not None else None)


def test_argument_errors(ctx):
    D, T = 2, 4
    like, prior = box_model(D, 0.1)
    betas = np.linspace(0.0, 1.0, T)
    props = box_props(betas, D, 0.1)
    x0 = np.full(D, 0.5)
    good = dict(nladders=8, nbin=5, nsteps=20, swap_every=1)
    E = lambda **kw: pytest.raises(InvalidArgument)  # noqa: E731
    for kw in (dict(nladders=0), dict(nsteps=0), dict(nbin=-1), dict(swap_every=-1), dict(ladder_offset=1 << 43),
               dict(nbin=(1 << 31) - 20)):
        with E():
            evidence.evidence_tempered(like, prior, props, betas, x0, ctx=ctx, **{**good, **kw})
    for bad in ([1.0], np.linspace(0.0, 1.0, 33), [0.0, 0.5, 0.5, 1.0], [0.0, 0.6, 0.5, 1.0], [-0.1, 0.2, 0.5, 1.0],
                [0.0, 0.2, 0.5, 0.9], [0.0, np.nan, 0.5, 1.0], [0.0, 0.2, np.inf, 1.0]):
        with E():
            evidence.evidence_tempered(like, prior, props[0], bad, x0, ctx=ctx, **good)
    with E():                                           # a proposal of another dimension
        evidence.evidence_tempered(like, prior, props[:3] + [P.box_proposal([0.1])], betas, x0, ctx=ctx, **good)
    with E():                                           # a prior of another dimension
        evidence.evidence_tempered(like, P.box(np.zeros(3), np.ones(3)), props, betas, x0, ctx=ctx, **good)
    big = P.gauss_diag(np.full(65, 0.5), np.full(65, 0.1))
    with E():                                           # D above 64
        evidence.evidence_tempered(big, P.box(np.zeros(65), np.ones(65)), P.box_proposal(np.full(65, 0.1)), betas,
                                   np.full(65, 0.5), ctx=ctx, **good)
    cfg = _abi.mg_tempered_cfg(8, T, D, 5, 20, 1, 0, 1, 0)
    out = _abi.mg_tempered_out()
    for args in ((None, betas, x0, out), (props, None, x0, out), (props, betas, None, out), (props, betas, x0, None)):
        assert _raw_call(ctx, like, prior, args[0], args[1], cfg, args[2], args[3]) == _abi.MG_EINVAL
        assert "evidence_tempered" in ctx.lib.mg_last_error(ctx.h).decode()
    assert _raw_call(ctx, like, prior, props, betas, cfg, x0, out) == _abi.MG_OK   # the context still works
    assert np.isfinite(out.log_z_ss)


def test_counters_and_epoch(ctx):
    """one call key, the context's accept / reject counters unchanged"""
    D, T = 2, 3
    like, prior = box_model(D, 0.1)
    betas = np.linspace(0.0, 1.0, T)
    ctx.set_seed(4)
    ctx.lib.mg_reset_counters(ctx.h)
    e0 = ctx.epoch
    evidence.evidence_tempered(like, prior, box_props(betas, D, 0.1), betas, np.full(D, 0.5), nladders=5, nbin=3,
                               nsteps=10, ctx=ctx)
    assert ctx.epoch == e0 + 1
    a, r = C.c_int64(), C.c_int64()
    ctx.lib.mg_get_counters(ctx.h, C.byref(a), C.byref(r))
    assert a.value == 0 and r.value == 0


def test_one_rank_communicator_is_the_single_gpu_call(ctx):
    comm = Comm(ctx, 1, 0)
    try:
        D, T, M = 5, 9, 70
        like, prior = box_model(D, 0.1)
        betas = (np.arange(T) / (T - 1.0)) ** 2
        props = box_props(betas, D, 0.1)
        x0 = np.random.default_rng(9).uniform(0.3, 0.7, (M, D))
        kw = dict(nladders=M, nbin=10, nsteps=100, swap_every=1)
        ctx.set_seed(55)
        a = evidence.evidence_tempered(like, prior, props, betas, x0, ctx=ctx, **kw)
        ctx.set_seed(55)
        b = comm.evidence_tempered(like, prior, props, betas, x0, **kw)
        for key in ("mean_ll", "mean_ll_err", "accept", "swaps_accepted", "swaps_tried", "final", "ladder_mean_ll",
                    "log_z_ss", "log_z_ss_err", "log_z_ti", "log_z_ti_err"):
            assert np.array_equal(getattr(a, key), getattr(b, key)), key
        with pytest.raises(InvalidArgument, match="evidence_tempered"):
            comm.evidence_tempered(like, prior, props, betas, x0, **{**kw, "nsteps": 0})
        c = comm.evidence_tempered(like, prior, props, betas, x0, **kw)       # the communicator still works
        assert np.isfinite(c.log_z_ss)
    finally:
        comm.close()
