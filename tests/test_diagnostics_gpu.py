"""Ensemble convergence diagnostics on the GPU (mg_stats_chain_diagnostics*, csrc/diagnostics.cu) against the numpy
transcription oracle/diagnostics_np.py: parity over shapes, a device-generated config-2 block, known answers, the
NaN / inf rules, a block of more than 2^31 elements and the one-rank communicator."""
import numpy as np
import pytest

from oracle import diagnostics_np as dg

pytestmark = pytest.mark.gpu

NEAR_CUT = 1e-9      # a pair sum this close to 0 may close the window on one side and not the other


def _rho_tol(x, split, var_plus):
    """the one-pass sums are about each sequence's first value: their rounding scales with (1/N) sum (x - pivot)^2"""
    seqs, N = dg.sequences(x, split)
    m2 = ((seqs - seqs[:, :, :1]) ** 2).mean(axis=(1, 2))
    return 1e-12 * np.maximum(m2 / np.where(var_plus > 0, var_plus, 1.0), 1.0)


def _assert_parity(got, want, x, split, what=""):
    F = x.shape[1]
    np.testing.assert_array_equal(got.window_closed, want.window_closed, err_msg=what)
    for k in ("rhat", "ess", "tau"):
        np.testing.assert_allclose(getattr(got, k), getattr(want, k), rtol=1e-10, atol=0, err_msg=f"{what} {k}")
    tol = _rho_tol(x, split, want.var_plus)
    for f in range(F):
        np.testing.assert_allclose(got.rho[f], want.rho[f], rtol=0, atol=tol[f], err_msg=f"{what} rho field {f}")
    if want.seq_tau is not None:
        P = want.seq_pairs
        ties = 0
        for f in range(F):
            for m in range(want.seq_tau.shape[1]):
                a, b = got.seq_tau[f, m], want.seq_tau[f, m]
                if np.isnan(b):
                    assert np.isnan(a), (what, f, m)
                    continue
                if np.isclose(a, b, rtol=1e-10, atol=1e-12):
                    continue
                pk = P[f, m]
                cut = np.nonzero(pk <= 0)[0]
                K = int(cut[0]) if cut.size else len(pk) - 1
                assert np.any(np.abs(pk[:K + 1]) < NEAR_CUT), (f"{what}: seq_tau[{f}][{m}] {a!r} != {b!r} "
                                                                f"and no pair sum is a near-tie")
                ties += 1
        if ties:
            print(f"[parity] {what}: {ties} sequences differ in tau at a near-zero pair sum")


def _block(n, F, C, seed, drift=0.0, phi=0.6):
    x = dg.ar1_block(n, F, C, phi, seed=seed) + 100.0 + np.linspace(-0.1, 0.1, C)[None, None, :]
    if drift:
        x += drift * np.arange(n)[:, None, None] * (1 + np.arange(C) % 3)[None, None, :]
    return x


SHAPES = [  # n, D, C, L, split, drift
    (200, 1, 1, 12, True, 0.0),
    (201, 1, 33, 16, True, 0.0),
    (97, 2, 1000, 8, True, 0.0),
    (301, 3, 64, 2, True, 0.0),
    (41, 1, 40, 19, True, 0.0),          # L = N - 1 (N = 20)
    (60, 1, 7, 59, False, 0.0),          # L = N - 1 without split
    (150, 20, 40, 24, True, 0.0),
    (400, 4, 96, 100, True, 0.0),
    (600, 2, 50, 256, True, 0.0),        # two register blocks per warp, the largest window
    (300, 2, 70, 40, True, 0.05),        # strong drift
    (300, 2, 70, 40, False, 0.05),
]


@pytest.mark.parametrize("n,D,C,L,split,drift", SHAPES)
def test_parity_with_the_oracle(ctx, n, D, C, L, split, drift):
    from mcmc_ocaml_b200 import stats
    x = _block(n, D + 2, C, seed=n + 7 * C + L, drift=drift)
    got = stats.chain_diagnostics(x, L, split=split, per_sequence=True, ctx=ctx)
    want = dg.chain_diagnostics(x, L, split=split, per_sequence=True, exact=C * (D + 2) * L <= 200_000)
    _assert_parity(got, want, x, split, what=f"n={n} D={D} C={C} L={L} split={split}")


def test_chain_major_samples_are_transposed(ctx):
    from mcmc_ocaml_b200 import stats
    from mcmc_ocaml_b200.mcmc import McmcSamples
    x = _block(120, 3, 10, seed=1)
    a = stats.chain_diagnostics(x, 10, ctx=ctx)
    s = McmcSamples(np.ascontiguousarray(np.transpose(x, (2, 0, 1))), 1, "chain", None, None)
    b = stats.chain_diagnostics(s, 10, ctx=ctx)
    np.testing.assert_array_equal(a.rho, b.rho)
    np.testing.assert_array_equal(a.tau, b.tau)


def test_config2_block_from_the_device_sampler(ctx):
    """C = 4096, n = 2000 of the headline model (flat prior: log_prior is constant -> NaN field)"""
    import torch

    from mcmc_ocaml_b200 import mcmc, stats, plugins as P
    D, C, n, L = 10, 4096, 2000, 48
    mu = np.arange(D) / 10.0
    cov = 0.7 ** np.abs(np.subtract.outer(np.arange(D), np.arange(D)))
    like, prior, prop = P.gauss_corr(mu, cov), P.zero(D), P.box_proposal(np.full(D, 0.5))
    dev = torch.device("cuda", 0)
    state = torch.zeros((D + 2, C), dtype=torch.float64, device=dev)
    state[:D] = torch.tensor(mu, device=dev)[:, None] + torch.randn((D, C), dtype=torch.float64, device=dev,
                                                                   generator=torch.Generator(dev).manual_seed(3))
    blk = torch.empty((n, D + 2, C), dtype=torch.float64, device=dev)
    torch.cuda.synchronize()
    mcmc.mcmc_array_dev(like, prior, prop, nchains=C, n=n, nbin=50, nskip=1, state_ptr=state.data_ptr(),
                        samples_ptr=blk.data_ptr(), ctx=ctx)
    ctx.sync()
    before = blk.clone()
    seq = torch.full((D + 2, 2 * C), -1.0, dtype=torch.float64, device=dev)
    torch.cuda.synchronize()                                      # the library works on its own stream
    got = stats.chain_diagnostics_dev(blk.data_ptr(), n, D, C, L, seq_tau_ptr=seq.data_ptr(), ctx=ctx)
    ctx.sync()
    assert torch.equal(blk.view(torch.int64), before.view(torch.int64)), "the block was modified"
    x = blk.cpu().numpy()
    host = stats.chain_diagnostics(x, L, per_sequence=True, ctx=ctx)
    for k in ("rhat", "ess", "tau", "window_closed", "rho"):
        np.testing.assert_array_equal(getattr(got, k), getattr(host, k), err_msg=k)
    np.testing.assert_array_equal(seq.cpu().numpy(), host.seq_tau)
    want = dg.chain_diagnostics(x, L, per_sequence=True, exact=False)
    _assert_parity(host, want, x, True, what="config 2")
    assert np.isnan(got.rhat[D + 1]) and np.isnan(got.tau[D + 1]) and np.isnan(got.rho[D + 1]).all()
    assert np.isfinite(got.rhat[:D + 1]).all() and np.isfinite(got.ess[:D + 1]).all()
    assert np.isnan(host.seq_tau[D + 1]).all()


def test_ar1_and_offset_known_answers(ctx):
    from mcmc_ocaml_b200 import stats
    phis = np.array([0.0, 0.5, 0.9, -0.5])
    x = dg.ar1_block(5000, 4, 1000, phis, seed=11)                # M N = 5e6 per field
    r = stats.chain_diagnostics(x, 64, ctx=ctx)
    want = (1 + phis) / (1 - phis)
    np.testing.assert_allclose(r.tau, want, rtol=0.04)
    np.testing.assert_allclose(r.ess, 2000 * 2500 / want, rtol=0.04)
    C, n = 2000, 5000                                             # M N = 1e7
    off = np.zeros((3, C))
    off[0, C // 2:] = 1.0                                         # delta = sigma: sqrt(1.25)
    off[1, C // 2:] = 2.0                                         # delta = 2 sigma: sqrt(2)
    y = dg.ar1_block(n, 3, C, 0.0, seed=5, offset=off)
    r = stats.chain_diagnostics(y, 8, split=False, ctx=ctx)
    np.testing.assert_allclose(r.rhat, [np.sqrt(1.25), np.sqrt(2.0), 1.0], rtol=3e-3)


def test_stuck_chains_and_non_finite_values(ctx):
    from mcmc_ocaml_b200 import stats
    x = _block(200, 3, 40, seed=9)
    x[:, 0, :] = np.arange(40.0)[None, :]                         # every chain stuck at its own value
    x[:, 1, :] = 2.5                                              # constant field
    x[77, 2, 5] = np.nan
    r = stats.chain_diagnostics(x, 10, per_sequence=True, ctx=ctx)
    assert r.rhat[0] == np.inf
    assert np.isnan(r.rhat[1]) and np.isnan(r.ess[1]) and np.isnan(r.rho[1]).all()
    assert np.isnan(r.rhat[2]) and np.isnan(r.tau[2]) and np.isnan(r.seq_tau[2, 5])
    assert np.isnan(r.seq_tau[0]).all() and np.isnan(r.seq_tau[1]).all()
    assert np.isfinite(r.seq_tau[2, :5]).all()


@pytest.mark.parametrize("n,L,split", [(100, 1, True), (100, 50, True), (100, 100, False), (3, 2, True),
                                        (2000, 257, True)])
def test_invalid_configurations_raise(ctx, n, L, split):
    from mcmc_ocaml_b200 import InvalidArgument, stats
    with pytest.raises(InvalidArgument):
        stats.chain_diagnostics(np.zeros((n, 3, 4)), L, split=split, ctx=ctx)


def test_block_of_more_than_2_31_elements(ctx):
    """C = 65536, F = 12, n = 3000: 2.36e9 elements (18.9 GB); tau of the last 64 chains against the oracle"""
    import torch

    from mcmc_ocaml_b200 import stats
    D, C, n, L = 10, 65536, 3000, 16
    dev = torch.device("cuda", 0)
    g = torch.Generator(dev).manual_seed(17)
    blk = torch.randn((n, D + 2, C), dtype=torch.float64, device=dev, generator=g)
    blk[1:] += 0.5 * blk[:-1].clone()                             # some autocorrelation
    assert blk.numel() > 2 ** 31
    seq = torch.empty((D + 2, 2 * C), dtype=torch.float64, device=dev)
    torch.cuda.synchronize()
    got = stats.chain_diagnostics_dev(blk.data_ptr(), n, D, C, L, seq_tau_ptr=seq.data_ptr(), ctx=ctx)
    ctx.sync()
    tail = blk[:, :, C - 64:].cpu().numpy()
    s = seq.cpu().numpy()
    got_tail = np.concatenate([s[:, C - 64:C], s[:, 2 * C - 64:]], axis=1)
    want = dg.chain_diagnostics(tail, L, per_sequence=True, exact=True)
    bad = ~np.isclose(got_tail, want.seq_tau, rtol=1e-10, atol=1e-12)
    for f, m in zip(*np.nonzero(bad)):
        pk = want.seq_pairs[f, m]
        assert np.any(np.abs(pk) < NEAR_CUT), (f, m, got_tail[f, m], want.seq_tau[f, m])
    assert np.isfinite(got.rhat).all() and (np.abs(got.rhat - 1) < 1e-2).all()
    del blk


def test_one_rank_communicator_is_the_single_gpu_call(ctx):
    import torch

    from mcmc_ocaml_b200 import stats
    from mcmc_ocaml_b200.comm import Comm
    x = _block(500, 4, 300, seed=21)
    d = torch.tensor(x, device="cuda:0")
    torch.cuda.synchronize()
    one = stats.chain_diagnostics_dev(d.data_ptr(), 500, 2, 300, 40, ctx=ctx)
    comm = Comm(ctx, 1, 0)
    try:
        cm = comm.chain_diagnostics(d.data_ptr(), 500, 2, 300, 40)
    finally:
        comm.close()
    for k in ("rhat", "ess", "tau", "window_closed", "rho"):
        np.testing.assert_array_equal(getattr(cm, k), getattr(one, k), err_msg=k)
