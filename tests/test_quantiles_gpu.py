"""Exact order statistics and quantiles on the GPU (mg_stats_quantiles*, mg_stats_order_statistics_dev,
mg_comm_quantiles; csrc/quantiles.cu) against the numpy transcription oracle/quantiles_np.py, bit for bit: shapes,
an unaligned block base, hard data, non-finite values, both resolution paths, a config-2 block from the device
sampler, a field of more than 2^31 values and the one-rank communicator."""
import numpy as np
import pytest

from oracle import quantiles_np as qn

pytestmark = pytest.mark.gpu

P5 = [0.025, 0.16, 0.5, 0.84, 0.975]


def _same_bits(got, want, what=""):
    got, want = np.asarray(got), np.asarray(want)
    assert got.shape == want.shape, what
    np.testing.assert_array_equal(got.view(np.uint64), want.view(np.uint64), err_msg=what)


def _dev(x):
    import torch
    d = torch.tensor(x, device="cuda:0")
    torch.cuda.synchronize()
    return d


SHAPES = [  # n, D, C, probs
    (1, 1, 1, [0.0, 0.5, 1.0]),                           # N = 1
    (2, 1, 1, [0.0, 0.3, 0.5, 1.0]),                      # N = 2
    (1, 1, 2, [0.5]),
    (37, 1, 33, P5),
    (300, 2, 1000, list(np.linspace(0.0, 1.0, 64))),      # nq = 64 with p = 0 and 1
    (500, 3, 64, [0.5]),                                  # nq = 1
    (64, 20, 7, P5 + [0.0, 1.0]),
]


@pytest.mark.parametrize("n,D,C,probs", SHAPES)
def test_parity_with_the_oracle(ctx, n, D, C, probs):
    from mcmc_ocaml_b200 import stats
    rng = np.random.default_rng(n * 31 + C)
    x = rng.standard_normal((n, D + 2, C))
    x[:, 1] = x[:, 1] * 1e-3 + 1e8                         # offset 1e8, sigma 1e-3
    x[:, 2] *= 10.0 ** rng.integers(-200, 200, size=(n, C))  # mixed magnitudes
    want = qn.quantiles(x, probs)
    _same_bits(stats.quantiles(x, probs, ctx=ctx), want, "host")
    d = _dev(x)
    _same_bits(stats.quantiles_dev(d.data_ptr(), n, D, C, probs, ctx=ctx), want, "device")
    N = n * C
    ranks = sorted({0, N - 1, N // 2, N // 3})
    _same_bits(stats.order_statistics_dev(d.data_ptr(), n, D, C, ranks, ctx=ctx), qn.order_statistics(x, ranks))


def _hard_block(n, C, seed):
    """[n][3][C]: offset 1e8 with sigma 1e-3, mixed magnitudes, normal"""
    rng = np.random.default_rng(seed)
    x = rng.standard_normal((n, 3, C))
    x[:, 0] = x[:, 0] * 1e-3 + 1e8
    x[:, 1] *= 10.0 ** rng.integers(-200, 200, size=(n, C))
    return x


SUBSAMPLED = [  # n, C, probs, every field resolved by its brackets (candidate select), no fallback
    (1101, 1001, P5, True),
    (1101, 1001, list(np.linspace(0.0, 1.0, 64)), False),  # nq = 64: the brackets may overflow the budget
    (1_100_001, 1, P5 + [0.0, 1.0], True),
    (33_401, 33, P5, True),
]


@pytest.mark.parametrize("n,C,probs,bracketed", SUBSAMPLED)
def test_parity_subsampled_from_row_one(ctx, capfd, monkeypatch, n, C, probs, bracketed):
    """N > 2^20, so the sample is a subsample and the brackets are wide: the candidate buffer and its radix select
    run, on hard data, from row 1 of the block (odd C and F = 3 make the base 8 but not 16-byte aligned)"""
    from mcmc_ocaml_b200 import stats
    D = 1
    x = _hard_block(n, C, seed=n + C)
    assert (n - 1) * C > 2 ** 20
    d = _dev(x)
    ptr = d.data_ptr() + 8 * (D + 2) * C
    assert ptr % 16 == 8
    monkeypatch.setenv("MCMC_GPU_DEBUG", "1")
    capfd.readouterr()
    got = stats.quantiles_dev(ptr, n - 1, D, C, probs, ctx=ctx)
    err = capfd.readouterr().err
    _same_bits(got, qn.quantiles(x[1:], probs))
    if bracketed:
        for f in range(D + 2):
            assert f"quantiles: field {f}: bracket, 1 full read" in err, err
    N = (n - 1) * C
    ranks = [0, 1, N // 3, N // 2, N - 2, N - 1]
    _same_bits(stats.order_statistics_dev(ptr, n - 1, D, C, ranks, ctx=ctx), qn.order_statistics(x[1:], ranks))


def test_unaligned_block_from_row_one(ctx):
    """a burn-in of one row with odd C and F: the block base is 8 but not 16-byte aligned"""
    from mcmc_ocaml_b200 import stats
    n, D, C = 401, 1, 1001
    x = np.random.default_rng(3).standard_normal((n, D + 2, C))
    d = _dev(x)
    ptr = d.data_ptr() + 8 * (D + 2) * C
    assert ptr % 16 == 8
    _same_bits(stats.quantiles_dev(ptr, n - 1, D, C, P5, ctx=ctx), qn.quantiles(x[1:], P5))


def test_non_finite_values(ctx):
    from mcmc_ocaml_b200 import stats
    n, D, C = 50, 3, 40
    rng = np.random.default_rng(5)
    x = rng.standard_normal((n, D + 2, C))
    x[7, 0, 3] = np.nan                                   # field 0 only
    x[:, 1].flat[rng.choice(n * C, 2, replace=False)] = [-np.inf, np.inf]
    x[:, 2] = rng.choice([-0.0, 0.0, 1.0], size=(n, C))   # signed zeros
    x[:, 3].flat[:3] = -np.inf
    x[:, 3].flat[3:6] = np.inf
    N = n * C
    probs = [0.0, 0.5 / (N - 1), 0.3, 0.5, 1.0 - 0.5 / (N - 1), 1.0]
    got = stats.quantiles(x, probs, ctx=ctx)
    want = qn.quantiles(x, probs)
    _same_bits(got, want)
    assert np.isnan(got[0]).all() and not np.isnan(got[1:]).any()
    assert got[1, 0] == -np.inf and got[1, 1] == -np.inf and got[1, -1] == np.inf and got[1, -2] == np.inf
    assert not np.signbit(got[2][got[2] == 0.0]).any()
    d = _dev(x)
    o = stats.order_statistics_dev(d.data_ptr(), n, D, C, [0, 1, N - 1], ctx=ctx)
    _same_bits(o, qn.order_statistics(x, [0, 1, N - 1]))


def test_both_paths_are_exercised(ctx, capfd, monkeypatch):
    """N > 2^20: the sample is a subsample.  A smooth field resolves by its brackets in one read; a field half of
    whose values are equal, at the median, overflows the candidate budget and takes the radix-select fallback."""
    from mcmc_ocaml_b200 import stats
    n, D, C = 1100, 1, 1000
    rng = np.random.default_rng(9)
    x = np.empty((n, D + 2, C))
    x[:, 0] = rng.standard_normal((n, C))
    x[:, 1] = rng.random((n, C))
    x[:, 1].flat[rng.choice(n * C, n * C // 2, replace=False)] = 0.0     # half the pool ties at the minimum
    x[:, 2] = -3.0                                                       # constant
    d = _dev(x)
    monkeypatch.setenv("MCMC_GPU_DEBUG", "1")
    capfd.readouterr()
    got = stats.quantiles_dev(d.data_ptr(), n, D, C, P5, ctx=ctx)
    err = capfd.readouterr().err
    assert "quantiles: field 0: bracket, 1 full read" in err, err
    assert "quantiles: field 1: fallback, 9 full reads" in err, err
    assert "quantiles: field 2: bracket, 1 full read" in err, err
    _same_bits(got, qn.quantiles(x, P5))
    ranks = [0, 1, n * C // 2 - 1, n * C // 2, n * C - 1]
    _same_bits(stats.order_statistics_dev(d.data_ptr(), n, D, C, ranks, ctx=ctx), qn.order_statistics(x, ranks))


def test_config2_block_from_the_device_sampler(ctx):
    """C = 4096, n = 2000 of the headline model (flat prior: log_prior is constant)"""
    import torch

    from mcmc_ocaml_b200 import mcmc, stats, plugins as P
    D, C, n = 10, 4096, 2000
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
    torch.cuda.synchronize()
    got = stats.quantiles_dev(blk.data_ptr(), n, D, C, P5, ctx=ctx)
    ctx.sync()
    assert torch.equal(blk.view(torch.int64), before.view(torch.int64)), "the block was modified"
    x = blk.cpu().numpy()
    _same_bits(stats.quantiles(x, P5, ctx=ctx), got, "host vs device")
    _same_bits(got, qn.quantiles(x, P5), "oracle")
    assert (got[D + 1] == x[0, D + 1, 0]).all()


def test_field_of_more_than_2_31_values(ctx):
    """field 1 is a permutation i a mod N of 0 .. N-1 made on the device: x_(k) = k exactly"""
    import torch

    from mcmc_ocaml_b200 import stats
    D, C, n = 1, 1024, 2 ** 21 + 3
    N = n * C
    assert N > 2 ** 31
    a = 1_000_003                                          # prime, not a factor of N
    assert np.gcd(a, N) == 1
    dev = torch.device("cuda", 0)
    blk = torch.zeros((n, D + 2, C), dtype=torch.float64, device=dev)
    blk[:, 2] = 0.25
    step = 1 << 27
    flat = blk[:, 1, :]
    for s0 in range(0, n, step // C):
        s1 = min(n, s0 + step // C)
        i = torch.arange(s0 * C, s1 * C, dtype=torch.int64, device=dev)
        flat[s0:s1] = ((i * a) % N).to(torch.float64).view(s1 - s0, C)
    torch.cuda.synchronize()
    ranks = [0, 1, 12345, N // 2, N - 2, N - 1]
    o = stats.order_statistics_dev(blk.data_ptr(), n, D, C, ranks, ctx=ctx)
    np.testing.assert_array_equal(o[1], np.array(ranks, dtype=np.float64))
    np.testing.assert_array_equal(o[2], 0.25)
    probs = [0.0, 0.1, 0.5, 0.975, 1.0]
    q = stats.quantiles_dev(blk.data_ptr(), n, D, C, probs, ctx=ctx)
    want = []
    for p in probs:                                       # the definition on x_(k) = k
        h = np.float64(N - 1) * np.float64(p)
        lo = int(np.floor(h))
        g = h - np.float64(lo)
        av, bv = np.float64(lo), np.float64(min(lo + 1, N - 1))
        want.append(av if (g == 0.0 or av == bv) else av + g * (bv - av))
    np.testing.assert_array_equal(q[1], np.array(want))
    np.testing.assert_array_equal(q[0], 0.0)
    del blk, flat


@pytest.mark.parametrize("n,D,C,probs", [(0, 1, 4, [0.5]), (4, 0, 4, [0.5]), (4, 1, 0, [0.5]), (4, 1, 4, []),
                                         (4, 1, 4, [0.5] * 65), (4, 1, 4, [1.5]), (4, 1, 4, [-0.1]),
                                         (4, 1, 4, [float("nan")]), (4, 2 ** 31 - 2, 4, [0.5])])
def test_invalid_arguments_raise(ctx, n, D, C, probs):
    from mcmc_ocaml_b200 import InvalidArgument, _abi
    x = np.zeros(64)                      # every case is rejected before the block or out is touched
    p = np.asarray(probs or [0.5], dtype=np.float64)
    out = np.empty(3 * 65)
    with pytest.raises(InvalidArgument):
        ctx.check(ctx.lib.mg_stats_quantiles(ctx.h, _abi.ptr(x), n, D, C, _abi.ptr(p), len(probs), _abi.ptr(out)))


@pytest.mark.parametrize("rank", [-1, 24])
def test_invalid_ranks_raise(ctx, rank):
    from mcmc_ocaml_b200 import InvalidArgument, stats
    d = _dev(np.zeros((4, 3, 6)))
    with pytest.raises(InvalidArgument):
        stats.order_statistics_dev(d.data_ptr(), 4, 1, 6, [0, rank], ctx=ctx)


def test_one_rank_communicator_is_the_single_gpu_call(ctx):
    from mcmc_ocaml_b200 import stats
    from mcmc_ocaml_b200.comm import Comm
    x = np.random.default_rng(21).standard_normal((500, 4, 300))
    d = _dev(x)
    one = stats.quantiles_dev(d.data_ptr(), 500, 2, 300, P5, ctx=ctx)
    comm = Comm(ctx, 1, 0)
    try:
        cm = comm.quantiles(d.data_ptr(), 500, 2, 300, P5)
    finally:
        comm.close()
    _same_bits(cm, one)
