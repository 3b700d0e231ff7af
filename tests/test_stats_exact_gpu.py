"""Stats reductions (csrc/stats.cu) against exactly summed references, at the shapes, data and edges where a parallel
reduction goes wrong.

Error models behind the tolerances (eps = 2^-52):
  * mean: every thread keeps a compensated partial and each block partial is rounded once, so
      |got - ref| <= 4 eps |ref| + 4 eps sum|x| / n.
  * std of a table: the variance pass is a compensated sum of rounded squares about the mean it is given (the
    caller's, or the kernel's own multi_mean), so it matches the exact sum about that same mean to 1e-13 relative.
  * std of a sample block: one pass about a pivot taken from the data; the cancellation in S2 - S1^2/N costs
    eps (mean - pivot)^2 / var, small whatever one outlying sample does, so 1e-13 relative against the exact variance.
  * the resident sampler's running moments are plain per-chain sums over n samples: the 1e-12 the project states.
Non-finite values follow the reference's left-to-right fold: a NaN, or both infinities, make the mean NaN, one
infinity makes it that infinity, and any non-finite value makes the std NaN (inf - inf); N = 1 gives std 0/0 = NaN.
"""
import ctypes as C
import itertools
import math
from fractions import Fraction

import numpy as np
import pytest

from mcmc_ocaml_b200 import InvalidArgument, stats

EPS = 2.0 ** -52
_CHUNK = 1 << 20


# ---- exact references -----------------------------------------------------------------------------------------

def _fsum(x):
    """Exactly rounded sum of a float64 array of any size (math.fsum fed in chunks, one running exact sum)."""
    x = np.asarray(x, dtype=np.float64).ravel()
    return math.fsum(itertools.chain.from_iterable(x[i:i + _CHUNK].tolist() for i in range(0, x.size, _CHUNK)))


def _fsum_sq_dev(x, m):
    """(fsum((x - m)^2), fsum(x - m)) with the deviations and squares rounded as float64, in chunks."""
    x = np.asarray(x, dtype=np.float64).ravel()
    d1 = (lambda: ((x[i:i + _CHUNK] - m).tolist() for i in range(0, x.size, _CHUNK)))
    d2 = (lambda: (((x[i:i + _CHUNK] - m) ** 2).tolist() for i in range(0, x.size, _CHUNK)))
    return math.fsum(itertools.chain.from_iterable(d2())), math.fsum(itertools.chain.from_iterable(d1()))


def _nonfinite_mean(x):
    """The reference fold's mean when x holds a non-finite value, else None."""
    if np.all(np.isfinite(x)):
        return None
    if np.isnan(x).any() or (np.isposinf(x).any() and np.isneginf(x).any()):
        return math.nan
    return math.inf if np.isposinf(x).any() else -math.inf


def ref_mean(x):
    """fsum(x) / n, with the reference's rules for NaN and +-inf."""
    x = np.asarray(x, dtype=np.float64).ravel()
    nf = _nonfinite_mean(x)
    return nf if nf is not None else _fsum(x) / x.size


def ref_std(x, mean=None):
    """sqrt(sum (x - m)^2 / (n - 1)).  With ``mean`` given, m is exactly that value.  Without, m is the exact mean:
    fsum((x - m)^2) about the rounded fsum mean m, less n (m - exact mean)^2 = fsum(x - m)^2 / n (the corrected
    two-pass form), so that the reference does not carry the rounding of m into the variance."""
    x = np.asarray(x, dtype=np.float64).ravel()
    n = x.size
    m = ref_mean(x) if mean is None else float(mean)
    with np.errstate(invalid="ignore", over="ignore"):
        d2 = (x - m) ** 2
    if np.isnan(d2).any():
        return math.nan
    if np.isinf(d2).any():
        return math.inf if n > 1 else math.nan
    if n == 1:
        return math.nan                      # 0 / 0
    s2, s1 = _fsum_sq_dev(x, m)
    if mean is None:
        s2 -= s1 * s1 / n
    return math.sqrt(max(s2, 0.0) / (n - 1))


def mean_tol(x, ref):
    x = np.asarray(x, dtype=np.float64).ravel()
    return 4 * EPS * abs(ref) + 4 * EPS * _fsum(np.abs(x)) / x.size


def same_nonfinite(got, want):
    return (math.isnan(got) and math.isnan(want)) or got == want


def dyadic_moments(values, counts):
    """Exact mean and std (n - 1) of a multiset given by distinct values and their counts, in rational arithmetic."""
    vals = [Fraction(float(v)) for v in values]
    n = sum(int(c) for c in counts)
    m = sum(v * int(c) for v, c in zip(vals, counts)) / n
    var = sum((v - m) ** 2 * int(c) for v, c in zip(vals, counts)) / (n - 1)
    return float(m), math.sqrt(var)


def hard_columns(rng, n, D):
    """Column d: kind d % 3 -- offset 1e8 with sigma 1e-3; mean ~0 with sigma 1e6; mixed magnitudes 1e-8..1e8."""
    xs = np.empty((n, D))
    for d in range(D):
        k = d % 3
        if k == 0:
            xs[:, d] = 1e8 + 1e-3 * rng.standard_normal(n)
        elif k == 1:
            xs[:, d] = 1e6 * rng.standard_normal(n)
        else:
            xs[:, d] = rng.choice([-1.0, 1.0], n) * 10.0 ** rng.uniform(-8, 8, n)
    return xs


# ---- CPU checks of the references themselves ------------------------------------------------------------------

def test_reference_rules_nonfinite():
    assert math.isnan(ref_mean([1.0, math.nan, 2.0])) and math.isnan(ref_std([1.0, math.nan, 2.0]))
    assert ref_mean([1.0, math.inf]) == math.inf and math.isnan(ref_std([1.0, math.inf]))
    assert ref_mean([-math.inf, 1.0]) == -math.inf and math.isnan(ref_std([-math.inf, 1.0]))
    assert math.isnan(ref_mean([math.inf, -math.inf])) and math.isnan(ref_std([math.inf, -math.inf]))
    assert ref_std([1.0, math.inf], mean=0.0) == math.inf            # about a given finite mean: inf
    assert ref_mean([3.5]) == 3.5 and math.isnan(ref_std([3.5]))     # N = 1: 0 / 0


def test_reference_exact_on_hard_data():
    """The corrected two-pass std equals the rational-arithmetic std to a few ulp where the plain two-pass form,
    about the rounded mean, is off by (rounding of m)^2 / var."""
    rng = np.random.default_rng(1)
    for x in (1e8 + 1e-3 * rng.standard_normal(3001), 1e6 * rng.standard_normal(2000), hard_columns(rng, 999, 3)[:, 2]):
        fr = [Fraction(float(v)) for v in x]
        m = sum(fr) / len(fr)
        exact = math.sqrt(sum((v - m) ** 2 for v in fr) / (len(fr) - 1))
        assert abs(ref_mean(x) - float(m)) <= math.ulp(float(m))        # two roundings: the sum, then / n
        assert abs(ref_std(x) - exact) <= 4 * EPS * exact


def test_reference_fsum_chunks_and_dyadic_closed_form():
    rng = np.random.default_rng(2)
    x = rng.standard_normal(3 * _CHUNK + 17) * 10.0 ** rng.uniform(-5, 5, 3 * _CHUNK + 17)
    assert _fsum(x) == math.fsum(x.tolist())
    vals, counts = np.array([-3.0, -2.75, 0.5, 7.25]), np.array([5, 11, 2, 9])
    m, s = dyadic_moments(vals, counts)
    flat = np.repeat(vals, counts)
    assert m == ref_mean(flat) and abs(s - ref_std(flat)) <= 2 * EPS * s


# ---- host-table reductions: mg_stats_multi_mean / multi_std / mean / std --------------------------------------

def _block(D):
    return D * (256 // D)


@pytest.mark.gpu
@pytest.mark.parametrize("D", [1, 7, 255, 256])
def test_table_mean_std_hard_data(ctx, D):
    bs = _block(D)
    rng = np.random.default_rng(100 + D)
    for n in (1, 2, 3, bs // D + 1, 5 * bs + 3, 4099):
        xs = hard_columns(rng, n, D)
        got = stats.multi_mean(xs, ctx=ctx)
        for d in range(D):
            ref = ref_mean(xs[:, d])
            assert abs(got[d] - ref) <= mean_tol(xs[:, d], ref), (n, d, got[d], ref)
        if n < 2:
            with pytest.raises(InvalidArgument):
                stats.multi_std(xs, ctx=ctx)
            continue
        sd = stats.multi_std(xs, ctx=ctx)
        user = xs[0] + 0.25 * (np.abs(xs[0]) + 1.0)              # a caller's mean, used exactly
        sdu = stats.multi_std(xs, mean=user, ctx=ctx)
        for d in range(D):
            ref = ref_std(xs[:, d], mean=got[d])               # about the mean the kernel computed (= multi_mean)
            assert abs(sd[d] - ref) <= 1e-13 * ref, (n, d, sd[d], ref)
            refu = ref_std(xs[:, d], mean=user[d])
            assert abs(sdu[d] - refu) <= 1e-13 * refu, (n, d, sdu[d], refu)


@pytest.mark.gpu
def test_scalar_mean_std_well_conditioned_large(ctx):
    """n = 2^24 + 3 positive values: a lost compensation shows as an error of many ulp."""
    n = (1 << 24) + 3
    x = np.random.default_rng(5).uniform(1.0, 2.0, n)
    x[::7] += 1e6
    ref = ref_mean(x)
    got = stats.mean(x, ctx=ctx)
    assert abs(got - ref) <= 4 * EPS * ref, (got, ref, (got - ref) / ref)
    s = stats.std(x, ctx=ctx)
    refs = ref_std(x, mean=got)
    assert abs(s - refs) <= 1e-13 * refs
    s = stats.std(x, mean=1.5, ctx=ctx)
    refs = ref_std(x, mean=1.5)
    assert abs(s - refs) <= 1e-13 * refs


@pytest.mark.gpu
def test_table_nonfinite_field_by_field(ctx):
    rng = np.random.default_rng(6)
    n, D = 1000, 8
    xs = rng.standard_normal((n, D)) + np.arange(D)
    xs[17, 1] = math.nan
    xs[500, 2] = math.inf
    xs[999, 3] = -math.inf
    xs[3, 4], xs[900, 4] = math.inf, -math.inf
    xs[0, 5], xs[1, 5] = math.inf, math.nan
    xs[0, 6] = math.inf                                          # the first value itself
    m = stats.multi_mean(xs, ctx=ctx)
    s = stats.multi_std(xs, ctx=ctx)
    given = np.full(D, 0.5)
    su = stats.multi_std(xs, mean=given, ctx=ctx)
    for d in range(D):
        col = xs[:, d]
        ref = ref_mean(col)
        if np.all(np.isfinite(col)):
            assert abs(m[d] - ref) <= mean_tol(col, ref)
            r = ref_std(col, mean=m[d])
            assert abs(s[d] - r) <= 1e-13 * r
        else:
            assert same_nonfinite(m[d], ref), (d, m[d], ref)
            assert same_nonfinite(s[d], ref_std(col, mean=m[d])), (d, s[d])
        assert same_nonfinite(su[d], ref_std(col, mean=0.5)) or abs(su[d] - ref_std(col, mean=0.5)) <= 1e-13 * su[d], d
    assert same_nonfinite(stats.mean(xs[:, 2], ctx=ctx), math.inf)
    assert math.isnan(stats.std(xs[:, 3], ctx=ctx))


# ---- device sample block: mg_stats_sample_block_dev -----------------------------------------------------------

def _torch():
    import torch
    return torch


def block_stats(ctx, t, n, D, C):
    _torch().cuda.synchronize()        # the library reads on its own stream: torch's writes must have landed
    return stats.sample_block_stats(t.data_ptr(), n, D, C, ctx=ctx)


def check_block(blk, got_mean, got_std, std_rtol=1e-13):
    """blk: host [n][F][C]; every field against the exact reference."""
    n, F, C = blk.shape
    worst = 0.0
    for f in range(F):
        x = blk[:, f, :]
        rm, rs = ref_mean(x), ref_std(x)
        if not np.all(np.isfinite(x)) or x.size == 1:
            assert same_nonfinite(got_mean[f], rm) or got_mean[f] == rm, (f, got_mean[f], rm)
            assert same_nonfinite(got_std[f], rs), (f, got_std[f], rs)
            continue
        assert abs(got_mean[f] - rm) <= mean_tol(x, rm), (f, got_mean[f], rm)
        err = abs(got_std[f] - rs) / rs if rs > 0 else abs(got_std[f])
        worst = max(worst, err)
        assert err <= std_rtol, (f, got_std[f], rs, err)
    return worst


def field_data(rng, n, F, C):
    """Field f: offset / scale by f % 3 -- (0, 1), (1e8, 1e-3), (-3e5, 1e6)."""
    off = np.array([0.0, 1e8, -3e5])[np.arange(F) % 3]
    sc = np.array([1.0, 1e-3, 1e6])[np.arange(F) % 3]
    return off[None, :, None] + sc[None, :, None] * rng.standard_normal((n, F, C))


@pytest.mark.gpu
@pytest.mark.parametrize("n,D,C", [(1, 1, 2), (5, 1, 4096), (3, 64, 1001), (4000, 1, 1), (2500, 64, 2), (700, 1, 257),
                                   (1, 64, 3000), (9, 1, 1)])
def test_sample_block_shapes(ctx, n, D, C):
    """C even (double2 loads), odd and 1 (scalar loads); n = 1, n below the grid (8 CTAs per SM), n far above it;
    F = 3 and 66."""
    torch = _torch()
    blk = field_data(np.random.default_rng(n * 7 + D * 3 + C), n, D + 2, C)
    t = torch.from_numpy(blk).cuda()
    m, s = block_stats(ctx, t, n, D, C)
    check_block(blk, m, s)


@pytest.mark.gpu
def test_sample_block_unaligned_base(ctx):
    """A block that starts 8 bytes past a 16-byte boundary (buf[1:] of a tensor), C even: the double2 path must not
    be taken."""
    torch = _torch()
    n, D, C = 300, 3, 1000
    blk = field_data(np.random.default_rng(8), n, D + 2, C)
    buf = torch.empty(blk.size + 1, dtype=torch.float64, device="cuda")
    assert buf.data_ptr() % 16 == 0
    buf[1:] = torch.from_numpy(blk.ravel()).cuda()
    t = buf[1:]
    assert t.data_ptr() % 16 == 8
    m, s = block_stats(ctx, t, n, D, C)
    check_block(blk, m, s)


@pytest.mark.gpu
def test_sample_block_constant_field_and_single_value(ctx):
    torch = _torch()
    n, D, C = 40, 2, 333
    blk = field_data(np.random.default_rng(9), n, D + 2, C)
    blk[:, 1, :] = 0.1
    m, s = block_stats(ctx, torch.from_numpy(blk).cuda(), n, D, C)
    assert s[1] == 0.0 and m[1] == 0.1
    check_block(np.delete(blk, 1, axis=1), np.delete(m, 1), np.delete(s, 1))
    one = np.array([[[2.5]], [[-1.0]], [[1e300]]]).reshape(1, 3, 1)
    m, s = block_stats(ctx, torch.from_numpy(one).cuda(), 1, 1, 1)
    assert np.array_equal(m, one.ravel()) and np.all(np.isnan(s))     # N = 1: 0 / 0


@pytest.mark.gpu
@pytest.mark.parametrize("k", [1e3, 3e3])
def test_sample_block_outlying_first_sample(ctx, k):
    """Chain 0's slot-0 value k sigma out (an outlying start point with no burn-in), N = 4.2e6 per field: the
    std stays within 1e-13 of the exact one."""
    torch = _torch()
    n, D, C = 64, 1, 65536
    blk = field_data(np.random.default_rng(int(k)), n, D + 2, C)
    sig = np.array([1.0, 1e-3, 1e6])
    blk[0, :, 0] += k * sig
    m, s = block_stats(ctx, torch.from_numpy(blk).cuda(), n, D, C)
    worst = check_block(blk, m, s)
    print(f"outlier {k:g} sigma: worst std rel err {worst:.2e} (tol 1e-13)")


@pytest.mark.gpu
@pytest.mark.parametrize("C", [1, 7, 64])
def test_sample_block_nonfinite(ctx, C):
    """Field 0 clean; 1 NaN; 2 +inf; 3 -inf; 4 both infinities; 5..7 NaN / +inf / -inf in the first value of the
    block (sample 0, chain 0), 8 +inf first and NaN later.  Other fields are unaffected."""
    torch = _torch()
    n, D = 50, 7
    blk = np.random.default_rng(10 + C).standard_normal((n, D + 2, C)) + 3.0
    blk[n // 2, 1, C // 2] = math.nan
    blk[n - 1, 2, C - 1] = math.inf
    blk[1, 3, 0] = -math.inf
    blk[2, 4, 0], blk[n - 2, 4, C - 1] = math.inf, -math.inf
    blk[0, 5, 0], blk[0, 6, 0], blk[0, 7, 0] = math.nan, math.inf, -math.inf
    blk[0, 8, 0], blk[n - 1, 8, C // 2] = math.inf, math.nan
    m, s = block_stats(ctx, torch.from_numpy(blk).cuda(), n, D, C)
    check_block(blk, m, s)
    assert np.isfinite(m[0]) and np.isfinite(s[0])
    assert m[2] == math.inf and m[3] == -math.inf and m[6] == math.inf and m[7] == -math.inf
    assert np.all(np.isnan(m[[1, 4, 5, 8]])) and np.all(np.isnan(s[1:]))


@pytest.mark.gpu
def test_sample_block_many_fields(ctx):
    """F = 65,540 fields: more than a grid's y extent."""
    torch = _torch()
    n, D, C = 2, 65538, 3
    blk = np.random.default_rng(11).standard_normal((n, D + 2, C)) * np.arange(1, D + 3)[None, :, None]
    m, s = block_stats(ctx, torch.from_numpy(blk).cuda(), n, D, C)
    x = blk.transpose(1, 0, 2).reshape(D + 2, -1)
    for f in range(0, D + 2, 997):
        assert abs(m[f] - ref_mean(x[f])) <= mean_tol(x[f], ref_mean(x[f]))
        assert abs(s[f] - ref_std(x[f])) <= 1e-13 * ref_std(x[f])
    assert abs(s[-1] - ref_std(x[-1])) <= 1e-13 * ref_std(x[-1])
    # every field, at the precision numpy's pairwise sums reach (far inside a wrong field's error)
    np.testing.assert_allclose(m, x.mean(axis=1), rtol=1e-12, atol=1e-12 * np.abs(x).mean(axis=1).max())
    np.testing.assert_allclose(s, x.std(axis=1, ddof=1), rtol=1e-12)


@pytest.mark.gpu
def test_sample_block_over_2_31_elements(ctx):
    """n * F * C = 2.15e9 elements (17.2 GB) on a dyadic grid: row s of field f is pattern[s % 4][f], so every
    value's count is known and the exact mean and std follow in rational arithmetic without a host copy."""
    torch = _torch()
    n, D, C = 4 * 2736, 1, 65538
    F = D + 2
    assert n * F * C > 2 ** 31
    c = np.arange(C)
    pat = np.empty((4, F, C))
    for r in range(4):
        for f in range(F):
            pat[r, f] = ((r + c) % 4) * 0.25 + ((r * c) % 3) * 1.5 - 3.0 + 8.0 * f
    pt = torch.from_numpy(pat).cuda()
    blk = torch.empty((n // 4, 4, F, C), dtype=torch.float64, device="cuda")
    blk.copy_(pt.unsqueeze(0).expand_as(blk))
    m, s = block_stats(ctx, blk, n, D, C)
    for f in range(F):
        vals, counts = np.unique(pat[:, f, :], return_counts=True)
        em, es = dyadic_moments(vals, counts * (n // 4))
        assert abs(m[f] - em) <= 4 * EPS * abs(em) + 4 * EPS * float(np.abs(vals) @ counts) / counts.sum(), (f, m[f], em)
        assert abs(s[f] - es) <= 1e-13 * es, (f, s[f], es)
    del blk


# ---- mg_mcmc_array_resident: block statistics and running moments --------------------------------------------

def _resident(ctx, D, Cn, n, x0, seed, nbin=0, nskip=1):
    torch = _torch()
    from mcmc_ocaml_b200 import _abi, plugins as P
    mu = np.arange(D) / 10.0
    cov = 0.7 ** np.abs(np.subtract.outer(np.arange(D), np.arange(D)))
    like, prior, prop = P.gauss_corr(mu, cov), P.zero(D), P.box_proposal(np.full(D, 0.5))
    F = D + 2
    blk = torch.empty((n, F, Cn), dtype=torch.float64, device="cuda")
    final = np.empty((Cn, F)); acc = np.empty(Cn, np.int64); rej = np.empty(Cn, np.int64)
    mean = np.empty(F); std = np.empty(F)
    cfg = _abi.mg_mcmc_cfg(Cn, D, 0, nbin, nskip, n, 0, 0, 0)          # x0_shared = 0: x0 is [C][D]
    ls, ps, js = like.spec(), prior.spec(), prop.spec()
    ctx.set_seed(seed)
    x0 = _abi.as_f64(x0)
    ctx.check(ctx.lib.mg_mcmc_array_resident(ctx.h, C.byref(ls), C.byref(ps), C.byref(js), C.byref(cfg), _abi.ptr(x0),
                                             C.c_void_p(blk.data_ptr()), _abi.ptr(final),
                                             _abi.ptr(acc, _abi.c_int64_p), _abi.ptr(rej, _abi.c_int64_p),
                                             _abi.ptr(mean), _abi.ptr(std)))
    torch.cuda.synchronize()
    host = blk.cpu().numpy()
    del blk
    return host, mean, std


def _far_start(D, Cn, k, seed):
    x0 = np.arange(D)[None, :] / 10.0 + np.random.default_rng(seed).uniform(-1, 1, (Cn, D))
    x0[0] = np.arange(D) / 10.0 + k                   # unit marginal variances: k sigma out in every coordinate
    return x0


def check_resident(host, mean, std, rtol):
    n, F, Cn = host.shape
    worst_m = worst_s = 0.0
    for f in range(F):
        x = host[:, f, :]
        rm, rs = ref_mean(x), ref_std(x)
        if rs == 0.0:                                  # a constant field (the flat prior's log_prior)
            assert mean[f] == rm and std[f] == 0.0
            continue
        scale = abs(rm) + float(np.abs(x).mean())
        worst_m = max(worst_m, abs(mean[f] - rm) / scale)
        worst_s = max(worst_s, abs(std[f] - rs) / rs)
    print(f"resident n={n} C={Cn}: worst mean err {worst_m:.2e} of (|mean| + mean|x|), worst std rel err "
          f"{worst_s:.2e} (tol {rtol:g})")
    assert worst_m <= rtol and worst_s <= rtol


@pytest.mark.gpu
@pytest.mark.parametrize("k", [1e3, 3e3])
def test_resident_block_path_far_start(ctx, k):
    """512 chains take the static sampler and the one-pass block statistics; no burn-in, chain 0 starts k out."""
    D, Cn, n = 10, 512, 700
    host, mean, std = _resident(ctx, D, Cn, n, _far_start(D, Cn, k, 1), 0x5A1)
    assert host[0, 0, 0] == k
    check_resident(host, mean, std, 1e-13)


@pytest.mark.gpu
def test_resident_running_moments_far_start(ctx):
    """19,951 chains and 599 steps take the balanced sampler's per-chain running moments; chain 0 starts 1e3 out."""
    D, n = 10, 600
    Cn = 592 * 32 + 1007
    host, mean, std = _resident(ctx, D, Cn, n, _far_start(D, Cn, 1e3, 2), 0x5A2)
    check_resident(host, mean, std, 1e-12)


@pytest.mark.gpu
def test_resident_running_moments_headline_length(ctx):
    """n = 10^4 recorded samples per chain (the headline run's length) through the running moments, D = 2 so that
    the block is 6.4 GB."""
    D, n = 2, 10_000
    Cn = 592 * 32 + 1007
    host, mean, std = _resident(ctx, D, Cn, n, _far_start(D, Cn, 1e3, 3), 0x5A3)
    check_resident(host, mean, std, 1e-12)


# ---- mg_stats_autocorrelation ---------------------------------------------------------------------------------

@pytest.mark.gpu
def test_autocorrelation_many_lags(ctx):
    """nslides = 70,000 (more than a grid's y extent) on an AR(1) series of 140,001 values."""
    n, nslides = 140_001, 70_000
    rng = np.random.default_rng(12)
    e = rng.standard_normal(n)
    x = np.empty(n)
    x[0] = e[0]
    for i in range(1, n):
        x[i] = 0.9 * x[i - 1] + e[i]
    x += 5.0
    r, _ = stats.autocorrelation(x, nslides, ctx=ctx)
    mu = ref_mean(x)
    sig2 = ref_std(x) ** 2
    d = x - mu
    for lag in (0, 1, 65_535, 65_536, nslides - 1):
        want = _fsum(d[: n - lag] * d[lag:]) / sig2 / (n - lag)
        assert abs(r[lag] - want) <= 1e-12, (lag, r[lag], want)
    assert np.all(np.isfinite(r))
