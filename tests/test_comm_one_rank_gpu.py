"""Every rank-pooled entry point of the C ABI (mg_comm_*, the *_sharded calls, the distributed kd-tree build and the tree
broadcast) on a one-rank communicator: the result is that of the single-GPU call, to the tolerance each call documents,
and an argument error comes back as MG_EINVAL naming the call, after which the communicator still works.  The
communicator's own exchanges carry every rank's status, so the one-rank error path is the path a failing rank takes in
a larger job.  The library is called directly where the Python wrapper would validate the arguments first."""
import ctypes as C

import numpy as np
import pytest

from mcmc_ocaml_b200 import InvalidArgument, _abi, evidence, mcmc, plugins as P, stats
from mcmc_ocaml_b200.comm import Comm
from mcmc_ocaml_b200.kd_tree import KdTree

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def comm(ctx):
    c = Comm(ctx, 1, 0)
    yield c
    c.close()


@pytest.fixture(scope="module")
def samples(ctx):
    """MH-like evidence input on the device: rows in [0, 1]^3 with repeats, their ll and lp"""
    import torch
    rng = np.random.default_rng(31)
    N, D = 20000, 3
    pts = rng.normal(0.5, 0.1, (N, D)).clip(0, 1)
    pts[1::3] = pts[0::3][: pts[1::3].shape[0]]            # exact repeats, as rejected MH steps give
    ll = (-0.5 * ((pts - 0.5) / 0.1) ** 2).sum(1)
    lp = -0.1 * pts.sum(1)
    dev = torch.device("cuda", 0)
    t = [torch.as_tensor(a, device=dev) for a in (pts, ll, lp)]
    torch.cuda.synchronize()
    return N, D, t


def _ptrs(samples):
    return tuple(x.data_ptr() for x in samples[2])


def _bits(x):
    return np.float64(x).view(np.int64)


def test_sharded_evidence_is_the_single_gpu_call(ctx, comm, samples):
    N, D, _ = samples
    for n, eps in ((64, 0.1), (16, 1e9)):
        one = evidence.evidence_lebesgue_dev(*_ptrs(samples), N, D, n=n, eps=eps, ctx=ctx)
        got = comm.evidence_lebesgue(*_ptrs(samples), N, D, n=n, eps=eps)
        assert _bits(got) == _bits(one)
        one = evidence.evidence_direct_dev(*_ptrs(samples), N, D, n=n, ctx=ctx)
        got = comm.evidence_direct(*_ptrs(samples), N, D, n=n)
        assert _bits(got) == _bits(one)


def test_harmonic_mean_sharded_within_2_ulp(ctx, comm, samples):
    N, _, t = samples
    ll = t[1].cpu().numpy()
    one = evidence.evidence_harmonic_mean(ll=ll, ctx=ctx)
    got = comm.evidence_harmonic_mean(t[1].data_ptr(), N)
    assert abs(int(_bits(got)) - int(_bits(one))) <= 2
    print(f"harmonic_mean_sharded bits {int(_bits(got)) & (2 ** 64 - 1):016x} value {got!r}")


@pytest.mark.parametrize("min_split", [2, 64])
def test_distributed_build_is_the_single_gpu_build(ctx, comm, samples, min_split):
    N, D, t = samples
    lo, hi = np.zeros(D), np.ones(D)
    td = comm.build_tree(t[0].data_ptr(), N, D, lo, hi, min_split=min_split)
    ts = KdTree.from_device(t[0].data_ptr(), N, D, lo, hi, min_split=min_split, ctx=ctx)
    try:
        ad, as_ = td.export(), ts.export()
        assert set(ad) == set(as_)
        for k in as_:
            np.testing.assert_array_equal(ad[k], as_[k], err_msg=k)
        assert (td.nnodes, td.nlevels) == (ts.nnodes, ts.nlevels)
    finally:
        td.close()
        ts.close()


def test_broadcast_returns_the_roots_tree(ctx, comm, samples):
    N, D, t = samples
    tree = KdTree.from_device(t[0].data_ptr(), N, D, np.zeros(D), np.ones(D), ctx=ctx)
    try:
        out = C.c_void_p()
        ctx.check(ctx.lib.mg_kdtree_broadcast(comm.h, tree.h, C.c_int32(0), C.byref(out)))
        assert out.value == tree.h.value
    finally:
        tree.close()


def _pool_moments_one_rank(n_local, mean_local, std_local):
    """mg_comm_pool_moments on one rank, operation for operation"""
    F = mean_local.size
    m2_local = std_local * std_local * (np.float64(n_local) - 1.0) if n_local > 1 else np.zeros(F)
    n, mean, m2 = np.float64(0.0), np.zeros(F), np.zeros(F)
    cnt = np.float64(n_local)
    if cnt != 0.0:
        tot = n + cnt
        delta = mean_local - mean
        mean = mean + delta * (cnt / tot)
        m2 = m2 + m2_local + delta * delta * (n * cnt / tot)
        n = tot
    std = np.sqrt(m2 / (n - 1.0)) if n > 1.0 else np.zeros(F)
    return int(n), mean, std


@pytest.mark.parametrize("n_local", [0, 1, 2, 12345])
def test_pool_moments_is_its_one_rank_arithmetic(comm, n_local):
    rng = np.random.default_rng(n_local)
    mean, std = rng.normal(0.0, 3.0, 7), rng.random(7) * 2.0
    got = comm.pool_moments(n_local, mean, std)
    want = _pool_moments_one_rank(n_local, mean, std)
    assert got[0] == want[0]
    np.testing.assert_array_equal(got[1].view(np.int64), want[1].view(np.int64))
    np.testing.assert_array_equal(got[2].view(np.int64), want[2].view(np.int64))


def _rj_models():
    mu1, s1, mu2, s2 = 0.31, 0.62, 0.77, 0.45
    g1, g2 = P.gauss_diag([mu1], [s1]), P.gauss_diag([mu2], [s2])
    A = mcmc.RjModel(g1.scaled(0.5), g1.scaled(0.5), P.indep_gauss_proposal([mu1], [s1]), 0.1, into_gauss=([mu1], [s1]))
    B = mcmc.RjModel(g2.scaled(0.3), g2.scaled(0.7), P.indep_gauss_proposal([mu2], [s2]), 0.9, into_gauss=([mu2], [s2]))
    return A, B, [mu1], [mu2]


def test_rjmcmc_sharded_counts_are_the_single_gpu_counts(ctx, comm):
    A, B, a0, b0 = _rj_models()
    ctx.set_seed(77)
    one = mcmc.rjmcmc_array(40, A, B, a0, b0, nskip=3, nchains=3000, ctx=ctx)
    ctx.set_seed(77)
    got = comm.rjmcmc_array(40, A, B, a0, b0, nskip=3, nchains=3000)
    assert got.counts == one.counts
    assert got.cross == one.cross
    assert got.shard == (0, 3000)


# ---- argument errors: MG_EINVAL naming the call, then a valid call on the same communicator ---------------------------

def _evidence_call(ctx, comm, samples, fn, root=0, n=16, out=True):
    N, D, _ = samples
    res = C.c_double()
    extra = (C.c_double(0.1),) if fn == "mg_evidence_lebesgue_sharded" else ()
    return getattr(ctx.lib, fn)(comm.h, C.c_int32(root), *[C.c_void_p(p) for p in _ptrs(samples)], C.c_int64(N),
                                C.c_int32(D), C.c_int32(n), *extra, C.byref(res) if out else None)


def _harmonic_call(ctx, comm, samples, n=None, out=True):
    N, _, t = samples
    res = C.c_double()
    return ctx.lib.mg_evidence_harmonic_mean_sharded(comm.h, C.c_void_p(t[1].data_ptr()), C.c_int64(N if n is None else n),
                                                     C.byref(res) if out else None)


def _rj_call(ctx, comm, cfg=True):
    A, B, a0, b0 = _rj_models()
    sa, sb = A.spec(), B.spec()
    a0, b0 = _abi.as_f64(a0), _abi.as_f64(b0)
    c = _abi.mg_rjmcmc_cfg(64, 0, 1, 4, 0, 0, 0)
    counts = (C.c_int64 * 2)()
    return ctx.lib.mg_rjmcmc_array_sharded(comm.h, C.byref(sa), C.byref(sb), C.byref(c) if cfg else None, _abi.ptr(a0),
                                           _abi.ptr(b0), None, None, counts, None, None)


def _pool_call(ctx, comm, F=4):
    m, s = np.zeros(4), np.ones(4)
    om, os_ = np.empty(4), np.empty(4)
    return ctx.lib.mg_comm_pool_moments(comm.h, C.c_int64(10), _abi.ptr(m), _abi.ptr(s), C.c_int32(F), None,
                                        _abi.ptr(om), _abi.ptr(os_))


@pytest.fixture(scope="module")
def block():
    import torch
    x = np.random.default_rng(5).standard_normal((64, 3, 40))
    d = torch.as_tensor(x, device=torch.device("cuda", 0))
    torch.cuda.synchronize()
    return d


def _diag_call(ctx, comm, block, maxlag=8):
    cfg = stats._diag_cfg(64, 1, 40, maxlag, True)
    outs = stats._diag_outputs(1, max(maxlag, 1))
    return stats._diag_call(ctx.lib.mg_comm_chain_diagnostics, comm.h, C.c_void_p(block.data_ptr()), cfg, outs, None)


def _quantiles_call(ctx, comm, block, p=0.5, n=64):
    probs = np.array([0.1, p])
    out = np.empty((3, 2))
    return ctx.lib.mg_comm_quantiles(comm.h, block.data_ptr(), n, 1, 40, _abi.ptr(probs), 2, _abi.ptr(out))


def _build_call(ctx, comm, samples, out=True):
    N, D, t = samples
    lo, hi = np.zeros(D), np.ones(D)
    h = C.c_void_p()
    rc = ctx.lib.mg_kdtree_build_distributed(comm.h, C.c_void_p(t[0].data_ptr()), C.c_int64(N), C.c_int32(D),
                                             _abi.ptr(lo), _abi.ptr(hi), C.c_int32(2), C.byref(h) if out else None)
    if h.value:
        ctx.lib.mg_kdtree_destroy(h)
    return rc


def _broadcast_call(ctx, comm, samples, root=0):
    N, D, t = samples
    tree = KdTree.from_device(t[0].data_ptr(), N, D, np.zeros(D), np.ones(D), ctx=ctx)
    try:
        out = C.c_void_p()
        return ctx.lib.mg_kdtree_broadcast(comm.h, tree.h, C.c_int32(root), C.byref(out))
    finally:
        tree.close()


CASES = {
    # case: (name in the message, bad call, good call)
    "lebesgue_bad_root": ("evidence (sharded)", lambda c, m, s, b: _evidence_call(c, m, s, "mg_evidence_lebesgue_sharded", root=1),
                          lambda c, m, s, b: _evidence_call(c, m, s, "mg_evidence_lebesgue_sharded")),
    "lebesgue_n_0": ("evidence (sharded)", lambda c, m, s, b: _evidence_call(c, m, s, "mg_evidence_lebesgue_sharded", n=0),
                     lambda c, m, s, b: _evidence_call(c, m, s, "mg_evidence_lebesgue_sharded")),
    "direct_null_out": ("evidence (sharded)", lambda c, m, s, b: _evidence_call(c, m, s, "mg_evidence_direct_sharded", out=False),
                        lambda c, m, s, b: _evidence_call(c, m, s, "mg_evidence_direct_sharded")),
    "harmonic_null_out": ("evidence_harmonic_mean", lambda c, m, s, b: _harmonic_call(c, m, s, out=False),
                          lambda c, m, s, b: _harmonic_call(c, m, s)),
    "harmonic_negative_n": ("evidence_harmonic_mean", lambda c, m, s, b: _harmonic_call(c, m, s, n=-1),
                            lambda c, m, s, b: _harmonic_call(c, m, s)),
    "rjmcmc_null_cfg": ("rjmcmc_array", lambda c, m, s, b: _rj_call(c, m, cfg=False), lambda c, m, s, b: _rj_call(c, m)),
    "pool_moments_F_0": ("pool_moments", lambda c, m, s, b: _pool_call(c, m, F=0), lambda c, m, s, b: _pool_call(c, m)),
    "diagnostics_maxlag_1": ("chain_diagnostics", lambda c, m, s, b: _diag_call(c, m, b, maxlag=1),
                             lambda c, m, s, b: _diag_call(c, m, b)),
    "diagnostics_maxlag_above_N": ("chain_diagnostics", lambda c, m, s, b: _diag_call(c, m, b, maxlag=32),
                                   lambda c, m, s, b: _diag_call(c, m, b)),
    "quantiles_p_above_1": ("quantiles", lambda c, m, s, b: _quantiles_call(c, m, b, p=1.5),
                            lambda c, m, s, b: _quantiles_call(c, m, b)),
    "quantiles_n_0": ("quantiles", lambda c, m, s, b: _quantiles_call(c, m, b, n=0), lambda c, m, s, b: _quantiles_call(c, m, b)),
    "build_null_out": ("kd-tree (distributed)", lambda c, m, s, b: _build_call(c, m, s, out=False),
                       lambda c, m, s, b: _build_call(c, m, s)),
    "broadcast_bad_root": ("kdtree_broadcast", lambda c, m, s, b: _broadcast_call(c, m, s, root=1),
                           lambda c, m, s, b: _broadcast_call(c, m, s)),
}


@pytest.mark.parametrize("case", sorted(CASES))
def test_argument_error_then_a_valid_call(ctx, comm, samples, block, case):
    name, bad, good = CASES[case]
    with pytest.raises(InvalidArgument) as e:
        ctx.check(bad(ctx, comm, samples, block))
    assert name in str(e.value)
    ctx.check(good(ctx, comm, samples, block))
