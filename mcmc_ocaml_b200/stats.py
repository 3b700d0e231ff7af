"""Host-side mirror of the ``Stats`` functions on the hot path (stats.mli:20-110)."""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass

import numpy as np

from . import _abi
from .context import Context, default_context


def mean(xs, *, ctx: Context | None = None) -> float:
    """``Stats.mean`` (stats.ml:17-23)."""
    ctx = ctx or default_context()
    xs = _abi.as_f64(xs)
    out = C.c_double()
    ctx.check(ctx.lib.mg_stats_mean(ctx.h, _abi.ptr(xs), C.c_int64(xs.size), C.byref(out)))
    return out.value


def std(xs, mean=None, *, ctx: Context | None = None) -> float:
    """``Stats.std ?mean`` (stats.ml:35-43), n-1 in the denominator."""
    ctx = ctx or default_context()
    xs = _abi.as_f64(xs)
    out = C.c_double()
    ctx.check(ctx.lib.mg_stats_std(ctx.h, _abi.ptr(xs), C.c_int64(xs.size), C.c_int(0 if mean is None else 1),
                                   C.c_double(0.0 if mean is None else mean), C.byref(out)))
    return out.value


def multi_mean(xs, *, ctx: Context | None = None) -> np.ndarray:
    """``Stats.multi_mean`` (stats.ml:58-70); xs [n][D]."""
    ctx = ctx or default_context()
    xs = _abi.as_f64(xs)
    out = np.empty(xs.shape[1])
    ctx.check(ctx.lib.mg_stats_multi_mean(ctx.h, _abi.ptr(xs), C.c_int64(xs.shape[0]), C.c_int32(xs.shape[1]),
                                          _abi.ptr(out)))
    return out


def multi_std(xs, mean=None, *, ctx: Context | None = None) -> np.ndarray:
    """``Stats.multi_std ?mean`` (stats.ml:72-87)."""
    ctx = ctx or default_context()
    xs = _abi.as_f64(xs)
    out = np.empty(xs.shape[1])
    m = None if mean is None else _abi.as_f64(mean)
    ctx.check(ctx.lib.mg_stats_multi_std(ctx.h, _abi.ptr(xs), C.c_int64(xs.shape[0]), C.c_int32(xs.shape[1]),
                                         _abi.ptr(m), _abi.ptr(out)))
    return out


def slow_autocorrelation(nslides: int, x, *, ctx: Context | None = None) -> np.ndarray:
    """``Stats.slow_autocorrelation nslides x`` (stats.ml:223-238), lags
    0..nslides-1 (SURVEY F6: parity unpinned)."""
    return autocorrelation(x, nslides, ctx=ctx)[0]


def autocorrelation(x, nslides: int, *, ctx: Context | None = None):
    """(r[0..nslides), integrated autocorrelation length)."""
    ctx = ctx or default_context()
    x = _abi.as_f64(x)
    r = np.empty(nslides)
    L = C.c_double()
    ctx.check(ctx.lib.mg_stats_autocorrelation(ctx.h, _abi.ptr(x), C.c_int64(x.size), C.c_int32(nslides), _abi.ptr(r),
                                               C.byref(L)))
    return r, L.value


def sample_block_stats(samples_ptr: int, n: int, D: int, nchains: int, *, ctx: Context | None = None):
    """Per-field mean / std over a device sample block [n][D+2][C] (all chains pooled)."""
    ctx = ctx or default_context()
    m, s = np.empty(D + 2), np.empty(D + 2)
    ctx.check(ctx.lib.mg_stats_sample_block_dev(ctx.h, C.c_void_p(samples_ptr), C.c_int64(n), C.c_int32(D),
                                                C.c_int64(nchains), _abi.ptr(m), _abi.ptr(s)))
    return m, s


# --- ensemble convergence diagnostics (an addition beyond the reference, DESIGN.md 4b) ---------------------------

@dataclass
class ChainDiagnostics:
    """Per field (0..D-1 values, D log_likelihood, D+1 log_prior): split-Rhat, effective sample size, integrated
    autocorrelation time (Geyer's initial monotone sequence), whether a non-positive pair closed the lag window, the
    ensemble autocorrelation rho[F][L]; ``seq_tau[F][M]`` (per sequence) when asked for."""
    rhat: np.ndarray
    ess: np.ndarray
    tau: np.ndarray
    window_closed: np.ndarray
    rho: np.ndarray
    seq_tau: np.ndarray | None = None


def _diag_cfg(n: int, D: int, nchains: int, maxlag: int, split: bool):
    return _abi.mg_diag_cfg(n=int(n), nchains=int(nchains), dim=int(D), maxlag=int(maxlag), split=1 if split else 0,
                            reserved=0)


def _diag_outputs(D: int, maxlag: int):
    F = D + 2
    return (np.empty(F), np.empty(F), np.empty(F), np.empty(F, dtype=np.int32), np.empty((F, int(maxlag))))


def _diag_call(fn, handle, ptr_arg, cfg, outs, seq_tau_arg):
    rh, es, ta, wc, rho = outs
    return fn(handle, ptr_arg, C.byref(cfg), _abi.ptr(rh), _abi.ptr(es), _abi.ptr(ta), _abi.ptr(wc, _abi.c_int32_p),
              _abi.ptr(rho), seq_tau_arg)


def chain_diagnostics(samples, maxlag: int, *, split: bool = True, per_sequence: bool = False,
                      ctx: Context | None = None) -> ChainDiagnostics:
    """Diagnostics of a host sample block: an ``McmcSamples`` (a chain-major block is transposed here) or an array
    [n][D+2][C].  ``per_sequence`` adds tau of every sequence ([F][M], M = 2C with ``split``)."""
    ctx = ctx or default_context()
    if hasattr(samples, "layout"):
        blk = samples.block if samples.layout == "step" else np.transpose(samples.block, (1, 2, 0))
    else:
        blk = samples
    blk = _abi.as_f64(blk)
    if blk.ndim != 3 or blk.shape[1] < 3:
        raise _abi.InvalidArgument("chain_diagnostics: the block must be [n][D+2][C] with D >= 1")
    n, F, nc = blk.shape
    D = F - 2
    cfg = _diag_cfg(n, D, nc, maxlag, split)
    outs = _diag_outputs(D, maxlag)
    seq = np.empty((F, (2 if split else 1) * nc)) if per_sequence else None
    ctx.check(_diag_call(ctx.lib.mg_stats_chain_diagnostics, ctx.h, _abi.ptr(blk), cfg, outs, _abi.ptr(seq)))
    return ChainDiagnostics(*outs, seq)


def chain_diagnostics_dev(samples_ptr: int, n: int, D: int, nchains: int, maxlag: int, *, split: bool = True,
                          seq_tau_ptr: int | None = None, ctx: Context | None = None) -> ChainDiagnostics:
    """The same over a device sample block [n][D+2][C] (``mg_mcmc_array_dev`` / ``_resident``), which is not
    modified; per-sequence tau goes to the device array ``seq_tau_ptr`` ([D+2][M] float64) when given."""
    ctx = ctx or default_context()
    cfg = _diag_cfg(n, D, nchains, maxlag, split)
    outs = _diag_outputs(D, maxlag)
    ctx.check(_diag_call(ctx.lib.mg_stats_chain_diagnostics_dev, ctx.h, C.c_void_p(samples_ptr), cfg, outs,
                         C.c_void_p(seq_tau_ptr) if seq_tau_ptr else None))
    return ChainDiagnostics(*outs)


# --- order statistics and quantiles of a sample block (DESIGN.md 4c) ------------------------------------------------

QUANT_MAX = _abi.QUANT_MAX


def _probs(probs) -> np.ndarray:
    p = _abi.as_f64(probs).ravel()
    if not 1 <= p.size <= QUANT_MAX:
        raise _abi.InvalidArgument(f"quantiles: need 1 to {QUANT_MAX} probabilities")
    return p


def quantiles(samples, probs, *, ctx: Context | None = None) -> np.ndarray:
    """Exact per-field quantiles [D+2][nq] of a host sample block: an ``McmcSamples`` (a chain-major block is
    transposed here) or an array [n][D+2][C]; all chains pooled, numpy's "linear" rule (include/mcmc_gpu.h)."""
    ctx = ctx or default_context()
    if hasattr(samples, "layout"):
        blk = samples.block if samples.layout == "step" else np.transpose(samples.block, (1, 2, 0))
    else:
        blk = samples
    blk = _abi.as_f64(blk)
    if blk.ndim != 3 or blk.shape[1] < 3:
        raise _abi.InvalidArgument("quantiles: the block must be [n][D+2][C] with D >= 1")
    n, F, nc = blk.shape
    p = _probs(probs)
    out = np.empty((F, p.size))
    ctx.check(ctx.lib.mg_stats_quantiles(ctx.h, _abi.ptr(blk), n, F - 2, nc, _abi.ptr(p), p.size, _abi.ptr(out)))
    return out


def quantiles_dev(samples_ptr: int, n: int, D: int, nchains: int, probs, *, ctx: Context | None = None) -> np.ndarray:
    """The same over a device sample block [n][D+2][C] (``mg_mcmc_array_dev`` / ``_resident``), which is not modified."""
    ctx = ctx or default_context()
    p = _probs(probs)
    out = np.empty((D + 2, p.size))
    ctx.check(ctx.lib.mg_stats_quantiles_dev(ctx.h, samples_ptr, n, D, nchains, _abi.ptr(p), p.size, _abi.ptr(out)))
    return out


def order_statistics_dev(samples_ptr: int, n: int, D: int, nchains: int, ranks, *,
                         ctx: Context | None = None) -> np.ndarray:
    """Exact order statistics [D+2][nk] (0-based ranks into the n C pooled values of each field) of a device block."""
    ctx = ctx or default_context()
    r = np.ascontiguousarray(ranks, dtype=np.int64).ravel()
    if not 1 <= r.size <= QUANT_MAX:
        raise _abi.InvalidArgument(f"order_statistics: need 1 to {QUANT_MAX} ranks")
    out = np.empty((D + 2, r.size))
    ctx.check(ctx.lib.mg_stats_order_statistics_dev(ctx.h, samples_ptr, n, D, nchains, _abi.ptr(r, _abi.c_int64_p),
                                                    r.size, _abi.ptr(out)))
    return out


# --- draws and densities (stats.ml:89-128, 240-248) ------------------------------------------------------------

DRAW_UNIFORM, DRAW_GAUSSIAN, DRAW_CAUCHY = 0, 1, 2


def _draw(kind: int, a: float, b: float, n: int, ctx: Context | None) -> np.ndarray:
    ctx = ctx or default_context()
    out = np.empty(int(n))
    ctx.check(ctx.lib.mg_stats_draw(ctx.h, C.c_int32(kind), C.c_double(a), C.c_double(b), C.c_int64(n), _abi.ptr(out)))
    return out


def draw_uniform(a: float, b: float, n: int = 1, *, ctx: Context | None = None) -> np.ndarray:
    """``Stats.draw_uniform a b`` (stats.ml:126-128), n draws from the context's Philox stream."""
    return _draw(DRAW_UNIFORM, a, b, n, ctx)


def draw_gaussian(mu: float, sigma: float, n: int = 1, *, ctx: Context | None = None) -> np.ndarray:
    """``Stats.draw_gaussian mu sigma`` (Leva's ratio of uniforms, stats.ml:113-124)."""
    return _draw(DRAW_GAUSSIAN, mu, sigma, n, ctx)


def draw_cauchy(x0: float, gamma: float, n: int = 1, *, ctx: Context | None = None) -> np.ndarray:
    """``Stats.draw_cauchy x0 gamma`` (stats.ml:89-91)."""
    return _draw(DRAW_CAUCHY, x0, gamma, n, ctx)


def log_gaussian(mu, sigma, x):
    """``Stats.log_gaussian`` (stats.ml:98-101) on the host; the device body is the GAUSS_DIAG plugin."""
    dx = (np.asarray(x, dtype=np.float64) - mu) / sigma
    return -0.91893853320467274178 - np.log(sigma) - 0.5 * dx * dx


def log_cauchy(x0, gamma, x):
    """``Stats.log_cauchy`` (stats.ml:93-96) on the host; the device body is the CAUCHY_DATA plugin."""
    dx = (np.asarray(x, dtype=np.float64) - x0) / gamma
    return 0.0 - np.log(np.pi * gamma) - np.log(1.0 + dx * dx)


def log_multi_gaussian(mu, sigma, x) -> float:
    """``Stats.log_multi_gaussian`` (stats.ml:103-108): sequential sum over the coordinates."""
    result = 0.0
    for m, s, v in zip(np.asarray(mu, dtype=np.float64), np.asarray(sigma, dtype=np.float64), np.asarray(x, dtype=np.float64)):
        result = result + float(log_gaussian(m, s, v))
    return result + 0.0


def log_sum_logs(a: float, b: float) -> float:
    """``Stats.log_sum_logs`` (stats.ml:240-248): log(e^a + e^b) without overflow."""
    if a == -np.inf and b == -np.inf:
        return -np.inf
    if b > a:
        a, b = b, a
    return float(a + np.log1p(np.exp(b - a)))
