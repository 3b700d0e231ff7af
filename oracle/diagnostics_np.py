"""Ensemble convergence diagnostics of a sample block, written out directly from
their definitions (DESIGN.md section 4b).  An addition beyond the reference, in
the same standing as the integrated autocorrelation length of
mg_stats_autocorrelation (SURVEY F6).  This is the reference the GPU kernel
(mcmc_ocaml_b200/csrc/diagnostics.cu) is compared with.

Block x[s][f][c], s < n, f < F = D + 2, c < C.

Sequences: split -> N = n // 2, M = 2C; sequence c is rows [0, N) of chain c,
sequence C + c rows [n - N, n) of chain c (the middle row of an odd n is
dropped).  No split -> N = n, M = C.

Per sequence m and field f:
  xbar_m = (1/N) sum_s x_s
  gamma_m(t) = (1/N) sum_{s=0}^{N-1-t} (x_s - xbar_m)(x_{s+t} - xbar_m),  t = 0..L-1
  s2_m = N/(N-1) gamma_m(0)
Pooled:
  W = mean_m s2_m,  B = N/(M-1) sum_m (xbar_m - xbar)^2  (B = 0 when M = 1)
  var+ = (N-1)/N W + B/N,  Rhat = sqrt(var+ / W)  (NaN when M = 1)
  rho_0 = 1,  rho_t = 1 - (W - mean_m gamma_m(t)) / var+
Geyer (1992), initial monotone sequence:
  P_k = rho_2k + rho_2k+1, k < L // 2; K = first k with P_k <= 0, else L // 2
  (window_closed = 0); P'_0 = P_0, P'_k = min(P_k, P'_k-1);
  tau = -1 + 2 sum_{k<K} P'_k,  ESS = M N / tau (no cap).
Per sequence: the same rule on rho_m(t) = gamma_m(t) / gamma_m(0) gives tau_m.

Edge cases: a field constant over the block (var+ = 0) -> Rhat, ESS, tau, rho
NaN; W = 0 with differing chain means -> Rhat = +inf; a non-finite value in a
field -> that field's pooled outputs NaN.  tau_m is NaN for a sequence that is
constant (gamma_m(0) = 0) or holds a non-finite value.

`exact=True` sums every mean and lag product with math.fsum (slow: small
blocks).  `exact=False` sums the same centred products with numpy's pairwise
float64 sums (error ~ 1e-15 gamma_m(0)), for blocks of millions of values.
"""
from __future__ import annotations

import math
from dataclasses import dataclass

import numpy as np


@dataclass
class Diagnostics:
    rhat: np.ndarray            # [F]
    ess: np.ndarray             # [F]
    tau: np.ndarray             # [F]
    window_closed: np.ndarray   # int32 [F]
    rho: np.ndarray             # [F][L]
    seq_tau: np.ndarray | None  # [F][M] or None
    # intermediate values, for the tests
    W: np.ndarray | None = None
    B: np.ndarray | None = None
    var_plus: np.ndarray | None = None
    seq_pairs: np.ndarray | None = None   # [F][M][L // 2] pair sums P_k of every sequence (per_sequence only)


def sequences(x: np.ndarray, split: bool) -> tuple[np.ndarray, int]:
    """x [n][F][C] -> sequences [F][M][N] (numpy copy), N"""
    n = x.shape[0]
    if split:
        N = n // 2
        seq = np.concatenate([x[:N], x[n - N:]], axis=2)   # [N][F][2C]: chains, then second halves
    else:
        N = n
        seq = x
    return np.ascontiguousarray(np.transpose(seq, (1, 2, 0))), N


def geyer(rho) -> tuple[float, int, list]:
    """tau, window_closed, pair sums of an autocorrelation sequence rho[0..L)"""
    L = len(rho)
    npairs = L // 2
    P = [rho[2 * k] + rho[2 * k + 1] for k in range(npairs)]
    K, closed = npairs, 0
    for k in range(npairs):
        if P[k] <= 0.0:
            K, closed = k, 1
            break
    total = 0.0
    prev = 0.0
    for k in range(K):
        cur = P[k] if k == 0 else (P[k] if P[k] < prev else prev)
        total += cur
        prev = cur
    return -1.0 + 2.0 * total, closed, P


def _gammas(seq: np.ndarray, N: int, L: int, exact: bool):
    """seq [M][N] -> means [M], gamma [M][L]"""
    M = seq.shape[0]
    if exact:
        means = np.array([math.fsum(seq[m]) / N for m in range(M)])
        dev = seq - means[:, None]
        gam = np.array([[math.fsum(dev[m, :N - t] * dev[m, t:]) / N for t in range(L)] for m in range(M)])
    else:
        means = seq.sum(axis=1) / N
        dev = seq - means[:, None]
        gam = np.empty((M, L))
        for t in range(L):
            gam[:, t] = np.einsum("ms,ms->m", dev[:, :N - t], dev[:, t:]) / N
    return means, gam


def chain_diagnostics(x, maxlag: int, split: bool = True, per_sequence: bool = False, exact: bool = True) -> Diagnostics:
    x = np.asarray(x, dtype=np.float64)
    if x.ndim != 3:
        raise ValueError("x must be [n][F][C]")
    n, F, C = x.shape
    L = int(maxlag)
    if split and n < 4:
        raise ValueError("split needs n >= 4")
    seqs, N = sequences(x, split)
    M = seqs.shape[1]
    if L < 2 or L >= N:
        raise ValueError("need 2 <= maxlag <= N - 1")
    rhat, ess, tau = np.empty(F), np.empty(F), np.empty(F)
    closed = np.zeros(F, dtype=np.int32)
    rho = np.empty((F, L))
    Ws, Bs, Vs = np.empty(F), np.empty(F), np.empty(F)
    seq_tau = np.empty((F, M)) if per_sequence else None
    seq_pairs = np.empty((F, M, L // 2)) if per_sequence else None
    for f in range(F):
        s = seqs[f]
        finite = bool(np.isfinite(s).all())
        with np.errstate(all="ignore"):
            means, gam = _gammas(s, N, L, exact) if finite else (np.full(M, np.nan), np.full((M, L), np.nan))
            s2 = N / (N - 1) * gam[:, 0]
            W = (math.fsum(s2) if finite else np.nan) / M
            if M > 1:
                grand = (math.fsum(means) if finite else np.nan) / M
                B = N / (M - 1) * (math.fsum((means - grand) ** 2) if finite else np.nan)
            else:
                B = 0.0
            vp = (N - 1) / N * W + B / N
            Ws[f], Bs[f], Vs[f] = W, B, vp
            bad = not finite or not (vp > 0.0)
            if bad:
                rhat[f] = ess[f] = tau[f] = np.nan
                rho[f] = np.nan
                closed[f] = 0
            else:
                rhat[f] = np.nan if M == 1 else (math.sqrt(vp / W) if W > 0.0 else np.inf)
                gbar = np.array([math.fsum(gam[:, t]) / M for t in range(L)])
                r = 1.0 - (W - gbar) / vp
                r[0] = 1.0
                rho[f] = r
                tau[f], closed[f], _ = geyer(list(r))
                ess[f] = M * N / tau[f]
            if per_sequence:
                for m in range(M):
                    g0 = gam[m, 0]
                    if not (np.isfinite(g0) and g0 > 0.0):
                        seq_tau[f, m] = np.nan
                        seq_pairs[f, m] = np.nan
                        continue
                    rm = gam[m] / g0
                    seq_tau[f, m], _, P = geyer(list(rm))
                    seq_pairs[f, m] = P
    return Diagnostics(rhat, ess, tau, closed, rho, seq_tau, Ws, Bs, Vs, seq_pairs)


def ar1_block(n: int, F: int, C: int, phi, seed: int = 0, offset=None) -> np.ndarray:
    """[n][F][C] block of stationary AR(1) chains x_s = phi x_{s-1} + e_s, unit innovations; phi per field (scalar or
    [F]); offset[F][C] added to every chain (group means for the Rhat known answers)."""
    rng = np.random.default_rng(seed)
    phi = np.broadcast_to(np.asarray(phi, dtype=np.float64), (F,))[None, :, None]
    x = np.empty((n, F, C))
    x[0] = rng.standard_normal((F, C)) / np.sqrt(1.0 - phi[0] ** 2)
    for s in range(1, n):
        x[s] = phi[0] * x[s - 1] + rng.standard_normal((F, C))
    if offset is not None:
        x += np.asarray(offset, dtype=np.float64)[None]
    return x
