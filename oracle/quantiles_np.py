"""numpy transcription of the order statistics and quantiles of a sample block (include/mcmc_gpu.h, DESIGN.md 4c),
line by line: np.sort of the f64_to_ordered keys and scalar float64 arithmetic."""
from __future__ import annotations

import numpy as np

_TOP = np.uint64(0x8000000000000000)


def ordered_keys(x) -> np.ndarray:
    """f64_to_ordered: -0.0 -> +0.0, then the bits with the sign bit set (x >= 0) or all bits flipped (x < 0)."""
    x = np.array(x, dtype=np.float64, copy=True).ravel()
    x[x == 0.0] = 0.0
    b = x.view(np.uint64)
    return np.where(b >> np.uint64(63) == 1, ~b, b | _TOP)


def from_keys(k) -> np.ndarray:
    k = np.asarray(k, dtype=np.uint64)
    b = np.where(k >> np.uint64(63) == 1, k & ~_TOP, ~k)
    return b.view(np.float64)


def field_pools(block) -> list[np.ndarray]:
    """block [n][F][C] -> per field its N = n C values as an [n][C] slice (unsorted)"""
    block = np.asarray(block, dtype=np.float64)
    return [block[:, f, :] for f in range(block.shape[1])]


def order_statistic(sorted_keys: np.ndarray, k: int) -> float:
    return float(from_keys(sorted_keys[k:k + 1])[0])


def quantile_of_sorted(sorted_keys: np.ndarray, p: float) -> float:
    N = sorted_keys.size
    h = np.float64(N - 1) * np.float64(p)
    lo = int(np.floor(h))
    g = h - np.float64(lo)
    a = np.float64(order_statistic(sorted_keys, lo))
    b = np.float64(order_statistic(sorted_keys, min(lo + 1, N - 1)))
    if g == 0.0 or a == b:
        return float(a)
    if a == -np.inf:
        return float("nan") if b == np.inf else float("-inf")
    if b == np.inf:
        return float("inf")
    return float(a + g * (b - a))


def quantiles(block, probs) -> np.ndarray:
    """[F][nq]; a field holding a NaN gives NaN throughout"""
    out = []
    for pool in field_pools(block):
        if np.isnan(pool).any():
            out.append([float("nan")] * len(probs))
            continue
        k = np.sort(ordered_keys(pool))
        out.append([quantile_of_sorted(k, p) for p in probs])
    return np.array(out, dtype=np.float64).reshape(len(out), len(probs))


def order_statistics(block, ranks) -> np.ndarray:
    """[F][nk]"""
    out = []
    for pool in field_pools(block):
        if np.isnan(pool).any():
            out.append([float("nan")] * len(ranks))
            continue
        k = np.sort(ordered_keys(pool))
        out.append([order_statistic(k, int(r)) for r in ranks])
    return np.array(out, dtype=np.float64).reshape(len(out), len(ranks))
