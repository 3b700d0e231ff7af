"""Multi-GPU plumbing: one process per GPU, ``torch.distributed`` for the
collectives (NCCL over NVLink on the GPU box, gloo in the CPU tests).

The hot path shards without any data-path collective (SURVEY.md 8e):
  * MH / RJ chains are independent: rank r runs global chain ids
    [r*C, (r+1)*C); Philox is keyed by the global id, so results do not depend
    on the number of ranks;
  * point-location / density / draw queries are independent: the kd-tree is
    built on one rank and broadcast as ONE contiguous device blob;
  * per-rank statistics (counts, sums, partial evidence terms) are tens of
    bytes: all-gathered and combined in rank order, so the result is
    deterministic.
"""
from __future__ import annotations

import numpy as np


def shard_range(n: int, rank: int, world: int) -> tuple[int, int]:
    """Contiguous [begin, end) of n items owned by `rank` (sizes differ by at most 1)."""
    base, rem = divmod(n, world)
    b = rank * base + min(rank, rem)
    return b, b + base + (1 if rank < rem else 0)


def combine_moments(counts, means, m2s):
    """Pooled mean and std (n-1) from per-rank (count, mean, sum of squared
    deviations) -- Chan et al. pairwise update applied in rank order."""
    n = 0.0
    mean = np.zeros_like(np.asarray(means[0], dtype=np.float64))
    m2 = np.zeros_like(mean)
    for c, mu, s in zip(counts, means, m2s):
        c = float(c)
        if c == 0:
            continue
        mu, s = np.asarray(mu, np.float64), np.asarray(s, np.float64)
        delta = mu - mean
        tot = n + c
        mean = mean + delta * (c / tot)
        m2 = m2 + s + delta * delta * (n * c / tot)
        n = tot
    return n, mean, np.sqrt(m2 / (n - 1.0))


def all_gather_array(x: np.ndarray, device=None) -> np.ndarray:
    """All-gather a small float64 array from every rank; returns [world, ...]."""
    import torch
    import torch.distributed as dist
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size() == 1:
        return np.asarray(x, np.float64)[None]
    t = torch.as_tensor(np.ascontiguousarray(x, dtype=np.float64))
    if device is not None:
        t = t.to(device)
    out = [torch.empty_like(t) for _ in range(dist.get_world_size())]
    dist.all_gather(out, t)
    return np.stack([o.cpu().numpy() for o in out])


def gather_ensemble_stats(n_samples: int, mean: np.ndarray, std: np.ndarray, accept: int, reject: int, device=None):
    """Combine per-rank sample-block statistics of a sharded ensemble run."""
    mean, std = np.asarray(mean, np.float64), np.asarray(std, np.float64)
    m2 = std * std * (n_samples - 1.0)
    payload = np.concatenate([[float(n_samples), float(accept), float(reject)], mean, m2])
    g = all_gather_array(payload, device)
    F = mean.size
    n, mu, sd = combine_moments(g[:, 0], g[:, 3:3 + F], g[:, 3 + F:3 + 2 * F])
    return dict(n=n, mean=mu, std=sd, accept=int(g[:, 1].sum()), reject=int(g[:, 2].sum()))


def combine_harmonic(counts, evidences) -> float:
    """Harmonic-mean evidence of pooled samples from per-rank shards (evidence.ml:101-107): shard r reports
    n_r and Z_r = n_r / sum_i 1/L_i, so the pooled estimate is (sum n_r) / sum_r (n_r / Z_r), summed in rank order."""
    n, inv = 0.0, 0.0
    for c, z in zip(counts, evidences):
        if c > 0:
            n += float(c)
            inv += float(c) / float(z)
    return n / inv


def harmonic_mean_sharded(log_likelihoods_shard, ctx=None, device=None) -> float:
    """``Evidence.evidence_harmonic_mean`` over samples sharded across ranks: each rank reduces its own shard on
    its GPU, the (count, estimate) pairs are all-gathered and combined in rank order."""
    from . import evidence
    ll = np.asarray(log_likelihoods_shard, dtype=np.float64)
    z = evidence.evidence_harmonic_mean(ll=ll, ctx=ctx) if ll.size else 0.0
    g = all_gather_array(np.array([float(ll.size), z]), device)
    return combine_harmonic(g[:, 0], g[:, 1])


def combine_model_counts(counts_a_b, device=None):
    """``Mcmc.rjmcmc_model_counts`` / ``rjmcmc_evidence_ratio`` (mcmc.ml:141-153) of an ensemble sharded across ranks."""
    g = all_gather_array(np.asarray(counts_a_b, dtype=np.float64), device)
    na, nb = int(g[:, 0].sum()), int(g[:, 1].sum())
    return na, nb, (na / nb if nb else float("inf"))


def broadcast_tree(tree, src: int = 0, ctx=None):
    """Replicate a KdTree built on rank `src` to every rank: one broadcast of
    the serialised device blob (SURVEY.md 8e).  Returns the local KdTree."""
    import torch
    import torch.distributed as dist

    from .kd_tree import KdTree
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size() == 1:
        return tree
    rank = dist.get_rank()
    ctx = ctx or (tree.ctx if tree is not None else None)
    dev = torch.device("cuda", ctx.device)
    nbytes = torch.zeros(1, dtype=torch.int64, device=dev)
    if rank == src:
        p, n = tree.blob()
        nbytes[0] = n
    dist.broadcast(nbytes, src)
    n = int(nbytes.item())
    buf = torch.empty(n, dtype=torch.uint8, device=dev)
    if rank == src:
        import ctypes as C
        ctx.sync()
        ctx.check(ctx.lib.mg_memcpy_d2d(ctx.h, C.c_void_p(buf.data_ptr()), C.c_void_p(p), C.c_int64(n)))
    dist.broadcast(buf, src)
    if rank == src:
        return tree
    torch.cuda.synchronize(dev)
    return KdTree.from_blob(buf.data_ptr(), n, ctx=ctx)


# ---- distributed kd-tree build: the numbering rule of mg_kdtree_build_distributed (csrc/comm.cu) on the host -------------
def tree_levels(left: np.ndarray) -> list[int]:
    """First node of every level (and the node count at the end) of a breadth-first tree with adjacent children:
    the next level ends two past the largest `left` of the level."""
    lb, b, e = [0], 0, 1
    while b < e:
        last = int(left[b:e].max())
        b, e = e, (last + 2 if last >= 0 else e)
        lb.append(b)
    return lb


def graft_subtrees(top: dict, subs: list[dict]) -> dict:
    """``top``: arrays of the tree truncated at 2^k leaves (a complete k-level tree); ``subs[r]``: arrays of the complete
    tree over the rows of leaf r taken in the top's order.  Returns the arrays of the whole tree: level L >= k of the
    whole tree is the ranks' levels L - k side by side, children adjacent; local point ids map back through the top's
    order.  This is what the unpack kernels of ``mg_kdtree_build_distributed`` compute; ``tests/test_distributed_cpu.py``
    checks it against the oracle's own whole tree."""
    R = len(subs)
    assert len(top["left"]) == 2 * R - 1, "the top must be a complete tree with one leaf per rank"
    lbs = [tree_levels(s["left"]) for s in subs]
    maxl = max(len(lb) - 1 for lb in lbs)
    cnt = lambda r, l: (lbs[r][l + 1] - lbs[r][l]) if l + 1 < len(lbs[r]) else 0
    gbase, goff = [R - 1], [[0] * (maxl + 1) for _ in range(R)]
    for l in range(maxl + 1):
        tot = 0
        for r in range(R):
            goff[r][l] = tot
            tot += cnt(r, l)
        gbase.append(gbase[-1] + tot)
    nn = gbase[maxl]
    out = {k: np.empty(nn, top[k].dtype) for k in ("split_dim", "split_val", "left", "begin", "end")}
    for k in out:
        out[k][:R - 1] = top[k][:R - 1]
    perm = np.empty_like(top["perm"])
    for r, s in enumerate(subs):
        pb = int(top["begin"][R - 1 + r])
        lb = lbs[r]
        for l in range(len(lb) - 1):
            i = np.arange(lb[l], lb[l + 1])
            gid = gbase[l] + goff[r][l] + (i - lb[l])
            lf = s["left"][i]
            nxt = lb[l + 1]
            out["left"][gid] = np.where(lf >= 0, gbase[l + 1] + (goff[r][l + 1] if l + 1 <= maxl else 0) + (lf - nxt), -1)
            out["split_dim"][gid], out["split_val"][gid] = s["split_dim"][i], s["split_val"][i]
            out["begin"][gid], out["end"][gid] = pb + s["begin"][i], pb + s["end"][i]
        n_r = int(top["end"][R - 1 + r]) - pb
        perm[pb:pb + n_r] = top["perm"][pb + s["perm"][:n_r]]
    out["perm"] = perm
    return out
