"""The kd-tree blob (csrc/kdtree.cuh) as both builders write it: header, section offsets and size, the contents of the
root-box and point sections, and a round trip through mg_kdtree_from_blob_dev."""
import ctypes as C

import numpy as np
import pytest

from mcmc_ocaml_b200 import kd_tree
from tests.test_kdtree_gpu import assert_same_tree

pytestmark = pytest.mark.gpu

# KdHeader: magic, N, nnodes, nbytes, D, nlevels, min_split, pad, off_low .. off_pts
HEADER = np.dtype([("magic", "<u8"), ("N", "<i8"), ("nnodes", "<i8"), ("nbytes", "<i8"), ("D", "<i4"),
                   ("nlevels", "<i4"), ("min_split", "<i4"), ("pad", "<i4"), ("off", "<i8", 7)])
KD_MAGIC = 0x6b64747265653031
HANDED_BACK = "second builder handed the input back"


def expected_layout(N, D, nnodes):
    """offsets of low, high, nodes, count, begin, perm, pts and the blob size: every section 256-byte aligned"""
    up = lambda x: (x + 255) // 256 * 256
    off, offs = up(HEADER.itemsize), []
    for size in (8 * D, 8 * D, 16 * nnodes, 4 * nnodes, 4 * nnodes, 4 * N, 8 * N * D):
        offs.append(off)
        off = up(off + size)
    return offs, off


def d2h(ctx, ptr, nbytes):
    out = np.empty(nbytes, np.uint8)
    ctx.check(ctx.lib.mg_memcpy_d2h(ctx.h, out.ctypes.data_as(C.c_void_p), C.c_void_p(ptr), C.c_int64(nbytes)))
    return out


def tie_heavy():
    """90 % of every coordinate is 0.0, the rest scaled by 10^(8 - d): the zeros tie, so the largest node of level 7
    still holds ~9,600 points, more than a subtree of the second builder takes at D = 8 (2,048) at the last level
    it tries (4 + 3)"""
    rng = np.random.default_rng(0)
    P = rng.random((20000, 8))
    for d in range(8):
        zero = np.zeros(20000, bool)
        zero[rng.permutation(20000)[:18000]] = True
        P[zero, d] = 0.0
        P[~zero, d] *= 10.0 ** (8 - d)
    return P


@pytest.mark.parametrize("case", ["random", "truncated", "ties"])
def test_blob_layout(ctx, og, monkeypatch, capfd, case):
    if case == "ties":
        P, min_split = tie_heavy(), 2
    else:
        P, min_split = np.random.default_rng(5).random((5000, 7)), (2 if case == "random" else 64)
    N, D = P.shape
    lo, hi = P.min(0) - 0.25, P.max(0) + 0.25
    monkeypatch.setenv("MCMC_GPU_DEBUG", "1")
    capfd.readouterr()
    t = kd_tree.KdTree(P, lo, hi, min_split=min_split, ctx=ctx)
    # which builder wrote the blob: the tie-heavy input must reach the first one, the others stay with the second
    assert (HANDED_BACK in capfd.readouterr().err) == (case == "ties")
    o = og.Tree(P, lo, hi, min_split=min_split)
    assert_same_tree(t, o)

    p, nbytes = t.blob()
    h = d2h(ctx, p, HEADER.itemsize).view(HEADER)[0]
    offs, size = expected_layout(N, D, t.nnodes)
    assert nbytes == size == h["nbytes"]
    assert [int(x) for x in h["off"]] == offs
    assert (int(h["magic"]), h["N"], h["nnodes"], h["D"], h["nlevels"], h["min_split"]) == \
        (KD_MAGIC, N, t.nnodes, D, t.nlevels, min_split)
    blob = d2h(ctx, p, nbytes)
    section = lambda i, n: blob[offs[i]:offs[i] + 8 * n].view("<f8")
    assert np.array_equal(section(0, D), lo) and np.array_equal(section(1, D), hi)
    assert np.array_equal(section(6, N * D), P.ravel())

    r = kd_tree.KdTree.from_blob(p, nbytes, ctx=ctx)
    assert_same_tree(r, o)
    assert np.array_equal(d2h(ctx, r.blob()[0], nbytes), blob)
