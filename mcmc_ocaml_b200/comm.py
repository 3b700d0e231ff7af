"""Host-side wrapper of the multi-GPU entry points of the C ABI (``mg_comm_*``, include/mcmc_gpu.h): one process
per GPU, one NCCL communicator per context.  The collectives themselves (tree broadcast, all-gathers) run inside
libmcmcgpu.so; the host program only has to hand the 128-byte NCCL id from one rank to the others -- here through
``torch.distributed`` (gloo on CPU, NCCL on the GPU box), a file, or any callable."""
from __future__ import annotations

import ctypes as C
import os
import time

import numpy as np

from . import _abi
from .context import Context

ID_BYTES = 128


def exchange_id_torch(make_id, rank: int, src: int = 0) -> bytes:
    """Rank ``src`` calls ``make_id()``; the bytes reach every rank through the default torch process group."""
    import torch
    import torch.distributed as dist
    t = torch.zeros(ID_BYTES, dtype=torch.uint8)
    if rank == src:
        t = torch.frombuffer(bytearray(make_id()), dtype=torch.uint8).clone()
    if dist.get_backend() == "nccl":
        t = t.cuda()
    dist.broadcast(t, src)
    return bytes(t.cpu().numpy().tobytes())


def exchange_id_file(make_id, rank: int, path: str, src: int = 0, timeout: float = 120.0) -> bytes:
    """The same through a file on a shared file system (what an OCaml host without MPI would do)."""
    if rank == src:
        tmp = path + ".tmp"
        with open(tmp, "wb") as f:
            f.write(make_id())
        os.replace(tmp, path)
    t0 = time.time()
    while not os.path.exists(path):
        if time.time() - t0 > timeout:
            raise _abi.Failure(f"comm: no NCCL id appeared at {path}")
        time.sleep(0.01)
    with open(path, "rb") as f:
        return f.read()


class Comm:
    """``mg_comm``: the ranks of one job, one per GPU.  Every method is collective."""

    def __init__(self, ctx: Context, nranks: int, rank: int, unique_id: bytes | None = None):
        self.ctx, self.nranks, self.rank = ctx, int(nranks), int(rank)
        h = C.c_void_p()
        idbuf = (C.c_uint8 * ID_BYTES).from_buffer_copy(unique_id) if unique_id is not None else None
        ctx.check(ctx.lib.mg_comm_create(ctx.h, C.c_int32(nranks), C.c_int32(rank), idbuf, C.byref(h)))
        self.h = h

    @staticmethod
    def make_unique_id() -> bytes:
        buf = (C.c_uint8 * ID_BYTES)()
        if _abi.load_library().mg_comm_get_unique_id(buf) != _abi.MG_OK:
            raise _abi.Failure("nccl: cannot create a unique id (libnccl.so.2 missing?)")
        return bytes(buf)

    @classmethod
    def from_torch(cls, ctx: Context):
        """Ranks and id exchange from the default torch.distributed process group."""
        import torch.distributed as dist
        if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size() == 1:
            return cls(ctx, 1, 0, None)
        rank, world = dist.get_rank(), dist.get_world_size()
        return cls(ctx, world, rank, exchange_id_torch(cls.make_unique_id, rank))

    def close(self):
        if getattr(self, "h", None) and getattr(self.ctx, "h", None):
            self.ctx.lib.mg_comm_destroy(self.h)
        self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def last_collective_ms(self) -> float:
        self.ctx.lib.mg_comm_last_collective_ms.restype = C.c_double
        return float(self.ctx.lib.mg_comm_last_collective_ms(self.h))

    def barrier(self):
        self.ctx.check(self.ctx.lib.mg_comm_barrier(self.h))

    def allgather(self, x: np.ndarray) -> np.ndarray:
        """[nranks, ...] of a small array contributed by every rank."""
        x = np.ascontiguousarray(x)
        out = np.empty((self.nranks,) + x.shape, dtype=x.dtype)
        self.ctx.check(self.ctx.lib.mg_comm_allgather(self.h, x.ctypes.data_as(C.c_void_p), out.ctypes.data_as(C.c_void_p),
                                                      C.c_int64(x.nbytes)))
        return out

    def broadcast_tree(self, tree, root: int = 0):
        """``Interp.make`` on ``root``, the tree replicated on every rank (one NCCL broadcast of the blob)."""
        from .kd_tree import KdTree
        out = C.c_void_p()
        self.ctx.check(self.ctx.lib.mg_kdtree_broadcast(self.h, tree.h if tree is not None else None, C.c_int32(root),
                                                        C.byref(out)))
        if self.rank == root or self.nranks == 1:
            return tree
        return KdTree(None, None, None, ctx=self.ctx, _handle=out)

    def build_tree(self, pts_ptr: int, N: int, D: int, low, high, *, min_split: int = 2):
        """``Kd_tree.tree_of_objects`` built by all ranks together (``mg_kdtree_build_distributed``): ``pts_ptr`` is the
        same [N][D] device array on every rank; every rank receives the whole tree, bit-identical to the one-GPU build."""
        from .kd_tree import KdTree
        low, high = _abi.as_f64(low), _abi.as_f64(high)
        out = C.c_void_p()
        self.ctx.check(self.ctx.lib.mg_kdtree_build_distributed(self.h, C.c_void_p(pts_ptr), C.c_int64(N), C.c_int32(D),
                                                                _abi.ptr(low), _abi.ptr(high), C.c_int32(min_split), C.byref(out)))
        return KdTree(None, None, None, ctx=self.ctx, _handle=out)

    def _evidence(self, fn, root, pts_ptr, ll_ptr, lp_ptr, N, D, n, *extra):
        out = C.c_double()
        self.ctx.check(fn(self.h, C.c_int32(root), C.c_void_p(pts_ptr or 0), C.c_void_p(ll_ptr or 0), C.c_void_p(lp_ptr or 0),
                          C.c_int64(N), C.c_int32(D), C.c_int32(n), *extra, C.byref(out)))
        return out.value

    def evidence_lebesgue(self, pts_ptr, ll_ptr, lp_ptr, N: int, D: int, *, n: int = 64, eps: float = 0.1, root: int = 0) -> float:
        """``Evidence.evidence_lebesgue`` with the kd-cells shared out over the ranks; device pointers on ``root``."""
        return self._evidence(self.ctx.lib.mg_evidence_lebesgue_sharded, root, pts_ptr, ll_ptr, lp_ptr, N, D, n, C.c_double(eps))

    def evidence_direct(self, pts_ptr, ll_ptr, lp_ptr, N: int, D: int, *, n: int = 64, root: int = 0) -> float:
        return self._evidence(self.ctx.lib.mg_evidence_direct_sharded, root, pts_ptr, ll_ptr, lp_ptr, N, D, n)

    def evidence_harmonic_mean(self, ll_shard_ptr, n_shard: int) -> float:
        out = C.c_double()
        self.ctx.check(self.ctx.lib.mg_evidence_harmonic_mean_sharded(self.h, C.c_void_p(ll_shard_ptr or 0), C.c_int64(n_shard),
                                                                      C.byref(out)))
        return out.value

    def rjmcmc_array(self, n: int, A, B, a0, b0, *, nbin: int = 0, nskip: int = 1, nchains: int = 1, chain_offset: int = 0,
                     record_model: bool = False):
        """``Mcmc.rjmcmc_array`` for ``nchains`` chains cut into one contiguous range per rank; the returned counts
        are those of ALL ranks, ``model`` (if recorded) holds this rank's chains."""
        from .mcmc import RjSamples
        base, rem = divmod(nchains, self.nranks)
        mine = base + (1 if self.rank < rem else 0)
        cfg = _abi.mg_rjmcmc_cfg(nchains, nbin, nskip, n, chain_offset, 0, 0)
        model = np.empty((n, mine), np.uint8) if record_model else None
        counts = (C.c_int64 * 2)()
        sa, sb = A.spec(), B.spec()
        a0, b0 = _abi.as_f64(a0), _abi.as_f64(b0)
        if a0.size != A.like.dim or b0.size != B.like.dim:
            raise _abi.InvalidArgument("rjmcmc_array: start points must have the dimensions of their models")
        sb_, sc_ = C.c_int64(), C.c_int64()
        self.ctx.check(self.ctx.lib.mg_rjmcmc_array_sharded(self.h, C.byref(sa), C.byref(sb), C.byref(cfg), _abi.ptr(a0),
                                                            _abi.ptr(b0), _abi.ptr(model, _abi.c_uint8_p), None, counts,
                                                            C.byref(sb_), C.byref(sc_)))
        cp, ca = C.c_int64(), C.c_int64()
        self.ctx.lib.mg_rjmcmc_jump_counters(self.ctx.h, C.byref(cp), C.byref(ca))
        r = RjSamples(model, None, (int(counts[0]), int(counts[1])), (int(cp.value), int(ca.value)))
        r.shard = (int(sb_.value), int(sc_.value))
        return r

    def pool_moments(self, n_local: int, mean_local, std_local):
        """``Stats.multi_mean`` / ``multi_std`` of samples held by several ranks (pooled in rank order)."""
        m, s = _abi.as_f64(mean_local), _abi.as_f64(std_local)
        om, os_ = np.empty_like(m), np.empty_like(s)
        nt = C.c_int64()
        self.ctx.check(self.ctx.lib.mg_comm_pool_moments(self.h, C.c_int64(n_local), _abi.ptr(m), _abi.ptr(s), C.c_int32(m.size),
                                                         C.byref(nt), _abi.ptr(om), _abi.ptr(os_)))
        return int(nt.value), om, os_

    def chain_diagnostics(self, samples_ptr: int, n: int, D: int, nchains_local: int, maxlag: int, *, split: bool = True,
                          seq_tau_ptr: int | None = None):
        """``stats.chain_diagnostics_dev`` over chains sharded across the ranks (this rank's device block
        [n][D+2][C_r]); the pooled outputs are identical on every rank, ``seq_tau_ptr`` gets the local sequences."""
        from . import stats
        cfg = stats._diag_cfg(n, D, nchains_local, maxlag, split)
        outs = stats._diag_outputs(D, maxlag)
        self.ctx.check(stats._diag_call(self.ctx.lib.mg_comm_chain_diagnostics, self.h, C.c_void_p(samples_ptr), cfg,
                                        outs, C.c_void_p(seq_tau_ptr) if seq_tau_ptr else None))
        return stats.ChainDiagnostics(*outs)

    def quantiles(self, samples_ptr: int, n: int, D: int, nchains_local: int, probs) -> np.ndarray:
        """``stats.quantiles_dev`` of the union of every rank's device block [n][D+2][C_r] (same n, D and probs on
        every rank); the result [D+2][nq] is the same bytes on every rank."""
        from . import stats
        p = stats._probs(probs)
        out = np.empty((D + 2, p.size))
        self.ctx.check(self.ctx.lib.mg_comm_quantiles(self.h, samples_ptr, n, D, nchains_local, _abi.ptr(p), p.size,
                                                      _abi.ptr(out)))
        return out
