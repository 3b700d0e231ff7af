#!/usr/bin/env python
"""Multi-GPU check THROUGH THE C ABI (mg_comm_*; torchrun launches one rank per GPU, torch only carries the 128-byte
NCCL id and allocates the test data):
  1. kd-tree built on rank 0, replicated with mg_kdtree_broadcast (one ncclBroadcast of the blob); every rank
     evaluates Interpolate_pdf densities on ITS shard of the queries; the shards are compared bit for bit with
     rank 0's own evaluation of all queries; the broadcast is timed cold and in steady state.
  2. Evidence with the kd-cells shared out (mg_evidence_lebesgue_sharded / _direct_sharded): every rank's result
     must be bit-identical to the single-GPU call on rank 0 (and to the other ranks').
  3. harmonic mean over sharded samples (<= 2 ulp of the single-GPU value).
  4. MH ensemble sharded by global chain id, statistics pooled with mg_comm_pool_moments (1e-12 of the one-rank run).
  5. RJMCMC sharded (mg_rjmcmc_array_sharded): model counts equal to the one-rank run of all chains.
  6. kd-tree built by all ranks together (mg_kdtree_build_distributed): every array equal to the single-GPU tree's on
     every rank; both builds timed.
  7. ensemble diagnostics of the chains of step 4, sharded as there (mg_comm_chain_diagnostics): the same bytes on
     every rank, within 1e-12 of the one-GPU call on all chains.  It runs right after step 4, whose chains it uses.
  8. step 6 on data whose subtree on one rank the second kd-tree builder hands back to the first (a block of
     identical rows), so that the level table of that rank comes from the first builder.
  9. exact quantiles of a seeded block whose chains are shared unevenly over the ranks (mg_comm_quantiles): the same
     bytes on every rank, equal to the single-GPU call on the whole block.
Prints one JSON line on rank 0."""
from __future__ import annotations

import argparse
import json
import math
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--samples", dest="n", type=int, default=2_000_000, help="samples of the evidence / tree test")
    ap.add_argument("--dim", dest="d", type=int, default=8)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import numpy as np
    import torch
    import torch.distributed as dist

    from mcmc_ocaml_b200 import Context, comm as CM, distributed as D, evidence, interpolate_pdf, kd_tree, mcmc, plugins as P
    rank, local, world = int(os.environ.get("RANK", 0)), int(os.environ.get("LOCAL_RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
    if world > 1:
        dist.init_process_group("gloo")          # host-side channel for the NCCL id only
    ctx = Context(local, 2024)
    comm = CM.Comm.from_torch(ctx)
    out = {"world": world}
    import ctypes as C
    ver = C.c_int32()
    if ctx.lib.mg_comm_nccl_version(C.byref(ver)) == 0:
        out["nccl_version"] = ver.value
    # ---- 1. tree broadcast + sharded queries ---------------------------------
    N, Dm, M = a.n, a.d, 1_000_000
    rng = np.random.default_rng(7)
    q = rng.random((M, Dm)) * 0.4 + 0.3
    pts = rng.normal(0.5, 0.08, (N, Dm)).clip(0, 1)
    tree = kd_tree.KdTree(pts, np.zeros(Dm), np.ones(Dm), ctx=ctx) if rank == 0 else None
    times = []
    local_tree = None
    for rep in range(3):
        if local_tree is not None and rank != 0:
            local_tree.close()
        comm.barrier()
        t = time.perf_counter()
        local_tree = comm.broadcast_tree(tree, 0)
        ctx.sync()
        times.append(time.perf_counter() - t)
    nbytes = local_tree.blob()[1]
    out["tree_blob_MB"] = nbytes / 1e6
    out["tree_broadcast_first_s"], out["tree_broadcast_steady_s"] = times[0], min(times[1:])
    out["tree_broadcast_steady_GBps"] = nbytes / min(times[1:]) / 1e9
    out["tree_broadcast_device_ms"] = comm.last_collective_ms
    b, e = D.shard_range(M, rank, world)
    interp = interpolate_pdf.InterpPdf(None, None, None, tree=local_tree)
    mine = interp.jump_prob(q[b:e])
    ok_density = True
    if rank == 0:
        want = interp.jump_prob(q)
    g_ok = comm.allgather(np.array([1.0]))      # keeps the ranks in step
    wants = None
    if world > 1:
        # rank 0 checks every rank's shard: gather the shards through the C ABI (8 MB / rank)
        pad = np.zeros(-(-M // world))
        pad[:e - b] = mine
        allsh = comm.allgather(pad)
        if rank == 0:
            for r in range(world):
                rb, re_ = D.shard_range(M, r, world)
                ok_density &= bool(np.array_equal(allsh[r][:re_ - rb], want[rb:re_]))
    elif rank == 0:
        ok_density = bool(np.array_equal(mine, want))
    out["sharded_density_bit_exact"] = ok_density
    # ---- 2. evidence with the cells shared out ---------------------------------
    sig = 0.08
    ll = (-0.91893853320467274178 - math.log(sig) - 0.5 * ((pts - 0.5) / sig) ** 2).sum(1)
    lp = -0.1 * pts.sum(1)
    if rank == 0:
        tp, tl, tq = torch.as_tensor(pts, device=dev), torch.as_tensor(ll, device=dev), torch.as_tensor(lp, device=dev)
        torch.cuda.synchronize()
        args = (tp.data_ptr(), tl.data_ptr(), tq.data_ptr())
    else:
        args = (0, 0, 0)
    comm.barrier()
    t = time.perf_counter(); zl = comm.evidence_lebesgue(*args, N, Dm, n=64, eps=0.1); t_l = time.perf_counter() - t
    t = time.perf_counter(); zl = comm.evidence_lebesgue(*args, N, Dm, n=64, eps=0.1); t_l = min(t_l, time.perf_counter() - t)
    zd = comm.evidence_direct(*args, N, Dm, n=64)
    both = comm.allgather(np.array([zl, zd]))
    out["lebesgue_sharded"], out["direct_sharded"], out["lebesgue_sharded_s"] = zl, zd, t_l
    out["evidence_identical_on_all_ranks"] = bool(np.all(both == both[0]))
    if rank == 0:
        z1 = evidence.evidence_lebesgue_dev(*args, N, Dm, n=64, eps=0.1, ctx=ctx)
        t = time.perf_counter(); z1 = evidence.evidence_lebesgue_dev(*args, N, Dm, n=64, eps=0.1, ctx=ctx); out["lebesgue_single_s"] = time.perf_counter() - t
        d1 = evidence.evidence_direct_dev(*args, N, Dm, n=64, ctx=ctx)
        out["lebesgue_single"], out["direct_single"] = z1, d1
        out["evidence_bit_identical_to_single_gpu"] = bool(z1 == zl and d1 == zd)
    # ---- 3. harmonic mean, samples sharded ---------------------------------------
    sb, se = D.shard_range(N, rank, world)
    tll = torch.as_tensor(ll[sb:se], device=dev); torch.cuda.synchronize()
    zh = comm.evidence_harmonic_mean(tll.data_ptr(), se - sb)
    if rank == 0:
        zh1 = evidence.evidence_harmonic_mean(ll=ll, ctx=ctx)
        out["harmonic_sharded_rel_err"] = abs(zh - zh1) / abs(zh1)
    # ---- 4. sharded MH ensemble + pooled statistics ------------------------------
    Dd, Cn, n = 10, 4096, 200
    mu = np.arange(Dd) / 10.0
    cov = 0.7 ** np.abs(np.subtract.outer(np.arange(Dd), np.arange(Dd)))
    like, prior, prop = P.gauss_corr(mu, cov), P.zero(Dd), P.box_proposal(np.full(Dd, 0.5))
    cb, ce = D.shard_range(Cn, rank, world)
    ctx.set_seed(99)
    s = mcmc.mcmc_array(n, like, prior, prop, mu, nchains=ce - cb, chain_offset=cb, nbin=20, ctx=ctx)
    pooled = s.block.transpose(0, 2, 1).reshape(-1, Dd + 2)
    ntot, pm, ps = comm.pool_moments(pooled.shape[0], pooled.mean(0), pooled.std(0, ddof=1))
    acc = comm.allgather(np.array([int(s.accept.sum())], dtype=np.int64)).sum()
    if rank == 0:
        ctx.set_seed(99)
        ref = mcmc.mcmc_array(n, like, prior, prop, mu, nchains=Cn, chain_offset=0, nbin=20, ctx=ctx)
        rp = ref.block.transpose(0, 2, 1).reshape(-1, Dd + 2)
        out["ensemble_mean_err"] = float(np.max(np.abs(pm - rp.mean(0))))
        out["ensemble_std_err"] = float(np.max(np.abs(ps - rp.std(0, ddof=1))))
        out["accept_equal"] = bool(int(acc) == int(ref.accept.sum()) and ntot == rp.shape[0])
        out["shard_chains_bit_exact"] = bool(np.array_equal(ref.block[:, :, cb:ce], s.block))
    # ---- 7. ensemble diagnostics of the sharded chains (mg_comm_chain_diagnostics) ----------------
    # every rank diagnoses its own chains; the pooled outputs must be the same bytes on every rank and within 1e-12 of
    # the one-GPU call on all chains
    from mcmc_ocaml_b200 import stats
    dblk = torch.as_tensor(np.ascontiguousarray(s.block), device=dev); torch.cuda.synchronize()
    dgr = comm.chain_diagnostics(dblk.data_ptr(), n, Dd, ce - cb, 32)
    vec = np.concatenate([dgr.rhat, dgr.ess, dgr.tau, dgr.window_closed.astype(np.float64), dgr.rho.ravel()])
    allv = np.asarray(comm.allgather(vec)).reshape(world, -1)
    del dblk
    if rank == 0:
        one = stats.chain_diagnostics(ref.block, 32, ctx=ctx)
        ov = np.concatenate([one.rhat, one.ess, one.tau, one.window_closed.astype(np.float64), one.rho.ravel()])
        out["diagnostics_identical_on_all_ranks"] = bool(all(np.array_equal(allv[r_], allv[0], equal_nan=True)
                                                             for r_ in range(world)))
        out["diagnostics_within_1e12_of_single_gpu"] = bool(np.allclose(vec, ov, rtol=1e-12, atol=1e-12, equal_nan=True))
    # ---- 9. quantiles of chains sharded unevenly (mg_comm_quantiles) ----------------------------------
    # the same seeded block on every rank; rank r holds a share of the chains proportional to r + 1.  The result must be
    # the same bytes on every rank and equal to the single-GPU call on the whole block
    nq_, Dq, Cq = 300, 3, 1537
    xq = np.random.default_rng(1234).standard_normal((nq_, Dq + 2, Cq))
    xq[:, 1] *= 1e-3
    xq[:, 1] += 1e8
    xq[5, 2, 7] = np.nan
    xq[:, 3, :Cq // 2] = 0.5
    edges = [Cq * r_ * (r_ + 1) // (world * (world + 1)) for r_ in range(world + 1)]
    qb, qe = edges[rank], edges[rank + 1]
    probs = [0.0, 0.025, 0.16, 0.5, 0.84, 0.975, 1.0]
    dq = torch.as_tensor(np.ascontiguousarray(xq[:, :, qb:qe]), device=dev); torch.cuda.synchronize()
    qv = comm.quantiles(dq.data_ptr(), nq_, Dq, qe - qb, probs)
    allq = np.asarray(comm.allgather(qv.ravel().view(np.int64))).reshape(world, -1)
    del dq
    if rank == 0:
        one = stats.quantiles(xq, probs, ctx=ctx)
        out["quantiles_identical_on_all_ranks"] = bool(all(np.array_equal(allq[r_], allq[0]) for r_ in range(world)))
        out["quantiles_bit_identical_to_single_gpu"] = bool(np.array_equal(qv.view(np.int64), one.view(np.int64)))
    # ---- 5. sharded RJMCMC over the broadcast tree(s) ----------------------------
    d2 = Dm
    likeA = P.gauss_diag(np.full(d2, 0.5), np.full(d2, 0.08)); priorA = P.box(np.zeros(d2), np.ones(d2), 0.0)
    priorB = P.box(np.zeros(d2), np.ones(d2), -math.log(2.0))
    propA = P.wrap_proposal(np.zeros(d2), np.ones(d2), np.full(d2, 0.05))
    interp_l = interpolate_pdf.InterpPdf(None, None, None, tree=local_tree)
    A = mcmc.RjModel(likeA, priorA, propA, 0.5, interp=interp_l, nstop=64)
    B = mcmc.RjModel(likeA, priorB, propA, 0.5, interp=interp_l, nstop=64)
    a0 = np.full(d2, 0.5)
    ctx.set_seed(4711)
    r = comm.rjmcmc_array(51, A, B, a0, a0, nskip=4, nchains=20000)
    out["rj_counts_sharded"] = list(r.counts); out["rj_cross"] = list(r.cross)
    # ---- 6. distributed kd-tree build (mg_kdtree_build_distributed) ---------------------
    # every rank holds the rows; the top log2(world) levels are built everywhere, the subtrees one per rank, one
    # all-gather; the result must equal the single-GPU tree array for array, on every rank
    dpts = torch.from_numpy(pts).to(dev)
    lo_, hi_ = np.zeros(Dm), np.ones(Dm)
    for ms in (2, 64):
        dt_d, dt_s = [], []
        for rep in range(3):
            comm.barrier(); torch.cuda.synchronize()
            t = time.perf_counter()
            td = comm.build_tree(dpts.data_ptr(), N, Dm, lo_, hi_, min_split=ms)
            ctx.sync(); dt_d.append(time.perf_counter() - t)
            if rep < 2:
                td.close()
        for rep in range(3):
            comm.barrier(); torch.cuda.synchronize()
            t = time.perf_counter()
            ts = kd_tree.KdTree.from_device(dpts.data_ptr(), N, Dm, lo_, hi_, min_split=ms, ctx=ctx)
            ctx.sync(); dt_s.append(time.perf_counter() - t)
            if rep < 2:
                ts.close()
        ad, as_ = td.export(), ts.export()
        same = all(np.array_equal(ad[k_], as_[k_]) for k_ in as_) and td.nnodes == ts.nnodes and td.nlevels == ts.nlevels
        flags = comm.allgather(np.array([1.0 if same else 0.0]))
        out[f"dist_build_ms{ms}"] = dict(identical_to_single_gpu_on_every_rank=bool(flags.min() == 1.0), nnodes=int(td.nnodes),
                                         nlevels=int(td.nlevels), distributed_s=min(dt_d), single_gpu_s=min(dt_s),
                                         speedup=min(dt_s) / min(dt_d))
        td.close(); ts.close()
    # ---- 8. distributed build with one rank's subtree from the first builder ------------------------------------------
    # uniform rows with a block of identical rows at 0.25 (left of the root's split, so on rank 0 only): the node that
    # holds the block sheds only a few rows per level and stays larger than a shared-memory subtree (<= 2048 points)
    # past the second builder's level budget, which hands the input back (MCMC_GPU_DEBUG=1 prints
    # "second builder handed the input back" between the rank's "gather" and "subtree" phases)
    tp = np.random.default_rng(11).random((N, Dm))
    tp[:max(N // 128, 16384)] = 0.25
    dtp = torch.from_numpy(tp).to(dev)
    td = comm.build_tree(dtp.data_ptr(), N, Dm, lo_, hi_, min_split=2)
    ts = kd_tree.KdTree.from_device(dtp.data_ptr(), N, Dm, lo_, hi_, min_split=2, ctx=ctx)
    ad, as_ = td.export(), ts.export()
    same = all(np.array_equal(ad[k_], as_[k_]) for k_ in as_) and td.nnodes == ts.nnodes and td.nlevels == ts.nlevels
    flags = comm.allgather(np.array([1.0 if same else 0.0]))
    out["dist_build_first_builder"] = dict(identical_to_single_gpu_on_every_rank=bool(flags.min() == 1.0),
                                           nnodes=int(td.nnodes), nlevels=int(td.nlevels))
    td.close(); ts.close()
    del dpts, dtp
    if rank == 0:
        ctx.set_seed(4711)
        r1 = mcmc.rjmcmc_array(51, A, B, a0, a0, nskip=4, nchains=20000, record_model=False, ctx=ctx)
        out["rj_counts_single"] = list(r1.counts)
        out["rj_counts_equal"] = bool(tuple(r1.counts) == tuple(r.counts))
        out["ok"] = bool(out["sharded_density_bit_exact"] and out["accept_equal"] and out["shard_chains_bit_exact"]
                         and out["ensemble_mean_err"] < 1e-12 and out["ensemble_std_err"] < 1e-12
                         and out["harmonic_sharded_rel_err"] < 1e-14 and out["evidence_identical_on_all_ranks"]
                         and out["evidence_bit_identical_to_single_gpu"] and out["rj_counts_equal"]
                         and out["diagnostics_identical_on_all_ranks"] and out["diagnostics_within_1e12_of_single_gpu"]
                         and out["quantiles_identical_on_all_ranks"] and out["quantiles_bit_identical_to_single_gpu"]
                         and all(out[f"dist_build_ms{ms}"]["identical_to_single_gpu_on_every_rank"] for ms in (2, 64))
                         and out["dist_build_first_builder"]["identical_to_single_gpu_on_every_rank"])
        s_ = json.dumps(out)
        print(s_)
        if a.out:
            with open(a.out, "w") as f:
                f.write(s_ + "\n")
    comm.barrier()
    comm.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
