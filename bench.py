#!/usr/bin/env python
"""bench.py -- BASELINE.json's metric on B200: chain-steps/s and evidence samples/s at 1/2/4/8 GPUs, next to the
reference's CPU path timed on the box's host cores.

Headline workload ("step" = one pass of the hot path over one batch), BASELINE.json config 2: 65,536 independent
Metropolis-Hastings chains per GPU on a 10-D correlated Gaussian (mu_i = i/10, Sigma_ij = 0.7^|i-j|), box proposal
h = 0.5, flat prior, 10,000 steps per chain, every step recorded (nskip = 1) into a [n][D+2][C] float64 sample block
in HBM (62.9 GB per pass per GPU).  Weak scaling: every rank runs its own 65,536 chains with global chain ids.

  value       device-resident: state and sample block live in HBM, one kernel per pass.
  e2e         the C-ABI call mg_mcmc_array_resident with HOST buffers (pinned start points in; final states,
              counters and Stats mean / std of the 6.6e8 recorded samples out; the block stays in HBM for the GPU
              consumers that follow it); `e2e.mcmc_array_host` adds the plain Mcmc.mcmc_array-shaped call whose
              samples all return to the host (nskip = 100).
  evidence    the metric's second half, config 3: Weinberg (Lebesgue) kd-tree evidence of 1e7 synthetic 20-D
              posterior samples -- device-resident value, roofline of its dominant kernel, host-buffer e2e, CPU
              baseline; with --gpus N the kd-cells are shared out over the ranks (mg_evidence_lebesgue_sharded).
  rjmcmc      config 5 (2-D vs 4-D): kd-trees of 1e7 posterior draws built on rank 0, replicated with one NCCL
              broadcast each (mg_kdtree_broadcast), 1M reversible-jump chains shared out over the ranks.
  --impl reference   the CPU restatement of the OCaml reference (oracle/; no OCaml toolchain exists in this image)
              on all host threads, on a bounded sample of the headline workload.
  --dump-outputs DIR  what the last timed step of the headline workload computed (final states, accept counters, a
              seeded sample of the sample block) as .npy files, so that two builds can be compared output for output.
              Only rank 0's chains are written, and nothing of the evidence or rjmcmc legs.
Every multi-GPU step goes through the C ABI's communicator (mg_comm_*, NCCL); torch.distributed only launches the
ranks, carries the 128-byte NCCL id and takes the max of the timings.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import math
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

D = 10
NCHAINS = 65536
NSTEPS = 10000          # steps per chain per pass; n = NSTEPS + 1 samples, nskip = 1
SEED = 0x5EED0001
BYTES_PER_STEP = 8 * (D + 2)   # SURVEY.md 8d: one recorded sample per chain-step at nskip = 1
EV_N, EV_D = 10_000_000, 20    # config 3
DUMP_BYTES = 60_000_000        # --dump-outputs: data bytes of all files together (64 MB less room for the .npy headers)
DUMP_CHAINS = 65536            # --dump-outputs: chains whose final state and counter are written
DUMP_SEED = 20240601           # --dump-outputs: the chains and slots sampled from larger outputs


def model():
    from mcmc_ocaml_b200 import plugins as P
    mu = np.arange(D) / 10.0
    cov = 0.7 ** np.abs(np.subtract.outer(np.arange(D), np.arange(D)))
    return mu, P.gauss_corr(mu, cov), P.zero(D), P.box_proposal(np.full(D, 0.5))


def workload_config(Cn=NCHAINS, T=NSTEPS):
    n, F = T + 1, D + 2
    return {"workload": f"cfg2: {Cn} independent MH chains per GPU, {D}-D correlated Gaussian "
                        f"(Sigma_ij=0.7^|i-j|), box proposal h=0.5, {T} steps each, nskip=1, "
                        f"every sample recorded ([n][D+2][C] f64, {n * F * Cn * 8 / 1e9:.1f} GB/pass)",
            "chains_per_gpu": Cn, "dim": D, "steps_per_chain": T, "nskip": 1,
            "l2": "outputs (62.9 GB/pass) far exceed the 126 MB L2; no flush needed",
            "rng": "Philox4x32-10, 52 private bits per draw, 11 draws from 5 blocks (5 blocks per 10-D step)",
            "stores": "recorded samples leave through the TMA: one cp.async.bulk.tensor.3d store per 4 samples of a warp"}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return json.load(f), "measured"
    return {"hbm_gbs": 6650.0}, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.stop_flag, self.t = index, [], threading.Event(), None

    def _run(self):
        while not self.stop_flag.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                      "-i", str(self.index)], capture_output=True, text=True, timeout=5).stdout
                self.rows.append([x.strip() for x in out.strip().split(",")])
            except Exception:
                pass
            self.stop_flag.wait(0.1)

    def start(self):
        self.t = threading.Thread(target=self._run, daemon=True)
        self.t.start()

    def stop(self):
        self.stop_flag.set()
        if self.t:
            self.t.join(timeout=6)
        sm, mx, reasons = [], 0.0, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx = max(mx, float(r[1]))
                for nm, v in zip(names, r[2:6]):
                    if v.lower().startswith("active"):
                        reasons.add(nm)
            except Exception:
                continue
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx or None,
                "reasons": sorted(reasons), "samples": len(sm)}


def kernel_stats(ctx):
    """(name, launches, mean ms) of the dominant kernel of the last call: CUDA events around every launch, in the
    library (mg_ctx_last_kernel_stats)."""
    buf = C.create_string_buffer(512)
    n, ms = C.c_int64(), C.c_double()
    ctx.lib.mg_ctx_last_kernel_stats(ctx.h, buf, C.c_int64(512), C.byref(n), C.byref(ms))
    return buf.value.decode(), int(n.value), float(ms.value)


def traffic_of(kernel_name):
    """dram bytes per launch from the round's committed `ncu --set full` capture, only if it is of THIS kernel."""
    p = os.path.join(ROOT, "profiles", "r02", "ncu_traffic.json")
    try:
        rec = json.load(open(p))
        for r in rec.get("kernels", []):
            if kernel_name.startswith(r["kernel_prefix"]):
                return r["dram_bytes_per_launch"], r.get("source")
    except Exception:
        pass
    return None, None


def dump_outputs(path, state, samples, accept):
    """Writes what the timed call (mg_mcmc_array_dev) hands its caller after the last timed step, as float64 .npy
    files, so that two builds run with the same arguments can be compared value for value:
      final_state [D+2][k]  coordinates, log-likelihood and log-prior of k chains (all of them up to DUMP_CHAINS,
                            else a seeded sample), chain ids in final_state_chain [k]
      accept      [k]       accepted steps of the same chains over the warm-up and timed calls
      samples     [m][D+2]  a seeded sample of m (step, chain) slots of the [n][D+2][C] sample block, filling what is
                            left of DUMP_BYTES; step and chain of each row in samples_slot [m][2]."""
    import torch
    n, F, Cn = samples.shape
    rng = np.random.default_rng(DUMP_SEED)
    chains = np.arange(Cn) if Cn <= DUMP_CHAINS else np.sort(rng.choice(Cn, DUMP_CHAINS, replace=False))
    ci = torch.from_numpy(chains).to(state.device)
    out = {"final_state": state[:, ci], "final_state_chain": chains, "accept": accept[ci]}
    left = DUMP_BYTES - 8 * len(chains) * (F + 2)
    m = min(n * Cn, max(0, left // (8 * (F + 2))))
    slots = np.sort(rng.choice(n * Cn, m, replace=False))
    step, chain = slots // Cn, slots % Cn
    out["samples"] = samples[torch.from_numpy(step).to(state.device), :, torch.from_numpy(chain).to(state.device)]
    out["samples_slot"] = np.stack([step, chain], axis=1)
    os.makedirs(path, exist_ok=True)
    for name, a in out.items():
        a = a.cpu().numpy() if isinstance(a, torch.Tensor) else a
        np.save(os.path.join(path, name + ".npy"), np.ascontiguousarray(a, dtype=np.float64))


def cpu_reference(nthreads, target_seconds=12.0):
    """Time the CPU restatement on a bounded sample of the workload."""
    from oracle import oracle as og
    mu, like, prior, prop = model()
    og.lib()
    c0, n0 = max(nthreads * 4, 8), 201
    t = time.perf_counter()
    og.mcmc_array(SEED, 0, n0, like, prior, prop, mu, nchains=c0, nthreads=nthreads, record=False)
    dt = time.perf_counter() - t
    rate = c0 * (n0 - 1) / dt
    steps = NSTEPS    # the sample keeps the real chain length (1e4 steps) and bounds the number of chains
    chains = int(max(nthreads, min(NCHAINS, rate * target_seconds / steps)))
    chains = max(nthreads, (chains // nthreads) * nthreads)
    t = time.perf_counter()
    og.mcmc_array(SEED, 1, steps + 1, like, prior, prop, mu, nchains=chains, nthreads=nthreads, record=True)
    dt = time.perf_counter() - t
    return chains * steps / dt, f"{chains} chains x {steps} steps of the same model, samples recorded, {nthreads} threads"


def evidence_data_host(N, Dd, seed=12345):
    rng = np.random.default_rng(seed)
    x = rng.normal(0.5, 0.05, (N, Dd))
    ll = (-0.91893853320467274178 - math.log(0.05) - 0.5 * ((x - 0.5) / 0.05) ** 2).sum(1)
    return x, ll, np.zeros(N)


def cpu_evidence_baseline(budget_s=25.0):
    """The oracle's evidence_lebesgue (single thread: the reference is single-threaded and its list-based kd-tree
    cannot be run in parallel) at growing N x 20 until the time budget; the figure at 1e7 is an EXTRAPOLATION."""
    from oracle import oracle as og
    rows, t_used = [], 0.0
    for N in (10_000, 100_000, 1_000_000):
        x, ll, lp = evidence_data_host(N, EV_D)
        t = time.perf_counter()
        og.evidence_lebesgue(x, ll, lp, n=64, eps=0.1)
        dt = time.perf_counter() - t
        rows.append({"N": N, "seconds": dt, "samples_per_s": N / dt})
        t_used += dt
        if t_used > budget_s:
            break
    last = rows[-1]
    # cost ~ N log2 N: scale the largest measured run to 1e7
    scale = (EV_N * math.log2(EV_N)) / (last["N"] * math.log2(last["N"]))
    return {"value": last["samples_per_s"], "unit": "evidence samples/s", "cores": 1, "kind": "port",
            "sample": f"oracle evidence_lebesgue (n=64, eps=0.1) on {last['N']} x {EV_D} samples of the same distribution, 1 thread",
            "runs": rows,
            "extrapolated_1e7_seconds": last["seconds"] * scale,
            "extrapolated_1e7_samples_per_s": EV_N / (last["seconds"] * scale),
            "note": "C++ restatement of farr/mcmc-ocaml (oracle/), not OCaml; the 1e7 figure is an N log N extrapolation"}


def run_reference(args, rank, world):
    if rank != 0:
        return
    nthreads = os.cpu_count() or 1
    vals, sample = [], ""
    per_step = max(2.0, min(12.0, 120.0 / max(1, args.steps + args.warmup)))
    for _ in range(args.warmup):
        cpu_reference(nthreads, per_step)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        v, sample = cpu_reference(nthreads, per_step)
        vals.append(v)
    wall = time.perf_counter() - t0
    v = float(np.mean(vals))
    out = {
        "impl": "reference", "metric": "chain-steps/sec", "value": v, "unit": "chain-steps/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * wall / max(1, args.steps),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(args.chains, args.chain_steps),
        "cpu_baseline": {"value": v, "unit": "chain-steps/s", "cores": nthreads, "kind": "port", "sample": sample,
                         "note": "C++ restatement of farr/mcmc-ocaml (oracle/), not OCaml: no OCaml toolchain here; "
                                 "each step is a bounded sample of the workload in `config`"},
        "e2e": {"value": v, "unit": "chain-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    if not args.no_evidence:
        out["evidence"] = {"cpu_baseline": cpu_evidence_baseline(20.0)}
    print(json.dumps(out))


# ---------------------------------------------------------------------------------------------------------------------
def leg_evidence(args, ctx, comm, dev, rank, world, peak):
    """config 3: Lebesgue evidence of EV_N x EV_D samples held by rank 0."""
    import torch
    import torch.distributed as dist

    from mcmc_ocaml_b200 import evidence
    N, Dd = args.ev_n, EV_D
    out = {"workload": f"cfg3: Weinberg (Lebesgue) kd-tree evidence (n=64, eps=0.1) + harmonic mean of {N} synthetic "
                       f"{Dd}-D posterior samples (x ~ N(0.5, 0.05^2 I), ll = log_multi_gaussian, lp = 0)",
           "metric": "evidence samples/s", "N": N, "D": Dd, "n_gpus": world}
    if rank == 0:
        g = torch.Generator(device=dev); g.manual_seed(12345)
        x = torch.empty((N, Dd), dtype=torch.float64, device=dev).normal_(0.5, 0.05, generator=g)
        ll = (-0.91893853320467274178 - math.log(0.05) - 0.5 * ((x - 0.5) / 0.05) ** 2).sum(1)
        lp = torch.zeros(N, dtype=torch.float64, device=dev)
        torch.cuda.synchronize(dev)
        ptrs = (x.data_ptr(), ll.data_ptr(), lp.data_ptr())
    else:
        ptrs = (0, 0, 0)

    def call():
        if world > 1:
            return comm.evidence_lebesgue(*ptrs, N, Dd, n=64, eps=0.1, root=0)
        return evidence.evidence_lebesgue_dev(*ptrs, N, Dd, n=64, eps=0.1, ctx=ctx)

    def sync_all():
        if world > 1:
            comm.barrier()
        ctx.sync()

    for _ in range(2):
        z = call()
    reps, ts = 5, []
    l0 = ctx.launch_count
    for _ in range(reps):
        sync_all(); t = time.perf_counter(); z = call(); ctx.sync(); ts.append(time.perf_counter() - t)
    launches = (ctx.launch_count - l0) // reps
    kname, kn, kms = kernel_stats(ctx)
    tt = torch.tensor([float(np.mean(ts))], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    mean_s = float(tt.item())
    out.update({"value": N / mean_s, "unit": "evidence samples/s", "seconds": mean_s, "best_seconds": float(np.min(ts)),
                "lebesgue_Z": z, "gpu_launches_per_call": int(launches),
                "scaling": "strong (one data set: sort and prefix cut on rank 0, survivors broadcast, kd-tree built by all ranks together, kd-cells shared out)" if world > 1 else "n/a"})
    if world > 1:
        # the kd-tree of the same rows built by all ranks together (mg_kdtree_build_distributed): every rank holds the rows
        g2 = torch.Generator(device=dev); g2.manual_seed(12345)
        xr = x if rank == 0 else torch.empty((N, Dd), dtype=torch.float64, device=dev).normal_(0.5, 0.05, generator=g2)
        torch.cuda.synchronize(dev)
        lo_, hi_ = np.zeros(Dd), np.ones(Dd)
        tb = []
        for rep in range(4):
            sync_all(); t = time.perf_counter()
            trd = comm.build_tree(xr.data_ptr(), N, Dd, lo_, hi_)
            ctx.sync(); tb.append(time.perf_counter() - t)
            nn_, nl_ = trd.nnodes, trd.nlevels
            trd.close()
        tt2 = torch.tensor([float(np.min(tb[1:]))], dtype=torch.float64, device=dev)
        dist.all_reduce(tt2, op=dist.ReduceOp.MAX)
        out["kdtree_distributed_build"] = {"seconds": float(tt2.item()), "points_per_s": N / float(tt2.item()), "nodes": int(nn_),
                                           "levels": int(nl_), "note": "full tree (min_split 2) of the same rows, returned on every rank; "
                                                                        "bit-identical to the one-GPU tree (tools/multi_gpu_check.py)"}
        del xr
    if rank == 0:
        # roofline of the dominant kernel: SURVEY.md 8d, one level of a row-permuting build moves (2*8*D + 16) N bytes
        per_launch = (2 * 8 * Dd + 16) * N
        ach = per_launch / (kms * 1e-3) / 1e9 if kms > 0 else None
        tr, tr_src = traffic_of(kname)
        out["roofline"] = {"bound": "hbm", "kernel": kname, "launches_per_call": kn, "kernel_ms": kms,
                           "bytes_per_launch": per_launch, "bytes_per_sample_per_level": 2 * 8 * Dd + 16,
                           "achieved": ach, "peak": peak, "unit": "GB/s", "frac": (ach / peak) if ach else None,
                           "traffic": tr, "traffic_source": tr_src,
                           "whole_call_frac_of_hbm": ((2 * 8 * Dd + 16) * N * 18 + 8 * (Dd + 2) * N) / mean_s / 1e9 / peak,
                           "whole_call_bytes": "SURVEY 8d: 18 levels x (2*8*D+16) N + one 8 (D+2) N pass"}
        if world == 1:
            # the other estimators and the Interpolate_pdf kernels on the same data
            t = time.perf_counter(); zh = evidence.evidence_harmonic_mean_dev(ptrs[1], N, ctx=ctx); out["harmonic_s"] = time.perf_counter() - t
            evidence.evidence_direct_dev(*ptrs, N, Dd, n=64, ctx=ctx)
            t = time.perf_counter(); zd = evidence.evidence_direct_dev(*ptrs, N, Dd, n=64, ctx=ctx); out["direct_s"] = time.perf_counter() - t
            out["direct_Z"], out["harmonic_Z"] = zd, zh
            from mcmc_ocaml_b200 import kd_tree
            lo, hi = np.zeros(Dd), np.ones(Dd)
            kd_tree.KdTree.from_device(ptrs[0], N, Dd, lo, hi, ctx=ctx).close()
            t = time.perf_counter(); tr_ = kd_tree.KdTree.from_device(ptrs[0], N, Dd, lo, hi, ctx=ctx); out["kdtree_full_build_s"] = time.perf_counter() - t
            out["kdtree_nodes"], out["kdtree_levels"] = tr_.nnodes, tr_.nlevels
            out["kdtree_full_frac_of_hbm"] = ((2 * 8 * Dd + 16) * N * 25) / out["kdtree_full_build_s"] / 1e9 / peak
            tr_.close()
            # e2e: the C-ABI call with pinned HOST buffers (1.76 GB host -> device inside the timed region)
            xh = torch.empty((N, Dd), dtype=torch.float64).pin_memory(); xh.copy_(x)
            llh = torch.empty(N, dtype=torch.float64).pin_memory(); llh.copy_(ll)
            lph = torch.zeros(N, dtype=torch.float64).pin_memory()
            torch.cuda.synchronize(dev)
            zc = C.c_double()

            def host_call():
                ctx.check(ctx.lib.mg_evidence_lebesgue(ctx.h, C.c_void_p(xh.data_ptr()), C.c_void_p(llh.data_ptr()),
                                                       C.c_void_p(lph.data_ptr()), C.c_int64(N), C.c_int32(Dd), C.c_int32(64),
                                                       C.c_double(0.1), C.byref(zc)))
            host_call()
            te = []
            for _ in range(3):
                t = time.perf_counter(); host_call(); te.append(time.perf_counter() - t)
            out["e2e"] = {"value": N / float(np.mean(te)), "unit": "evidence samples/s", "seconds": float(np.mean(te)),
                          "h2d_bytes_per_step": N * (Dd + 2) * 8, "d2h_bytes_per_step": 8,
                          "call": "mg_evidence_lebesgue with pinned host pts / ll / lp", "same_result": bool(zc.value == z)}
            del xh, llh, lph
        del x, ll, lp
        torch.cuda.empty_cache()
    if world > 1:
        # weak scaling next to it: every rank integrates ITS OWN data set of N samples (e.g. one model per GPU), no
        # collective on the data path; value = world * N / slowest rank
        g2 = torch.Generator(device=dev); g2.manual_seed(1000 + rank)
        x2 = torch.empty((N, Dd), dtype=torch.float64, device=dev).normal_(0.5, 0.05, generator=g2)
        ll2 = (-0.91893853320467274178 - math.log(0.05) - 0.5 * ((x2 - 0.5) / 0.05) ** 2).sum(1)
        lp2 = torch.zeros(N, dtype=torch.float64, device=dev)
        torch.cuda.synchronize(dev)
        for _ in range(2):
            evidence.evidence_lebesgue_dev(x2.data_ptr(), ll2.data_ptr(), lp2.data_ptr(), N, Dd, n=64, eps=0.1, ctx=ctx)
        tw = []
        for _ in range(3):
            sync_all(); t = time.perf_counter()
            evidence.evidence_lebesgue_dev(x2.data_ptr(), ll2.data_ptr(), lp2.data_ptr(), N, Dd, n=64, eps=0.1, ctx=ctx)
            ctx.sync(); tw.append(time.perf_counter() - t)
        tt = torch.tensor([float(np.mean(tw))], dtype=torch.float64, device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        if rank == 0:
            out["weak"] = {"value": world * N / float(tt.item()), "unit": "evidence samples/s", "seconds": float(tt.item()),
                           "scaling": "weak (one data set of N samples per rank, no data-path collective)"}
        del x2, ll2, lp2
        torch.cuda.empty_cache()
    ctx.trim_pool()
    return out


def leg_rjmcmc(args, ctx, comm, dev, rank, world):
    """config 5 at (2,4)-D: trees on rank 0, one broadcast each, chains shared out."""
    import torch
    import torch.distributed as dist

    from mcmc_ocaml_b200 import interpolate_pdf, kd_tree, mcmc, plugins as P
    chains, steps, ntree, s = args.rj_chains, 1000, args.rj_ntree, 0.05
    out = {"workload": f"cfg5: {chains} two-model RJMCMC chains x {steps} steps (2-D vs 4-D isotropic Gaussian posteriors, "
                       f"Z_A / Z_B = 2), interpolated jumps from kd-trees of {ntree} posterior draws each",
           "metric": "chain-steps/s", "n_gpus": world}
    models, bcast, builds = [], [], []
    for d, logc in ((2, 0.0), (4, -math.log(2.0))):
        tree = None
        if rank == 0:
            g = torch.Generator(device=dev); g.manual_seed(d)
            pts = torch.empty((ntree, d), dtype=torch.float64, device=dev).normal_(0.5, s, generator=g).clamp_(0.0, 1.0)
            torch.cuda.synchronize(dev)
            kd_tree.KdTree.from_device(pts.data_ptr(), ntree, d, np.zeros(d), np.ones(d), ctx=ctx).close()   # warm (pool growth)
            t = time.perf_counter()
            tree = kd_tree.KdTree.from_device(pts.data_ptr(), ntree, d, np.zeros(d), np.ones(d), ctx=ctx)
            builds.append(time.perf_counter() - t)
            del pts
        if world > 1:
            tms = []
            local = None
            for rep in range(3):            # first broadcast warms NCCL up; steady state = the later ones
                if local is not None and rank != 0:
                    local.close()
                comm.barrier(); t = time.perf_counter()
                local = comm.broadcast_tree(tree, 0); ctx.sync()
                tms.append(time.perf_counter() - t)
            nbytes = local.blob()[1]
            bcast.append({"blob_GB": nbytes / 1e9, "first_s": tms[0], "steady_s": min(tms[1:]),
                          "steady_GBps": nbytes / min(tms[1:]) / 1e9, "device_ms": comm.last_collective_ms})
            tree = local
        interp = interpolate_pdf.InterpPdf(None, None, None, tree=tree)
        like = P.gauss_diag(np.full(d, 0.5), np.full(d, s))
        prior = P.box(np.zeros(d), np.ones(d), logc)
        prop = P.wrap_proposal(np.zeros(d), np.ones(d), np.full(d, 2.0 * s / math.sqrt(d)))
        models.append(mcmc.RjModel(like, prior, prop, 0.5, interp=interp))
    A, B = models
    a0, b0 = np.full(2, 0.5), np.full(4, 0.5)
    ctx.set_seed(20111104)
    comm.rjmcmc_array(2, A, B, a0, b0, nskip=10, nchains=chains)          # warm-up
    ts = []
    for rep in range(2):
        ctx.set_seed(20111104)
        if world > 1:
            comm.barrier()
        t = time.perf_counter()
        r = comm.rjmcmc_array(steps // 10 + 1, A, B, a0, b0, nskip=10, nchains=chains)
        ts.append(time.perf_counter() - t)
    tt = torch.tensor([min(ts)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    sec = float(tt.item())
    out.update({"value": chains * steps / sec, "unit": "chain-steps/s", "seconds": sec, "kernel_ms_this_rank": ctx.last_kernel_ms,
                "counts": list(r.counts), "ratio": r.counts[0] / max(1, r.counts[1]), "expected_ratio": 2.0,
                "cross_model_accept_rate": r.cross[1] / max(1, r.cross[0]), "scaling": "strong (chains shared out)",
                "tree_build_s_rank0": builds, "tree_broadcast": bcast})
    for m in models:
        if m.interp is not None and m.interp.tree is not None:
            m.interp.tree.close()
    ctx.trim_pool()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--chains", type=int, default=NCHAINS)
    ap.add_argument("--chain-steps", type=int, default=NSTEPS)
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline legs")
    ap.add_argument("--no-evidence", action="store_true", help="skip the config-3 evidence leg")
    ap.add_argument("--no-rjmcmc", action="store_true", help="skip the config-5 reversible-jump leg")
    ap.add_argument("--ev-n", type=int, default=EV_N)
    ap.add_argument("--rj-chains", type=int, default=1_000_000)
    ap.add_argument("--rj-ntree", type=int, default=10_000_000)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed to DIR/<name>.npy (rank 0; see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist

    from mcmc_ocaml_b200 import Context, _abi, comm as CM

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    mu, like, prior, prop = model()
    Cn, T = args.chains, args.chain_steps
    n, F = T + 1, D + 2
    ctx = Context(local_rank, SEED)
    stream = torch.cuda.Stream(dev)      # a real (non-NULL) stream shared by torch and the library
    torch.cuda.set_stream(stream)
    ctx.set_stream(stream.cuda_stream)   # time with torch events on the launching stream
    lib = ctx.lib
    comm = CM.Comm.from_torch(ctx)       # the C ABI's own NCCL communicator (id carried by torch.distributed)

    # device-resident buffers (sized for 180 GB HBM: 62.9 GB sample block)
    state = torch.empty((F, Cn), dtype=torch.float64, device=dev)
    state[:D] = torch.tensor(mu, dtype=torch.float64, device=dev)[:, None]
    samples = torch.empty((n, F, Cn), dtype=torch.float64, device=dev)
    accept = torch.zeros(Cn, dtype=torch.int32, device=dev)
    cfg = _abi.mg_mcmc_cfg(Cn, D, 0, 0, 1, n, rank * Cn, 0, 0)
    ls, ps, js = like.spec(), prior.spec(), prop.spec()

    def step_dev():
        ctx.check(lib.mg_mcmc_array_dev(ctx.h, C.byref(ls), C.byref(ps), C.byref(js), C.byref(cfg),
                                        C.c_void_p(state.data_ptr()), C.c_void_p(samples.data_ptr()),
                                        C.c_void_p(accept.data_ptr())))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    sampler = ClockSampler(local_rank)
    for _ in range(args.warmup):
        step_dev()
    barrier()
    if rank == 0:
        sampler.start()
    l0 = ctx.launch_count
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    marks = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
    e0.record(stream)
    marks[0].record(stream)
    for i in range(args.steps):
        step_dev()
        marks[i + 1].record(stream)
    e1.record(stream)
    barrier()
    total_ms = e0.elapsed_time(e1)
    launches = ctx.launch_count - l0
    # average launch duration of the dominant kernel: CUDA events on the launching stream around every launch of
    # the timed region (torch events here, the library's own events around the last launch as a cross-check)
    k_ms = float(np.mean([marks[i].elapsed_time(marks[i + 1]) for i in range(args.steps)]))
    k_name, k_n, k_ms_lib = kernel_stats(ctx)
    t = torch.tensor([total_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms = float(t.item())
    clocks = sampler.stop() if rank == 0 else None
    ms_per_step = total_ms / args.steps
    value = Cn * T * world / (ms_per_step * 1e-3)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, state, samples, accept)   # before the e2e calls below overwrite the block

    # ---- e2e: C-ABI call with host buffers -------------------------------
    x0 = torch.empty((Cn, D), dtype=torch.float64).pin_memory()
    x0[:] = torch.tensor(mu, dtype=torch.float64)
    final = torch.empty((Cn, F), dtype=torch.float64).pin_memory()
    acc_h = torch.empty(Cn, dtype=torch.int64).pin_memory()
    rej_h = torch.empty(Cn, dtype=torch.int64).pin_memory()
    mean_h = np.empty(F); std_h = np.empty(F)
    cfg_e = _abi.mg_mcmc_cfg(Cn, D, 0, 0, 1, n, rank * Cn, 0, 0)

    def step_e2e():
        ctx.check(lib.mg_mcmc_array_resident(
            ctx.h, C.byref(ls), C.byref(ps), C.byref(js), C.byref(cfg_e), C.c_void_p(x0.data_ptr()),
            C.c_void_p(samples.data_ptr()), C.c_void_p(final.data_ptr()), C.c_void_p(acc_h.data_ptr()),
            C.c_void_p(rej_h.data_ptr()), _abi.ptr(mean_h), _abi.ptr(std_h)))

    e2e_warm = min(args.warmup, 2)
    for _ in range(e2e_warm):
        step_e2e()
    barrier()
    t0 = time.perf_counter()
    e0.record(stream)
    for _ in range(args.steps):
        step_e2e()      # returns after its D2H copies completed
    e1.record(stream)
    barrier()
    e2e_ms = max(e0.elapsed_time(e1), 1e3 * (time.perf_counter() - t0))
    e2e_kernel_ms = ctx.last_kernel_ms   # the sampler launch inside the last call (library events)
    t = torch.tensor([e2e_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_ms = float(t.item())
    e2e_value = Cn * T * world / (e2e_ms / args.steps * 1e-3)
    h2d = Cn * D * 8
    d2h = Cn * F * 8 + Cn * 4 + 2 * F * 8

    # statistics of the whole job, gathered through the C ABI (ncclAllGather inside mg_comm_*)
    ntot, pmean, pstd = comm.pool_moments(n * Cn, mean_h, std_h)
    accs = comm.allgather(np.array([float(acc_h.sum()), float(rej_h.sum())]))
    rates = [float(a / (a + r)) for a, r in accs]

    # ---- e2e of the plain Mcmc.mcmc_array-shaped call: every recorded sample returns to the host --------------------
    host_e2e = None
    if world == 1 and Cn == NCHAINS:
        n_h, nskip_h = T // 100 + 1, 100
        out_h = torch.empty((n_h, F, Cn), dtype=torch.float64).pin_memory()
        cfg_h = _abi.mg_mcmc_cfg(Cn, D, 0, 0, nskip_h, n_h, 0, 0, 0)

        def step_host():
            ctx.check(lib.mg_mcmc_array(ctx.h, C.byref(ls), C.byref(ps), C.byref(js), C.byref(cfg_h), C.c_void_p(x0.data_ptr()),
                                        C.c_void_p(out_h.data_ptr()), C.c_void_p(acc_h.data_ptr()), C.c_void_p(rej_h.data_ptr())))
        step_host()
        th = []
        for _ in range(3):
            t0 = time.perf_counter(); step_host(); th.append(time.perf_counter() - t0)
        host_e2e = {"value": Cn * (n_h - 1) * nskip_h / float(np.mean(th)), "unit": "chain-steps/s", "seconds": float(np.mean(th)),
                    "call": f"mg_mcmc_array, nskip={nskip_h}, n={n_h}: pinned x0 in, all {n_h} x {F} x {Cn} recorded values out",
                    "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": n_h * F * Cn * 8 + 2 * Cn * 8,
                    "sampler_kernel_ms_last_segment": ctx.last_kernel_ms,
                    "note": "the run is cut into 8 segments; segment k's samples leave on a second stream while segment k + 1 computes"}
        del out_h

    out = None
    peaks, peak_kind = measured_peaks()
    peak = float(peaks.get("hbm_gbs", 6650.0))
    if rank == 0:
        achieved = BYTES_PER_STEP * Cn * T / (k_ms * 1e-3) / 1e9
        traffic, traffic_src = traffic_of(k_name)
        fp64 = C.c_double(0.0)
        store = C.c_double(0.0)
        lib.mg_measure_fp64_tflops(ctx.h, 3, C.byref(fp64))
        lib.mg_measure_store_gbs(ctx.h, C.c_int64(8 << 30), 3, C.byref(store))
        out = {
            "metric": "chain-steps/sec", "value": value, "unit": "chain-steps/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": workload_config(Cn, T),
            "e2e": {"value": e2e_value, "unit": "chain-steps/s", "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": d2h, "ms_per_step": e2e_ms / args.steps, "sampler_kernel_ms_in_call": e2e_kernel_ms,
                    "call": "mg_mcmc_array_resident: pinned x0 -> device, MH kernel (per-chain running moments kept in "
                            "registers), sample block stays in HBM, Stats mean/std pooled from the chain moments, "
                            "final states + counters + stats -> host",
                    "mcmc_array_host": host_e2e},
            "gpu_launches": int(launches),
            "clocks": clocks,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic, "traffic_source": traffic_src, "peak_source": f"{peak_kind} hbm_gbs (burst copy)",
                         "kernel": k_name, "kernel_source": "mg_ctx_last_kernel_stats (cudaFuncGetName of the launched function)",
                         "kernel_ms": k_ms, "kernel_ms_last_launch_lib_events": k_ms_lib, "bytes_per_chain_step": BYTES_PER_STEP,
                         "store_only_peak_gbs": store.value, "fp64_fma_tflops_measured": fp64.value,
                         "fp64_flops_per_chain_step": D * D + 8 * D + 3,
                         "fp64_tflops_achieved": (D * D + 8 * D + 3) * Cn * T / (k_ms * 1e-3) / 1e12},
            "accept_rate_per_rank": rates,
            "pooled_samples": ntot,
            "posterior_mean_err_max": float(np.max(np.abs(pmean[:D] - mu))),
            "posterior_std_err_max": float(np.max(np.abs(pstd[:D] - 1.0))),
        }
    # ---- the other half of the metric and config 5, at the same number of GPUs ----------------------------------------
    del samples, state
    torch.cuda.empty_cache()
    ctx.trim_pool()
    ctx.reserve_pool()
    if not args.no_evidence:
        try:
            ev = leg_evidence(args, ctx, comm, dev, rank, world, peak)
            if rank == 0:
                out["evidence"] = ev
        except Exception as e:  # the headline line must still be printed
            if rank == 0:
                out["evidence"] = {"error": repr(e)}
    if not args.no_rjmcmc:
        try:
            rj = leg_rjmcmc(args, ctx, comm, dev, rank, world)
            if rank == 0:
                out["rjmcmc"] = rj
        except Exception as e:
            if rank == 0:
                out["rjmcmc"] = {"error": repr(e)}
    if rank == 0:
        if world == 1 and not args.no_cpu:
            nthreads = os.cpu_count() or 1
            v, sample = cpu_reference(nthreads, 12.0)
            out["cpu_baseline"] = {"value": v, "unit": "chain-steps/s", "cores": nthreads, "kind": "port",
                                   "sample": sample,
                                   "note": "C++ restatement of farr/mcmc-ocaml (oracle/), not OCaml"}
            if "evidence" in out and "error" not in out["evidence"]:
                out["evidence"]["cpu_baseline"] = cpu_evidence_baseline(20.0)
        print(json.dumps(out))
    comm.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
