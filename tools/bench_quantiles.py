"""Timing of the exact quantiles (mg_stats_quantiles_dev, csrc/quantiles.cu) on the config-2 block.

The block -- 65,536 chains x 10,001 rows x 12 fields, nskip = 1, 62.9 GB -- is generated on the device by
mg_mcmc_array_dev (the headline model of bench.py).  For nq = 1, 5 and 32 (the median; the 2.5 / 16 / 50 / 84 /
97.5 % points; 32 evenly spaced points in [0.01, 0.99]) the call is warmed up and timed --reps times with a host clock
(the call ends in a synchronise: its result is on the host), and the block-pass kernel with CUDA events
(mg_ctx_last_kernel_ms).  One more call under MCMC_GPU_DEBUG=1 counts the full reads of each field (1 when the
brackets resolve it, 9 when it takes the radix-select fallback).  The one-read HBM bound divides the bytes of the block
by the streaming-store rate measured in the same process (mg_measure_store_gbs): the library has no read
microbenchmark, so the read rate is approximated by the store rate.  The card's name and power limit are recorded.

  python tools/bench_quantiles.py --out profiles/quantiles.json [--chains 65536 --steps 10000 --reps 5]
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import re
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

PROBS = {1: [0.5], 5: [0.025, 0.16, 0.5, 0.84, 0.975], 32: list(np.linspace(0.01, 0.99, 32))}


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except Exception as e:  # noqa: BLE001
        return f"unknown ({e})"


def full_reads(call):
    """run call() with MCMC_GPU_DEBUG=1 and stderr captured: the per-field debug lines -> reads per field"""
    os.environ["MCMC_GPU_DEBUG"] = "1"
    sys.stderr.flush()
    saved = os.dup(2)
    with tempfile.TemporaryFile(mode="w+") as fh:
        os.dup2(fh.fileno(), 2)
        try:
            call()
        finally:
            os.dup2(saved, 2)
            os.close(saved)
            del os.environ["MCMC_GPU_DEBUG"]
        fh.seek(0)
        text = fh.read()
    return [int(m.group(2)) for m in re.finditer(r"quantiles: field (\d+): \w+, (\d+) full read", text)]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--chains", type=int, default=65536)
    ap.add_argument("--steps", type=int, default=10000)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    import torch

    from mcmc_ocaml_b200 import Context, mcmc, stats, plugins as P
    D, Cn, n = 10, a.chains, a.steps + 1
    F = D + 2
    mu = np.arange(D) / 10.0
    cov = 0.7 ** np.abs(np.subtract.outer(np.arange(D), np.arange(D)))
    like, prior, prop = P.gauss_corr(mu, cov), P.zero(D), P.box_proposal(np.full(D, 0.5))
    dev = torch.device("cuda", 0)
    nbytes = 8 * n * F * Cn
    rec = {"tool": "tools/bench_quantiles.py", "card": card(), "chains": Cn, "rows": n, "fields": F,
           "block_gb": nbytes / 1e9, "reps": a.reps,
           "hbm_bound": "bytes of the block (one read) / the measured streaming-store rate (the read rate is "
                        "approximated by the store rate of mg_measure_store_gbs)"}
    with Context(0, 0x5EED0002) as ctx:
        store = C.c_double()
        ctx.check(ctx.lib.mg_measure_store_gbs(ctx.h, C.c_int64(8 << 30), 3, C.byref(store)))
        rec["store_gbs_measured"] = store.value
        state = torch.zeros((F, Cn), dtype=torch.float64, device=dev)
        state[:D] = torch.tensor(mu, device=dev)[:, None]
        blk = torch.empty((n, F, Cn), dtype=torch.float64, device=dev)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        mcmc.mcmc_array_dev(like, prior, prop, nchains=Cn, n=n, nbin=0, nskip=1, state_ptr=state.data_ptr(),
                            samples_ptr=blk.data_ptr(), ctx=ctx)
        ctx.sync()
        rec["sampling_s"] = time.perf_counter() - t0
        t_bound = nbytes / (store.value * 1e9) * 1e3
        rows = []
        for nq, probs in PROBS.items():
            def call():
                return stats.quantiles_dev(blk.data_ptr(), n, D, Cn, probs, ctx=ctx)
            q = call()                                      # warm-up
            kms, wall = [], []
            for _ in range(a.reps):
                t0 = time.perf_counter()
                call()
                wall.append(1e3 * (time.perf_counter() - t0))
                kms.append(ctx.last_kernel_ms)
            reads = full_reads(call)
            c = float(np.median(wall))
            row = {"nq": nq, "call_ms": wall, "pass_kernel_ms": kms, "call_ms_median": c,
                   "call_ms_min": min(wall), "call_ms_max": max(wall), "pass_kernel_ms_median": float(np.median(kms)),
                   "full_reads_per_field": reads, "full_reads_total_bytes": 8 * n * Cn * int(sum(reads)),
                   "one_read_bound_ms": t_bound, "fraction_of_one_read_bound": t_bound / c,
                   "pass_kernel_fraction_of_one_read_bound": t_bound / float(np.median(kms)),
                   "quantiles": q.tolist()}
            rows.append(row)
            print(json.dumps({k: v for k, v in row.items() if k != "quantiles"}), flush=True)
        rec["runs"] = rows
    print(json.dumps({"card": rec["card"], "store_gbs": rec["store_gbs_measured"]}), flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            json.dump(rec, fh, indent=1)


if __name__ == "__main__":
    main()
