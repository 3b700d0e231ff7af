"""Timing of the ensemble diagnostics (mg_stats_chain_diagnostics_dev, csrc/diagnostics.cu) on the config-2 block.

The block -- 65,536 chains x 10,001 rows x 12 fields, nskip = 1, 62.9 GB -- is generated on the device by
mg_mcmc_array_dev (the headline model of bench.py).  For every maxlag L in --lags (split = 1) the call is warmed up and
timed --reps times: the kernel with CUDA events (mg_ctx_last_kernel_ms brackets the per-sequence kernel) and the whole
call with a host clock (it ends in a synchronise).  Work from shapes: bytes = the block once; FMAs = F M (N L - L(L-1)/2).
The peaks are re-measured in the same process (mg_measure_fp64_tflops, mg_measure_store_gbs) and the card's name and
power limit are recorded beside them.  The HBM bound divides the bytes read by the measured streaming-store rate: the
library has no read microbenchmark, so the read rate is approximated by the store rate.

  python tools/bench_diagnostics.py --out profiles/diagnostics.json [--chains 65536 --steps 10000 --lags 16,64,256]
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except Exception as e:  # noqa: BLE001
        return f"unknown ({e})"


def work(n, F, Cn, L, split=True):
    N = n // 2 if split else n
    M = 2 * Cn if split else Cn
    fma = F * M * (N * L - L * (L - 1) // 2)
    return 8 * n * F * Cn, fma


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--chains", type=int, default=65536)
    ap.add_argument("--steps", type=int, default=10000)
    ap.add_argument("--lags", default="16,64,256")
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
    rec = {"tool": "tools/bench_diagnostics.py", "card": card(), "chains": Cn, "rows": n, "fields": F,
           "block_gb": 8 * n * F * Cn / 1e9, "split": 1, "reps": a.reps,
           "hbm_bound": "bytes read / the measured streaming-store rate (the read rate is approximated by the store "
                        "rate of mg_measure_store_gbs)",
           "fma_bound": "2 F M (N L - L(L-1)/2) flop / the measured FP64 FMA rate of mg_measure_fp64_tflops"}
    with Context(0, 0x5EED0002) as ctx:
        fp64, store = C.c_double(), C.c_double()
        ctx.check(ctx.lib.mg_measure_fp64_tflops(ctx.h, 3, C.byref(fp64)))
        ctx.check(ctx.lib.mg_measure_store_gbs(ctx.h, C.c_int64(8 << 30), 3, C.byref(store)))
        rec["peaks_measured"] = {"fp64_fma_tflops": fp64.value, "store_gbs": store.value}
        state = torch.zeros((F, Cn), dtype=torch.float64, device=dev)
        state[:D] = torch.tensor(mu, device=dev)[:, None]
        blk = torch.empty((n, F, Cn), dtype=torch.float64, device=dev)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        mcmc.mcmc_array_dev(like, prior, prop, nchains=Cn, n=n, nbin=0, nskip=1, state_ptr=state.data_ptr(),
                            samples_ptr=blk.data_ptr(), ctx=ctx)
        ctx.sync()
        rec["sampling_s"] = time.perf_counter() - t0
        seq = torch.empty((F, 2 * Cn), dtype=torch.float64, device=dev)
        rows = []
        for L in [int(v) for v in a.lags.split(",")]:
            r = stats.chain_diagnostics_dev(blk.data_ptr(), n, D, Cn, L, seq_tau_ptr=seq.data_ptr(), ctx=ctx)  # warm-up
            kms, wall = [], []          # CUDA-event kernel times and host-clock call times of every repetition
            for _ in range(a.reps):
                t0 = time.perf_counter()
                stats.chain_diagnostics_dev(blk.data_ptr(), n, D, Cn, L, seq_tau_ptr=seq.data_ptr(), ctx=ctx)
                wall.append(1e3 * (time.perf_counter() - t0))
                kms.append(ctx.last_kernel_ms)
            nbytes, fma = work(n, F, Cn, L)
            k = float(np.median(kms))
            t_mem = nbytes / (store.value * 1e9) * 1e3
            t_fma = 2 * fma / (fp64.value * 1e12) * 1e3
            bound = "hbm" if t_mem >= t_fma else "fp64_fma"
            row = {"maxlag": L, "kernel_ms": kms, "call_ms": wall,
                   "kernel_ms_median": k, "kernel_ms_min": min(kms), "kernel_ms_max": max(kms),
                   "call_ms_median": float(np.median(wall)), "gb_per_s": nbytes / (k * 1e-3) / 1e9,
                   "fp64_tflops": 2 * fma / (k * 1e-3) / 1e12, "bound": bound,
                   "bound_ms": max(t_mem, t_fma), "fraction_of_bound": max(t_mem, t_fma) / k,
                   "rhat": [float(v) for v in r.rhat], "tau": [float(v) for v in r.tau],
                   "seq_tau_median": float(torch.nanmedian(seq[:D]).item())}
            rows.append(row)
            print(json.dumps({kk: v for kk, v in row.items() if kk not in ("rhat", "tau")}), flush=True)
        rec["runs"] = rows
    print(json.dumps({"card": rec["card"], "peaks": rec["peaks_measured"]}), flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            json.dump(rec, fh, indent=1)


if __name__ == "__main__":
    main()
