"""Parallel-tempering evidence (mg_evidence_tempered) on config 3's model, against the plain dynamic sampler.

Model: 20-D MG_FN_GAUSS_DIAG, N(0.5, 0.05^2) per coordinate, in an MG_FN_BOX_CLOSED prior on the unit box (analytic
log Z = 0 to 1e-20).  Ladder: T = 32, beta_k = (k / 31)^3; per-rung box proposals of half-width
min(0.5, 2.4 sigma / sqrt(beta_k D)) (0.5 at beta_0 = 0); M = 4096 ladders = 131,072 replicas; nbin = 2000,
nsteps = 10000, a swap round after every step.  Each timing is a host clock around a call that ends in a device
synchronise, after one warm-up call; five timed calls.

The like-for-like reference is mg_mcmc_array_dev with no sample block (d_samples = NULL) over C = 131,072 chains of the
same model and step count (one box proposal, the beta = 1 width), timed in the same process the same way.  Both
kernels read almost nothing from HBM: they are bound by instruction issue and FP64.  The card's name and power limit
are read in the same run.

  python tools/bench_tempered.py --out profiles/tempered.json [--ladders 4096 --nsteps 10000 --reps 5]
"""
from __future__ import annotations

import argparse
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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--ladders", type=int, default=4096)
    ap.add_argument("--temps", type=int, default=32)
    ap.add_argument("--nbin", type=int, default=2000)
    ap.add_argument("--nsteps", type=int, default=10000)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()

    import torch
    from scipy.stats import norm

    from mcmc_ocaml_b200 import Context, evidence, mcmc, plugins as P

    D, sigma, T, M = 20, 0.05, a.temps, a.ladders
    like = P.gauss_diag(np.full(D, 0.5), np.full(D, sigma))
    prior = P.box(np.zeros(D), np.ones(D), 0.0)
    betas = (np.arange(T) / (T - 1.0)) ** 3
    hw = [0.5 if b == 0 else min(0.5, 2.4 * sigma / np.sqrt(b * D)) for b in betas]
    props = [P.box_proposal(np.full(D, h)) for h in hw]
    steps = a.nbin + a.nsteps
    x0 = np.random.default_rng(1).uniform(0.0, 1.0, (M, D))
    rec = {"card": card(), "model": "config 3: 20-D gauss_diag sigma 0.05 in the closed unit box", "ladders": M,
           "temps": T, "replicas": M * T, "nbin": a.nbin, "nsteps": a.nsteps, "swap_every": 1,
           "betas": "(k/31)^3", "half_widths": hw}
    print(json.dumps({"card": rec["card"]}), flush=True)
    C = M * T
    with Context(0, 2024) as ctx:
        def tempered():
            return evidence.evidence_tempered(like, prior, props, betas, x0, nladders=M, nbin=a.nbin, nsteps=a.nsteps,
                                              swap_every=1, ctx=ctx)
        state = torch.empty((D + 2, C), dtype=torch.float64, device="cuda:0")

        def plain():
            state[:D].fill_(0.5)
            mcmc.mcmc_array_dev(like, prior, props[-1], nchains=C, n=1, nbin=steps, state_ptr=state.data_ptr(), ctx=ctx)
            torch.cuda.synchronize()

        r = tempered()          # warm-up
        plain()
        tt, tp = [], []
        for _ in range(a.reps):  # alternate the two, so that both see the same state of the card
            t0 = time.perf_counter(); r = tempered(); tt.append(time.perf_counter() - t0)
            t0 = time.perf_counter(); plain(); tp.append(time.perf_counter() - t0)
    rate_t = [C * steps / t for t in tt]
    rate_p = [C * steps / t for t in tp]
    rec.update({
        "tempered_s": tt, "plain_s": tp,
        "tempered_replica_steps_per_s": float(np.median(rate_t)),
        "plain_chain_steps_per_s": float(np.median(rate_p)),
        "ratio_tempered_to_plain": float(np.median(rate_t) / np.median(rate_p)),
        "log_z_ss": r.log_z_ss, "log_z_ss_err": r.log_z_ss_err, "log_z_ti": r.log_z_ti, "log_z_ti_err": r.log_z_ti_err,
        "log_z_exact": float(D * np.log(2.0 * norm.cdf(0.5 / sigma) - 1.0)),
        "swap_acceptance": (r.swaps_accepted / r.swaps_tried).tolist(),
        "mh_acceptance": (r.accept / (M * a.nsteps)).tolist(),
        "mean_ll": r.mean_ll.tolist(), "mean_ll_err": r.mean_ll_err.tolist(),
    })
    print(json.dumps({k: rec[k] for k in ("tempered_replica_steps_per_s", "plain_chain_steps_per_s",
                                           "ratio_tempered_to_plain", "log_z_ss", "log_z_ss_err", "log_z_ti",
                                           "log_z_ti_err")}), flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            json.dump(rec, fh, indent=1)


if __name__ == "__main__":
    main()
