"""The parallel-tempering evidence oracle (oracle/tempered_oracle.cpp) against closed forms, against og_mcmc_array, and its
swap bookkeeping against a hand count; the ABI structs of the call against gcc.

Model: D iid Gaussians N(0.5, sigma^2) under a flat prior on the unit box.  Under pi_beta each coordinate is a normal
of scale sigma / sqrt(beta) truncated to [0, 1] (uniform at beta = 0), so E_beta[ll] is known in closed form, and
log Z = D log(2 Phi(0.5 / sigma) - 1)."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np
import pytest
from scipy.stats import norm

from mcmc_ocaml_b200 import _abi, plugins as P
from oracle import tempered as ot


def box_model(D, sigma):
    like = P.gauss_diag(np.full(D, 0.5), np.full(D, sigma))
    prior = P.box(np.zeros(D), np.ones(D), 0.0)
    return like, prior


def box_props(betas, D, sigma):
    return [P.box_proposal(np.full(D, 0.5 if b == 0 else min(0.5, 2.4 * sigma / np.sqrt(b * D)))) for b in betas]


def exact_mean_ll(beta, D, sigma):
    """E_beta[ll] for the truncated model above"""
    if beta == 0:
        ez2 = 1.0 / 12.0
    else:
        s = sigma / np.sqrt(beta)
        c = 0.5 / s
        ez2 = s * s * (1.0 - 2.0 * c * norm.pdf(c) / (2.0 * norm.cdf(c) - 1.0))
    return D * (-0.91893853320467274178 - np.log(sigma) - 0.5 * ez2 / sigma ** 2)


@pytest.mark.parametrize("D,sigma,T", [(2, 0.1, 8), (5, 0.08, 12)])
def test_oracle_matches_closed_forms(D, sigma, T):
    like, prior = box_model(D, sigma)
    betas = (np.arange(T) / (T - 1.0)) ** 3
    r = ot.evidence_tempered(7, 0, like, prior, box_props(betas, D, sigma), betas, np.full(D, 0.5), nladders=64,
                             nbin=300, nsteps=3000, swap_every=1, nthreads=8)
    want = np.array([exact_mean_ll(b, D, sigma) for b in betas])
    z = (r["mean_ll"] - want) / r["mean_ll_err"]
    print("mean_ll z-scores", np.round(z, 2))
    assert np.all(np.abs(z) < 4.0), z
    log_z = D * np.log(2.0 * norm.cdf(0.5 / sigma) - 1.0)
    print(f"log_z_ss {r['log_z_ss']:.5f} +- {r['log_z_ss_err']:.5f}, exact {log_z:.5f}; log_z_ti {r['log_z_ti']:.5f}")
    assert abs(r["log_z_ss"] - log_z) < 4.0 * r["log_z_ss_err"]
    # TI is the trapezoid over the pooled curve
    ti = sum((betas[k + 1] - betas[k]) * (r["mean_ll"][k] + r["mean_ll"][k + 1]) / 2.0 for k in range(T - 1))
    assert r["log_z_ti"] == ti
    assert np.all(np.isfinite(r["ladder_mean_ll"])) and np.all(r["accept"] > 0) and np.all(r["swaps_accepted"] > 0)


def test_beta_one_rung_is_the_plain_sampler_without_swaps(og):
    """swap_every = 0: the rung at beta = 1 of ladder m is chain m T + T - 1 of og_mcmc_array, draw for draw"""
    D, sigma, T, M, nbin, nsteps = 3, 0.1, 5, 16, 40, 200
    like, prior = box_model(D, sigma)
    betas = np.linspace(0.0, 1.0, T)
    prop = P.box_proposal(np.full(D, 0.1))
    rng = np.random.default_rng(3)
    x0 = rng.uniform(0.3, 0.7, (M, D))
    r = ot.evidence_tempered(11, 4, like, prior, prop, betas, x0, nladders=M, nbin=nbin, nsteps=nsteps, swap_every=0)
    starts = np.repeat(x0, T, axis=0)                       # chain m T + k starts at x0_m
    out, acc, _ = og.mcmc_array(11, 4, 1, like, prior, prop, starts, nbin=nbin + nsteps, nchains=M * T)
    want = out[0].T.reshape(M, T, D + 2)
    assert np.array_equal(r["final"][:, T - 1], want[:, T - 1])
    assert np.all(r["swaps_accepted"] == 0) and np.all(r["swaps_tried"] == 0)


@pytest.mark.parametrize("T,nbin,nsteps,every", [(2, 0, 10, 1), (5, 3, 17, 1), (6, 4, 30, 7), (7, 13, 29, 3), (4, 5, 3, 9)])
def test_swap_bookkeeping_against_a_hand_count(T, nbin, nsteps, every):
    """round r follows step t with (t + 1) % every == 0, r = (t + 1) / every - 1, and tries the pairs k = r (mod 2);
    only the rounds after measured steps (t >= nbin) count"""
    D, M = 2, 3
    like, prior = box_model(D, 0.2)
    betas = np.linspace(0.0, 1.0, T)
    r = ot.evidence_tempered(5, 0, like, prior, P.box_proposal(np.full(D, 0.2)), betas, np.full(D, 0.5), nladders=M,
                             nbin=nbin, nsteps=nsteps, swap_every=every)
    tried = np.zeros(T - 1, np.int64)
    for t in range(nbin, nbin + nsteps):
        if (t + 1) % every == 0:
            rnd = (t + 1) // every - 1
            for k in range(rnd % 2, T - 1, 2):
                tried[k] += M
    assert np.array_equal(r["swaps_tried"], tried)
    assert np.all(r["swaps_accepted"] <= tried)


def test_minus_infinity_at_beta_zero_and_one_ladder():
    """A beta = 0 rung that measures ll = -inf (a prior draw outside the likelihood's support) gives mean_ll[0] and
    log_z_ti = -inf; SS stays finite.  M = 1 gives errors of NaN."""
    D = 1
    like = P.box(np.array([0.25]), np.array([0.75]), 0.0)      # support of L: half the prior's box
    prior = P.box(np.zeros(D), np.ones(D), 0.0)
    betas = np.array([0.0, 0.5, 1.0])
    r = ot.evidence_tempered(2, 0, like, prior, P.box_proposal([0.5]), betas, [0.5], nladders=1, nbin=0, nsteps=400,
                             swap_every=1)
    assert r["mean_ll"][0] == -np.inf and r["log_z_ti"] == -np.inf
    assert np.isfinite(r["log_z_ss"]) and abs(r["log_z_ss"] - np.log(0.5)) < 0.3
    assert np.isnan(r["log_z_ss_err"]) and np.isnan(r["log_z_ti_err"]) and np.isnan(r["mean_ll_err"][2])


def test_tempered_struct_layouts_match_the_header():
    root = os.path.dirname(os.path.dirname(os.path.abspath(_abi.__file__)))
    src = ('#include <stdio.h>\n#include "mcmc_gpu.h"\n'
           'int main(){printf("%zu %zu\\n",sizeof(mg_tempered_cfg),sizeof(mg_tempered_out));return 0;}')
    with tempfile.TemporaryDirectory() as d:
        open(os.path.join(d, "t.c"), "w").write(src)
        subprocess.check_call(["gcc", "-I", os.path.join(root, "include"), os.path.join(d, "t.c"), "-o", os.path.join(d, "t")])
        sizes = list(map(int, subprocess.check_output([os.path.join(d, "t")]).split()))
    assert sizes == [C.sizeof(_abi.mg_tempered_cfg), C.sizeof(_abi.mg_tempered_out)]
