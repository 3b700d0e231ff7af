"""ctypes binding of oracle/tempered_oracle.cpp (TEST INFRASTRUCTURE): the CPU restatement of mg_evidence_tempered.

The library is compiled on first use, with the flags of oracle/Makefile, into a temporary directory of this process,
so that the tree is never written to."""
from __future__ import annotations

import atexit
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

from mcmc_ocaml_b200 import _abi
from mcmc_ocaml_b200._abi import ptr

_HERE = os.path.dirname(os.path.abspath(__file__))
_lib = None


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        d = tempfile.mkdtemp(prefix="tempered_oracle_")
        atexit.register(shutil.rmtree, d, True)
        so = os.path.join(d, "libtempered_oracle.so")
        subprocess.check_call([os.environ.get("CXX", "g++"), "-O2", "-std=c++17", "-fPIC", "-ffp-contract=off", "-mfma",
                               "-Wall", "-pthread", "-shared", "-o", so, os.path.join(_HERE, "tempered_oracle.cpp")])
        L = C.CDLL(so)
        L.og_tempered_last_error.restype = C.c_char_p
        _lib = L
    return _lib


def evidence_tempered(seed, epoch, like, prior, props, betas, start, *, nladders, nbin, nsteps, swap_every=1,
                      ladder_offset=0, nthreads=1):
    """The definition of include/mcmc_gpu.h ladder by ladder.  props: one proposal or one per rung.  Returns a dict
    of the pooled outputs, the per-ladder means [M][T], the final states [M][T][D+2] and the near-tie margins [M][T]
    (the MH tests of the replica and the swap tests it took part in); swaps_tried is counted, not computed."""
    from mcmc_ocaml_b200.evidence import _tempered_args, _tempered_outputs
    cfg, pa, keep, x0, b = _tempered_args(like, prior, props, betas, start, nladders, nbin, nsteps, swap_every,
                                          ladder_offset)
    res, out = _tempered_outputs(cfg)
    mg = np.full((cfg.nladders, cfg.ntemps), np.inf)
    ls, ps = like.spec(), prior.spec()
    rc = lib().og_evidence_tempered(C.c_uint64(seed), C.c_uint64(epoch), C.byref(ls), C.byref(ps), pa, ptr(b),
                                    C.byref(cfg), ptr(x0), C.byref(out), ptr(mg), C.c_int(nthreads))
    if rc != 0:
        msg = lib().og_tempered_last_error().decode()
        raise _abi.InvalidArgument(msg) if rc == _abi.MG_EINVAL else RuntimeError(msg)
    res.update(log_z_ss=out.log_z_ss, log_z_ss_err=out.log_z_ss_err, log_z_ti=out.log_z_ti,
               log_z_ti_err=out.log_z_ti_err, margins=mg)
    return res
