"""bench.py --dump-outputs: what the timed path computed, written so that two builds can be compared value for value."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402


def _load(d):
    return {f[:-4]: np.load(os.path.join(d, f)) for f in sorted(os.listdir(d))}


@pytest.mark.parametrize("n,Cn", [(11, 300), (1001, 200_000)])
def test_dump_outputs_samples_within_budget(tmp_path, n, Cn):
    F = bench.D + 2
    g = torch.Generator().manual_seed(0)
    state = torch.randn(F, Cn, dtype=torch.float64, generator=g)
    # the [n][F][C] block as a view of n * F + C values: slot (s, f, c) holds base[s * F + f + c], so the large case
    # (over DUMP_CHAINS and over DUMP_BYTES; 19 GB if it were dense) needs no more host memory than the small one
    base = torch.randn(n * F + Cn, dtype=torch.float64, generator=g)
    samples = base.as_strided((n, F, Cn), (F, 1, 1))
    accept = torch.arange(Cn, dtype=torch.int32)
    bench.dump_outputs(str(tmp_path / "a"), state, samples, accept)
    bench.dump_outputs(str(tmp_path / "b"), state, samples, accept)
    a, b = _load(str(tmp_path / "a")), _load(str(tmp_path / "b"))
    assert set(a) == {"final_state", "final_state_chain", "accept", "samples", "samples_slot"}
    assert all(np.array_equal(a[k], b[k]) for k in a)
    assert all(v.dtype == np.float64 for v in a.values())
    assert sum(os.path.getsize(tmp_path / "a" / (k + ".npy")) for k in a) <= 64_000_000
    ch = a["final_state_chain"].astype(np.int64)
    assert len(ch) == min(Cn, bench.DUMP_CHAINS) and np.all(np.diff(ch) > 0)
    assert np.array_equal(a["final_state"], state.numpy()[:, ch])
    assert np.array_equal(a["accept"], ch.astype(np.float64))
    slot = a["samples_slot"].astype(np.int64)
    assert len(np.unique(slot[:, 0] * Cn + slot[:, 1])) == len(slot) > 0
    assert np.array_equal(a["samples"], base.numpy()[slot[:, :1] * F + np.arange(F) + slot[:, 1:]])
    if n * Cn * (F + 2) * 8 <= bench.DUMP_BYTES // 2:
        assert len(slot) == n * Cn                     # a small block is written whole


@pytest.mark.gpu
def test_bench_dump_outputs_repeat_and_follow_steps(tmp_path):
    """Two runs with the same arguments write identical outputs; one more timed step changes them."""
    def run(name, steps):
        d = str(tmp_path / name)
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(steps),
                            "--warmup", "1", "--chains", "2048", "--chain-steps", "100", "--no-cpu", "--no-evidence",
                            "--no-rjmcmc", "--dump-outputs", d], capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
        assert json.loads(r.stdout.strip().splitlines()[-1])["steps"] == steps
        return _load(d)

    a, b, c = run("a", 2), run("b", 2), run("c", 3)
    assert a["samples"].shape == (101 * 2048, bench.D + 2) and a["final_state"].shape == (bench.D + 2, 2048)
    assert all(np.array_equal(a[k], b[k]) for k in a)
    assert np.all(np.isfinite(a["samples"])) and a["accept"].max() > 0
    assert not np.array_equal(a["final_state"], c["final_state"])
