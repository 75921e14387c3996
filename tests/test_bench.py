"""bench.py --dump-outputs: what the last timed step computed, written as .npy files that the dump of another build can be
compared with element for element."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import bench

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dump_samples_large_arrays_at_fixed_positions(tmp_path):
    n = bench.DUMP_MAX_ELEMENTS + 1000
    big, small = torch.arange(n, dtype=torch.float64).reshape(2, -1), torch.arange(6, dtype=torch.int32).reshape(2, 3)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), {"big": big, "small": small})
    a, b = np.load(tmp_path / "a" / "big.npy"), np.load(tmp_path / "b" / "big.npy")
    assert a.dtype == np.float32 and a.shape == (bench.DUMP_MAX_ELEMENTS,)
    assert np.array_equal(a, b)                                     # the same positions in every run
    assert (np.diff(a) > 0).all() and a[0] >= 0 and a[-1] < n        # distinct elements of the array, in flat order
    s = np.load(tmp_path / "a" / "small.npy")
    assert s.dtype == np.float32 and np.array_equal(s, small.numpy())


def _bench_dump(out_dir, B):
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "0", "--batch", str(B),
           "--no-cpu-baseline", "--no-e2e", "--dump-outputs", str(out_dir)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert json.loads(r.stdout.strip().splitlines()[-1])["steps"] == 2
    return {f[:-4]: np.load(out_dir / f) for f in os.listdir(out_dir)}


@pytest.mark.gpu
def test_bench_dumps_the_last_timed_step(tmp_path):
    """R-MG-34 at batch 4: the output, loss, parameters (sampled: 32.9M) and their gradients of the second timed step, the
    same bits in two runs (each autotunes its kernel variants by timing: the choice must not change the result)"""
    B = 4
    d = _bench_dump(tmp_path / "a", B)
    again = _bench_dump(tmp_path / "b", B)
    assert sorted(d) == ["grad_parameters", "loss", "output", "parameters"]
    assert all(np.array_equal(d[k], again[k]) for k in d), "two runs with the same arguments must dump the same values"
    assert all(a.dtype == np.float32 and np.isfinite(a).all() for a in d.values())
    assert sum(a.nbytes for a in d.values()) <= 64 << 20
    assert d["output"].shape == (B, 1000) and d["parameters"].shape == d["grad_parameters"].shape == (bench.DUMP_MAX_ELEMENTS,)
    assert np.allclose(np.exp(d["output"]).sum(1), 1, atol=1e-2)     # log-probabilities
    # the loss is the mean NLL of the dumped log-probabilities on bench.py's seeded labels: both from the same step
    g = torch.Generator(device="cpu").manual_seed(100)
    torch.randn(B, 3, 224, 224, generator=g)
    t = torch.randint(1, 1001, (B,), generator=g).numpy()
    assert np.isclose(d["loss"][0], -d["output"][np.arange(B), t - 1].mean(), rtol=1e-3, atol=1e-4)
