"""bench.py --dump-outputs: what the timed SpMV computed, written so that two builds can be compared
output for output."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import bench

ROOT = os.path.normpath(os.path.join(os.path.dirname(__file__), ".."))


def test_dump_outputs_full_or_fixed_sample(tmp_path):
    small = np.random.default_rng(0).standard_normal(1000)
    bench.dump_outputs(str(tmp_path / "small"), small)
    assert np.array_equal(np.load(tmp_path / "small" / "y.npy"), small)
    # one element over the limit: a sample of fixed rows, the same from call to call, in row order
    big = np.arange(bench.DUMP_MAX_BYTES // 8 + 1, dtype=np.float64)
    bench.dump_outputs(str(tmp_path / "a"), big)
    bench.dump_outputs(str(tmp_path / "b"), big)
    a, b = np.load(tmp_path / "a" / "y.npy"), np.load(tmp_path / "b" / "y.npy")
    assert a.dtype == np.float64 and a.size == bench.DUMP_SAMPLE_ROWS and a.nbytes <= bench.DUMP_MAX_BYTES
    assert np.array_equal(a, b) and np.all(np.diff(a) > 0)


@pytest.mark.gpu
def test_bench_dump_is_the_timed_spmv(tmp_path):
    """y.npy of the b200 arm equals the oracle's product of the bench matrix (host twin of the device
    generator, same seed) and the bench's x, and the JSON line reports the requested step count."""
    import torch

    from oracle import oracle

    n, k = 200_000, 50
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--rows", str(n), "--nnz-per-row", str(k), "--steps", "3",
           "--warmup", "1", "--no-extras", "--dump-outputs", str(tmp_path)]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-3000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["steps"] == 3 and line["warmup"] == 1
    y = np.load(tmp_path / "y.npy")
    assert y.dtype == np.float64 and y.shape == (n,)
    g = torch.Generator(device="cuda")
    g.manual_seed(1)
    x = torch.rand(n, dtype=torch.float64, device="cuda", generator=g).cpu().numpy()
    p, c, v = oracle.random_csr(n, n, n * k, bench.SEED)
    want = oracle.spmv(p, c, v, x)
    assert np.linalg.norm(y - want) / np.linalg.norm(want) < 1e-10
