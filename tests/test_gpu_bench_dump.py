"""bench.py --dump-outputs on the GPU arm: the files hold the Cholesky factor that the last timed step computed from the
seeded input, as float64 arrays."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dump_outputs_hold_the_llt_factor(cuda_dev, oracle, tmp_path):
    import torch
    n = 2048  # small enough for every column to be written
    env = dict(os.environ)
    env.pop("RANK", None); env.pop("WORLD_SIZE", None)
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "2", "--warmup", "3", "--n", str(n),
                          "--no-e2e", "--no-cpu-baseline", "--dump-outputs", str(tmp_path)],
                         capture_output=True, text=True, timeout=600, env=env, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1])
    assert line["steps"] == 2
    diag = np.load(tmp_path / "llt_factor_diagonal.npy")
    cols = np.load(tmp_path / "llt_factor_columns.npy")
    assert diag.dtype == np.float64 and diag.shape == (n,)
    assert cols.dtype == np.float64 and cols.shape == (n, n)
    assert np.array_equal(np.diag(cols), diag) and not np.triu(cols, 1).any()
    # bench.py's input: A = G G^T + n I with G from torch's generator seeded 1234 on the device
    torch.manual_seed(1234)
    G = torch.randn((n, n), dtype=torch.float64, device=cuda_dev)
    A = np.asfortranarray(torch.addmm(n * torch.eye(n, dtype=torch.float64, device=cuda_dev), G, G.T).cpu().numpy())
    fail, _ = oracle.llt(A)
    assert fail == -1
    assert np.allclose(cols, np.tril(A), rtol=1e-10, atol=1e-10)
