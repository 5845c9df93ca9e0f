"""Feature-parallel minibatch training on 2 GPUs equals the single-GPU run (needs >= 2 GPUs; skipped otherwise)."""
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def gpu_count():
    try:
        out = subprocess.run(["nvidia-smi", "-L"], capture_output=True, text=True, timeout=30).stdout
        return sum(1 for l in out.splitlines() if l.startswith("GPU "))
    except Exception:
        return 0


@pytest.mark.skipif(gpu_count() < 2, reason="needs 2 GPUs")
def test_feature_parallel_equals_single_gpu():
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29611", os.path.join(ROOT, "tests", "multi_worker.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0 and "MULTI_OK" in r.stdout, r.stdout[-3000:] + r.stderr[-3000:]


@pytest.mark.skipif(gpu_count() < 2, reason="needs 2 GPUs")
def test_row_sharded_als_mcmc_equals_single_gpu():
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29612", os.path.join(ROOT, "tests", "multi_worker_als.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0 and "MULTI_ALS_OK" in r.stdout, r.stdout[-3000:] + r.stderr[-3000:]
