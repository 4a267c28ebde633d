"""lbbnn.vd.EnsemblePredictor(process_group=) against the single-process predictor, injected and native zeta on both GEMM
paths.  A one-rank group on any GPU box, and two ranks (skipped below 2 GPUs).  The checks live in
tests/vd_predict_dp_worker.py (one process per GPU under torch.distributed.run)."""
import os
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.parametrize("world", [1, 2])
def test_sharded_vd_ensemble_equals_single_process_run(world):
    if torch.cuda.device_count() < world:
        pytest.skip(f"needs {world} GPUs")
    port = 29500 + (os.getpid() + 300 + world) % 400
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(world), "--master-addr",
           "127.0.0.1", "--master-port", str(port), os.path.join(ROOT, "tests", "vd_predict_dp_worker.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    sys.stdout.write(r.stdout[-4000:])
    assert r.returncode == 0, r.stdout[-3000:] + "\n" + r.stderr[-6000:]
    assert r.stdout.count(" OK, ") == 4
