"""Data-parallel GraphedTrainer (MNF, MF and LRT networks) on 2 GPUs against the single-GPU trainer on the concatenated
minibatch.  Skipped below 2 GPUs.  The checks live in tests/dp_graphed_worker.py: first one plain process computes the
reference, then one process per GPU under torch.distributed.run runs the shards."""
import os
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
WORKER = os.path.join(ROOT, "tests", "dp_graphed_worker.py")


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_data_parallel_graphed_step_equals_single_gpu_step_on_the_concatenated_batch(tmp_path):
    r = subprocess.run([sys.executable, WORKER, "single", "--world", "2", "--out", str(tmp_path)],
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-3000:] + "\n" + r.stderr[-6000:]
    port = 29100 + os.getpid() % 300
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", str(port), WORKER, "dp", "--out", str(tmp_path)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    sys.stdout.write(r.stdout[-4000:])
    assert r.returncode == 0, r.stdout[-3000:] + "\n" + r.stderr[-6000:]
    assert r.stdout.count(" OK, ") == 2 * 7 + 2
