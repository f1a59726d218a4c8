"""Row-sharded training over REAL ranks (one process per GPU, NVLink peer memory + NCCL): launched with
torchrun when the machine has >= 2 GPUs (skipped on a single GPU; logs of 2- and 8-GPU runs in
profiles/).  The script compares against the CPU oracle on the global batch (tools/dist_sharded_check.py)."""
import os
import subprocess
import sys

import pytest
import torch

from conftest import ROOT

pytestmark = pytest.mark.gpu


def _ngpus():
    return torch.cuda.device_count() if torch.cuda.is_available() else 0


@pytest.mark.parametrize("model", ["DeepFM", "DLRM"])
@pytest.mark.parametrize("precision", ["fp32", "tf32x3"])
def test_sharded_training_matches_the_oracle_on_real_ranks(model, precision):
    n = _ngpus()
    if n < 2:
        pytest.skip("needs >= 2 GPUs")
    world = 8 if n >= 8 else (4 if n >= 4 else 2)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(world),
           "--master-addr", "127.0.0.1", "--master-port", "29611", os.path.join(ROOT, "tools", "dist_sharded_check.py"),
           "--model", model, "--precision", precision]
    r = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True, timeout=600)
    sys.stdout.write(r.stdout[-3000:])
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
