"""Sample-sharded multi-GPU parity (one rank per GPU, NCCL all-reduce of the partials)."""
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_two_ranks_match_oracle(tmp_path):
    import torch

    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs >= 2 GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
           "--master-addr", "127.0.0.1", "--master-port", "29631", os.path.join(ROOT, "tests", "mg_worker.py")]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    with open(tmp_path / "mg_worker.log", "w") as fh:
        fh.write(out.stdout[-20000:] + "\n--- stderr ---\n" + out.stderr[-5000:])
    assert out.returncode == 0 and "MG_OK" in out.stdout, out.stdout[-3000:] + out.stderr[-3000:]
