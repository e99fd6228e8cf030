"""Low-rank-corrected (MATLRC) operators on several GPUs: tests/mgpu_lrc_worker.py under torch.distributed.run, one rank
per GPU (4 ranks when there are 4), slab grids and row-partitioned CSR bases, compared with one GPU to 1e-12 relative and
with a second run at the same rank count bitwise.  Needs >= 2 GPUs; skipped on a one-GPU machine."""
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.gpu
def test_multi_gpu_lrc_matches_single_gpu():
    import torch
    ngpu = torch.cuda.device_count()
    if ngpu < 2:
        pytest.skip("needs >= 2 GPUs")
    world = 4 if ngpu >= 4 else 2
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(world), "--master-addr", "127.0.0.1", "--master-port", "29523",
                        os.path.join(ROOT, "tests", "mgpu_lrc_worker.py")], capture_output=True, text=True, timeout=1200)
    print(r.stdout[-4000:])
    assert r.returncode == 0, r.stdout[-6000:] + r.stderr[-6000:]
    assert "FAIL" not in r.stdout and r.stdout.count("-> OK") == 7
