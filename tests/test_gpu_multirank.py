"""GPU, N > 1 on real NCCL: two (or more) ranks extract their z-slabs, all-gather the counts from the device and gather
the mesh to rank 0 through the C ABI's NCCL entry points (ctr_comm_init / ctr_allgather_offsets / ctr_gather_mesh); rank 0
checks the gathered mesh against the single-GPU mesh of the same volume -- the arrays must be identical.
Skipped on a single-GPU box (the gloo tests in test_sharding_gloo.py cover the host logic there)."""
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))


def test_two_ranks_gathered_mesh_equals_single_gpu():
    import torch
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs two GPUs")
    world = 4 if n >= 4 else 2
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(world),
           "--master-addr", "127.0.0.1", "--master-port", "29533", os.path.join(HERE, "multirank_worker.py")]
    p = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert p.returncode == 0, p.stdout[-3000:] + "\n" + p.stderr[-3000:]
    assert "MULTIRANK OK: %d ranks" % world in p.stdout and "MULTIRANK OK (second round)" in p.stdout
