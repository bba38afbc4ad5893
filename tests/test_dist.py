"""Multi-process tests: world_size 2 on gloo (CPU, host logic) and one rank per GPU on NCCL."""
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _launch(mode, nproc, port):
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(nproc),
           "--master-addr", "127.0.0.1", "--master-port", str(port), os.path.join(ROOT, "tests", "dist_worker.py"), mode]
    return subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=600, cwd=ROOT)


def test_gloo_world2_host_logic():
    r = _launch("cpu", 2, 29631)
    assert r.returncode == 0 and "DIST_CPU_OK" in r.stdout, r.stdout[-3000:]


@pytest.mark.gpu
def test_nccl_root_sharding_and_data_parallel_updates():
    import torch
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs >= 2 GPUs")
    r = _launch("gpu", min(n, 4), 29641)
    assert r.returncode == 0 and "DIST_GPU_OK" in r.stdout, r.stdout[-3000:]
