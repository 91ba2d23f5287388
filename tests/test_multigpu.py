"""Multi-process parity: sharded BA across ranks == oracle. One GPU per rank over NCCL when the box has them; otherwise both
ranks share GPU 0 (gloo process group, CUDA-IPC mappings of a second process on the same device, cooperative grids limited to
a share of the SMs) - the same multi-process code path, so the test never skips."""
import os
import socket
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.gpu
def test_sharded_ba_matches_oracle_across_processes():
    import torch
    env = dict(os.environ)
    if torch.cuda.device_count() < 2:
        env["SE2GPU_BA_PK_GRID"] = "70"
        env["SE2GPU_BA_PEER_TIMEOUT_S"] = "60"
    with socket.socket() as s:          # a port nobody else on the host holds
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
           "--master-port", str(port), os.path.join(ROOT, "tests", "mgpu_ba_check.py")]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=900, env=env)
    assert res.returncode == 0, res.stdout[-3000:] + res.stderr[-3000:]
    assert "MISMATCH" not in res.stdout
    assert res.stdout.count("-> OK") == 4, res.stdout[-2000:]
