"""Multi-GPU results on hardware (skipped below 2 GPUs): the per-field argmin exchange (NCCL all-gather +
merge kernel) against the numpy rule, and plan_batch(distributed=True) against the single-process result."""
import os
import socket
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu


def test_exchange_and_sharded_plan_batch_on_two_or_more_gpus():
    import torch
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs >= 2 GPUs")
    n = 2 if n < 4 else (4 if n < 8 else 8)
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={n}", "--master-addr",
           "127.0.0.1", "--master-port", str(port), os.path.join(root, "tests", "_multi_gpu_worker.py")]
    # own process group: a timeout must take the ranks down with the launcher (they would keep the GPUs busy)
    p = subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, cwd=root, start_new_session=True)
    try:
        out, err = p.communicate(timeout=300)
    except subprocess.TimeoutExpired:
        import signal
        os.killpg(p.pid, signal.SIGKILL)
        out, err = p.communicate()
        raise AssertionError("multi-GPU worker timed out\n" + out[-2000:] + err[-4000:])
    assert p.returncode == 0 and "MULTI GPU CHECK OK" in out, out[-2000:] + err[-4000:]
