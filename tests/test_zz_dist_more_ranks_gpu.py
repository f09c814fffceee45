"""GPU, boxes with 4 or 8 devices: the sharded render equals the single-GPU render bit for bit at 4 and 8 ranks too
(tests/test_dist_gpu.py runs the same worker at 2 ranks; `bench.py` re-checks bit-identity at whatever N it runs on --
measured true at N = 2 and N = 8).  This worker has not been run on hardware at 4 or 8 ranks yet, so both cases are
xfail(strict=False); the worker runs under torchrun in its own processes."""
import os
import socket
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.xfail(strict=False, reason="this worker has not yet run on hardware at this rank count")
@pytest.mark.parametrize("n", [4, 8])
def test_sharded_render_equals_single_gpu_more_ranks(n):
    if torch.cuda.device_count() < n:
        pytest.skip(f"needs {n} GPUs")
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={n}", "--master-addr", "127.0.0.1",
           "--master-port", str(port), os.path.join(ROOT, "tests", "dist_worker.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, env=dict(os.environ, NCCL_DEBUG="WARN"), cwd=ROOT)
    tail = r.stdout[-3000:] + "\n" + r.stderr[-3000:]
    assert r.returncode == 0 and "DIST_WORKER_OK" in r.stdout, tail
