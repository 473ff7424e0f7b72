"""-m gpu, needs >= 2 devices on the box (skipped otherwise): N-rank frame-sharded gradients == 1-rank accumulated
gradients on real GPUs, through NCCL (eager and captured in the CUDA graph) and through the NVLS multicast path."""
import json
import os
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))


def test_sharded_gradients_equal_accumulated_gradients_on_hardware():
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs at least two GPUs")
    world = 2 if n < 4 else 4
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}", "--master-addr", "127.0.0.1",
           "--master-port", "29611", os.path.join(ROOT, "scripts", "multi_gpu_equivalence.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=240, cwd=ROOT)
    assert r.returncode == 0, (r.stdout[-3000:], r.stderr[-3000:])
    line = [l for l in r.stdout.splitlines() if l.startswith("{")][-1]
    out = json.loads(line)
    print(out)
    assert out["ok"] and out["eager_nccl"] < 2e-5 and out["graph_nccl"] < 2e-5
