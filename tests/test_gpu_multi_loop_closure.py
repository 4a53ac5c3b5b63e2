"""Loop closure sharded over 2 GPUs (NCCL): needs >= 2 visible GPUs, skipped otherwise."""
import json
import os
import subprocess
import sys

import pytest

from conftest import ROOT

pytestmark = pytest.mark.gpu


def gpu_count():
    import ctypes
    try:
        n = ctypes.c_int(0)
        return n.value if ctypes.CDLL("libcudart.so").cudaGetDeviceCount(ctypes.byref(n)) == 0 else 0
    except OSError:
        import torch
        return torch.cuda.device_count()


@pytest.mark.timeout(900)
def test_sharded_loop_closure_matches_single_gpu(tmp_path):
    if gpu_count() < 2:
        pytest.skip("needs 2 GPUs")
    out = tmp_path / "res.json"
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
           "--master-port", "29657", os.path.join(ROOT, "tests", "helpers", "loop_closure_worker.py"), str(out)]
    p = subprocess.run(cmd, env=dict(os.environ, MASTER_ADDR="127.0.0.1"), capture_output=True, text=True, timeout=880)
    assert p.returncode == 0, p.stderr[-3000:]
    r = json.load(open(out))
    r0, r1 = r["ranks"]
    # Q = 31 over 2 ranks: both ranks return the same records, byte-equal to one GPU closing every loop
    assert r0["sharded"] == r1["sharded"] == r0["single"] == r1["single"]
