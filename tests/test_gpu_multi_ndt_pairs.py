"""Batched NDT pair registration sharded over 2 GPUs (NCCL): needs >= 2 visible GPUs, skipped otherwise."""
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
def test_sharded_pairs_match_single_gpu(tmp_path):
    if gpu_count() < 2:
        pytest.skip("needs 2 GPUs")
    out = tmp_path / "res.json"
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
           "--master-port", "29653", os.path.join(ROOT, "tests", "helpers", "ndt_pairs_worker.py"), str(out)]
    p = subprocess.run(cmd, env=dict(os.environ, MASTER_ADDR="127.0.0.1"), capture_output=True, text=True, timeout=880)
    assert p.returncode == 0, p.stderr[-3000:]
    r = json.load(open(out))
    r0, r1 = r["ranks"]
    # P = 37 over 2 ranks: both ranks return the same records, bit-identical to one GPU registering every pair
    assert r0["sharded"] == r1["sharded"] == r0["single"] == r1["single"]
    # a pair that fails on its owner (rank 1) is reported in its own status on every rank; the rest is unchanged
    assert r0["bad"] == r1["bad"]
    assert r0["bad"]["status"][3] == -1
    assert [h for i, h in enumerate(r0["bad"]["records"]) if i != 3] == [h for i, h in enumerate(r0["single"]) if i != 3]
