"""Relocalization with NDT refinement sharded over 2 GPUs (NCCL): needs >= 2 visible GPUs, skipped otherwise."""
import json
import os
import subprocess
import sys

import pytest

from conftest import ROOT
from test_gpu_multi_ndt_pairs import gpu_count

pytestmark = pytest.mark.gpu


@pytest.mark.timeout(900)
def test_sharded_refine_matches_single_gpu(tmp_path):
    if gpu_count() < 2:
        pytest.skip("needs 2 GPUs")
    out = tmp_path / "res.json"
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
           "--master-port", "29673", os.path.join(ROOT, "tests", "helpers", "reloc_refine_worker.py"), "nccl", str(out)]
    p = subprocess.run(cmd, env=dict(os.environ, MASTER_ADDR="127.0.0.1"), capture_output=True, text=True, timeout=880)
    assert p.returncode == 0, p.stderr[-3000:]
    r = [json.load(open(f"{out}.{q}")) for q in range(2)]
    single = r[0]["single"]
    assert single == r[1]["single"] and single["n"] == 8 and single["best"] >= 0
    for name in ("contiguous", "interleaved", "empty"):
        # every rank returns the same code, winner and records, byte-equal to one GPU over the whole grid
        assert r[0]["runs"][name] == r[1]["runs"][name] == single, name
    # a rank passing h > 0 without poses: every rank returns B200_ERR_ARG, nobody hangs
    assert r[0]["null_poses"]["rc"] == r[1]["null_poses"]["rc"] == -1
    assert r[0]["null_poses"]["best"] == r[1]["null_poses"]["best"] == -1
    assert "rank 1" in r[0]["null_poses"]["error"] and "bad argument" in r[1]["null_poses"]["error"]
    assert r[0]["argmin"] == r[1]["argmin"]
