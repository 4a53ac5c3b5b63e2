"""Relocalization with NDT refinement (b200_reloc_refine) without a device: the two-exchange protocol over 2 gloo ranks against a
single-process computation, the ctypes mirror of the candidate record, argument checking and the C++ adaptor's build."""
import ctypes
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT, have_gpu

ERR_ARG = -1


@pytest.mark.timeout(600)
def test_two_rank_gloo_refine_protocol(tmp_path):
    out = tmp_path / "res.json"
    env = dict(os.environ, MASTER_ADDR="127.0.0.1", OMP_NUM_THREADS="2")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
           "--master-port", "29671", os.path.join(ROOT, "tests", "helpers", "reloc_refine_worker.py"), "gloo", str(out)]
    p = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=580)
    assert p.returncode == 0, p.stderr[-3000:]
    r = [json.load(open(f"{out}.{q}")) for q in range(2)]
    single = r[0]["single"]
    assert single == r[1]["single"] and len(single["candidates"]) == 8
    assert single["status"] == 0   # the scene's best starts converge
    for name in ("contiguous", "interleaved", "empty"):
        for q in range(2):
            run = r[q]["runs"][name]
            assert run["candidates"] == single["candidates"], (name, q)       # merged top K in (score desc, index asc) order
            assert run["dealt"] == [j for j in range(8) if j % 2 == q], (name, q)   # candidate j refined on rank j mod 2
            assert run["refined"] == single["refined"], (name, q)
            assert (run["status"], run["best"]) == (single["status"], single["best"]), (name, q)
    assert r[1]["runs"]["empty"]["n_local"] == 0
    assert r[0]["runs"]["contiguous"]["n_local"] == 38 and r[1]["runs"]["contiguous"]["n_local"] == 37
    # a rank that fails on its own makes every rank return its error
    assert r[0]["failing_rank"] == r[1]["failing_rank"] == dict(status=-1, best=-1)


def test_protocol_single_rank_order_and_edges(api):
    one = lambda t: t[None]
    poses = np.stack([np.eye(4, dtype=np.float32).T.reshape(16)] * 6)
    poses[:, 12] = np.arange(6)                    # x translation = local index: refine() recognises the candidate by its pose
    poses[4, 13] = np.nan                          # a non-finite pose never qualifies, whatever its score
    scores = np.array([0.5, 0.9, np.nan, 0.9, 2.0, -1.0])

    def refiner(status, tp):
        return lambda pose16: (status, tp[int(pose16[12])], 0.0)
    # 0.9 twice (ties: lower index first), then 0.5 and -1.0; the NaN score and the NaN pose are dropped
    out = api.reloc_refine_protocol_host(scores, poses, 10, 1, 8, 1, 0, one, refiner(0, {0: 0.3, 1: 0.7, 3: 0.7, 5: 0.1}))
    assert [c[0] for c in out["candidates"]] == [11, 13, 10, 15]
    assert out["dealt"] == [0, 1, 2, 3]
    assert (out["status"], out["best"]) == (0, 11)  # equal probabilities: the lower hypothesis wins
    # top_k below the number of finite scores; none converged: the highest probability and NOT_CONVERGED
    out = api.reloc_refine_protocol_host(scores, poses, 10, 1, 2, 1, 0, one, refiner(2, {1: 0.1, 3: 0.5}))
    assert [c[0] for c in out["candidates"]] == [11, 13] and (out["status"], out["best"]) == (2, 13)
    # no hypothesis at all
    out = api.reloc_refine_protocol_host(np.zeros(0), np.zeros((0, 16), np.float32), 0, 1, 4, 1, 0, one, refiner(0, {}))
    assert (out["status"], out["best"], out["candidates"]) == (1, -1, [])


def test_candidate_layout_matches_the_c_struct(api, tmp_path):
    """The ctypes RelocCandidate has the size and field offsets gcc gives b200_reloc_candidate (the header compiles as C99)."""
    src = tmp_path / "layout.c"
    fields = ["hypothesis", "initial_score", "refined"]
    body = ['printf("size %zu\\n", sizeof(b200_reloc_candidate));']
    body += [f'printf("{f} %zu\\n", offsetof(b200_reloc_candidate, {f}));' for f in fields]
    src.write_text('#include <stddef.h>\n#include <stdio.h>\n#include "b200reg.h"\nint main(void) {\n' + "\n".join(body) + "\nreturn 0;\n}\n")
    exe = tmp_path / "layout"
    p = subprocess.run(["gcc", "-std=c99", "-Wall", "-Wextra", "-pedantic", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)],
                       capture_output=True, text=True)
    assert p.returncode == 0, p.stderr
    got = dict(line.split() for line in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.splitlines())
    assert int(got["size"]) == ctypes.sizeof(api.RelocCandidate) == 480
    for f in fields:
        assert int(got[f]) == getattr(api.RelocCandidate, f).offset, f


def test_refine_bad_arguments_are_rejected(api):
    lib = api.lib()
    res = (api.RelocCandidate * 4)()
    best, nc = ctypes.c_int64(0), ctypes.c_int64(0)
    poses = np.zeros((2, 16), np.float32)
    p = poses.ctypes.data_as(ctypes.c_void_p)
    refine = lib.b200_reloc_refine
    assert refine(None, None, p, 2, 0, 1, 4, 1.0, ctypes.byref(best), res, ctypes.byref(nc), None) == ERR_ARG   # no handle
    assert b"bad argument" in lib.b200_last_error()


def build_adaptor(tmp_path, api):
    exe = str(tmp_path / "reloc_refine_smoke")
    libdir = os.path.dirname(api.lib_path())
    cmd = ["g++", "-std=c++17", "-O1", "-Wall", "-I", os.path.join(ROOT, "include"), "-I", os.path.join(libdir, "host"),
           os.path.join(ROOT, "tests", "helpers", "reloc_refine_smoke.cpp"), "-o", exe, "-L", libdir, "-lb200reg", f"-Wl,-rpath,{libdir}",
           "-L/usr/local/cuda/lib64", "-Wl,-rpath,/usr/local/cuda/lib64"]
    p = subprocess.run(cmd, capture_output=True, text=True)
    assert p.returncode == 0, p.stderr[-3000:]
    return exe


def test_refine_adaptor_compiles_and_fails_loudly_without_gpu(tmp_path, api):
    exe = build_adaptor(tmp_path, api)
    if have_gpu():
        pytest.skip("the GPU run is tests/test_gpu_reloc_refine.py")
    p = subprocess.run([exe], capture_output=True, text=True)
    assert p.returncode == 10 and "FAILED LOUDLY" in p.stdout and "no CUDA device" in p.stdout, p.stdout + p.stderr
