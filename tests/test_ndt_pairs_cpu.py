"""Batched NDT pair registration (b200_ndt_pairs_*) without a device: argument checking, the ctypes mirror of the result
record, the C++ adaptor's build, and the refusal to run without a GPU."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT, have_gpu

ERR_ARG = -1


def test_pairs_handle_fails_loudly_without_gpu(api):
    if have_gpu():
        pytest.skip("only meaningful on a box without a GPU")
    with pytest.raises(api.B200Error, match="no CUDA device"):
        api.NdtPairBatch()


def test_pairs_bad_arguments_are_rejected(api):
    lib = api.lib()
    prm = api.NdtParams(1.0, 0.1, 0.55, 0.01, 35, 7, 6, 0.01)
    assert lib.b200_ndt_pairs_create(None, 0, None) == ERR_ARG
    assert lib.b200_ndt_pairs_create(ctypes.byref(prm), 0, None) == ERR_ARG
    assert lib.b200_ndt_pairs_destroy(None) == 0
    xyz = np.zeros((8, 3), np.float32)
    off = np.array([0, 4], np.int64)
    res = (api.NdtPairResult * 2)()
    p = xyz.ctypes.data_as(ctypes.c_void_p)
    o = off.ctypes.data_as(ctypes.c_void_p)
    align = lib.b200_ndt_pairs_align
    assert align(None, None, p, o, p, o, 12, 1, None, 1.0, res) == ERR_ARG           # no handle
    assert b"bad argument" in lib.b200_last_error()
    assert align(None, None, None, o, p, o, 12, 1, None, 1.0, res) == ERR_ARG        # no source cloud
    assert align(None, None, p, o, p, None, 12, 1, None, 1.0, res) == ERR_ARG        # no target offsets
    assert align(None, None, p, o, p, o, 12, 0, None, 1.0, res) == ERR_ARG           # P = 0
    assert align(None, None, p, o, p, o, 8, 1, None, 1.0, res) == ERR_ARG            # stride below 12
    assert align(None, None, p, o, p, o, 12, 1, None, 1.0, None) == ERR_ARG          # no result array
    assert lib.b200_ndt_pairs_leaves(None, 0, 0, None, None, None, None, None) == -1


def test_pair_result_layout_matches_the_c_struct(api, tmp_path):
    """The ctypes NdtPairResult has the size and field offsets gcc gives b200_ndt_pair_result."""
    src = tmp_path / "layout.c"
    fields = ["status", "ndt", "fitness", "n_in_range", "final16"]
    inner = ["converged", "iters", "evals", "hess_evals", "trans_probability", "hessian", "score", "p_final", "gpu_ms"]
    body = ['printf("size %zu\\n", sizeof(b200_ndt_pair_result));', 'printf("inner %zu\\n", sizeof(b200_ndt_result));']
    body += [f'printf("{f} %zu\\n", offsetof(b200_ndt_pair_result, {f}));' for f in fields]
    body += [f'printf("ndt.{f} %zu\\n", offsetof(b200_ndt_result, {f}));' for f in inner]
    src.write_text('#include <stddef.h>\n#include <stdio.h>\n#include "b200reg.h"\nint main(void) {\n' + "\n".join(body) + "\nreturn 0;\n}\n")
    exe = tmp_path / "layout"
    p = subprocess.run(["gcc", "-std=c99", "-Wall", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], capture_output=True, text=True)
    assert p.returncode == 0, p.stderr
    got = dict(line.split() for line in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.splitlines())
    assert int(got["size"]) == ctypes.sizeof(api.NdtPairResult)
    assert int(got["inner"]) == ctypes.sizeof(api.NdtResult)
    for f in fields:
        assert int(got[f]) == getattr(api.NdtPairResult, f).offset, f
    for f in inner:
        assert int(got["ndt." + f]) == getattr(api.NdtResult, f).offset, f


def build_adaptor(tmp_path, api):
    exe = str(tmp_path / "ndt_pairs_smoke")
    libdir = os.path.dirname(api.lib_path())
    cmd = ["g++", "-std=c++17", "-O1", "-Wall", "-I", os.path.join(ROOT, "include"), "-I", os.path.join(libdir, "host"),
           os.path.join(ROOT, "tests", "helpers", "ndt_pairs_smoke.cpp"), "-o", exe, "-L", libdir, "-lb200reg", f"-Wl,-rpath,{libdir}",
           "-L/usr/local/cuda/lib64", "-Wl,-rpath,/usr/local/cuda/lib64"]
    p = subprocess.run(cmd, capture_output=True, text=True)
    assert p.returncode == 0, p.stderr[-3000:]
    return exe


def test_pairs_adaptor_compiles_and_fails_loudly_without_gpu(tmp_path, api):
    exe = build_adaptor(tmp_path, api)
    if have_gpu():
        pytest.skip("the GPU run is tests/test_gpu_ndt_pairs.py")
    p = subprocess.run([exe], capture_output=True, text=True)
    assert p.returncode == 10 and "FAILED LOUDLY" in p.stdout and "no CUDA device" in p.stdout, p.stdout + p.stderr
