"""Loop closure from the device keyframe store without a device: the oracle's candidate search and submap assembly against
numpy restatements, argument checking of the b200_keyframes_* / b200_loop_* entry points, the ctypes mirrors of the records,
the C++ adaptor's build, and the refusal to run without a GPU."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT, have_gpu

ERR_ARG, ERR_CUDA = -1, -2


@pytest.fixture(scope="module")
def loop_oracle():
    from oracle import loop_binding
    loop_binding.build()
    return loop_binding


def detect_numpy(poses6, times, cur, radius, gap):
    """detectLoopClosureDistance in fp32 numpy: (q - j) per axis, squares summed x, y, z left to right, strict radius test,
    time gap strict, nearest with ties to the lower index."""
    P = np.asarray(poses6, np.float32)
    r2 = np.float32(np.float64(radius) * np.float64(radius))
    pre, d2 = [], []
    for c in cur:
        d = P[c, :3][None, :] - P[:c, :3]
        s = (d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1]) + d[:, 2] * d[:, 2]
        ok = (s < r2) & (np.abs(np.asarray(times)[:c] - times[c]) > gap)
        if not ok.any():
            pre.append(-1); d2.append(np.float32(0)); continue
        j = np.flatnonzero(ok)
        k = j[np.argmin(s[j])]   # argmin returns the first (lowest index) minimum
        pre.append(k); d2.append(s[k])
    return np.array(pre, np.int64), np.array(d2, np.float32)


def pcl_matrix_f32(p6):
    """pcl::getTransformation in float with correctly rounded sin / cos."""
    f = np.float32
    roll, pitch, yaw = (f(v) for v in p6[3:6])
    cs = lambda a: (f(np.cos(np.float64(a))), f(np.sin(np.float64(a))))
    (A, B), (C, D), (E, F) = cs(yaw), cs(pitch), cs(roll)
    DE, DF = D * E, D * F
    return np.array([[A * C, A * DF - B * E, B * F + A * DE, f(p6[0])],
                     [B * C, A * E + B * DF, B * DE - A * F, f(p6[1])],
                     [-D, C * F, C * E, f(p6[2])]], np.float32)


def submap_numpy(clouds, poses6, key, num):
    out = []
    for k in range(max(0, key - num), min(len(clouds) - 1, key + num) + 1):
        T, p = pcl_matrix_f32(poses6[k]), np.asarray(clouds[k], np.float32)
        xyz = [((T[r, 0] * p[:, 0] + T[r, 1] * p[:, 1]) + T[r, 2] * p[:, 2]) + T[r, 3] for r in range(3)]
        out.append(np.stack(xyz + [p[:, 3]], 1))
    return np.concatenate(out, 0) if out else np.zeros((0, 4), np.float32)


def test_detect_oracle_matches_numpy(loop_oracle, synth):
    s = synth.loop_session(K=240, n_points=16, laps=2)
    P, t = s["poses"].copy(), s["times"].copy()
    cur = np.arange(0, 240, 3)
    radius, gap = 2.0, 30.0
    pre_o, d_o = loop_oracle.loop_detect(P, t, cur, radius, gap)
    pre_n, d_n = detect_numpy(P, t, cur, radius, gap)
    np.testing.assert_array_equal(pre_o, pre_n)
    assert d_o.view(np.uint32).tolist() == d_n.view(np.uint32).tolist()
    assert (pre_o >= 0).sum() > 20 and (pre_o < 0).sum() > 10   # both outcomes are exercised


def test_detect_boundaries(loop_oracle):
    """Ties go to the lower index; a keyframe exactly on r^2 and one exactly at the time gap are not candidates."""
    P = np.zeros((8, 6), np.float32)
    t = np.array([0.0, 1.0, 2.0, 3.0, 4.0, 5.0, 6.0, 40.0])
    P[0, :3] = [1.0, 0.0, 0.0]     # d2 = 1 = r^2 exactly (radius 1): outside
    P[1, :3] = [0.0, 0.5, 0.0]     # d2 = 0.25: tie with 2
    P[2, :3] = [0.0, -0.5, 0.0]    # d2 = 0.25
    P[3, :3] = [0.0, 0.0, 0.1]     # nearest, but only 37 s before the query
    P[4, :3] = [5.0, 5.0, 5.0]
    # gap 37: keyframe 3 sits exactly on the gap, 1 and 2 tie; gap 39: 1 sits on the gap and 0 on the radius
    for gap, want in [(37.0, 1), (36.5, 3), (38.5, 1), (39.0, -1)]:
        pre_o, d_o = loop_oracle.loop_detect(P, t, [7], 1.0, gap)
        pre_n, d_n = detect_numpy(P, t, [7], 1.0, gap)
        assert pre_o[0] == pre_n[0] == want, (gap, pre_o, pre_n)
        assert d_o[0] == d_n[0]
    pre, _ = loop_oracle.loop_detect(P, t, [0], 1.0, 0.0)     # the first keyframe has no history
    assert pre[0] == -1


def test_submap_oracle_matches_numpy_and_voxel_grid(loop_oracle, oracle, synth):
    s = synth.loop_session(K=30, n_points=400, laps=1)
    clouds = list(s["clouds"])
    clouds[5] = np.zeros((0, 4), np.float32)                     # an empty keyframe
    clouds[6] = clouds[6].copy()
    clouds[6][::7, 1] = np.nan                                   # NaN points are dropped by the downsample
    kf = loop_oracle.Keyframes(clouds, s["poses"])
    for key, num in [(0, 3), (29, 4), (6, 2), (15, 0), (15, 25)]:
        raw, ds, cnt = kf.submap(key, num, 0.4)
        ref = submap_numpy(clouds, s["poses"], key, num)
        assert raw.shape == ref.shape
        assert raw.view(np.uint32).tolist() == ref.view(np.uint32).tolist(), (key, num)
        vg, vc = oracle.voxel_grid(raw, 0.4, 0)
        assert ds.view(np.uint32).tolist() == vg.view(np.uint32).tolist() and cnt.tolist() == vc.tolist(), (key, num)


def test_keyframes_handle_fails_loudly_without_gpu(api):
    if have_gpu():
        pytest.skip("only meaningful on a box without a GPU")
    lib = api.lib()
    h = ctypes.c_void_p()
    assert lib.b200_keyframes_create(0, ctypes.byref(h)) == ERR_CUDA
    assert b"no CUDA device" in lib.b200_last_error()
    with pytest.raises(api.B200Error, match="no CUDA device"):
        api.KeyframeStore()


def test_loop_bad_arguments_are_rejected(api):
    lib = api.lib()
    prm = api.KeyframeStore.params()
    cur = np.array([3], np.int64)
    pre = np.array([0], np.int64)
    d2 = np.zeros(1, np.float32)
    out = np.zeros((4, 4), np.float32)
    n = ctypes.c_int64()
    res = (api.LoopResult * 1)()
    p = lambda a: a.ctypes.data_as(ctypes.c_void_p)
    assert lib.b200_keyframes_create(0, None) == ERR_ARG
    assert lib.b200_keyframes_destroy(None) == 0
    assert lib.b200_keyframes_count(None) == -1
    xyz = np.zeros((4, 4), np.float32)
    pose = np.zeros(6, np.float32)
    assert lib.b200_keyframes_add(None, p(xyz), 4, 16, p(pose), 0.0, None) == ERR_ARG
    assert lib.b200_keyframes_set_poses(None, 0, 1, p(pose)) == ERR_ARG
    assert lib.b200_loop_detect(None, p(cur), 1, ctypes.byref(prm), p(pre), p(d2)) == ERR_ARG
    assert lib.b200_loop_submap(None, 0, 2, 0.4, p(out), 4, ctypes.byref(n)) == ERR_ARG
    assert lib.b200_loop_close(None, None, None, p(cur), None, 1, ctypes.byref(prm), res) == ERR_ARG
    assert b"bad argument" in lib.b200_last_error()


def test_loop_records_match_the_c_structs(api, tmp_path):
    """The ctypes LoopParams / LoopResult have the sizes and field offsets gcc gives the C structs."""
    src = tmp_path / "layout.c"
    pf = ["search_radius", "time_gap", "search_num", "leaf", "min_source_points", "min_target_points", "max_range"]
    rf = ["cur", "pre", "pre_sqdist", "n_source", "n_target", "reg"]
    body = ['printf("psize %zu\\n", sizeof(b200_loop_params));', 'printf("rsize %zu\\n", sizeof(b200_loop_result));']
    body += [f'printf("p.{f} %zu\\n", offsetof(b200_loop_params, {f}));' for f in pf]
    body += [f'printf("r.{f} %zu\\n", offsetof(b200_loop_result, {f}));' for f in rf]
    src.write_text('#include <stddef.h>\n#include <stdio.h>\n#include "b200reg.h"\nint main(void) {\n' + "\n".join(body) + "\nreturn 0;\n}\n")
    exe = tmp_path / "layout"
    r = subprocess.run(["gcc", "-std=c99", "-Wall", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    got = dict(line.split() for line in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.splitlines())
    assert int(got["psize"]) == ctypes.sizeof(api.LoopParams) and int(got["rsize"]) == ctypes.sizeof(api.LoopResult)
    for f in pf:
        assert int(got["p." + f]) == getattr(api.LoopParams, f).offset, f
    for f in rf:
        assert int(got["r." + f]) == getattr(api.LoopResult, f).offset, f


def build_adaptor(tmp_path, api):
    exe = str(tmp_path / "loop_closure_smoke")
    libdir = os.path.dirname(api.lib_path())
    cmd = ["g++", "-std=c++17", "-O1", "-Wall", "-I", os.path.join(ROOT, "include"), "-I", os.path.join(libdir, "host"),
           os.path.join(ROOT, "tests", "helpers", "loop_closure_smoke.cpp"), "-o", exe, "-L", libdir, "-lb200reg", f"-Wl,-rpath,{libdir}",
           "-L/usr/local/cuda/lib64", "-Wl,-rpath,/usr/local/cuda/lib64"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    return exe


def test_loop_adaptor_compiles_and_fails_loudly_without_gpu(tmp_path, api):
    exe = build_adaptor(tmp_path, api)
    if have_gpu():
        pytest.skip("the GPU run is tests/test_gpu_loop_closure.py")
    r = subprocess.run([exe], capture_output=True, text=True)
    assert r.returncode == 10 and "FAILED LOUDLY" in r.stdout and "no CUDA device" in r.stdout, r.stdout + r.stderr
