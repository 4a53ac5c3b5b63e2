"""The LOAM local map from the device keyframe store without a device: the oracle's extractSurroundingKeyFrames against an
independent numpy restatement (radius hits, key-pose VoxelGrid, nearest keyframe, the 10 s walk, the distance gate, corner /
surf assembly and the two VoxelGrids), argument checking of the new entry points, the ctypes mirrors of the new records, the
C++ adaptor's build, and the refusal to run without a GPU."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT, have_gpu
from test_loop_cpu import pcl_matrix_f32

ERR_ARG, ERR_CUDA = -1, -2
F = np.float32


@pytest.fixture(scope="module")
def surround_oracle():
    from oracle import surround_binding
    surround_binding.build()
    return surround_binding


def sqd(a, b):
    """FLANN's squared distance in fp32: differences, squares summed x, y, z left to right."""
    d = (np.asarray(a, F) - np.asarray(b, F)).astype(F)
    return (d[..., 0] * d[..., 0] + d[..., 1] * d[..., 1]) + d[..., 2] * d[..., 2]


def voxel_f32(p, leaf):
    """pcl::VoxelGrid (min points 0) on finite [n, 3] float32 positions: fp32 sums in input order, ascending leaf order."""
    p = np.asarray(p, F)
    if len(p) == 0:
        return np.zeros((0, 3), F)
    inv = F(1.0) / F(leaf)
    min_b = np.floor(p.min(0) * inv).astype(np.int64)
    div_b = np.floor(p.max(0) * inv).astype(np.int64) - min_b + 1
    ijk = (np.floor(p * inv) - min_b.astype(F)).astype(np.int64)
    idx = ijk[:, 0] + ijk[:, 1] * div_b[0] + ijk[:, 2] * div_b[0] * div_b[1]
    out = []
    for k in np.unique(idx):
        s = np.zeros(3, F)
        members = np.flatnonzero(idx == k)
        for i in members:
            s = (s + p[i]).astype(F)
        out.append((s / F(len(members))).astype(F))
    return np.array(out, F)


def surrounding_numpy(clouds, n_corner, poses6, times, cur, time_cur, radius, density):
    """extractSurroundingKeyFrames restated: (list after the gate, list length, raw corner map, raw surf map)."""
    P = np.asarray(poses6, F)[: cur + 1, :3]
    q = P[cur]
    r2 = F(np.float64(radius) * np.float64(radius))
    d2 = sqd(P, q[None, :])
    hits = [j for j in range(cur + 1) if d2[j] < r2]
    hits.sort(key=lambda j: (d2[j], j))
    entries = []
    for c in voxel_f32(P[hits], density):
        dc = sqd(P, c[None, :])
        entries.append((int(np.argmin(dc)), c))      # argmin: the first (lowest index) minimum
    for j in range(cur, -1, -1):
        if not (time_cur - times[j] < 10.0):
            break
        entries.append((j, P[j]))
    keys = [k for k, pt in entries if not (np.sqrt(sqd(pt, q)) > F(radius))]
    corner, surf = [], []
    for k in keys:
        T, c = pcl_matrix_f32(poses6[k]), np.asarray(clouds[k], F)
        xyz = [((T[r, 0] * c[:, 0] + T[r, 1] * c[:, 1]) + T[r, 2] * c[:, 2]) + T[r, 3] for r in range(3)]
        moved = np.stack(xyz + [c[:, 3]], 1).astype(F)
        corner.append(moved[: n_corner[k]])
        surf.append(moved[n_corner[k]:])
    cat = lambda a: np.concatenate(a, 0) if a else np.zeros((0, 4), F)
    return np.array(keys, np.int64), len(entries), cat(corner), cat(surf)


def check_session(surround_oracle, oracle, clouds, n_corner, poses6, times, cur, time_cur, radius, density, leaves=(0.2, 0.4)):
    kf = surround_oracle.Keyframes(clouds, poses6, times, n_corner)
    keys, n_list, co, so = kf.surrounding(cur, time_cur, search_radius=radius, density=density, corner_leaf=leaves[0], surf_leaf=leaves[1])
    keys_n, n_list_n, raw_c, raw_s = surrounding_numpy(clouds, n_corner, poses6, times, cur, time_cur, radius, density)
    assert keys.tolist() == keys_n.tolist() and n_list == n_list_n, (cur, keys, keys_n)
    for got, raw, leaf in ((co, raw_c, leaves[0]), (so, raw_s, leaves[1])):
        ref = oracle.voxel_grid(raw, leaf, 0)[0] if len(raw) else np.zeros((0, 4), F)
        assert got.view(np.uint32).tolist() == ref.view(np.uint32).tolist(), cur
    return keys, n_list


def split_session(synth, K, n_points, seed_mod=5):
    s = synth.loop_session(K=K, n_points=n_points, laps=2)
    clouds = [np.asarray(c, F) for c in s["clouds"]]
    n_corner = np.array([len(c) // seed_mod for c in clouds], np.int64)
    return s, clouds, n_corner


def test_oracle_matches_numpy_on_a_two_lap_session(surround_oracle, oracle, synth):
    s, clouds, n_corner = split_session(synth, 80, 120)
    clouds[7] = clouds[7][:0]                               # an empty keyframe
    n_corner[7] = 0
    n_corner[9] = 0                                          # no corner cloud
    n_corner[11] = len(clouds[11])                           # no surf cloud
    seen_dup = False
    for radius in (6.0, 14.0):
        for cur in (0, 5, 39, 41, 60, 79):                   # cur before the end of the store, first keyframe, second lap
            keys, n_list = check_session(surround_oracle, oracle, clouds, n_corner, s["poses"], s["times"], cur, s["times"][cur] + 0.5, radius, 2.0)
            seen_dup |= len(set(keys.tolist())) < len(keys)
    assert seen_dup                                          # recent keyframes also listed as a centroid's nearest


def test_boundaries(surround_oracle, oracle):
    """The radius is strict, equal positions go to the lower index, a centroid rounded beyond the radius is skipped, the walk
    stops at time_cur - t == 10.0, and a recent keyframe that is also a centroid's nearest is listed twice."""
    P = np.zeros((8, 6), F)
    P[0, :3] = [3.0, 0.0, 0.0]                               # d2 == r^2 (radius 3): not a hit
    P[1, :3] = [1.9116278886795044, -2.297743558883667, 0.25700733065605164]   # 1 and 2: one leaf whose fp32 centroid
    P[2, :3] = [1.9116290807724, -2.2977428436279297, 0.2570052146911621]      # lies beyond the radius
    P[3, :3] = [-1.0, 1.0, 0.5]                              # 3 and 4 share a position: the nearest is 3
    P[4, :3] = [-1.0, 1.0, 0.5]
    P[5, :3] = [0.5, 0.5, 0.0]
    P[6, :3] = [0.0, -1.5, 0.0]                              # a leaf of its own
    P[7, :3] = [0.0, 0.0, 0.0]                               # the newest keyframe
    t = np.array([0.0, 1.0, 2.0, 3.0, 4.0, 6.0, 8.0, 16.0])
    rng = np.random.default_rng(3)
    clouds = [rng.normal(0, 3, (20 + k, 4)).astype(F) for k in range(8)]
    n_corner = np.array([5] * 8, np.int64)
    for time_cur, recent in ((16.0, [7, 6]), (18.0, [7]), (17.5, [7, 6])):   # 18.0: keyframe 6 is exactly 10 s old
        keys, n_list = check_session(surround_oracle, oracle, clouds, n_corner, P, t, 7, time_cur, 3.0, 2.0)
        k = keys.tolist()
        assert 0 not in k and 4 not in k and 3 in k
        assert 1 not in k and 2 not in k                     # their centroid's entry is skipped by the gate
        assert k[-len(recent):] == recent and k.count(6) == 1 + (6 in recent)
        assert n_list == len(k) + 1


def test_local_map_handle_fails_loudly_without_gpu(api):
    if have_gpu():
        pytest.skip("only meaningful on a box without a GPU")
    with pytest.raises(api.B200Error, match="no CUDA device"):
        api.KeyframeStore()


def test_local_map_bad_arguments_are_rejected(api):
    lib = api.lib()
    prm = api.KeyframeStore.surround_params()
    info = api.SurroundInfo()
    n, m = ctypes.c_int64(), ctypes.c_int64()
    keys = np.zeros(4, np.int64)
    out = np.zeros((4, 4), F)
    pose = np.zeros(6, F)
    p = lambda a: a.ctypes.data_as(ctypes.c_void_p)
    assert lib.b200_keyframes_add_features(None, p(out), 4, 16, p(out), 4, 16, p(pose), 0.0, None) == ERR_ARG
    assert lib.b200_keyframes_surrounding(None, -1, 0.0, ctypes.byref(prm), p(keys), 4, ctypes.byref(n)) == ERR_ARG
    assert lib.b200_keyframes_surrounding_map(None, -1, 0.0, ctypes.byref(prm), p(out), 4, ctypes.byref(n), p(out), 4, ctypes.byref(m)) == ERR_ARG
    assert lib.b200_loam_set_map_from_keyframes(None, None, -1, 0.0, ctypes.byref(prm), ctypes.byref(info)) == ERR_ARG
    assert b"bad argument" in lib.b200_last_error()
    with pytest.raises(TypeError):
        api.KeyframeStore.surround_params(radius=3.0)


def test_local_map_records_match_the_c_structs(api, tmp_path):
    """The ctypes SurroundParams / SurroundInfo have the sizes and field offsets gcc gives the C structs."""
    src = tmp_path / "layout.c"
    pf = [f for f, _ in api.SurroundParams._fields_]
    inf = [f for f, _ in api.SurroundInfo._fields_]
    body = ['printf("psize %zu\\n", sizeof(b200_surround_params));', 'printf("isize %zu\\n", sizeof(b200_surround_info));']
    body += [f'printf("p.{f} %zu\\n", offsetof(b200_surround_params, {f}));' for f in pf]
    body += [f'printf("i.{f} %zu\\n", offsetof(b200_surround_info, {f}));' for f in inf]
    src.write_text('#include <stddef.h>\n#include <stdio.h>\n#include "b200reg.h"\nint main(void) {\n' + "\n".join(body) + "\nreturn 0;\n}\n")
    exe = tmp_path / "layout"
    r = subprocess.run(["gcc", "-std=c99", "-Wall", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    got = dict(line.split() for line in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.splitlines())
    assert int(got["psize"]) == ctypes.sizeof(api.SurroundParams) and int(got["isize"]) == ctypes.sizeof(api.SurroundInfo)
    for f in pf:
        assert int(got["p." + f]) == getattr(api.SurroundParams, f).offset, f
    for f in inf:
        assert int(got["i." + f]) == getattr(api.SurroundInfo, f).offset, f


def build_adaptor(tmp_path, api):
    exe = str(tmp_path / "loam_local_map_smoke")
    libdir = os.path.dirname(api.lib_path())
    cmd = ["g++", "-std=c++17", "-O1", "-Wall", "-I", os.path.join(ROOT, "include"), "-I", os.path.join(libdir, "host"),
           os.path.join(ROOT, "tests", "helpers", "loam_local_map_smoke.cpp"), "-o", exe, "-L", libdir, "-lb200reg", f"-Wl,-rpath,{libdir}",
           "-L/usr/local/cuda/lib64", "-Wl,-rpath,/usr/local/cuda/lib64"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    return exe


def test_local_map_adaptor_compiles_and_fails_loudly_without_gpu(tmp_path, api):
    exe = build_adaptor(tmp_path, api)
    if have_gpu():
        pytest.skip("the GPU run is tests/test_gpu_loam_local_map.py")
    r = subprocess.run([exe], capture_output=True, text=True)
    assert r.returncode == 10 and "FAILED LOUDLY" in r.stdout and "no CUDA device" in r.stdout, r.stdout + r.stderr
