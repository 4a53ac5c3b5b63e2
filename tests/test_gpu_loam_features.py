"""The LOAM front end on the device (b200_features_*) against the CPU oracle, byte for byte on every probe; no state between
scans; the device hand-offs to scan-to-map and the keyframe store against their host paths; error codes."""
import os
import subprocess
from dataclasses import asdict

import numpy as np
import pytest

import feature_scans
from conftest import ROOT

pytestmark = pytest.mark.gpu

PROBES = ("cloud", "col", "range", "start", "end", "curvature", "label", "picked", "corner", "surface", "corner_ds", "surf_ds")


@pytest.fixture(scope="module")
def api():
    from pointcloud_slam_b200 import api
    return api


@pytest.fixture(scope="module")
def oracle():
    from oracle import feature_binding
    feature_binding.build()
    return feature_binding


def device_run(api, fx, scan):
    rec, stride, io, ro, rb, _ = scan
    rc = fx.extract(rec, stride, io, ro, rb)
    cloud, col, rng, start, end = fx.cloud_info()
    curv, label, picked = fx.labels()
    out = dict(cloud=cloud, col=col, range=rng, start=start, end=end, curvature=curv, label=label, picked=picked)
    for k, w in (("corner", fx.CORNER), ("surface", fx.SURFACE), ("corner_ds", fx.CORNER_DS), ("surf_ds", fx.SURF_DS)):
        out[k] = fx.cloud(w)
    return rc, out


def check_parity(api, oracle, scan, fx=None):
    rec, stride, io, ro, rb, prm = scan
    own = fx is None
    fx = fx or api.FeatureExtraction(**asdict(prm))
    try:
        rc, got = device_run(api, fx, scan)
        want = oracle.features(rec, stride, io, ro, rb, prm)
        for k in PROBES:
            a, b = np.ascontiguousarray(got[k]), np.ascontiguousarray(want[k], dtype=got[k].dtype)
            assert a.shape == b.shape, (k, a.shape, b.shape)
            assert a.tobytes() == b.tobytes(), (k, np.flatnonzero((a != b).reshape(len(a), -1).any(1))[:10] if a.ndim else None)
        info = fx.info
        assert (info.dropped_nonfinite, info.dropped_range, info.dropped_row, info.dropped_col, info.dropped_dup) == (
            want["dropped_nonfinite"], want["dropped_range"], want["dropped_row"], want["dropped_col"], want["dropped_dup"])
        assert rc == (1 if want["n_extracted"] == 0 else 0)
        return got, want
    finally:
        if own:
            fx.close()


@pytest.mark.parametrize("n_scan,H", [(16, 1800), (32, 1800), (64, 1024), (128, 2048), (16, 1024)])
def test_spinning_parity(api, oracle, n_scan, H):
    got, _ = check_parity(api, oracle, feature_scans.spinning(n_scan=n_scan, H=H, seed=n_scan + H))
    assert len(got["corner"]) > 0 and len(got["surf_ds"]) > 0


def test_duplicates_junk_and_rate(api, oracle):
    check_parity(api, oracle, feature_scans.spinning(n_scan=16, H=1800, seed=3, dup=0.3, junk=0.05))
    check_parity(api, oracle, feature_scans.spinning(n_scan=32, H=1800, seed=4, rate=2, junk=0.02))


def test_livox_and_quirk_scans(api, oracle):
    check_parity(api, oracle, feature_scans.livox())
    check_parity(api, oracle, feature_scans.livox(n_lines=6, per_line=20000, H=4000, seed=9))
    got, _ = check_parity(api, oracle, feature_scans.quirks())
    assert len(got["corner"]) > 0
    check_parity(api, oracle, feature_scans.spinning(n_scan=8, H=360, seed=0))


def test_tiny_and_empty_scans(api, oracle):
    rec, stride, io, ro, rb, prm = feature_scans.spinning(n_scan=4, H=120, seed=5)
    fx = api.FeatureExtraction(**asdict(prm))
    try:
        for k in (0, 1, 5, 11, 12, 40):
            check_parity(api, oracle, (rec[:k], stride, io, ro, rb, prm), fx)
        assert fx.extract(rec[:0], stride, io, ro, rb) == 1 and fx.cloud(fx.SURF_DS).shape == (0, 4)
    finally:
        fx.close()


def test_no_state_between_scans(api, oracle):
    a = feature_scans.spinning(n_scan=16, H=1800, seed=11, dup=0.1)
    fx = api.FeatureExtraction(**asdict(a[-1]))
    try:
        _, first = device_run(api, fx, a)
        device_run(api, fx, feature_scans.spinning(n_scan=16, H=1800, seed=12, junk=0.1))
        _, again = device_run(api, fx, a)
        for k in PROBES:
            assert first[k].tobytes() == again[k].tobytes(), k
    finally:
        fx.close()


def test_handoffs_match_host_path(api, oracle):
    scan = feature_scans.spinning(n_scan=32, H=1800, seed=21)
    rec, stride, io, ro, rb, prm = scan
    fx = api.FeatureExtraction(**asdict(prm))
    s2m = api.ScanToMap(max_map_points=200_000)
    st_h, st_d = api.KeyframeStore(), api.KeyframeStore()
    try:
        assert fx.extract(rec, stride, io, ro, rb) == 0
        cds, sds = fx.cloud(fx.CORNER_DS), fx.cloud(fx.SURF_DS)
        s2m.setInputCloud(cds[:, :3], sds[:, :3])
        t0 = np.array([0.01, -0.02, 0.015, 0.3, -0.2, 0.1], np.float32)
        t_h, rc_h = s2m.scan2MapOptimization(cds, sds, t0, 30)
        st_host = (s2m.stats.iters, s2m.stats.n_sel, s2m.stats.converged, s2m.stats.degenerate, bytes(s2m.stats.AtA_first))
        t_d, rc_d = s2m.scan2MapOptimization_device(fx.device_cloud(fx.CORNER_DS), fx.device_cloud(fx.SURF_DS), t0, 30)
        st_dev = (s2m.stats.iters, s2m.stats.n_sel, s2m.stats.converged, s2m.stats.degenerate, bytes(s2m.stats.AtA_first))
        assert rc_h == rc_d and t_h.tobytes() == t_d.tobytes() and st_host == st_dev
        # the keyframe store: three keyframes from three scans, host copies vs device clouds
        for k in range(3):
            sc = feature_scans.spinning(n_scan=32, H=1800, seed=30 + k)
            assert fx.extract(*sc[:5]) == 0
            pose = np.array([0.7 * k, 0.1 * k, 0.0, 0.0, 0.0, 0.05 * k], np.float32)
            kh = st_h.add_features(fx.cloud(fx.CORNER_DS), fx.cloud(fx.SURF_DS), pose, float(k))
            kd = st_d.add_features_device(fx.device_cloud(fx.CORNER_DS), fx.device_cloud(fx.SURF_DS), pose, float(k))
            assert kh == kd == k
        mh, md = st_h.surrounding_map(-1, 2.5), st_d.surrounding_map(-1, 2.5)
        for a, b in zip(mh, md):
            assert a.tobytes() == b.tobytes()
        assert st_h.submap(1, 1, 0.4).tobytes() == st_d.submap(1, 1, 0.4).tobytes()
    finally:
        fx.close()
        s2m.close()
        st_h.close()
        st_d.close()


def test_error_cases(api, oracle):
    base = feature_scans.spinning(n_scan=16, H=360, seed=7)
    rec, stride, io, ro, rb, prm = base
    for bad in (dict(n_scan=0), dict(n_scan=1025), dict(n_scan=1024, horizon_scan=65537), dict(odometry_surf_leaf=0.0), dict(mapping_corner_leaf=-1.0),
                dict(downsample_rate=0), dict(sensor=2)):
        with pytest.raises(api.B200Error, match="error -1"):
            api.FeatureExtraction(**dict(asdict(prm), **bad))
    fx = api.FeatureExtraction(**asdict(prm))
    try:
        for args in ((rec, 10, io, ro, rb), (rec, stride, 2, ro, rb), (rec, stride, io, ro, 3), (rec, stride, io, stride - 1, 2)):
            with pytest.raises(api.B200Error, match="error -1"):
                fx.extract(*args)
        check_parity(api, oracle, base, fx)  # still usable
        tiny = api.FeatureExtraction(**dict(asdict(prm), mapping_surf_leaf=1e-12))
        try:
            with pytest.raises(api.B200Error, match="error -4"):
                tiny.extract(rec, stride, io, ro, rb)
        finally:
            tiny.close()
        check_parity(api, oracle, base, fx)
        # host memory where device clouds are expected
        host = np.zeros((4, 4), np.float32)
        s2m = api.ScanToMap(max_map_points=1000)
        st = api.KeyframeStore()
        try:
            s2m.setInputCloud(host[:, :3] + 1, host[:, :3] + 2)
            with pytest.raises(api.B200Error, match="error -1"):
                s2m.scan2MapOptimization_device((host.ctypes.data, 4), (host.ctypes.data, 4), np.zeros(6), 5)
            with pytest.raises(api.B200Error, match="error -1"):
                st.add_features_device((host.ctypes.data, 4), (None, 0), np.zeros(6), 0.0)
            assert lib_count(api, st) == 0
        finally:
            s2m.close()
            st.close()
    finally:
        fx.close()


def lib_count(api, st):
    return int(api.lib().b200_keyframes_count(st.h))


def test_cpp_chain_runs(tmp_path, api):
    exe = str(tmp_path / "loam_features_smoke")
    libdir = os.path.dirname(api.lib_path())
    cmd = ["g++", "-std=c++17", "-O1", "-Wall", "-I", os.path.join(ROOT, "include"), "-I", os.path.join(libdir, "host"),
           os.path.join(ROOT, "tests", "helpers", "loam_features_smoke.cpp"), "-o", exe, "-L", libdir, "-lb200reg", f"-Wl,-rpath,{libdir}",
           "-L/usr/local/cuda/lib64", "-Wl,-rpath,/usr/local/cuda/lib64"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    r = subprocess.run([exe], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "features chain ok" in r.stdout, r.stdout + r.stderr
