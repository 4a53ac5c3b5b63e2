"""Loop closure from the device keyframe store (b200_keyframes_*, b200_loop_detect / submap / close) against the CPU oracle,
b200_voxel_downsample, b200_ndt_pairs_align on the downloaded submaps, itself (determinism) and the synthetic ground truth.

Bars: detection and submaps bit-exact; a loop record byte-equal (gpu_ms zeroed) to b200_ndt_pairs_align's record for the same
two clouds; align / fitness against the oracle with the bars of test_gpu_ndt_pairs.py.
"""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT

pytestmark = pytest.mark.gpu

NDT = dict(resolution=1.0, trans_eps=0.01, step_size=0.1, max_iter=35)
LOOP = dict(search_radius=5.0, time_gap=30.0, search_num=25, leaf=0.4, min_source_points=100, min_target_points=1000)
NO_EFFECTIVE_POINTS = 1


@pytest.fixture(scope="module")
def loop_oracle():
    from oracle import loop_binding
    loop_binding.build()
    return loop_binding


@pytest.fixture(scope="module")
def session(synth):
    return synth.loop_session(K=2000, n_points=500, laps=2)


def make_store(api, clouds, poses, times):
    st = api.KeyframeStore()
    for k, c in enumerate(clouds):
        assert st.add(c, poses[k], times[k]) == k
    return st


@pytest.fixture(scope="module")
def store(api, session):
    return make_store(api, session["clouds"], session["poses"], session["times"])


@pytest.fixture(scope="module")
def queries(store):
    cur = np.arange(1030, 2000, 24)
    pre, _ = store.detect(cur, **LOOP)
    assert (pre >= 0).sum() >= 30
    return cur


def reg_bytes(rec):
    r = type(rec).from_buffer_copy(rec)
    r.ndt.gpu_ms = 0.0
    return bytes(memoryview(r).cast("B"))


def test_detect_equals_oracle(api, loop_oracle, store, session):
    cur = np.arange(len(session["clouds"]))
    pre, d2 = store.detect(cur, **LOOP)
    pre0, d20 = loop_oracle.loop_detect(session["poses"], session["times"], cur, LOOP["search_radius"], LOOP["time_gap"])
    np.testing.assert_array_equal(pre, pre0)
    assert d2.view(np.uint32).tolist() == d20.view(np.uint32).tolist()
    assert (pre >= 0).sum() > 1000 and (pre < 0).sum() >= 20   # both outcomes are exercised


def test_detect_ties_and_boundaries(api, loop_oracle):
    P = np.zeros((8, 6), np.float32)
    t = np.array([0.0, 1.0, 2.0, 3.0, 4.0, 5.0, 6.0, 40.0])
    P[0, :3] = [1.0, 0.0, 0.0]     # exactly on r^2 = 1
    P[1, :3] = [0.0, 0.5, 0.0]     # tie with 2
    P[2, :3] = [0.0, -0.5, 0.0]
    P[3, :3] = [0.0, 0.0, 0.1]     # nearest, 37 s before the query
    P[4, :3] = [5.0, 5.0, 5.0]
    st = make_store(api, [np.ones((3, 4), np.float32)] * 8, P, t)
    for gap, want in [(37.0, 1), (36.5, 3), (38.5, 1), (39.0, -1)]:
        pre, d2 = st.detect(np.arange(8), **dict(LOOP, search_radius=1.0, time_gap=gap))
        pre0, d20 = loop_oracle.loop_detect(P, t, np.arange(8), 1.0, gap)
        np.testing.assert_array_equal(pre, pre0)
        np.testing.assert_array_equal(d2, d20)
        assert pre[7] == want, gap


def submap_checks(api, st, kf, key, num, leaf):
    raw, ds0, _ = kf.submap(key, num, leaf)
    ds = st.submap(key, num, leaf)
    assert ds.shape == ds0.shape, (key, num)
    assert ds.view(np.uint32).tolist() == ds0.view(np.uint32).tolist(), (key, num)
    if len(raw):
        vg = api.VoxelGrid()
        vg.setLeafSize(leaf)
        vg.setInputCloud(raw)
        c1, _ = vg.filter()
        assert ds.view(np.uint32).tolist() == c1.view(np.uint32).tolist(), (key, num)
    return ds


def test_submap_bit_exact(api, loop_oracle, store, session):
    kf = loop_oracle.Keyframes(session["clouds"], session["poses"])
    for key in (0, 3, 24, 1000, 1976, 1999):
        submap_checks(api, store, kf, key, 25, 0.4)
    submap_checks(api, store, kf, 700, 0, 0.4)


def test_submap_empty_nan_and_huge_grid(api, loop_oracle, session):
    clouds = [c.copy() for c in session["clouds"][:40]]
    clouds[10] = np.zeros((0, 4), np.float32)
    clouds[11][::5, 0] = np.nan
    clouds[12][::9, 2] = np.inf
    clouds[20] = np.full((6, 4), np.nan, np.float32)
    st = make_store(api, clouds, session["poses"][:40], session["times"][:40])
    kf = loop_oracle.Keyframes(clouds, session["poses"][:40])
    for key, num in [(10, 0), (11, 2), (10, 3), (20, 0), (39, 5)]:
        submap_checks(api, st, kf, key, num, 0.4)
    assert len(st.submap(20, 0, 0.4)) == 0 and len(st.submap(10, 0, 0.4)) == 0
    ds = submap_checks(api, st, kf, 30, 3, 0.002)   # a leaf grid of far more than 2^32 cells
    raw, _, _ = kf.submap(30, 3, 0.002)
    ext = (raw[:, :3].max(0) - raw[:, :3].min(0)) / 0.002
    assert np.prod(ext.astype(np.float64)) > 2.0 ** 32 and len(ds) > 0


@pytest.mark.parametrize("search", [7, 1, 0])
def test_close_equals_pairs_on_downloaded_submaps(api, oracle, store, queries, search):
    b = api.NdtPairBatch(search=search, **NDT)
    r = b.close_loops(store, queries, **LOOP)
    live = [q for q in range(len(queries)) if r["pre"][q] >= 0 and r["status"][q] != NO_EFFECTIVE_POINTS]
    assert len(live) >= 25
    srcs = [store.submap(int(queries[q]), 0, LOOP["leaf"]) for q in live]
    tgts = [store.submap(int(r["pre"][q]), LOOP["search_num"], LOOP["leaf"]) for q in live]
    for k, q in enumerate(live):
        assert (r["n_source"][q], r["n_target"][q]) == (len(srcs[k]), len(tgts[k]))
    rp = api.NdtPairBatch(search=search, **NDT).align(srcs, tgts)
    for k, q in enumerate(live):
        assert reg_bytes(r["loop_records"][q].reg) == reg_bytes(rp["records"][k]), q
    for k in range(0, len(live), 4 if search == 7 else 8):
        q = live[k]
        o = oracle.OracleNdt(search=search, **NDT)
        o.set_target(tgts[k][:, :3])
        o.set_source(srcs[k][:, :3])
        rc0, T0, r0 = o.align(np.eye(4, dtype=np.float32))
        assert r["status"][q] == rc0 and r["converged"][q] == r0.converged, q
        assert (r["iters"][q], r["evals"][q], r["hess_evals"][q]) == (r0.iters, r0.evals, r0.hess_evals), q
        assert np.abs(r["p_final"][q] - np.array(r0.p_final)).max() < 1e-4, q
        assert abs(r["trans_probability"][q] - r0.trans_probability) <= 1e-6 * abs(r0.trans_probability), q
        s0, n0 = o.fitness(r["final"][q])
        assert r["n_in_range"][q] == n0 and abs(r["fitness"][q] - s0) <= 1e-12 * abs(s0), q


def test_determinism(api, store, queries, session, tmp_path):
    """A query's record is bit-identical alone, in a shuffled batch and with 3 queries per chunk in a fresh process."""
    full = api.NdtPairBatch(**NDT).close_loops(store, queries, **LOOP)

    def rb(res, k):
        x = type(res["loop_records"][k]).from_buffer_copy(res["loop_records"][k])
        x.reg.ndt.gpu_ms = 0.0
        return bytes(memoryview(x).cast("B"))
    base = [rb(full, k) for k in range(len(queries))]
    perm = np.random.default_rng(4).permutation(len(queries))
    shuf = api.NdtPairBatch(**NDT).close_loops(store, queries[perm], **LOOP)
    for k, p in enumerate(perm):
        assert rb(shuf, k) == base[p], p
    for p in (0, 5, len(queries) - 1):
        alone = api.NdtPairBatch(**NDT).close_loops(store, queries[p:p + 1], **LOOP)
        assert rb(alone, 0) == base[p], p
    np.savez(tmp_path / "s.npz", poses=session["poses"], times=session["times"], cur=queries,
             **{f"c{k}": c for k, c in enumerate(session["clouds"])})
    script = f"""
import sys, numpy as np
sys.path.insert(0, {ROOT!r})
from pointcloud_slam_b200 import api
d = np.load({str(tmp_path / 's.npz')!r})
st = api.KeyframeStore()
for k in range(len(d["poses"])):
    st.add(d[f"c{{k}}"], d["poses"][k], d["times"][k])
r = api.NdtPairBatch(**{NDT!r}).close_loops(st, d["cur"], **{LOOP!r})
out = []
for x in r["loop_records"][: len(d["cur"])]:
    y = type(x).from_buffer_copy(x)
    y.reg.ndt.gpu_ms = 0.0
    out.append(bytes(memoryview(y).cast("B")).hex())
print("\\n".join(out))
"""
    p = subprocess.run([sys.executable, "-c", script], env=dict(os.environ, B200_NDT_PAIRS_CHUNK="3"), capture_output=True, text=True, timeout=600)
    assert p.returncode == 0, p.stderr[-3000:]
    assert [bytes.fromhex(h) for h in p.stdout.split()] == base


def test_explicit_pre_gates_and_set_poses(api, loop_oracle, session, queries):
    st = make_store(api, session["clouds"], session["poses"], session["times"])
    b = api.NdtPairBatch(**NDT)
    det = b.close_loops(st, queries, **LOOP)
    # an explicit partner overrides the detection; -1 registers nothing
    pre = det["pre"].copy()
    pre[0], pre[1] = int(queries[0]) - 1000, -1
    r = b.close_loops(st, queries, pre=pre, **LOOP)
    assert r["pre"].tolist() == pre.tolist() and r["status"][1] == NO_EFFECTIVE_POINTS and r["n_source"][1] == 0
    assert r["n_target"][0] > 0
    for q in range(2, len(queries)):
        assert r["loop_records"][q].reg.status == det["loop_records"][q].reg.status
    # size gates: reported with the sizes, not registered
    g = b.close_loops(st, queries[:4], pre=det["pre"][:4], **dict(LOOP, min_source_points=10 ** 6))
    assert (g["status"] == NO_EFFECTIVE_POINTS).all() and (g["iters"] == 0).all()
    assert (g["n_source"][det["pre"][:4] >= 0] > 0).all()
    g = b.close_loops(st, queries[:4], pre=det["pre"][:4], **dict(LOOP, min_target_points=10 ** 6))
    assert (g["status"] == NO_EFFECTIVE_POINTS).all()
    # correctPoses: detection and submaps follow the new poses
    poses = session["poses"].copy()
    poses[1000:, :2] -= np.float32(0.7)
    poses[1000:, 5] += np.float32(0.01)
    st.set_poses(1000, poses[1000:])
    cur = np.arange(1000, 2000, 7)
    pre1, d21 = st.detect(cur, **LOOP)
    pre0, d20 = loop_oracle.loop_detect(poses, session["times"], cur, LOOP["search_radius"], LOOP["time_gap"])
    np.testing.assert_array_equal(pre1, pre0)
    np.testing.assert_array_equal(d21, d20)
    kf = loop_oracle.Keyframes(session["clouds"], poses)
    for key in (990, 1500):
        submap_checks(api, st, kf, key, 25, 0.4)


def test_ground_truth(api, oracle, store, queries, session):
    """Accepted loops undo the injected drift as well as the oracle's own align does."""
    r = api.NdtPairBatch(**NDT).close_loops(store, queries, **LOOP)
    Tt, Td = session["T_true"], session["T_drift"]
    yaw = lambda M: np.arctan2(M[1, 0], M[0, 0])
    n = 0
    for q in range(0, len(queries), 3):
        if r["status"][q] != 0:
            continue
        c, p = int(queries[q]), int(r["pre"][q])
        C = (Td[p] @ np.linalg.inv(Tt[p])) @ (Tt[c] @ np.linalg.inv(Td[c]))
        o = oracle.OracleNdt(search=7, **NDT)
        o.set_target(store.submap(p, LOOP["search_num"], LOOP["leaf"])[:, :3])
        o.set_source(store.submap(c, 0, LOOP["leaf"])[:, :3])
        _, T0, _ = o.align(np.eye(4, dtype=np.float32))
        e_dev, e_orc = np.abs(r["final"][q][:3, 3] - C[:3, 3]).max(), np.abs(T0[:3, 3] - C[:3, 3]).max()
        assert e_dev <= e_orc + 1e-4, (q, e_dev, e_orc)
        assert abs(yaw(r["final"][q]) - yaw(C)) <= abs(yaw(T0) - yaw(C)) + 1e-4, q
        n += 1
    assert n >= 8


def test_store_arguments(api, store):
    lib = api.lib()
    prm = api.KeyframeStore.params(**LOOP)
    pre = np.zeros(1, np.int64)
    d2 = np.zeros(1, np.float32)
    n = ctypes.c_int64()
    res = (api.LoopResult * 1)()
    p = lambda a: a.ctypes.data_as(ctypes.c_void_p)
    bad = np.array([len(store)], np.int64)
    assert lib.b200_loop_detect(store.h, p(bad), 1, ctypes.byref(prm), p(pre), p(d2)) == -1        # key out of range
    assert lib.b200_loop_detect(store.h, p(pre), 0, ctypes.byref(prm), p(pre), p(d2)) == -1         # Q < 1
    assert lib.b200_loop_submap(store.h, 0, 2, 0.0, None, 0, ctypes.byref(n)) == -1                 # leaf <= 0
    assert lib.b200_loop_submap(store.h, -1, 2, 0.4, None, 0, ctypes.byref(n)) == -1
    b = api.NdtPairBatch(**NDT)
    assert lib.b200_loop_close(None, b.h, store.h, p(bad), None, 1, ctypes.byref(prm), res) == -1
    assert lib.b200_loop_close(None, b.h, store.h, p(pre), p(bad), 1, ctypes.byref(prm), res) == -1  # partner out of range
    bad_leaf = api.KeyframeStore.params(**dict(LOOP, leaf=-1.0))
    assert lib.b200_loop_close(None, b.h, store.h, p(pre), None, 1, ctypes.byref(bad_leaf), res) == -1
    assert lib.b200_loop_close(None, b.h, store.h, p(pre), None, 0, ctypes.byref(prm), res) == -1
    assert lib.b200_keyframes_set_poses(store.h, len(store), 1, p(np.zeros(6, np.float32))) == -1
    import torch
    if torch.cuda.device_count() >= 2:   # store and pairs handle on different devices
        st1 = api.KeyframeStore(device=1)
        st1.add(np.ones((4, 4), np.float32), np.zeros(6, np.float32), 0.0)
        assert lib.b200_loop_close(None, b.h, st1.h, p(pre), None, 1, ctypes.byref(prm), res) == -1
        assert b"different devices" in lib.b200_last_error()


def test_cpp_adaptor_closes_a_loop(tmp_path, api):
    from test_loop_cpu import build_adaptor
    exe = build_adaptor(tmp_path, api)
    p = subprocess.run([exe], capture_output=True, text=True)
    assert p.returncode == 0 and "loop closure adaptor ok" in p.stdout, p.stdout + p.stderr
