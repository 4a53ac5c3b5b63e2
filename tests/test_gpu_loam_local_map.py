"""The LOAM local map built from the device keyframe store (b200_keyframes_surrounding[_map], b200_loam_set_map_from_keyframes):
the keyframe list and both downsampled maps bit-exact against the oracle, the LOAM handle afterwards byte-equal to
b200_loam_set_map with the same clouds, an end-to-end scan-to-map run, pose updates, the error cases, and loop-closure results
independent of the add call that built the store."""
import subprocess

import numpy as np
import pytest

from test_loam_local_map_cpu import build_adaptor

pytestmark = pytest.mark.gpu
F = np.float32
NO_EFFECTIVE_POINTS, ERR_ARG, ERR_CAPACITY = 1, -1, -5


@pytest.fixture(scope="module")
def surround_oracle():
    from oracle import surround_binding
    surround_binding.build()
    return surround_binding


@pytest.fixture(scope="module")
def session(synth):
    """Two laps of 160 keyframes, each cloud split into a corner head (a fifth) and a surf tail; a few degenerate splits."""
    s = synth.loop_session(K=160, n_points=1500, laps=2)
    clouds = [np.asarray(c, F) for c in s["clouds"]]
    n_corner = np.array([len(c) // 5 for c in clouds], np.int64)
    clouds[3] = clouds[3][:0]
    n_corner[3] = 0
    n_corner[10] = 0
    n_corner[20] = len(clouds[20])
    return dict(clouds=clouds, n_corner=n_corner, poses=s["poses"].copy(), times=s["times"].copy())


def make_store(api, sess, features=True):
    st = api.KeyframeStore()
    for c, nc, p, t in zip(sess["clouds"], sess["n_corner"], sess["poses"], sess["times"]):
        if features:
            st.add_features(c[:nc], c[nc:], p, t)
        else:
            st.add(c, p, t)
    return st


@pytest.fixture(scope="module")
def store(api, session):
    return make_store(api, session)


def oracle_map(surround_oracle, sess, cur, time_cur, **kw):
    kf = surround_oracle.Keyframes(sess["clouds"], sess["poses"], sess["times"], sess["n_corner"])
    return kf.surrounding(cur, time_cur, **kw)


def bits(a):
    return np.ascontiguousarray(a, F).view(np.uint32)


@pytest.mark.parametrize("radius", [8.0, 50.0])
def test_list_and_maps_bit_exact_against_the_oracle(api, surround_oracle, session, store, radius):
    for cur in (0, 1, 17, 79, 80, 81, 120, 159):
        tc = session["times"][cur] + 0.25
        keys_o, n_list_o, co, so = oracle_map(surround_oracle, session, cur, tc, search_radius=radius)
        keys = store.surrounding(cur, tc, search_radius=radius)
        assert keys.tolist() == keys_o.tolist(), (radius, cur)
        gc, gs = store.surrounding_map(cur, tc, search_radius=radius)
        assert np.array_equal(bits(gc), bits(co)) and np.array_equal(bits(gs), bits(so)), (radius, cur)
    assert len(store.surrounding(-1, session["times"][-1], search_radius=radius)) > 0


def test_loam_maps_byte_equal_to_set_map(api, oracle, session, store):
    cur = 150
    tc = session["times"][cur] + 0.1
    co, so = store.surrounding_map(cur, tc)
    a, b = api.ScanToMap(max_map_points=400_000), api.ScanToMap(max_map_points=400_000)
    info = a.extractSurroundingKeyFrames(store, cur, tc)
    b.setInputCloud(co[:, :3], so[:, :3])
    assert info.n_corner == len(co) and info.n_surf == len(so) and info.n_kept <= info.n_list and info.gpu_ms > 0
    assert info.n_corner_raw >= len(co) and info.n_surf_raw >= len(so)
    o = oracle.OracleLoam()
    o.set_map(co[:, :3], so[:, :3])
    # a scan: keyframe cur's own features, seen from a perturbed pose
    c = session["clouds"][cur]
    nc = session["n_corner"][cur]
    p = session["poses"][cur]
    t_true = np.array([p[3], p[4], p[5], p[0], p[1], p[2]], F)
    corner, surf = np.ascontiguousarray(c[:nc, :3]), np.ascontiguousarray(c[nc:, :3])
    for d in ([0, 0, 0, 0, 0, 0], [0.01, -0.01, 0.02, 0.15, -0.1, 0.05]):
        t6 = t_true + np.array(d, F)
        n1, f1, c1 = a.features(corner, surf, t6)
        n2, f2, c2 = b.features(corner, surf, t6)
        n0, f0, c0 = o.features(corner, surf, t6)
        assert n1 == n2 == n0
        assert f1.tobytes() == f2.tobytes() and c1.tobytes() == c2.tobytes()
        np.testing.assert_array_equal(c1, c0)
    guess = t_true + np.array([0.01, -0.01, 0.02, 0.15, -0.1, 0.05], F)
    t1, rc1 = a.scan2MapOptimization(corner, surf, guess)
    s1 = (a.stats.iters, a.stats.n_sel, a.stats.converged)
    t2, rc2 = b.scan2MapOptimization(corner, surf, guess)
    assert rc1 == rc2 and t1.tobytes() == t2.tobytes() and s1 == (b.stats.iters, b.stats.n_sel, b.stats.converged)
    t0, s0 = o.optimize(corner, surf, guess)
    assert a.stats.iters == s0["iters"] and a.stats.n_sel == s0["n_sel"]
    np.testing.assert_allclose(t1, t0, rtol=0, atol=1e-6)


def test_end_to_end_scan_to_map(api, synth):
    """Keyframes of the LOAM scene's maps along a short trajectory, then the scene's scan from a perturbed guess."""
    sc = synth.loam_scene()
    st = api.KeyframeStore()
    t_true = sc["t_true"]
    for k in range(12):
        pos = np.array([t_true[3] - 6.0 + k, t_true[4] + 0.3 * np.sin(k), t_true[5]], F)
        sel_c = np.linalg.norm(sc["corner_map"] - pos, axis=1) < 30
        sel_s = np.linalg.norm(sc["surf_map"] - pos, axis=1) < 30
        st.add_features((sc["corner_map"][sel_c] - pos).astype(F), (sc["surf_map"][sel_s] - pos).astype(F), [pos[0], pos[1], pos[2], 0, 0, 0], float(k))
    g = api.ScanToMap(max_map_points=400_000)
    info = g.extractSurroundingKeyFrames(st, -1, 12.0)
    assert info.n_corner > 1000 and info.n_surf > 1000
    guess = t_true + np.array([0.01, -0.01, 0.02, 0.15, -0.1, 0.05], F)
    t1, rc = g.scan2MapOptimization(sc["corner"], sc["surf"], guess)
    assert rc == 0
    assert np.abs(t1[3:] - t_true[3:]).max() < 0.01


def test_set_poses_between_calls(api, surround_oracle, session):
    st = make_store(api, session)
    sess = dict(session, poses=session["poses"].copy())
    cur, tc = 140, session["times"][140] + 0.5
    before = st.surrounding_map(cur, tc)
    rng = np.random.default_rng(9)
    new = sess["poses"][60:150].copy()
    new[:, :2] += rng.normal(0, 0.3, (len(new), 2)).astype(F)
    new[:, 5] += F(0.01)
    st.set_poses(60, new)
    sess["poses"][60:150] = new
    keys_o, _, co, so = oracle_map(surround_oracle, sess, cur, tc)
    assert st.surrounding(cur, tc).tolist() == keys_o.tolist()
    gc, gs = st.surrounding_map(cur, tc)
    assert np.array_equal(bits(gc), bits(co)) and np.array_equal(bits(gs), bits(so))
    assert gc.tobytes() != before[0].tobytes()


def test_error_cases(api, session, store):
    lib = api.lib()
    prm = api.KeyframeStore.surround_params()
    info = api.SurroundInfo()
    g = api.ScanToMap(max_map_points=400_000)
    cur, tc = 100, session["times"][100] + 0.1
    co, so = store.surrounding_map(cur, tc)
    g.extractSurroundingKeyFrames(store, cur, tc)
    c = session["clouds"][cur]
    nc = session["n_corner"][cur]
    p = session["poses"][cur]
    t6 = np.array([p[3], p[4], p[5], p[0], p[1], p[2]], F)
    ref = g.features(c[:nc, :3], c[nc:, :3], t6)
    # an empty store: NO_EFFECTIVE_POINTS, the maps stay
    empty = api.KeyframeStore()
    assert lib.b200_loam_set_map_from_keyframes(g.h, empty.h, -1, 0.0, prm, info) == NO_EFFECTIVE_POINTS
    assert g.extractSurroundingKeyFrames(empty, -1, 0.0) is None and empty.surrounding(-1, 0.0) is None
    got = g.features(c[:nc, :3], c[nc:, :3], t6)
    assert got[0] == ref[0] and got[1].tobytes() == ref[1].tobytes() and got[2].tobytes() == ref[2].tobytes()
    # a map larger than max_map_points: CAPACITY before the maps are cleared
    small = api.ScanToMap(max_map_points=max(16, min(len(co), len(so)) - 1))
    small.setInputCloud(co[:10, :3], so[:10, :3])
    n0 = small.features(c[:nc, :3], c[nc:, :3], t6)
    assert lib.b200_loam_set_map_from_keyframes(small.h, store.h, cur, tc, prm, info) == ERR_CAPACITY
    n1 = small.features(c[:nc, :3], c[nc:, :3], t6)
    assert n0[1].tobytes() == n1[1].tobytes() and n0[2].tobytes() == n1[2].tobytes()
    # a keyframe without a split
    plain = api.KeyframeStore()
    for k in range(5):
        plain.add(session["clouds"][k], session["poses"][k], session["times"][k])
    assert lib.b200_loam_set_map_from_keyframes(g.h, plain.h, -1, 5.0, prm, info) == ERR_ARG
    assert b"split" in lib.b200_last_error()
    # bad arguments
    assert lib.b200_loam_set_map_from_keyframes(g.h, store.h, len(session["clouds"]), tc, prm, info) == ERR_ARG
    assert lib.b200_loam_set_map_from_keyframes(g.h, store.h, cur, tc, api.KeyframeStore.surround_params(density=0.0), info) == ERR_ARG
    got = g.features(c[:nc, :3], c[nc:, :3], t6)
    assert got[1].tobytes() == ref[1].tobytes() and got[2].tobytes() == ref[2].tobytes()


def test_loop_closure_independent_of_the_add_call(api, session, store):
    plain = make_store(api, session, features=False)
    for key, num in [(0, 3), (40, 5), (159, 25)]:
        a, b = store.submap(key, num, 0.4), plain.submap(key, num, 0.4)
        assert a.tobytes() == b.tobytes()
    pa, da = store.detect(np.arange(100, 160, 7), search_radius=15.0, time_gap=30.0)
    pb, db = plain.detect(np.arange(100, 160, 7), search_radius=15.0, time_gap=30.0)
    assert pa.tolist() == pb.tolist() and da.tobytes() == db.tobytes()
    ndt = api.NdtPairBatch()
    ra = ndt.close_loops(store, np.arange(100, 160, 7))
    rb = ndt.close_loops(plain, np.arange(100, 160, 7))
    def record(x):   # the record without its timing
        y = type(x).from_buffer_copy(x)
        y.reg.ndt.gpu_ms = 0.0
        return bytes(y)
    assert [record(x) for x in ra["loop_records"]] == [record(x) for x in rb["loop_records"]]
    assert (ra["status"] != 1).sum() > 0


def test_cpp_adaptor_runs(tmp_path, api):
    exe = build_adaptor(tmp_path, api)
    r = subprocess.run([exe], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "local map adaptor ok" in r.stdout, r.stdout + r.stderr
