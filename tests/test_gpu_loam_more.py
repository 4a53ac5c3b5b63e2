"""GPU LOAM scan-to-map (b200_loam_*) beyond the one well-conditioned scene of test_gpu_loam.py: large rotations, a
degenerate corridor, the host's convergence polling, map replacement on one handle (both insert paths, capacity), every
candidate walk of the search, strided records, empty feature classes, more features than one grid pass covers, and the exact
range gate and distance ties.  Each case is compared with the fp32 oracle (bit for bit where the operation order is the same)
and with the fp64 restatement of tests/loam_ref.py."""
import os
import subprocess
import sys

import numpy as np
import pytest

import loam_ref as lr

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GUESS = np.array([0.01, -0.01, 0.02, 0.15, -0.1, 0.05], np.float32)
EMPTY = np.zeros((0, 3), np.float32)


def handle(oracle, api, corner_map, surf_map, max_map_points=200_000):
    o = oracle.OracleLoam()
    o.set_map(corner_map, surf_map)
    g = api.ScanToMap(max_map_points=max_map_points)
    g.setInputCloud(corner_map, surf_map)
    return o, g


def features_equal(o, g, corner, surf, t6):
    n0, f0, c0 = o.features(corner, surf, t6)
    n1, f1, c1 = g.features(corner, surf, t6)
    assert n1 == n0
    np.testing.assert_array_equal(f1, f0)
    np.testing.assert_array_equal(c1, c0)
    return f1, c1


def optimize_equal(o, g, corner, surf, guess, iter_num=30):
    t0, s0 = o.optimize(corner, surf, guess, iter_num=iter_num)
    t1, rc = g.scan2MapOptimization(corner, surf, guess, iter_num=iter_num)
    st = g.stats
    assert rc == (0 if s0["converged"] else 2)
    assert (st.iters, st.converged, st.degenerate, st.n_sel) == (s0["iters"], int(s0["converged"]), int(s0["degenerate"]), s0["n_sel"])
    np.testing.assert_allclose(t1, t0, rtol=0, atol=1e-6)
    return t1, rc, np.array(st.AtA_first).reshape(6, 6)


@pytest.fixture(scope="module")
def scene(synth):
    return synth.loam_scene()


@pytest.fixture(scope="module", params=lr.LARGE_ANGLE_POSES, ids=lambda t: "rpy=%g,%g,%g" % t[:3])
def rotated(request, synth):
    return synth.loam_scene(t_true=request.param)


def test_large_rotation_features(oracle, api, rotated):
    sc = rotated
    o, g = handle(oracle, api, sc["corner_map"], sc["surf_map"])
    for t6 in (sc["t_true"], sc["t_true"] + GUESS):
        flags, coeff = features_equal(o, g, sc["corner"], sc["surf"], t6)
        lr.check_features(lr.Pass(sc["corner_map"], sc["surf_map"], sc["corner"], sc["surf"], t6), flags, coeff)


def test_large_rotation_optimize(oracle, api, rotated):
    sc = rotated
    o, g = handle(oracle, api, sc["corner_map"], sc["surf_map"])
    guess = sc["t_true"] + GUESS
    t1, rc, AtA = optimize_equal(o, g, sc["corner"], sc["surf"], guess)
    _, flags, coeff = g.features(sc["corner"], sc["surf"], guess)
    assert lr.rel_err(AtA, lr.jtj(sc["corner"], sc["surf"], flags, coeff, guess)) <= 1e-5
    if sc["t_true"][1] > 1.0:   # pitch 1.3: no convergence within the 30 passes
        assert rc == 2 and g.stats.iters == 30
    else:
        assert rc == 0 and np.abs(t1[3:] - sc["t_true"][3:]).max() < 0.01


def test_degenerate_corridor_projects_the_step(oracle, api):
    sc = lr.corridor()
    o, g = handle(oracle, api, sc["corner_map"], sc["surf_map"])
    guess = sc["t_true"] + GUESS
    features_equal(o, g, sc["corner"], sc["surf"], guess)
    t, rc, _ = optimize_equal(o, g, sc["corner"], sc["surf"], guess)
    assert g.stats.degenerate == 1 and rc == 0
    assert abs(t[3] - guess[3]) < 1e-3        # the weak direction (x, along the corridor) is left alone
    t1, _, AtA = optimize_equal(o, g, sc["corner"], sc["surf"], guess, iter_num=1)
    lam = np.linalg.eigvalsh(AtA)
    assert lam[0] < 100 < lam[1]
    assert lr.weak_step_fraction(AtA, guess, t1) <= 1e-5


def test_poll_batches(oracle, api, synth):
    """The host polls the done flag after 6, 10, 14 ... passes: iteration counts on both sides of each boundary."""
    for pose, conv_at in ((lr.LARGE_ANGLE_POSES[0], 11), (lr.LARGE_ANGLE_POSES[2], 10)):
        sc = synth.loam_scene(t_true=pose)
        o, g = handle(oracle, api, sc["corner_map"], sc["surf_map"])
        guess = sc["t_true"] + GUESS
        optimize_equal(o, g, sc["corner"], sc["surf"], guess)
        assert g.stats.iters == conv_at and g.stats.converged
        if conv_at == 11:
            for it in (1, 5, 6, 7, 10, 11):
                _, rc, _ = optimize_equal(o, g, sc["corner"], sc["surf"], guess, iter_num=it)
                assert g.stats.iters == it and rc == (0 if it == 11 else 2)


def test_map_lifecycle_on_one_handle(oracle, api, synth, scene):
    big = synth.loam_scene(n_surf_map=250_000)["surf_map"]
    _, nvox, mx = lr.stencil_candidates(big, big[:1])
    assert len(big) > 6 * nvox      # dense enough for the cooperative walk (mode 1)
    cm, s60 = scene["corner_map"], scene["surf_map"]
    maps = (("250k", cm, big), ("60k", cm, s60), ("no corner map", EMPTY, s60), ("65536", cm, big[:65536]),
            ("65537", cm, big[:65537]), ("small", cm[::4], s60[::20]))
    g = api.ScanToMap(max_map_points=len(big))
    guess = scene["t_true"] + GUESS
    for name, c, s in maps:
        g.setInputCloud(c, s)
        o = oracle.OracleLoam()
        o.set_map(c, s)
        for t6 in (scene["t_true"], guess):
            flags, coeff = features_equal(o, g, scene["corner"], scene["surf"], t6)
        if name == "no corner map":
            assert not flags[:len(scene["corner"])].any()
        if name in ("60k", "65537", "small"):
            optimize_equal(o, g, scene["corner"], scene["surf"], guess)
    # one point over the capacity is refused and leaves the previous maps in force
    with pytest.raises(api.B200Error):
        g.setInputCloud(cm, np.concatenate([big, big[:1]]))
    with pytest.raises(api.B200Error):
        g.setInputCloud(np.concatenate([big, big[:1]]), s60)
    _, f1, c1 = g.features(scene["corner"], scene["surf"], guess)
    np.testing.assert_array_equal(f1, flags)
    np.testing.assert_array_equal(c1, coeff)


def run_mode(mode, path):
    env = dict(os.environ)
    env.pop("B200_KNN_MODE", None)
    if mode is not None:
        env["B200_KNN_MODE"] = str(mode)
    p = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "helpers", "loam_mode_worker.py"), str(path)], env=env,
                       capture_output=True, text=True, timeout=600)
    assert p.returncode == 0, p.stderr[-2000:]
    return dict(np.load(path))


def test_walk_variants_agree(oracle, tmp_path):
    scenes = lr.mode_scenes()
    # regimes on numpy voxel counts: the sparse surf map takes the lane-owned walk (0) and fits the flat list of walk 5, the
    # dense one takes the cooperative walk (1) and overflows the flat list (64 candidates) on almost every query
    for name, sc in scenes.items():
        q = lr.to_world(sc["surf"], sc["guess"]).astype(np.float32)
        cand, nvox, mx = lr.stencil_candidates(sc["surf_map"], q)
        dense = len(sc["surf_map"]) > 6 * nvox or mx > 32
        if name == "sparse":
            assert not dense and (cand > 64).mean() < 0.01
        else:
            assert dense and (cand > 64).mean() > 0.9
    ref = {}
    for name, sc in scenes.items():
        o = oracle.OracleLoam()
        o.set_map(sc["corner_map"], sc["surf_map"])
        _, ref[name + "_flags"], ref[name + "_coeff"] = o.features(sc["corner"], sc["surf"], sc["guess"])
        ref[name + "_t6"], s0 = o.optimize(sc["corner"], sc["surf"], sc["guess"])
        ref[name + "_stats"] = [0 if s0["converged"] else 2, s0["iters"], s0["n_sel"], int(s0["converged"]), int(s0["degenerate"])]
    first = None
    for mode in (None, 0, 1, 5):
        got = run_mode(mode, tmp_path / f"mode_{mode}.npz")
        for name in scenes:
            for k in ("flags", "coeff", "stats"):
                np.testing.assert_array_equal(got[f"{name}_{k}"], ref[f"{name}_{k}"], err_msg=f"{mode} {name} {k}")
            np.testing.assert_allclose(got[f"{name}_t6"], ref[f"{name}_t6"], rtol=0, atol=1e-6, err_msg=f"{mode} {name}")
        if first is None:
            first = got
        for k in got:    # identical across the walks, bit for bit (t6 and A^T A included)
            np.testing.assert_array_equal(got[k], first[k], err_msg=f"{mode} {k}")


def test_record_layouts(oracle, api, scene):
    """16-byte and 32-byte point records (x, y, z, then padding / intensity ...) give what packed 12-byte records give."""
    rng = np.random.default_rng(3)

    def widen(a, cols):
        w = rng.standard_normal((len(a), cols)).astype(np.float32) * 1e3
        w[:, :3] = a
        return w

    guess = scene["t_true"] + GUESS
    o, g = handle(oracle, api, scene["corner_map"], scene["surf_map"])
    _, f0, c0 = g.features(scene["corner"], scene["surf"], guess)
    t0, rc0 = g.scan2MapOptimization(scene["corner"], scene["surf"], guess)
    A0 = np.array(g.stats.AtA_first)
    for cols in (4, 8):
        g.setInputCloud(widen(scene["corner_map"], cols), widen(scene["surf_map"], cols))
        wc, ws = widen(scene["corner"], cols), widen(scene["surf"], cols)
        assert wc.strides[0] == 4 * cols
        _, f1, c1 = g.features(wc, ws, guess)
        np.testing.assert_array_equal(f1, f0)
        np.testing.assert_array_equal(c1, c0)
        t1, rc1 = g.scan2MapOptimization(wc, ws, guess)
        assert rc1 == rc0
        np.testing.assert_array_equal(t1, t0)
        np.testing.assert_array_equal(np.array(g.stats.AtA_first), A0)
        _, f2, c2 = g.features(wc[:, :3], ws[:, :3], guess)      # a strided view of the wide records
        np.testing.assert_array_equal(f2, f0)
        np.testing.assert_array_equal(c2, c0)


def test_empty_feature_classes(oracle, api, scene):
    o, g = handle(oracle, api, scene["corner_map"], scene["surf_map"])
    guess = scene["t_true"] + GUESS
    for corner, surf in ((EMPTY, scene["surf"]), (scene["corner"], EMPTY)):
        features_equal(o, g, corner, surf, guess)
        optimize_equal(o, g, corner, surf, guess)


def test_more_features_than_one_grid_pass(oracle, api, synth, scene):
    """> MAXB x 256 = 262144 feature points: every accumulation thread takes several points (grid-stride loop)."""
    surf_map = synth.loam_scene(n_surf_map=20_000)["surf_map"]
    rng = np.random.default_rng(7)
    near = surf_map[np.linalg.norm(surf_map - scene["t_true"][3:], axis=1) < 25]
    pw = near[rng.integers(0, len(near), 280_000)] + rng.normal(0, 0.01, (280_000, 3)).astype(np.float32)
    surf = lr.to_body(pw, scene["t_true"])
    corner = scene["corner"]
    assert len(corner) + len(surf) > 1024 * 256
    o, g = handle(oracle, api, scene["corner_map"], surf_map)
    guess = scene["t_true"] + GUESS
    flags, coeff = features_equal(o, g, corner, surf, guess)
    assert flags[1024 * 256:].sum() > 1000       # selected features past the first grid pass
    _, _, AtA = optimize_equal(o, g, corner, surf, guess, iter_num=1)
    assert lr.rel_err(AtA, lr.jtj(corner, surf, flags, coeff, guess)) <= 1e-5


def test_range_gate_and_ties(oracle, api):
    surf_map, scan = lr.lattice()
    t0 = np.zeros(6, np.float32)
    o, g = handle(oracle, api, EMPTY, surf_map)
    n0, f0, c0 = o.features(EMPTY, scan, t0)
    n1, f1, c1 = g.features(EMPTY, scan, t0)
    # the 5th neighbour at exactly d2 = 1.0 fails the gate, one at the float below 1.0 passes; numpy agrees
    d5 = np.array([np.sort(lr.fp32_d2(surf_map, q))[4] for q in scan[:2]])
    assert d5[0] == np.float32(1) and d5[1] == np.nextafter(np.float32(1), np.float32(0))
    np.testing.assert_array_equal(f0[:2], [0, 1])
    np.testing.assert_array_equal(f1[:2], [0, 1])
    np.testing.assert_array_equal(c1[:2], c0[:2])    # no ties: same neighbours in the same order
    # ties inside the five: the same set, but the device orders tied neighbours by (stencil cell, in-voxel index) and the
    # oracle by map index, so the plane fit sees its rows in another order: equal up to fp32 rounding
    assert f1[2] == f0[2] == 1
    np.testing.assert_allclose(c1[2], c0[2], rtol=0, atol=1e-6)
    # a tie between the 5th and the 6th neighbour: FLANN leaves the choice open, the device must return a valid 5-NN set
    base = [lr.TIE56_Q, (29.5, 0, 5), (30, 0.5, 5), (30, -0.5, 5)]
    q = np.array(lr.TIE56_Q, np.float64)
    options = []
    for extra in (lr.TIE56_A, lr.TIE56_B):
        sel, co, _ = lr.Pass._surf(np.array(base + [extra], np.float64), q)
        options.append((1, co) if sel else (0, np.zeros(4)))
    assert options[0][0] != options[1][0] or np.abs(options[0][1] - options[1][1]).max() > 1e-3   # the choice is visible
    assert any(f1[3] == fl and np.abs(c1[3] - co).max() < 1e-5 for fl, co in options), (f1[3], c1[3], options)
