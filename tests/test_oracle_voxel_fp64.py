"""The voxel-grid and undistortion oracles (fp32, the device's operation order) against an independent fp64 restatement
(tests/voxel_ref.py): the PCL partition, counts and order at leaves 0.01 / 0.1 / 1.0 near the origin and kilometres
away, min_points, the max-corner voxel of a grid above 2^53 leaves, the full-map builder and the closed-form motions of
the undistortion.  With the device-to-oracle parity of the GPU tests this ties the device to fp64 math."""
import numpy as np
import pytest

import voxel_ref as vr

LEAVES = (0.01, 0.1, 1.0)


def hall(synth, offset=(0.0, 0.0, 0.0)):
    from test_gpu_voxel import make_frames
    frames, _ = make_frames(synth, k=1, n=6000)
    f = frames[0].copy()
    f[:, :3] = (f[:, :3].astype(np.float64) + offset).astype(np.float32)
    return f


def lattice(leaf):
    """Points on exact float32 leaf multiples, negative and straddling 0, plus a jittered copy."""
    k = np.arange(-12, 13, dtype=np.float64)
    g = np.stack(np.meshgrid(k, k[::3], k[::4], indexing="ij"), -1).reshape(-1, 3) * leaf
    rng = np.random.default_rng(11)
    jit = g + rng.uniform(-0.5, 0.5, g.shape) * leaf
    p = np.concatenate([g, jit]).astype(np.float32)
    return np.concatenate([p, rng.uniform(0, 255, (len(p), 1)).astype(np.float32)], 1)


CLOUDS = {
    "hall": lambda synth: hall(synth),
    "lattice": None,
    "hall_2km": lambda synth: hall(synth, (2000.0, 300.0, 0.0)),
    "hall_50km": lambda synth: hall(synth, (50000.0, -50000.0, 10.0)),
}


def cloud(name, synth, leaf):
    return lattice(leaf) if name == "lattice" else CLOUDS[name](synth)


def check_against_ref(c0, n0, xyzi, leaf, min_points=0):
    cent, cnt, _ = vr.voxel_grid(xyzi, leaf, min_points)
    np.testing.assert_array_equal(n0, cnt)                     # same partition, same order (counts in leaf-index order)
    xyz, inten = vr._records(xyzi)
    a = np.concatenate([xyz, inten[:, None]], 1)[np.isfinite(xyz).all(1)]
    maxabs = np.abs(a).max(0) if len(a) else np.zeros(4)
    bound = vr.running_sum_bound(cnt, 1.0)[:, None] * maxabs[None, :]   # fp32 running sums of coordinates (and intensity)
    assert (np.abs(c0 - cent) <= bound).all()
    return cent, cnt


@pytest.mark.parametrize("leaf", LEAVES)
@pytest.mark.parametrize("name", list(CLOUDS))
def test_partition_matches_fp64(oracle, synth, name, leaf):
    p = cloud(name, synth, leaf)
    c0, n0 = oracle.voxel_grid(p, leaf)
    check_against_ref(c0, n0, p, leaf)
    assert n0.sum() == len(p)


@pytest.mark.parametrize("min_points", [0, 1, 2, 5, 1_000_000])
def test_min_points_matches_fp64(oracle, synth, min_points):
    p = hall(synth)
    c0, n0 = oracle.voxel_grid(p, 0.2, min_points)
    check_against_ref(c0, n0, p, 0.2, min_points)
    assert (n0 >= min_points).all()


def test_max_corner_voxel_kept_above_2_53_leaves(oracle):
    """(0,0,0) and (3000,3000,3000) at leaf 0.01: 300001^3 = 27000270000900001 leaves, which rounds to ...900000 in double,
    the index of the max-corner leaf.  Both voxels exist."""
    p = np.array([[0, 0, 0, 1], [3000, 3000, 3000, 2]], np.float32)
    cells = 300001 ** 3
    assert cells > 2 ** 53 and int(float(cells)) == cells - 1
    cent, cnt, idx = vr.voxel_grid(p, 0.01)
    assert list(cnt) == [1, 1] and idx[-1] == cells - 1
    c0, n0 = oracle.voxel_grid(p, 0.01)
    np.testing.assert_array_equal(n0, [1, 1])
    np.testing.assert_array_equal(c0, p)


@pytest.mark.parametrize("offset", [(0.0, 0.0, 0.0), (2000.0, 300.0, 0.0)], ids=["origin", "2km"])
def test_full_map_matches_fp64(oracle, synth, offset):
    from test_gpu_voxel import make_frames
    frames, poses = make_frames(synth, k=4, n=3000)
    poses[:, :3] += offset
    c0, n0 = oracle.full_map(frames, poses, 0.1)
    ref = vr.map_build(frames, poses, 0.1)
    np.testing.assert_array_equal(n0, ref["counts"])
    assert ref["out_of_range"] == 0
    maxabs = np.abs(ref["pts"]).max(0).astype(np.float64)
    # the oracle sums absolute fp32 coordinates: the running-sum bound grows with the distance from the origin
    assert (np.abs(c0 - ref["cent"]) <= vr.running_sum_bound(ref["counts"], 1.0)[:, None] * maxabs[None, :]).all()


def timed_scan(n, T, seed, t_min_ms=0.5):
    rng = np.random.default_rng(seed)
    pts = np.zeros((n, 12), np.float32)
    pts[:, :3] = rng.uniform(-30, 30, (n, 3))
    pts[:, 8] = rng.uniform(0, 255, n)
    pts[:, 9] = rng.uniform(t_min_ms, T * 1000.0, n)
    return pts


MOTIONS = {"rest": {}, "velocity": dict(vel=(1.5, -0.4, 0.2)), "yaw": dict(yaw_rate=0.9, ext_t=(0.04, -0.02, 0.1))}


@pytest.mark.parametrize("motion", list(MOTIONS))
def test_undistort_closed_forms(oracle, motion):
    kw = MOTIONS[motion]
    poses, x_end, T = vr.imu_motion(0.01 * np.arange(11), **kw)
    # the last 4 ms lie after the last pose; with the velocity the earliest point is in segment 5 of 10
    pts = timed_scan(4000, T + 0.004, seed=21, t_min_ms=55.0 if motion == "velocity" else 0.5)
    out, order = oracle.undistort(pts, 9, 8, poses, x_end)
    t = pts[order, 9].astype(np.float64) / 1000.0
    ref = vr.undistort_closed_form(pts[order, :3], t, T, **kw)
    # fp64 chain narrowed to fp32 (half an ulp of a 30-50 m coordinate is <= 1.9e-6) and libm sin/cos: 4e-6 m
    np.testing.assert_allclose(out[1:, :3], ref[1:], rtol=0, atol=4e-6)
    if motion == "rest":
        np.testing.assert_array_equal(out[:, :3], pts[order, :3])
    if motion == "velocity":
        # the earliest point is compensated again by every earlier segment (imu_processing.hpp:279-281): with a pure
        # translation, once per segment up to its own
        lo = int(np.searchsorted(poses[:, 0], t[0], side="left")) - 1
        assert lo == 5
        shift = (ref[0] - pts[order[0], :3]) * (lo + 1)
        np.testing.assert_allclose(out[0, :3], pts[order[0], :3] + shift, rtol=0, atol=4e-6)
