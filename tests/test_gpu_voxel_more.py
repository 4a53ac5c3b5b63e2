"""csrc/voxel.cu where the first tests never ran it: the scan downsample on grids above 2^53 leaves, far from the origin, at
scale and with every record stride; the undistortion at its time edges; the full-map builder at its key range, its
capacity, far from the origin, with a keyframe large enough for the grid-stride loop and in every batching.  Each case
is checked against the oracle (bit for bit where the operation order is the same) and against the fp64 reference
tests/voxel_ref.py, with the tolerance stated where it is used."""
import ctypes as C
import os
import signal
import subprocess
import sys
import json

import numpy as np
import pytest

import voxel_ref as vr
from conftest import ROOT
from test_gpu_voxel import imu_scene, make_frames
from test_oracle_voxel_fp64 import CLOUDS, LEAVES, MOTIONS, check_against_ref, cloud, timed_scan

pytestmark = pytest.mark.gpu

ERR_ARG, ERR_RANGE = -1, -4
IDENTITY7 = np.array([0.0, 0.0, 0.0, 1.0, 0.0, 0.0, 0.0])


def downsample(api, vg, rec, leaf, min_points=0, max_out=None):
    """b200_voxel_downsample on the records at their own stride: (rc, n_out, centroids, counts, rows past max_out)."""
    a = np.ascontiguousarray(rec, np.float32)
    cap = len(a) if max_out is None else max_out
    out = np.full((cap + 4, 4), np.nan, np.float32)
    cnt = np.full(cap + 4, -1, np.int32)
    m = C.c_int64(-7)
    rc = api.lib().b200_voxel_downsample(vg.h, api._p(a), len(a), a.strides[0], leaf, min_points, api._p(out), api._p(cnt), cap, C.byref(m))
    k = min(m.value, cap) if rc == 0 else 0
    return rc, m.value, out[:k], cnt[:k], (out[k:], cnt[k:])


def assert_downsample_parity(oracle, api, vg, rec, leaf, min_points=0):
    rc, m, c1, n1, _ = downsample(api, vg, rec, leaf, min_points)
    assert rc == 0 and m == len(c1)
    c0, n0 = oracle.voxel_grid(rec, leaf, min_points)
    np.testing.assert_array_equal(n1, n0)
    np.testing.assert_array_equal(c1, c0)          # the same fp32 sums in the same (input) order
    check_against_ref(c1, n1, np.asarray(rec, np.float32), leaf, min_points)
    return c1, n1


# ------------------------------------------------------------------ downsample
GRIDS = {  # name: (points, leaf); the extents' product is the number of leaves
    "3000m_1cm": ([[0, 0, 0], [3000, 3000, 3000]], 0.01),              # 300001^3: double rounds down onto the last index
    "650m_2.5mm": ([[0, 0, 0], [650, 650, 650]], 0.0025),              # 260001^3: the same
    "under_2^53": ([[0, 0, 0], [262144.5, 262144.5, 131070.5]], 1.0),   # 262145^2 * 131071 = 2^53 - 393217
    "over_2^53": ([[0, 0, 0], [262144.5, 262146.5, 131070.5]], 1.0),    # 262145 * 262147 * 131071 = 2^53 + 68718821373
}


@pytest.mark.parametrize("name", list(GRIDS))
def test_downsample_max_corner_voxel_near_2_53_leaves(oracle, api, name):
    pts, leaf = GRIDS[name]
    p = np.array(pts, np.float32)
    rng = np.random.default_rng(1)
    p = np.concatenate([p, p[1] * rng.uniform(0, 1, (200, 3)).astype(np.float32)])   # points inside as well
    p = np.concatenate([p, np.arange(len(p), dtype=np.float32)[:, None]], 1)
    c, n = assert_downsample_parity(oracle, api, api.VoxelGrid(), p, leaf)
    assert n.sum() == len(p)
    np.testing.assert_array_equal(c[-1, :3], p[1, :3])        # the max-corner voxel holds the far point alone


@pytest.mark.parametrize("extent, leaf", [(3000.0, 1e-4), (2100.0, 1e-3)], ids=["over_2^64", "over_9e18"])
def test_downsample_refuses_more_than_9e18_leaves(api, extent, leaf):
    """(3e7 + 1)^3 leaves overflow 64 bits; 2100000^3 = 9.26e18 fits in 64 bits but is above the 9e18 limit."""
    p = np.array([[0, 0, 0], [extent] * 3], np.float32)
    div = int(np.floor(np.float32(extent) * (np.float32(1) / np.float32(leaf)))) + 1
    assert 9e18 < div ** 3 and (div ** 3 < 2 ** 64) == (extent == 2100.0)
    with pytest.raises(OverflowError):
        vr.voxel_grid(p, leaf)
    rc, *_ = downsample(api, api.VoxelGrid(), p, leaf)
    assert rc == ERR_RANGE


@pytest.mark.parametrize("leaf", LEAVES)
@pytest.mark.parametrize("name", list(CLOUDS))
def test_downsample_far_and_on_leaf_multiples(oracle, api, synth, name, leaf):
    assert_downsample_parity(oracle, api, api.VoxelGrid(), cloud(name, synth, leaf), leaf)


def test_downsample_two_million_points_and_a_dense_voxel(oracle, api):
    """k_minmax's grid-stride loop iterates (> 151k points), k_keys / k_centroids run 7.8k blocks, one voxel holds 120k points."""
    rng = np.random.default_rng(5)
    p = np.empty((2_000_000, 4), np.float32)
    p[:, :3] = rng.uniform((-20, -20, -1), (20, 20, 4), (len(p), 3))
    p[:120_000, :3] = rng.uniform(3.01, 3.24, (120_000, 3))       # one 0.25 m voxel: [3.0, 3.25)^3
    p[:, 3] = rng.uniform(0, 255, len(p))
    rng.shuffle(p)
    c, n = assert_downsample_parity(oracle, api, api.VoxelGrid(), p, 0.25)
    assert n.max() >= 120_000


@pytest.mark.parametrize("min_points", [0, 1, 2, 3, 100_000])
def test_downsample_min_points(oracle, api, synth, min_points):
    p = cloud("hall", synth, 0.2)
    c, n = assert_downsample_parity(oracle, api, api.VoxelGrid(), p, 0.2, min_points)
    assert (n >= min_points).all() and (len(n) == 0) == (min_points == 100_000)


def test_negative_min_points_is_refused(api, synth):
    """pcl::VoxelGrid's setter is unsigned: a negative count is refused rather than read as 0 (the device) or 2^32 - k (PCL)."""
    vg = api.VoxelGrid()
    rc, *_ = downsample(api, vg, cloud("hall", synth, 0.2), 0.2, min_points=-1)
    assert rc == ERR_ARG
    pts, poses, x_end = imu_scene(synth, n=2000)
    vg.undistort(pts, 9, 8, poses, x_end)
    m = C.c_int64(0)
    assert api.lib().b200_voxel_downsample_staged(vg.h, 0.2, -3, C.byref(m)) == ERR_ARG
    assert api.lib().b200_voxel_downsample_staged(vg.h, 0.2, 0, C.byref(m)) == 0 and m.value > 0   # the staged scan is intact


@pytest.mark.parametrize("stride_floats", [3, 4, 12])
def test_downsample_record_strides_and_short_output(oracle, api, synth, stride_floats):
    h = cloud("hall", synth, 0.1)
    rec = np.random.default_rng(2).uniform(-1e3, 1e3, (len(h), stride_floats)).astype(np.float32)   # junk past x y z [i]
    rec[:, : min(4, stride_floats)] = h[:, : min(4, stride_floats)]
    vg = api.VoxelGrid()
    c, n = assert_downsample_parity(oracle, api, vg, rec, 0.1)
    if stride_floats == 3:
        assert (c[:, 3] == 0).all()
    # max_out below the voxel count: n_out is still the full count, only max_out voxels are written
    k = len(c) // 3
    rc, m, c2, n2, (tail_c, tail_n) = downsample(api, vg, rec, 0.1, max_out=k)
    assert rc == 0 and m == len(c)
    np.testing.assert_array_equal(c2, c[:k])
    np.testing.assert_array_equal(n2, n[:k])
    assert np.isnan(tail_c).all() and (tail_n == -1).all()


def test_downsampler_reuse_big_small_big(oracle, api, synth):
    """Buffers sized for a big cloud, then a small one, then a bigger one (reallocation): each equals a fresh downsampler."""
    rng = np.random.default_rng(9)
    big = np.concatenate([rng.uniform(-30, 30, (300_000, 3)), rng.uniform(0, 255, (300_000, 1))], 1).astype(np.float32)
    small = cloud("lattice", synth, 0.1)
    bigger = np.concatenate([big, big + np.float32(0.05)])
    vg = api.VoxelGrid()
    for rec in (big, small, bigger, small):
        _, m, c, n, _ = downsample(api, vg, rec, 0.1)
        _, m0, c0, n0, _ = downsample(api, api.VoxelGrid(), rec, 0.1)
        assert m == m0
        np.testing.assert_array_equal(n, n0)
        np.testing.assert_array_equal(c, c0)


def test_staged_scan_is_gone_after_a_host_filter(api, synth):
    """undistort(8000) -> filter(100 host points) -> filter_staged: the host cloud overwrote the staged scan in the
    device buffer, so there is nothing staged any more."""
    pts, poses, x_end = imu_scene(synth, n=8000)
    vg = api.VoxelGrid()
    vg.setLeafSize(0.5)
    vg.undistort(pts, 9, 8, poses, x_end)
    m_staged = vg.filter_staged()
    vg.setInputCloud(pts[:100, :3])
    vg.filter()
    with pytest.raises(api.B200Error, match="nothing staged"):
        vg.filter_staged()
    vg.undistort(pts, 9, 8, poses, x_end)                      # a new undistort stages again
    assert vg.filter_staged() == m_staged


# ------------------------------------------------------------------ undistortion
def assert_undistort_parity(oracle, api, pts, poses, x_end, intensity_index=8):
    o_xyzi, o_order = oracle.undistort(pts, 9, intensity_index, poses, x_end)
    g_xyzi, g_order = api.VoxelGrid().undistort(pts, 9, intensity_index, poses, x_end)
    np.testing.assert_array_equal(g_order, o_order)            # ascending time, ties in input order
    np.testing.assert_array_equal(g_xyzi[:, 3], o_xyzi[:, 3])
    # fp64 chain narrowed to fp32: device sin/cos may differ from libm in the last bit of the double
    np.testing.assert_allclose(g_xyzi[:, :3], o_xyzi[:, :3], rtol=0, atol=4e-6)
    assert (g_xyzi[:, :3] == o_xyzi[:, :3]).mean() > 0.999
    return g_xyzi, g_order


@pytest.mark.parametrize("K", [1, 2])
def test_undistort_one_and_two_poses(oracle, api, synth, K):
    pts, poses, x_end = imu_scene(synth, n=3000)
    g, order = assert_undistort_parity(oracle, api, pts, poses[:K], x_end)
    if K == 1:
        np.testing.assert_array_equal(g[:, :3], pts[order, :3])   # no segment: nothing moves


def test_undistort_times_equal_to_pose_offsets(oracle, api, synth):
    """Pose offsets built as (double)float_ms / 1000 like the point times: a point at exactly a pose's offset belongs to
    the segment that ends there (strict <).  The IMU samples are noisy, so the two segments give different points."""
    pts, poses, x_end = imu_scene(synth, n=3000)
    ms = (5.0 * np.arange(len(poses)) + 0.3).astype(np.float32)
    poses[:, 0] = ms.astype(np.float64) / 1000.0
    pts[: 3 * len(ms), 9] = np.repeat(ms, 3)
    g, order = assert_undistort_parity(oracle, api, pts, poses, x_end)
    assert np.abs(g[:, :3] - pts[order, :3]).max() > 0.05


@pytest.mark.parametrize("case", ["after_last_pose", "negative", "one_time", "late_first"])
def test_undistort_time_edges(oracle, api, synth, case):
    pts, poses, x_end = imu_scene(synth, n=3000)
    t = pts[:, 9]
    if case == "after_last_pose":
        t[::3] = np.float32(100.0) + np.arange(len(t[::3]), dtype=np.float32) * np.float32(0.01)   # poses end at 100 ms
    elif case == "negative":
        t[::4] = -t[::4] - np.float32(0.5)
    elif case == "one_time":
        t[:] = np.float32(47.25)
    else:
        t[:] = np.float32(60.0) + t * np.float32(0.4)            # the earliest point is in segment 12 of 20
    g, order = assert_undistort_parity(oracle, api, pts, poses, x_end)
    if case == "negative":
        untouched = pts[order, 9] <= 0
        np.testing.assert_array_equal(g[untouched, :3], pts[order][untouched, :3])


def test_undistort_mixed_signed_zero_times(oracle, api, synth):
    """+0.0 and -0.0 stamps compare equal: they tie and keep their input order, as in a stable sort on `<`."""
    pts, poses, x_end = imu_scene(synth, n=2000)
    pts[0:40:2, 9] = np.float32(0.0)
    pts[1:40:2, 9] = np.float32(-0.0)
    pts[40:44, 9] = [np.float32(-0.0), np.float32(0.0), np.float32(-1.0), np.float32(-0.0)]
    assert np.signbit(pts[1, 9]) and not np.signbit(pts[0, 9])
    assert_undistort_parity(oracle, api, pts, poses, x_end)


def test_undistort_without_intensity(oracle, api, synth):
    pts, poses, x_end = imu_scene(synth, n=2000)
    g, order = assert_undistort_parity(oracle, api, pts, poses, x_end, intensity_index=-1)
    assert (g[:, 3] == 0).all()
    g8, _ = api.VoxelGrid().undistort(pts, 9, 8, poses, x_end)
    np.testing.assert_array_equal(g[:, :3], g8[:, :3])


@pytest.mark.parametrize("motion", list(MOTIONS))
def test_undistort_closed_forms(oracle, api, motion):
    kw = MOTIONS[motion]
    poses, x_end, T = vr.imu_motion(0.01 * np.arange(11), **kw)
    pts = timed_scan(4000, T + 0.004, seed=21, t_min_ms=55.0 if motion == "velocity" else 0.5)
    g, order = assert_undistort_parity(oracle, api, pts, poses, x_end)
    t = pts[order, 9].astype(np.float64) / 1000.0
    ref = vr.undistort_closed_form(pts[order, :3], t, T, **kw)
    # half an ulp of a <= 52 m coordinate (1.9e-6) plus the fp64 chain: 4e-6 m; the earliest point is the quirk
    # (compensated again by every earlier segment), pinned against the oracle above
    np.testing.assert_allclose(g[1:, :3], ref[1:], rtol=0, atol=4e-6)


# ------------------------------------------------------------------ map builder
def build(api, frames, poses, leaf=0.1, capacity=2_000_000):
    b = api.FullMapBuilder(leaf=leaf, capacity_voxels=capacity)
    for f, p in zip(frames, poses):
        b.add_keyframe(f, p)
    return b


def assert_map_matches_ref(c, n, ref, leaf, max_intensity):
    """Counts equal, centroids within one fp32 ulp of the fp64 mean (the final narrowing) plus the running-sum bound of the
    corner-relative fp32 offsets (< one leaf each); intensity within the running-sum bound of an absolute fp32 sum."""
    np.testing.assert_array_equal(n, ref["counts"])
    m = ref["cent"]
    assert (np.abs(c[:, :3] - m[:, :3]) <= vr.ulp32(m[:, :3]) + vr.running_sum_bound(n, leaf)[:, None]).all()
    assert (np.abs(c[:, 3] - m[:, 3]) <= vr.running_sum_bound(n, max_intensity) + vr.ulp32(m[:, 3])).all()


def assert_same_map(c, n, c0, n0, leaf, max_intensity):
    """Two builds of the same keyframes: the same voxels and counts; fp32 atomics in another order change each sum by at
    most twice the running-sum bound, and the narrowed centroid by one more ulp."""
    np.testing.assert_array_equal(n, n0)
    assert (np.abs(c[:, :3] - c0[:, :3]) <= vr.ulp32(c0[:, :3]) + 2 * vr.running_sum_bound(n0, leaf)[:, None]).all()
    assert (np.abs(c[:, 3] - c0[:, 3]) <= 2 * vr.running_sum_bound(n0, max_intensity) + vr.ulp32(c0[:, 3])).all()


@pytest.mark.parametrize("offset", [(2000.0, 300.0, 0.0), (100000.0, 0.0, 0.0)], ids=["2km", "100km"])
def test_full_map_far_from_the_origin(oracle, api, synth, offset, record_property):
    """Sums relative to the voxel corner keep the centroid exact far from the origin: within one ulp of the fp64 mean of the
    fp32-moved points and equal to its fp32 rounding for >= 99 % of the voxels.  The oracle sums absolute fp32 coordinates
    (pcl::CentroidPoint), which drift by (count + 1) * 2^-24 * |coordinate| - several ulps here - so it is the reference
    for the partition and the counts only; its drift is recorded, not asserted."""
    frames, poses = make_frames(synth)
    poses[:, :3] += offset
    ref = vr.map_build(frames, poses, 0.1)
    c0, n0 = oracle.full_map(frames, poses, 0.1)
    c, n = build(api, frames, poses).extract()
    np.testing.assert_array_equal(n, n0)
    assert_map_matches_ref(c, n, ref, 0.1, 100.0)
    m = ref["cent"][:, :3]
    # where the corner-relative sums' running-sum bound is below half an ulp of the coordinate - every x here, kilometres
    # out - the centroid is within one ulp; near 0 (the floor's z) an ulp is far below the offsets' own fp32 rounding
    # (2^-24 * leaf), and assert_map_matches_ref's bound applies
    far = 0.5 * vr.ulp32(m) >= vr.running_sum_bound(n, 0.1)[:, None]
    assert far[:, 0].all()
    assert (np.abs(c[:, :3] - m)[far] <= vr.ulp32(m)[far]).all()
    assert (c[:, :3] == m.astype(np.float32))[far].mean() >= 0.99
    drift = np.abs(c0[:, :3] - m)[far] / vr.ulp32(m)[far]
    record_property("oracle_drift_ulp_max", float(drift.max()))
    record_property("oracle_drift_ulp_mean", float(drift.mean()))
    print(f"oracle fp32 drift at {offset}: max {drift.max():.1f} ulp, mean {drift.mean():.2f} ulp, device max "
          f"{(np.abs(c[:, :3] - m)[far] / vr.ulp32(m)[far]).max():.2f} ulp")


def test_full_map_key_range(oracle, api):
    """Cells -2^20 .. 2^20 - 1 per axis are accepted (+-1048 km at a 1 m leaf, +-104.8 km at 0.1 m); NaN and Inf points are
    skipped like the oracle skips them."""
    lim = float(1 << 20)
    f = np.array([[lim - 0.5, 0.5, 0.5, 1], [0.5, lim - 0.5, -lim, 2], [-lim, -lim + 0.25, lim - 0.75, 3], [0.25, 0.5, 0.75, 4],
                  [np.nan, 0, 0, 5], [np.inf, 0, 0, 6], [0, -np.inf, 0, 7], [0, 0, np.nan, 8]], np.float32)
    ref = vr.map_build([f], [IDENTITY7], 1.0)
    assert ref["out_of_range"] == 0 and len(ref["counts"]) == 4
    assert ref["cells"].min() == -(1 << 20) and ref["cells"].max() == (1 << 20) - 1
    b = build(api, [f], [IDENTITY7], leaf=1.0, capacity=16)
    assert b.num_voxels() == 4
    c, n = b.extract()
    c0, n0 = oracle.full_map([f], [IDENTITY7], 1.0)
    np.testing.assert_array_equal(n, n0)
    np.testing.assert_array_equal(c, c0)          # one point per voxel: both exact
    np.testing.assert_array_equal(c, ref["cent"].astype(np.float32))


@pytest.mark.parametrize("bad", [(1 << 20, 0.5, 0.5), (0.5, 0.5, -(1 << 20) - 0.5)], ids=["x=2^20", "z=-2^20-1"])
def test_full_map_key_range_refused_and_sticky(api, bad):
    """A point one cell beyond the key range is refused with B200_ERR_RANGE.  The error stays raised for the builder's life:
    after later keyframes, counts, single-rank merges and extractions all fail, and a new builder is needed."""
    f = np.array([[0.5, 0.5, 0.5, 1], list(bad) + [2]], np.float32)
    b = build(api, [f], [IDENTITY7], leaf=1.0, capacity=16)
    with pytest.raises(api.B200Error, match="key range"):
        b.num_voxels()
    assert api.lib().b200_mapbuild_num_voxels(b.h) == -1
    b.add_keyframe(f[:1], IDENTITY7)
    with pytest.raises(api.B200Error, match="key range"):
        b.num_voxels()
    with pytest.raises(api.B200Error, match="key range"):
        b.merge(None)
    with pytest.raises(api.B200Error):
        b.extract()
    assert build(api, [f[:1]], [IDENTITY7], leaf=1.0, capacity=16).num_voxels() == 1


def test_full_map_capacity_is_exact(api, synth):
    frames, poses = make_frames(synth, k=3, n=4000)
    m = len(vr.map_build(frames, poses, 0.1)["counts"])
    c, n = build(api, frames, poses, capacity=m).extract()
    assert len(n) == m
    c2, n2 = build(api, frames, poses, capacity=4 * m).extract()
    np.testing.assert_array_equal(n, n2)
    with pytest.raises(api.B200Error, match="capacity"):
        build(api, frames, poses, capacity=m - 1).num_voxels()


def big_scene(synth):
    """62 keyframes: the hall's, ragged, with 1-point frames among them, and one 1.2M-point frame (k_accumulate's grid-stride
    loop covers 303k points per pass) with a 20k-point voxel of intensities 0..255."""
    base, bposes = make_frames(synth)
    rng = np.random.default_rng(17)
    frames, poses = [], []
    for i in range(62):
        p = bposes[i % 12].copy()
        p[0] += 0.013 * i
        if i == 30:
            f = np.empty((1_200_000, 4), np.float32)
            f[:, :3] = rng.uniform((-20, -8, 0), (20, 8, 4), (len(f), 3))
            f[:20_000, :3] = rng.uniform(3.01, 3.09, (20_000, 3))     # the voxel [3.0, 3.1)^3 under the identity pose
            f[:, 3] = rng.uniform(0, 255, len(f))
            p = IDENTITY7.copy()
        elif i % 7 == 3:
            f = base[i % 12][i:i + 1]
        else:
            f = base[i % 12][: len(base[i % 12]) - 37 * (i % 5)]
        frames.append(np.ascontiguousarray(f))
        poses.append(p)
    return frames, np.array(poses)


@pytest.fixture(scope="module")
def big(synth):
    frames, poses = big_scene(synth)
    return frames, poses, vr.map_build(frames, poses, 0.1)


def test_full_map_big_keyframe_matches_fp64(oracle, api, big):
    frames, poses, ref = big
    c, n = build(api, frames, poses).extract()
    c0, n0 = oracle.full_map(frames, poses, 0.1)
    np.testing.assert_array_equal(n, n0)
    assert_map_matches_ref(c, n, ref, 0.1, 255.0)
    dense = n >= 20_000
    assert dense.sum() == 1


def test_full_map_batching_and_order_do_not_matter(api, big):
    import torch
    frames, poses, ref = big
    c_ref, n_ref = build(api, frames, poses).extract()
    dev = [torch.from_numpy(f).cuda() for f in frames]
    for chunk in (23, 24, 25, 48):
        b = api.FullMapBuilder(leaf=0.1, capacity_voxels=2_000_000)
        for s in range(0, len(frames), chunk):
            b.add_keyframes_device([d.data_ptr() for d in dev[s:s + chunk]], [len(f) for f in frames[s:s + chunk]], poses[s:s + chunk])
        c, n = b.extract()
        assert_same_map(c, n, c_ref, n_ref, 0.1, 255.0)
        assert_map_matches_ref(c, n, ref, 0.1, 255.0)
    c, n = build(api, frames[::-1], poses[::-1]).extract()
    assert_same_map(c, n, c_ref, n_ref, 0.1, 255.0)
    torch.cuda.synchronize()


def test_full_map_extract_then_more_keyframes(api, synth):
    frames, poses = make_frames(synth)
    b = build(api, frames[:5], poses[:5])
    c5, n5 = b.extract()
    assert_map_matches_ref(c5, n5, vr.map_build(frames[:5], poses[:5], 0.1), 0.1, 100.0)
    for f, p in zip(frames[5:], poses[5:]):
        b.add_keyframe(f, p)
    c, n = b.extract()
    c0, n0 = build(api, frames, poses).extract()
    assert_same_map(c, n, c0, n0, 0.1, 100.0)
    assert_map_matches_ref(c, n, vr.map_build(frames, poses, 0.1), 0.1, 100.0)


# ------------------------------------------------------------------ two GPUs
def gpu_count():
    import torch
    return torch.cuda.device_count()


def stop_launch(p, pid_dir, grace=60):
    """Leaves no process of a torch.distributed.run launch behind.  The launcher starts every worker in a session of its own,
    so killing the launcher's group would orphan them: it gets SIGTERM, on which it terminates each worker's group, and a
    bounded wait.  Workers still alive after that (a launcher that had to be killed) are killed by the pid they wrote."""
    if p.poll() is None:
        p.terminate()
        try:
            p.wait(timeout=grace)
        except subprocess.TimeoutExpired:
            p.kill()
            p.wait()
    for f in pid_dir.glob("worker*.pid"):
        pid = int(f.read_text())
        try:
            with open(f"/proc/{pid}/cmdline", "rb") as fh:
                alive = b"mapbuild_worker.py" in fh.read()      # still our worker, not a reused pid
        except OSError:
            continue
        if alive:
            try:
                os.kill(pid, signal.SIGKILL)
            except ProcessLookupError:
                pass


def launch_mapbuild_worker(tmp_path, world, port, timeout=300):
    out = tmp_path / "res.json"
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}", "--master-addr", "127.0.0.1",
           "--master-port", str(port), os.path.join(ROOT, "tests", "helpers", "mapbuild_worker.py"), str(out)]
    p = subprocess.Popen(cmd, env=dict(os.environ, MASTER_ADDR="127.0.0.1"), stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
    err = ""
    try:
        _, err = p.communicate(timeout=timeout)
    except subprocess.TimeoutExpired:
        err = f"timed out after {timeout} s"
    finally:
        stop_launch(p, tmp_path)
    assert p.returncode == 0, err[-3000:]
    return json.load(open(out))


def test_two_gpu_merge_far_keyframes_empty_rank_and_second_merge(tmp_path):
    """tests/helpers/mapbuild_worker.py on two ranks: far-coordinate keyframes all on rank 0 (rank 1 has none), merge, more
    keyframes on both ranks, merge again.  Each rank's voxels must be exactly the fp64 reference's voxels it owns."""
    if gpu_count() < 2:
        pytest.skip("needs 2 GPUs")
    r = launch_mapbuild_worker(tmp_path, 2, 29667)
    assert r["ok"] and r["world"] == 2, r


def test_mapbuild_worker_on_one_rank(tmp_path):
    """The same worker on one rank (both merges are local): the worker's own checks and the launcher's cleanup run on any
    machine with a GPU."""
    r = launch_mapbuild_worker(tmp_path, 1, 29669)
    assert r["ok"] and r["world"] == 1, r
