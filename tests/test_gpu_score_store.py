"""calculateScore reads each NDT leaf from the score store that set_target builds next to the leaf records: three arrays
indexed by leaf slot, {mean, icov00}, {icov01 + icov10, icov02 + icov20, icov11, icov12 + icov21} and {icov22}, and the
quadratic form is evaluated from the symmetric form with fused multiply-adds.  Only rounding changes, so:

- scores stay within 1e-12 relative of the CPU oracle in every neighbourhood search mode (KDTREE, DIRECT1, DIRECT7,
  DIRECT26), at random yaws, under roll / pitch and at poses that put points outside the target grid (where DIRECT7
  resolves the neighbourhood cell by cell instead of through the per-cell table);
- maps with leaves below min_points and leaves rejected by the eigenvalue check score like the oracle (such leaves are
  never referenced);
- a second set_target with a smaller map leaves nothing of the first map's store behind;
- a hypothesis's score is bit-identical however the batch is cut.
"""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

RTOL = 1e-12
MODES = [0, 1, 7, 27]   # KDTREE, DIRECT1, DIRECT7, DIRECT26


@pytest.fixture(scope="module")
def scene(synth):
    world = synth.make_world(synth.SEED, beams=True)
    mp = synth.sample_map(300_000, synth.SEED, world=world)
    p_true = np.array([3.0, -2.0, 1.2, 0.0, 0.0, 0.6])
    T = synth.pose_vec_to_matrix(p_true)
    dirs = synth.livox_dirs(5000, synth.SEED)
    scan = np.ascontiguousarray(synth.raycast(T[:3, 3], T[:3, :3], dirs, world, seed=synth.SEED)[:4000])
    return dict(map=mp, scan=scan, p_true=p_true)


@pytest.fixture(scope="module")
def far_scene(synth):
    """A map 3e7 m out along x: there fp32 coordinates are 2 m apart, every occupied 1 m cell holds copies of one point,
    and the leaf covariance is fp64 rounding noise on top of Leaf()'s identity start.  Some leaves get a negative
    eigenvalue and are rejected; most cells hold fewer than min_points points."""
    world = synth.make_world(synth.SEED, beams=True)
    mp = synth.sample_map(60_000, synth.SEED, world=world)
    off = np.array([3e7, 0.0, 0.0])
    mp = (mp.astype(np.float64) + off).astype(np.float32)
    rng = np.random.default_rng(2)
    scan = np.ascontiguousarray(mp[rng.choice(len(mp), 3000, replace=False)] + rng.normal(0, 0.05, (3000, 3)).astype(np.float32))
    poses = []
    for _ in range(24):   # a small rotation about the map's own region and a shift of up to a few cells
        R = rotation(0.0, 0.0, rng.uniform(-0.05, 0.05))
        t = off - R @ off + [rng.uniform(-1.5, 1.5), rng.uniform(-1.5, 1.5), rng.uniform(-0.5, 0.5)]
        poses.append(matrix_pose(R, t))
    return dict(map=mp, scan=scan, poses=np.ascontiguousarray(np.stack(poses)))


def rotation(roll, pitch, yaw):
    cr, sr, cp, sp, cy, sy = np.cos(roll), np.sin(roll), np.cos(pitch), np.sin(pitch), np.cos(yaw), np.sin(yaw)
    Rx = np.array([[1, 0, 0], [0, cr, -sr], [0, sr, cr]])
    Ry = np.array([[cp, 0, sp], [0, 1, 0], [-sp, 0, cp]])
    Rz = np.array([[cy, -sy, 0], [sy, cy, 0], [0, 0, 1]])
    return Rx @ Ry @ Rz


def matrix_pose(R, t):
    """column-major fp32 4x4, the layout calculateScore takes"""
    A = np.eye(4)
    A[:3, :3] = R
    A[:3, 3] = t
    return A.astype(np.float32).T.reshape(16)


def engines(oracle, api, mp, scan, search):
    o = oracle.OracleNdt(resolution=1.0, search=search)
    o.set_target(mp)
    o.set_source(scan)
    g = api.NormalDistributionsTransform()
    g.setNeighborhoodSearchMethod(search)
    g.setInputTarget(mp)
    g.setInputSource(scan)
    return o, g


def wide_poses(p, n=48, seed=21):
    """Random yaws, roll / pitch up to 0.3 rad and shifts of up to 30 m in x / y and 1 m in z: the scan hangs over the
    grid's edges (the map spans 120 x 80 x 8 m)."""
    rng = np.random.default_rng(seed)
    out = []
    for k in range(n):
        R = rotation(*rng.uniform(-0.3, 0.3, 2), rng.uniform(-np.pi, np.pi))
        t = np.asarray(p[:3]) + rng.uniform(-1, 1, 3) * [30, 30, 1]
        if k == 0:
            R, t = rotation(*p[3:]), np.asarray(p[:3])
        out.append(matrix_pose(R, t))
    return np.ascontiguousarray(np.stack(out))


def cells_of(scan, poses):
    """The kernel's cell of every (pose, point): pcl::transformPointCloud's fp32 order, then floor(t / 1 m)."""
    M = poses.reshape(-1, 4, 4).transpose(0, 2, 1).astype(np.float32)
    x = scan.astype(np.float32)
    t = ((M[:, None, :3, 0] * x[None, :, 0:1] + M[:, None, :3, 1] * x[None, :, 1:2]) + M[:, None, :3, 2] * x[None, :, 2:3]) + M[:, None, :3, 3]
    return np.floor(t).astype(np.int64)


def assert_oracle(o, g, poses):
    s0 = o.score_batch(poses)
    s1 = g.calculateScore(poses)
    np.testing.assert_allclose(s1, s0, rtol=RTOL, atol=1e-14)
    return s1


def assert_batch_independent(g, poses):
    full = g.calculateScore(poses)
    alone = np.array([g.calculateScore(poses[i:i + 1])[0] for i in range(len(poses))])
    np.testing.assert_array_equal(alone, full)
    np.testing.assert_array_equal(g.calculateScore(poses[::-1])[::-1], full)
    for k in (3, 5):
        np.testing.assert_array_equal(np.concatenate([g.calculateScore(c) for c in np.array_split(poses, k)]), full)
        inter = np.empty_like(full)
        for r in range(k):
            inter[r::k] = g.calculateScore(poses[r::k])
        np.testing.assert_array_equal(inter, full)
    return full


@pytest.mark.parametrize("search", MODES)
def test_modes_match_oracle_and_batch_cut(oracle, api, scene, search):
    o, g = engines(oracle, api, scene["map"], scene["scan"], search)
    poses = wide_poses(scene["p_true"])
    # the poses put points just outside the grid, where a face neighbour can still hold a leaf
    mn, dv = (np.asarray(a, np.int64) for a in o.grid())
    c = cells_of(scene["scan"], poses)
    outside = ((c < mn) | (c > mn + dv - 1)).any(-1)
    near = ((c >= mn - 1) & (c <= mn + dv)).all(-1)
    assert (outside & near).sum() > 1000 and (~outside).sum() > 10000
    s = assert_oracle(o, g, poses)
    assert np.isfinite(s).all() and int(np.argmax(s)) == 0
    assert_batch_independent(g, poses)


@pytest.mark.parametrize("search", MODES)
def test_sparse_and_rejected_leaves(oracle, api, far_scene, search):
    mp = far_scene["map"]
    o, g = engines(oracle, api, mp, far_scene["scan"], search)
    _, cnt = np.unique(np.floor(mp.astype(np.float64)).astype(np.int64), axis=0, return_counts=True)
    Lo, Lg = o.leaves(), g.leaves()
    np.testing.assert_array_equal(Lg["ids"], Lo["ids"])
    assert ((cnt > 0) & (cnt < 6)).sum() > 1000              # below min_points
    assert (cnt >= 6).sum() - len(Lo["ids"]) > 20            # rejected by the eigenvalue check
    s = assert_oracle(o, g, far_scene["poses"])
    assert np.isfinite(s).all() and (s > 0).all()
    assert_batch_independent(g, far_scene["poses"])


@pytest.mark.parametrize("search", MODES)
def test_second_smaller_target(oracle, api, scene, search):
    """set_target again with a map of fewer leaves on another grid: the store's slots past the new leaf count still hold
    the first map's leaves, and nothing may read them."""
    poses = wide_poses(scene["p_true"], n=24, seed=22)
    big = scene["map"]
    small = np.ascontiguousarray(big[(big[:, 0] < 25) & (big[:, 1] > -30)][::2])
    o, g = engines(oracle, api, big, scene["scan"], search)
    first = g.calculateScore(poses)
    g.setInputTarget(small)
    o.set_target(small)
    s = assert_oracle(o, g, poses)
    _, fresh = engines(oracle, api, small, scene["scan"], search)
    np.testing.assert_array_equal(fresh.calculateScore(poses), s)
    assert not np.array_equal(s, first)
    g.setInputTarget(big)   # and back
    np.testing.assert_array_equal(g.calculateScore(poses), first)
