"""Relocalization screens every hypothesis with a certified fp32 score interval and rescores only the hypotheses that can
still win in fp64.  So:

- the interval of every hypothesis contains its calculateScore value, in every neighbourhood search mode, on a
  relocalization grid, at random yaws with roll / pitch, at poses hanging over the grid's edges and on a map 3e7 m out
  with sparse and rejected leaves;
- relocalize returns the same (best, score) bits and code with the screen on and off, equal to argmax(calculateScore):
  duplicated poses (ties go to the lowest index), poses one fp32 ulp apart, all poses non-finite, an empty slice,
  contiguous and interleaved slices, and more survivors than the rescore kernel's 64 block rows;
- on a relocalization grid only a handful of hypotheses survive the screen.
"""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

MODES = [0, 1, 7, 27]   # KDTREE, DIRECT1, DIRECT7, DIRECT26
# survivors allowed on the 4096-pose grid: the winner's interval must separate it from all but its closest competitors
MAX_GRID_SURVIVORS = 16


def rotation(roll, pitch, yaw):
    cr, sr, cp, sp, cy, sy = np.cos(roll), np.sin(roll), np.cos(pitch), np.sin(pitch), np.cos(yaw), np.sin(yaw)
    Rx = np.array([[1, 0, 0], [0, cr, -sr], [0, sr, cr]])
    Ry = np.array([[cp, 0, sp], [0, 1, 0], [-sp, 0, cp]])
    Rz = np.array([[cy, -sy, 0], [sy, cy, 0], [0, 0, 1]])
    return Rx @ Ry @ Rz


def matrix_pose(R, t):
    A = np.eye(4)
    A[:3, :3] = R
    A[:3, 3] = t
    return A.astype(np.float32).T.reshape(16)


@pytest.fixture(scope="module")
def scene(synth):
    world = synth.make_world(synth.SEED, beams=True)
    mp = synth.sample_map(300_000, synth.SEED, world=world)
    p_true = np.array([3.0, -2.0, 1.2, 0.0, 0.0, 0.6])
    T = synth.pose_vec_to_matrix(p_true)
    dirs = synth.livox_dirs(5000, synth.SEED)
    scan = np.ascontiguousarray(synth.raycast(T[:3, 3], T[:3, :3], dirs, world, seed=synth.SEED)[:4000])
    grid = synth.hypothesis_grid(p_true, 32, 32, 4, 1.0)
    rng = np.random.default_rng(31)
    wide = []
    for k in range(64):   # random yaws, roll / pitch up to 0.3 rad, shifts of up to 30 m: the scan hangs over the grid's edges
        R = rotation(*rng.uniform(-0.3, 0.3, 2), rng.uniform(-np.pi, np.pi))
        wide.append(matrix_pose(R, p_true[:3] + rng.uniform(-1, 1, 3) * [30, 30, 1]))
    return dict(map=mp, scan=scan, p_true=p_true, grid=grid, wide=np.ascontiguousarray(np.stack(wide)))


@pytest.fixture(scope="module")
def far_scene(synth):
    """3e7 m out along x: fp32 coordinates 2 m apart, most cells below min_points, some leaves rejected."""
    world = synth.make_world(synth.SEED, beams=True)
    mp = synth.sample_map(60_000, synth.SEED, world=world)
    off = np.array([3e7, 0.0, 0.0])
    mp = (mp.astype(np.float64) + off).astype(np.float32)
    rng = np.random.default_rng(2)
    scan = np.ascontiguousarray(mp[rng.choice(len(mp), 3000, replace=False)] + rng.normal(0, 0.05, (3000, 3)).astype(np.float32))
    poses = []
    for _ in range(24):
        R = rotation(0.0, 0.0, rng.uniform(-0.05, 0.05))
        poses.append(matrix_pose(R, off - R @ off + [rng.uniform(-1.5, 1.5), rng.uniform(-1.5, 1.5), rng.uniform(-0.5, 0.5)]))
    return dict(map=mp, scan=scan, poses=np.ascontiguousarray(np.stack(poses)))


def engine(api, mp, scan, search=7):
    g = api.NormalDistributionsTransform()
    g.setNeighborhoodSearchMethod(search)
    g.setInputTarget(mp)
    g.setInputSource(scan)
    return g


def reloc(api, g, poses, screen, h_begin=0, h_stride=1):
    """(code, best, score bits) of b200_reloc_argmin_strided with the screen on or off"""
    g.setRelocScreen(screen)
    poses = np.ascontiguousarray(poses, dtype=np.float32).reshape(-1, 16)
    best, score, ms = C.c_int64(-1), C.c_double(0), C.c_float(0)
    rc = api.lib().b200_reloc_argmin_strided(None, g._handle(), poses.ctypes.data_as(C.c_void_p) if len(poses) else None, len(poses),
                                             h_begin, h_stride, C.byref(best), C.byref(score), C.byref(ms))
    g.setRelocScreen(True)
    return rc, best.value, np.float64(score.value).tobytes()


def expected(g, poses, h_begin=0, h_stride=1):
    s = g.calculateScore(poses)
    ok = ~np.isnan(s)
    if not ok.any():
        return None
    i = int(np.flatnonzero(s == s[ok].max())[0])
    return h_begin + i * h_stride, np.float64(s[i]).tobytes()


def assert_same(api, g, poses, h_begin=0, h_stride=1):
    on = reloc(api, g, poses, True, h_begin, h_stride)
    off = reloc(api, g, poses, False, h_begin, h_stride)
    assert on == off
    exp = expected(g, poses, h_begin, h_stride) if len(poses) else None
    if exp is None:
        assert on[1] == -1 and on[0] != 0
    else:
        assert on[0] == 0 and (on[1], on[2]) == exp
    return on


def assert_contains(g, poses):
    s = g.calculateScore(poses)
    lo, hi = g.screenScore(poses)
    fin = np.isfinite(s)
    assert (lo[fin] <= s[fin]).all() and (s[fin] <= hi[fin]).all(), np.flatnonzero(~((lo <= s) & (s <= hi)))
    assert np.isfinite(lo[fin]).all() and np.isfinite(hi[fin]).all()
    return s, lo, hi


@pytest.mark.parametrize("search", MODES)
def test_intervals_contain_scores(api, scene, far_scene, search):
    g = engine(api, scene["map"], scene["scan"], search)
    for poses in (scene["grid"], scene["wide"]):
        s, lo, hi = assert_contains(g, poses)
        assert ((hi - lo) <= 1e-3 * np.abs(s) + 1e-12).all()   # tens of ppm of the score on these scenes
    gf = engine(api, far_scene["map"], far_scene["scan"], search)
    assert_contains(gf, far_scene["poses"])


def test_grid_survivors_are_few(api, scene):
    g = engine(api, scene["map"], scene["scan"])
    lo, hi = g.screenScore(scene["grid"])
    survivors = int((hi >= lo.max()).sum())
    print(f"grid survivors: {survivors} of {len(lo)}")
    assert 1 <= survivors <= MAX_GRID_SURVIVORS
    assert_same(api, g, scene["grid"])


@pytest.mark.parametrize("search", MODES)
def test_relocalize_same_bits(api, scene, search):
    g = engine(api, scene["map"], scene["scan"], search)
    grid = scene["grid"][::4] if search != 7 else scene["grid"]
    assert_same(api, g, grid)
    assert_same(api, g, scene["wide"])
    for r in range(3):   # interleaved slices of 3 ranks and contiguous slices
        assert_same(api, g, grid[r::3], h_begin=r, h_stride=3)
        part = np.array_split(np.arange(len(grid)), 3)[r]
        assert_same(api, g, grid[part], h_begin=int(part[0]))


def test_ties_ulps_and_many_survivors(api, scene):
    g = engine(api, scene["map"], scene["scan"])
    grid = scene["grid"]
    best = int(np.argmax(g.calculateScore(grid)))
    # exact duplicates of the winner: every copy survives and the lowest index wins
    dup = np.ascontiguousarray(np.concatenate([grid[:50], np.repeat(grid[best:best + 1], 5, 0), grid[50:100], grid[best:best + 1]]))
    rc, b, _ = assert_same(api, g, dup)
    assert rc == 0 and b == min(best, 50)
    # translations one fp32 ulp apart around the winner
    ulp = np.repeat(grid[best:best + 1], 9, 0)
    for k in range(9):
        for c in (12, 13):
            ulp[k, c] = np.nextafter(ulp[k, c], np.float32(np.inf) if k % 2 else np.float32(-np.inf)) if k else ulp[k, c]
    assert_same(api, g, np.ascontiguousarray(np.concatenate([grid[:20], ulp])))
    # more survivors than the rescore's 64 block rows: 150 copies of the winner among other poses
    many = np.ascontiguousarray(np.concatenate([grid[::7], np.repeat(grid[best:best + 1], 150, 0)]))
    lo, hi = g.screenScore(many)
    assert int((hi >= lo.max()).sum()) >= 150
    assert_same(api, g, many)


def test_non_finite_and_empty(api, scene):
    g = engine(api, scene["map"], scene["scan"])
    bad = scene["grid"][:40].copy()
    bad[:, 12] = np.nan
    lo, hi = g.screenScore(bad)
    s = g.calculateScore(bad)
    assert np.isnan(s).all() and (lo == -np.inf).all() and (hi == np.inf).all()
    rc, b, _ = assert_same(api, g, bad)
    assert rc == 1 and b == -1   # B200_NO_EFFECTIVE_POINTS
    mixed = scene["grid"][:40].copy()
    mixed[::3, 13] = np.inf
    mixed[1::5, 0] = np.nan
    assert_same(api, g, mixed)
    rc, b, _ = assert_same(api, g, np.zeros((0, 16), np.float32))
    assert b == -1
