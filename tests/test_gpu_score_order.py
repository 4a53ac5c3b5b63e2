"""calculateScore / relocalize read the scan in the Morton order of the pose's yaw bin (the score kernel picks the bin from
the pose's rotation alone; the ordering of a bin is built the first time a batch needs it and kept until the next
set_source).  Only the fp64 summation order changes, so:

- scores stay within 1e-12 relative of the CPU oracle at every yaw bin, at bin boundaries, near +-pi and under roll / pitch;
- a hypothesis's score is bit-identical however the batch is cut (alone, full, reversed, contiguous or interleaved slices),
  and relocalize returns argmax(calculateScore) with exactly that score;
- the orderings built so far, and the order they were built in, never change a score;
- set_source with another cloud replaces every ordering;
- NaN points, points beyond the Morton key's clamp range and scans of any length (also < 32 points) are handled.
"""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

RTOL = 1e-12


@pytest.fixture(scope="module")
def scene(synth):
    world = synth.make_world(synth.SEED, beams=True)
    mp = synth.sample_map(300_000, synth.SEED, world=world)
    p_true = np.array([3.0, -2.0, 1.2, 0.0, 0.0, 0.6])
    T = synth.pose_vec_to_matrix(p_true)
    dirs = synth.livox_dirs(5000, synth.SEED)
    scan = np.ascontiguousarray(synth.raycast(T[:3, 3], T[:3, :3], dirs, world, seed=synth.SEED)[:4000])
    return dict(map=mp, scan=scan, p_true=p_true)


def engines(oracle, api, mp, scan, search=7):
    o = oracle.OracleNdt(resolution=1.0, search=search)
    o.set_target(mp)
    o.set_source(scan)
    g = api.NormalDistributionsTransform()
    g.setNeighborhoodSearchMethod(search)
    g.setInputTarget(mp)
    g.setInputSource(scan)
    return o, g


def poses_from(synth, vecs):
    return np.ascontiguousarray(np.stack([synth.pose_vec_to_matrix(v).astype(np.float32).T.reshape(16) for v in vecs]))


def yaw_poses(synth, p, yaws, roll=0.0, pitch=0.0, dxy=(0.0, 0.0)):
    out = []
    for psi in yaws:
        v = np.array(p, dtype=np.float64)
        v[0] += dxy[0]
        v[1] += dxy[1]
        v[3], v[4], v[5] = roll, pitch, psi
        out.append(v)
    return poses_from(synth, out)


def boundary_yaws(bins=(256, 512)):
    """Bin centres and boundaries of 256 / 512 yaw bins (512 up to 32k scan points, 256 up to 64k), the fp32 neighbours
    (+-1 ulp) of every boundary, and yaws at +-pi."""
    ys = set()
    for nb in bins:
        for j in range(nb):
            ys.add(float(np.float32(2 * np.pi * j / nb)))
            b = np.float32(2 * np.pi * (j + 0.5) / nb)
            if b > np.pi:
                b = np.float32(b - 2 * np.pi)
            for y in (b, np.nextafter(b, np.float32(np.inf)), np.nextafter(b, np.float32(-np.inf))):
                ys.add(float(y))
    pi = np.float32(np.pi)
    for y in (pi, -pi, np.nextafter(pi, np.float32(0)), np.nextafter(-pi, np.float32(0)), 3.14159, -3.14159):
        ys.add(float(y))
    return sorted(ys)


def assert_oracle(o, g, poses):
    s0 = o.score_batch(poses)
    s1 = g.calculateScore(poses)
    np.testing.assert_allclose(s1, s0, rtol=RTOL, atol=1e-14)
    return s1


@pytest.mark.parametrize("search", [1, 7, 27])
def test_every_yaw_bin_and_boundary_matches_oracle(oracle, api, synth, scene, search):
    o, g = engines(oracle, api, scene["map"], scene["scan"], search)
    poses = yaw_poses(synth, scene["p_true"], boundary_yaws())
    s1 = assert_oracle(o, g, poses)
    assert np.isfinite(s1).all() and (s1 != 0).any()
    # the true pose still wins among its yaw neighbours
    near = yaw_poses(synth, scene["p_true"], 0.6 + np.linspace(-0.3, 0.3, 13))
    assert int(np.argmax(assert_oracle(o, g, near))) == 6


def test_roll_pitch_matches_oracle(oracle, api, synth, scene):
    o, g = engines(oracle, api, scene["map"], scene["scan"])
    yaws = np.linspace(-np.pi, np.pi, 12, endpoint=False) + 0.6
    poses = np.concatenate([yaw_poses(synth, scene["p_true"], yaws, roll=r, pitch=q, dxy=(0.4, -0.3))
                            for r, q in ((0.52, 0.0), (0.0, -0.52), (0.3, 0.3), (-0.52, 0.52), (0.1, -0.2))])
    assert_oracle(o, g, poses)


def mixed_poses(synth, p, n=96, seed=3):
    rng = np.random.default_rng(seed)
    vecs = []
    for _ in range(n):
        v = np.array(p, dtype=np.float64)
        v[:3] += rng.uniform(-2, 2, 3) * [1, 1, 0.2]
        v[3:5] = rng.uniform(-0.3, 0.3, 2)
        v[5] = rng.uniform(-np.pi, np.pi)
        vecs.append(v)
    vecs[n // 2] = np.array(p)
    return poses_from(synth, vecs)


def assert_batch_independent(api, g, poses):
    full = g.calculateScore(poses)
    alone = np.array([g.calculateScore(poses[i:i + 1])[0] for i in range(len(poses))])
    np.testing.assert_array_equal(alone, full)
    np.testing.assert_array_equal(g.calculateScore(poses[::-1])[::-1], full)
    for k in (2, 3, 7):
        parts = np.concatenate([g.calculateScore(c) for c in np.array_split(poses, k)])
        np.testing.assert_array_equal(parts, full)
        inter = np.empty_like(full)
        for r in range(k):
            inter[r::k] = g.calculateScore(poses[r::k])
        np.testing.assert_array_equal(inter, full)
    return full


def test_scores_independent_of_batch_cut(oracle, api, synth, scene):
    o, g = engines(oracle, api, scene["map"], scene["scan"])
    poses = mixed_poses(synth, scene["p_true"])
    full = assert_batch_independent(api, g, poses)
    np.testing.assert_allclose(full, o.score_batch(poses), rtol=RTOL, atol=1e-14)
    best, score, _ = api.relocalize(g, poses)
    assert best == int(np.argmax(full)) and score == full[best]
    wins = [api.relocalize(g, poses[r::5], h_begin=r, h_stride=5)[:2] for r in range(5)]
    assert max(wins, key=lambda w: (w[1], -w[0])) == (best, score)


def test_lazy_build_order_does_not_matter(api, synth, scene):
    """Bins built one call at a time (the ordering store grows and is copied), the bins of one batch, and every bin at
    once (a later batch of at least as many poses as bins) all give the same scores."""
    poses = np.concatenate([mixed_poses(synth, scene["p_true"], n=40, seed=4), yaw_poses(synth, scene["p_true"], boundary_yaws()[::23])])
    one = api.NormalDistributionsTransform()
    one.setInputTarget(scene["map"])
    one.setInputSource(scene["scan"])
    single = np.array([one.calculateScore(poses[i:i + 1])[0] for i in range(len(poses))])
    many = api.NormalDistributionsTransform()
    many.setInputTarget(scene["map"])
    many.setInputSource(scene["scan"])
    np.testing.assert_array_equal(many.calculateScore(poses), single)
    np.testing.assert_array_equal(one.calculateScore(poses[::-1])[::-1], single)
    every = api.NormalDistributionsTransform()
    every.setInputTarget(scene["map"])
    every.setInputSource(scene["scan"])
    big = np.concatenate([poses, yaw_poses(synth, scene["p_true"], np.linspace(-np.pi, np.pi, 600, endpoint=False))])
    np.testing.assert_array_equal(every.calculateScore(big[:3]), single[:3])   # first call on the source: its bins only
    np.testing.assert_array_equal(every.calculateScore(big)[:len(poses)], single)   # a later large batch: every bin at once
    np.testing.assert_array_equal(every.calculateScore(poses), single)
    np.testing.assert_array_equal(every.calculateScore(big), many.calculateScore(big))


def test_set_source_replaces_every_ordering(oracle, api, synth, scene):
    poses = mixed_poses(synth, scene["p_true"], n=64, seed=5)
    rng = np.random.default_rng(11)
    other = np.ascontiguousarray(scene["scan"][rng.permutation(len(scene["scan"]))[:1500]] + np.float32(0.05))
    o, g = engines(oracle, api, scene["map"], scene["scan"])
    g.calculateScore(poses)
    g.setInputSource(other)          # fewer points: no stale entries of the longer scan may be read
    o.set_source(other)
    s1 = assert_oracle(o, g, poses)
    _, fresh = engines(oracle, api, scene["map"], other)
    np.testing.assert_array_equal(fresh.calculateScore(poses), s1)
    g.setInputSource(scene["scan"])  # and back
    _, first = engines(oracle, api, scene["map"], scene["scan"])
    np.testing.assert_array_equal(g.calculateScore(poses), first.calculateScore(poses))


@pytest.mark.parametrize("n", [1, 17, 31, 32, 1023, 1025, 2049])
def test_scan_lengths(oracle, api, synth, scene, n):
    scan = np.ascontiguousarray(scene["scan"][:n])
    o, g = engines(oracle, api, scene["map"], scan)
    poses = mixed_poses(synth, scene["p_true"], n=24, seed=n)
    assert_oracle(o, g, poses)
    assert_batch_independent(api, g, poses)


@pytest.mark.parametrize("n", [40_000, (1 << 23) + 5])
def test_large_scans(oracle, api, synth, scene, n):
    """40k points: 256 yaw bins; over 8M points the orderings would exceed their memory bound and the scan is scored in
    its sensor order."""
    rng = np.random.default_rng(n)
    base = scene["scan"]
    scan = np.ascontiguousarray(base[rng.integers(0, len(base), n)] + rng.normal(0, 0.05, (n, 3)).astype(np.float32))
    o, g = engines(oracle, api, scene["map"], scan)
    poses = mixed_poses(synth, scene["p_true"], n=6 if n > 1e6 else 24, seed=7)
    assert_oracle(o, g, poses)
    full = g.calculateScore(poses)
    np.testing.assert_array_equal(np.array([g.calculateScore(poses[i:i + 1])[0] for i in range(len(poses))]), full)


def test_points_beyond_morton_clamp(oracle, api, synth, scene):
    scan = scene["scan"].copy()
    far = np.array([[700, 0, 0], [-900, 30, 2], [0, 5000, -1], [1e5, -1e5, 1e4], [-600, -600, 600]], np.float32)
    scan[::400][:len(far)] = far
    o, g = engines(oracle, api, scene["map"], scan)
    poses = np.concatenate([mixed_poses(synth, scene["p_true"], n=24, seed=8), yaw_poses(synth, scene["p_true"], boundary_yaws()[::9])])
    assert_oracle(o, g, poses)
    assert_batch_independent(api, g, poses[:24])


def test_scan_with_nan_points(oracle, api, synth, scene):
    scan = scene["scan"].copy()
    scan[3] = [np.nan, 0, 0]
    scan[1200] = [0, np.inf, 1]
    scan[2500] = [np.nan, np.nan, np.nan]
    g = api.NormalDistributionsTransform()
    g.setInputTarget(scene["map"])
    g.setInputSource(scan)
    poses = mixed_poses(synth, scene["p_true"], n=24, seed=9)
    s = assert_batch_independent(api, g, poses)
    fin = np.isfinite(s)
    if fin.any():   # relocalize ranks NaN below every real score
        best, score, _ = api.relocalize(g, poses)
        assert best == int(np.argmax(np.where(fin, s, -np.inf))) and score == s[best]


def test_align_derivatives_fitness_unchanged(api, synth):
    """The per-yaw orderings feed the score kernel only: derivatives, Hessian, align and fitness are bit-identical to the
    values tools/make_score_order_golden.py wrote with the build before the orderings existed."""
    import os
    import sys
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools"))
    import make_score_order_golden as mk
    gold = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "score_order_ndt.npz"))
    got = mk.compute(api, synth)
    assert sorted(got) == sorted(gold.files)
    for k in gold.files:
        np.testing.assert_array_equal(got[k], gold[k], err_msg=k)
