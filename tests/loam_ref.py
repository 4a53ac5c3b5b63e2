"""Plain float64 restatement of one LOAM scan-to-map pass (jueying_slam mapOptmization.cpp:1255-1558), independent of the
device and of the fp32 oracle: exact 5-NN by a k-d tree, the corner line and surf plane by numpy linear algebra, and the
Jacobian of the LM step by central differences.  Inputs are float32 arrays; everything after that is float64.

Also builds the scenes the LOAM tests share (a corridor that makes the LM step degenerate, lattice maps with exact
distances) so that the CPU and the GPU tests run the same recipes."""
import numpy as np
from scipy.spatial import cKDTree

LARGE_ANGLE_POSES = ((0.4, -0.5, 2.5, 3.0, -2.0, 1.2), (-0.3, 1.3, -3.0, 3.0, -2.0, 1.2), (3.0, 0.2, 0.1, 3.0, -2.0, 1.2))
CORRIDOR_T = (0.01, -0.02, 0.1, 1.0, 0.2, 1.2)


def pose_matrix(t6):
    """pcl::getTransformation(x, y, z, roll, pitch, yaw) for t6 = (roll, pitch, yaw, x, y, z): (R, t) in float64."""
    r, p, y = (float(v) for v in t6[:3])
    cr, sr, cp, sp, cy, sy = np.cos(r), np.sin(r), np.cos(p), np.sin(p), np.cos(y), np.sin(y)
    Rx = np.array([[1, 0, 0], [0, cr, -sr], [0, sr, cr]])
    Ry = np.array([[cp, 0, sp], [0, 1, 0], [-sp, 0, cp]])
    Rz = np.array([[cy, -sy, 0], [sy, cy, 0], [0, 0, 1]])
    return Rz @ Ry @ Rx, np.array([float(v) for v in t6[3:]])


def to_world(pts, t6):
    R, t = pose_matrix(t6)
    return np.asarray(pts, np.float64)[:, :3] @ R.T + t


class Pass:
    """One cornerOptimization + surfOptimization pass at t6 in float64.  Per point: flag, coeff (4), and `masked` = the point
    sits within rounding distance of one of the pass's decisions, where fp32 and fp64 may legitimately disagree."""

    def __init__(self, corner_map, surf_map, corner, surf, t6):
        corner, surf = np.asarray(corner, np.float32)[:, :3], np.asarray(surf, np.float32)[:, :3]
        self.nc, n = len(corner), len(corner) + len(surf)
        self.flags = np.zeros(n, np.uint8)
        self.coeff = np.zeros((n, 4))
        self.masked = np.zeros(n, bool)
        self.d2 = np.full((n, 5), np.inf)
        self.cond = np.ones(n)   # condition number of the surf plane fit's 5x3 system
        for base, pts, mp, fn in ((0, corner, corner_map, self._corner), (self.nc, surf, surf_map, self._surf)):
            if len(pts) == 0:
                continue
            mp = np.asarray(mp, np.float64)[:, :3]
            if len(mp) < 6:
                raise ValueError("the reference pass needs at least six map points per class")
            w = to_world(pts, t6)
            d, idx = cKDTree(mp).query(w, 6)
            self.d2[base:base + len(pts)] = d[:, :5] ** 2
            for i in range(len(pts)):
                k = base + i
                # the gate pointSearchSqDis[4] < 1.0, and the choice between the 5th and the 6th neighbour
                self.masked[k] = abs(d[i, 4] ** 2 - 1.0) < 1e-4 or d[i, 5] - d[i, 4] < 2e-5
                if not d[i, 4] ** 2 < 1.0:
                    continue
                if base:
                    self.cond[k] = np.linalg.cond(mp[idx[i, :5]])
                sel, co, near = fn(mp[idx[i, :5]], w[i])
                self.masked[k] |= near
                if sel:
                    self.flags[k] = 1
                    self.coeff[k] = co

    @staticmethod
    def _corner(nb, p):
        c = nb.mean(0)
        lam, V = np.linalg.eigh((nb - c).T @ (nb - c) / 5)
        l1, l2, v = lam[2], lam[1], V[:, 2]
        near = abs(l1 - 3 * l2) < 1e-3 * l1
        if not l1 > 3 * l2:
            return False, None, near
        r = (p - c) - np.dot(p - c, v) * v       # from the line c + s v to the point
        dist = np.linalg.norm(r)
        s = 1 - 0.9 * dist
        return s > 0.1, np.r_[s * r / dist, s * dist], near or abs(s - 0.1) < 1e-4

    @staticmethod
    def _surf(nb, p):
        X = np.linalg.lstsq(nb, -np.ones(5), rcond=None)[0]
        ps = np.linalg.norm(X)
        nrm, pd = X / ps, 1 / ps
        res = np.abs(nb @ nrm + pd)
        near = bool(np.any(np.abs(res - 0.2) < 1e-4))
        if np.any(res > 0.2):
            return False, None, near
        pd2 = nrm @ p + pd
        s = 1 - 0.9 * abs(pd2) / np.sqrt(np.linalg.norm(p))   # weighted by the world-frame point pointSel, as the device does
        return s > 0.1, np.r_[s * nrm, s * pd2], near or abs(s - 0.1) < 1e-4


def jtj(corner, surf, flags, coeff, t6, h=1e-6):
    """A^T A of LMOptimization at t6 for the selected points: rows d/d(roll, pitch, yaw, x, y, z) of coeff[:3] . (R p + t),
    by central differences in float64 (the rotation rows) and exactly (the translation rows)."""
    pts = np.concatenate([np.asarray(corner, np.float32)[:, :3], np.asarray(surf, np.float32)[:, :3]]).astype(np.float64)
    sel = np.asarray(flags).astype(bool)
    p, c = pts[sel], np.asarray(coeff, np.float64)[sel, :3]
    t6 = np.asarray(t6, np.float64)
    J = np.empty((len(p), 6))
    for k in range(3):
        e = np.zeros(6)
        e[k] = h
        dR = (pose_matrix(t6 + e)[0] - pose_matrix(t6 - e)[0]) / (2 * h)
        J[:, k] = np.einsum("ij,ij->i", c, p @ dR.T)
    J[:, 3:] = c
    return J.T @ J


def rel_err(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return np.abs(a - b).max() / np.abs(b).max()


def check_features(ref, flags, coeff):
    """The bars a pass computed in fp32 must meet against the fp64 pass (points on a decision threshold excluded)."""
    keep = ~ref.masked
    np.testing.assert_array_equal(np.asarray(flags)[keep], ref.flags[keep])
    both = keep & ref.flags.astype(bool)
    err = np.abs(np.asarray(coeff, np.float64) - ref.coeff).max(1)
    nc = ref.nc
    cm, sm = both.copy(), both.copy()
    cm[nc:] = False
    sm[:nc] = False
    if cm.any():
        # the distance to the line to 5e-5; the normal's direction to 5e-5 plus what a few-micrometre rounding of the
        # fp32 world coordinates (~20 m) turns into at the point's distance (scan corners lie 0.3 mm from their line)
        co = np.asarray(coeff, np.float64)[cm]
        assert np.abs(co[:, 3] - ref.coeff[cm, 3]).max() <= 5e-5
        dir_err = np.abs(co[:, :3] - ref.coeff[cm, :3]).max(1)
        bar = 5e-5 + 2e-5 / np.abs(ref.coeff[cm, 3])
        assert np.all(dir_err <= bar), (dir_err / bar).max()
    if sm.any():
        # plane fits of the form q X = -1 are ill-conditioned for planes that pass near the world origin (condition numbers
        # of 1e4 on the corridor's floor): there fp32 is held to its rounding times the condition number
        bar = 5e-4 + 1e-7 * ref.cond[sm]
        assert np.all(err[sm] <= bar), (err[sm] / bar).max()
        assert np.median(err[sm]) <= 1e-5, np.median(err[sm])
    return both


def weak_step_fraction(AtA, t_in, t_out, limit=100.0):
    """|component of the step along the eigenvectors of AtA with eigenvalue < limit| / |step|."""
    lam, V = np.linalg.eigh(np.asarray(AtA, np.float64))
    W = V[:, lam < limit]
    assert W.shape[1] > 0, lam
    d = np.asarray(t_out, np.float64) - np.asarray(t_in, np.float64)
    return np.linalg.norm(W.T @ d) / np.linalg.norm(d)


# ------------------------------------------------------------------ scenes
def to_body(pw, t6):
    R, t = pose_matrix(t6)
    return np.ascontiguousarray(((np.asarray(pw, np.float64) - t) @ R).astype(np.float32))


def corridor(seed=5, t_true=CORRIDOR_T):
    """A floor and two walls along x with four x-direction edges: translation along x and yaw-free sliding are only held by
    the few sparse features, so the first A^T A has eigenvalues below 100 (LMOptimization's degeneracy test fires)."""
    rng = np.random.default_rng(seed)
    n, sig = 40_000, 0.002
    x = lambda: rng.uniform(-30, 30, n)
    floor = np.stack([x(), rng.uniform(-2, 2, n), np.zeros(n)], 1)
    wall_l = np.stack([x(), np.full(n, -2.0), rng.uniform(0, 3, n)], 1)
    wall_r = np.stack([x(), np.full(n, 2.0), rng.uniform(0, 3, n)], 1)
    surf_map = np.concatenate([floor, wall_l, wall_r])
    surf_map = (surf_map + rng.normal(0, sig, surf_map.shape)).astype(np.float32)
    edges = [np.stack([rng.uniform(-30, 30, 3000), np.full(3000, y), np.full(3000, z)], 1) for y in (-2.0, 2.0) for z in (0.0, 3.0)]
    corner_map = np.concatenate(edges)
    corner_map = (corner_map + rng.normal(0, sig, corner_map.shape)).astype(np.float32)
    t_true = np.array(t_true, np.float32)
    t = t_true[3:].astype(np.float64)
    surf = to_body(surf_map[np.linalg.norm(surf_map - t, axis=1) < 20][::40], t_true)
    corner = to_body(corner_map[np.linalg.norm(corner_map - t, axis=1) < 20][::20], t_true)
    return dict(corner_map=corner_map, surf_map=surf_map, corner=corner, surf=surf, t_true=t_true)


GATE_Q, BELOW_Q, TIE5_Q, TIE56_Q = (0.0, 0.0, 5.0), (10.0, 0.0, 5.0), (20.0, 0.0, 5.0), (30.0, 0.0, 5.0)
TIE56_A, TIE56_B = (30.5, 0.0, 5.5), (30.5, 0.5, 5.0)


def lattice():
    """A surf map of small exact-binary point sets on the plane z = 5, one per query; at t6 = 0 the world point is the lidar
    point bit for bit, so every squared distance below is exact in fp32:
      GATE_Q   the query itself and four points at d2 = 1.0 exactly: the 5th neighbour fails the gate d2 < 1.0
      BELOW_Q  neighbours at 0, 0.0625, 0.140625, 0.25 and the 5th at d2 = 1 - 2^-24 (dx = 2^-12, dy = 1 - 2^-24), the
               largest float below 1.0: accepted
      TIE5_Q   four neighbours tied at d2 = 0.25 behind the query itself, the 6th at 0.8125: ties inside the five only
      TIE56_Q  neighbours at 0, 0.25 x 3, then TIE56_A (off the plane) and TIE56_B (on it) tied at d2 = 0.5 for 5th / 6th
    Returns (surf_map, surf scan)."""
    f = np.float32
    pts = [(0, 0, 5), (1, 0, 5), (-1, 0, 5), (0, 1, 5), (0, -1, 5),
           (10, 0, 5), (10.5, 0, 5), (9.75, 0, 5), (10, -0.375, 5), (f(10) + f(2.0 ** -12), f(1) - f(2.0 ** -24), 5),
           (20, 0, 5), (20.5, 0, 5), (19.5, 0, 5), (20, 0.5, 5), (20, -0.5, 5), (20.75, 0.5, 5),
           (30, 0, 5), (29.5, 0, 5), (30, 0.5, 5), (30, -0.5, 5), TIE56_A, TIE56_B]
    surf_map = np.array(pts, np.float32)
    scan = np.array([GATE_Q, BELOW_Q, TIE5_Q, TIE56_Q], np.float32)
    return surf_map, scan


def fp32_d2(mp, q):
    """The squared distances exactly as the search computes them: (dx*dx + dy*dy) + dz*dz, one rounding per fp32 op."""
    d = np.asarray(mp, np.float32) - np.asarray(q, np.float32)
    return (d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1]) + d[:, 2] * d[:, 2]


def mode_scenes():
    """The sparse and the dense scene of the walk-variant comparison (the dense scan is thinned to keep the oracle cheap)."""
    from pointcloud_slam_b200 import synth
    out = {}
    for name, n_map, step in (("sparse", 60_000, 1), ("dense", 250_000, 3)):
        sc = synth.loam_scene(n_surf_map=n_map)
        sc["surf"] = np.ascontiguousarray(sc["surf"][::step])
        sc["guess"] = sc["t_true"] + np.array([0.01, -0.01, 0.02, 0.15, -0.1, 0.05], np.float32)
        out[name] = sc
    return out


def stencil_candidates(mp, q):
    """Per query: the number of map points in the 27 cells around it on the LOAM index (1 m cells, cell = round(p))."""
    cells = np.round(np.asarray(mp, np.float32)[:, :3]).astype(np.int64)
    keys, cnt = np.unique(cells, axis=0, return_counts=True)
    occ = dict(zip(map(tuple, keys.tolist()), cnt.tolist()))
    offs = [(a, b, c) for a in (-1, 0, 1) for b in (-1, 0, 1) for c in (-1, 0, 1)]
    qc = np.round(np.asarray(q, np.float32)).astype(np.int64).tolist()
    return np.array([sum(occ.get((x + a, y + b, z + c), 0) for a, b, c in offs) for x, y, z in qc]), len(keys), int(cnt.max())
