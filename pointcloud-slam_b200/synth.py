"""Seeded synthetic worlds, maps and Livox-shaped scans (SURVEY.md §8d).

Everything the benchmarks and parity tests feed to the engine comes from here:
there is no network, no dataset, and the reference's own fixtures are absent
(SURVEY.md §4).  The world is an axis-aligned "warehouse": a 120 m x 80 m x 8 m
room with 40 interior box obstacles.  Maps are surface samples with Gaussian
noise along the normal; scans are ray casts from a sensor pose with range noise.
Coordinates are continuous float32, so exact distance ties have probability ~0.
"""
from __future__ import annotations

import numpy as np

SEED = 20261018
ROOM = np.array([[-60.0, -40.0, 0.0], [60.0, 40.0, 8.0]])


def make_world(seed: int = SEED, n_obstacles: int = 40, offset=(0.0, 0.0, 0.0), beams: bool = False):
    """Returns (room[2,3], boxes[n,2,3]) — axis-aligned obstacle boxes standing on the floor.
    beams=True adds a roof truss (0.4 m x 0.8 m beams hanging from the ceiling every 6 m in x and 8 m in y) so that
    an upward-looking scan, which sees mostly ceiling, still constrains x/y (used by the NDT configs)."""
    rng = np.random.default_rng(seed)
    size = rng.uniform(1.0, 6.0, size=(n_obstacles, 3))
    size[:, 2] = np.minimum(size[:, 2], 5.0)
    lo_xy = np.stack([rng.uniform(ROOM[0, 0] + 2, ROOM[1, 0] - 8, n_obstacles),
                      rng.uniform(ROOM[0, 1] + 2, ROOM[1, 1] - 8, n_obstacles)], 1)
    lo = np.concatenate([lo_xy, np.zeros((n_obstacles, 1))], 1)
    boxes = np.stack([lo, lo + size], 1)
    if beams:
        bl = []
        jit = rng.uniform(-1.0, 1.0, 64)
        for k, x0 in enumerate(np.arange(ROOM[0, 0] + 3.0, ROOM[1, 0] - 1.0, 6.0)):
            x0 = x0 + jit[k]
            bl.append([[x0, ROOM[0, 1], ROOM[1, 2] - 0.8], [x0 + 0.4, ROOM[1, 1], ROOM[1, 2]]])
        for k, y0 in enumerate(np.arange(ROOM[0, 1] + 4.0, ROOM[1, 1] - 1.0, 8.0)):
            y0 = y0 + jit[32 + k]
            bl.append([[ROOM[0, 0], y0, ROOM[1, 2] - 0.5], [ROOM[1, 0], y0 + 0.4, ROOM[1, 2]]])
        boxes = np.concatenate([boxes, np.array(bl)], 0)
    off = np.asarray(offset, dtype=np.float64)
    return ROOM + off, boxes + off


def _faces(room, boxes):
    """List of faces as (origin, edge_u, edge_v, normal, area)."""
    faces = []

    def add_box(lo, hi, inward):
        d = hi - lo
        for ax in range(3):
            u, v = (ax + 1) % 3, (ax + 2) % 3
            eu = np.zeros(3); eu[u] = d[u]
            ev = np.zeros(3); ev[v] = d[v]
            for side in (0, 1):
                o = lo.copy()
                if side:
                    o[ax] = hi[ax]
                nrm = np.zeros(3)
                nrm[ax] = (1.0 if side else -1.0) * (-1.0 if inward else 1.0)
                faces.append((o, eu, ev, nrm, d[u] * d[v]))

    add_box(room[0], room[1], True)
    for b in boxes:
        # the face of an obstacle that lies in the floor (or, for a roof beam, in the ceiling) is not a surface: skip it
        lo, hi = b
        on_floor = abs(lo[2] - room[0][2]) < 1e-9
        on_ceiling = abs(hi[2] - room[1][2]) < 1e-9
        d = hi - lo
        for ax in range(3):
            u, v = (ax + 1) % 3, (ax + 2) % 3
            eu = np.zeros(3); eu[u] = d[u]
            ev = np.zeros(3); ev[v] = d[v]
            for side in (0, 1):
                if ax == 2 and ((side == 0 and on_floor) or (side == 1 and on_ceiling)):
                    continue
                o = lo.copy()
                if side:
                    o[ax] = hi[ax]
                nrm = np.zeros(3)
                nrm[ax] = 1.0 if side else -1.0
                faces.append((o, eu, ev, nrm, d[u] * d[v]))
    return faces


def sample_map(n_points: int, seed: int = SEED, sigma: float = 0.01, world=None) -> np.ndarray:
    """n_points surface samples (float32 [n,3]), area-uniform, noise sigma along the face normal."""
    room, boxes = world if world is not None else make_world(seed)
    faces = _faces(room, boxes)
    rng = np.random.default_rng(seed + 1)
    areas = np.array([f[4] for f in faces])
    counts = rng.multinomial(n_points, areas / areas.sum())
    out = np.empty((n_points, 3), dtype=np.float64)
    k = 0
    for (o, eu, ev, nrm, _), c in zip(faces, counts):
        if c == 0:
            continue
        a = rng.random((c, 1)); b = rng.random((c, 1))
        out[k:k + c] = o + a * eu + b * ev + rng.normal(0.0, sigma, (c, 1)) * nrm
        k += c
    rng.shuffle(out, axis=0)
    return out.astype(np.float32)


def livox_dirs(n_rays: int, seed: int = SEED, fov_deg=(-7.0, 52.0)) -> np.ndarray:
    """Mid-360-shaped ray bundle: azimuth by golden-angle rosette + jitter, elevation uniform in fov."""
    rng = np.random.default_rng(seed + 2)
    i = np.arange(n_rays)
    az = (i * 2.399963229728653 + rng.uniform(-0.01, 0.01, n_rays)) % (2 * np.pi)
    el = np.deg2rad(rng.uniform(fov_deg[0], fov_deg[1], n_rays))
    return np.stack([np.cos(el) * np.cos(az), np.cos(el) * np.sin(az), np.sin(el)], 1)


def avia_dirs(n_rays: int, seed: int = SEED) -> np.ndarray:
    """Avia-shaped bundle: 70.4 deg x 77.2 deg forward FoV rosette."""
    rng = np.random.default_rng(seed + 3)
    az = np.deg2rad(rng.uniform(-35.2, 35.2, n_rays))
    el = np.deg2rad(rng.uniform(-38.6, 38.6, n_rays))
    return np.stack([np.cos(el) * np.cos(az), np.cos(el) * np.sin(az), np.sin(el)], 1)


def quat_to_R(q) -> np.ndarray:
    x, y, z, w = q
    return np.array([[1 - 2 * (y * y + z * z), 2 * (x * y - z * w), 2 * (x * z + y * w)],
                     [2 * (x * y + z * w), 1 - 2 * (x * x + z * z), 2 * (y * z - x * w)],
                     [2 * (x * z - y * w), 2 * (y * z + x * w), 1 - 2 * (x * x + y * y)]])


def quat_from_rotvec(r) -> np.ndarray:
    r = np.asarray(r, dtype=np.float64)
    th = np.linalg.norm(r)
    if th < 1e-12:
        return np.array([0.5 * r[0], 0.5 * r[1], 0.5 * r[2], 1.0])
    s = np.sin(th / 2) / th
    return np.array([r[0] * s, r[1] * s, r[2] * s, np.cos(th / 2)])


def quat_mul(a, b) -> np.ndarray:
    ax, ay, az, aw = a
    bx, by, bz, bw = b
    return np.array([aw * bx + ax * bw + ay * bz - az * by, aw * by + ay * bw + az * bx - ax * bz,
                     aw * bz + az * bw + ax * by - ay * bx, aw * bw - ax * bx - ay * by - az * bz])


def raycast(origin, R, dirs, world, rmin=0.1, rmax=40.0, sigma=0.02, seed=SEED) -> np.ndarray:
    """Casts sensor-frame dirs from (origin, R) into the world; returns sensor-frame hits float32 [m,3]."""
    room, boxes = world
    d = dirs @ R.T
    o = np.asarray(origin, dtype=np.float64)
    with np.errstate(divide="ignore", invalid="ignore"):
        inv = 1.0 / d
        # room: we are inside; exit distance
        t1 = (room[0] - o) * inv
        t2 = (room[1] - o) * inv
        t_exit = np.min(np.maximum(t1, t2), axis=1)
        t_hit = t_exit.copy()
        for b in boxes:
            ta = (b[0] - o) * inv
            tb = (b[1] - o) * inv
            tn = np.max(np.minimum(ta, tb), axis=1)
            tf = np.min(np.maximum(ta, tb), axis=1)
            ok = (tn <= tf) & (tn > 0)
            t_hit = np.where(ok & (tn < t_hit), tn, t_hit)
    rng = np.random.default_rng(seed + 4)
    t_hit = t_hit + rng.normal(0.0, sigma, t_hit.shape)
    keep = (t_hit >= rmin) & (t_hit <= rmax) & np.isfinite(t_hit)
    return (dirs[keep] * t_hit[keep, None]).astype(np.float32)


# ---- jueying_lio state helpers (26 doubles: pos rot(xyzw) offR(xyzw) offT vel bg ba grav) ----
EXT_T = np.array([0.1713, 0.0, 0.05925])  # config/livox.yaml:20 (SURVEY.md §8d)


def make_state(pos, rotvec, ext_t=EXT_T) -> np.ndarray:
    x = np.zeros(26)
    x[0:3] = pos
    x[3:7] = quat_from_rotvec(rotvec)
    x[7:11] = [0, 0, 0, 1]
    x[11:14] = ext_t
    x[23:26] = [0.0, 0.0, -9.809]
    return x


def init_cov(seed: int = SEED) -> np.ndarray:
    """IMU-init covariance (imu_processing.hpp:154-161) plus a small seeded SPD coupling term,
    standing in for 0.1 s of propagation (the IMU pipeline is out of scope, SURVEY.md §8f)."""
    d = np.ones(23)
    d[6:12] = 1e-5
    d[15:18] = 1e-4
    d[18:21] = 1e-3
    d[21:23] = 1e-5
    rng = np.random.default_rng(seed + 5)
    G = rng.normal(0.0, 1.0, (23, 4)) * np.sqrt(d)[:, None] * 0.3
    P = np.diag(d) + G @ G.T
    return 0.5 * (P + P.T)


def lidar_pose(x: np.ndarray):
    R = quat_to_R(x[3:7])
    Rl = R @ quat_to_R(x[7:11])
    return R @ x[11:14] + x[0:3], Rl


def perturb_state(x_true: np.ndarray, seed: int = SEED, dpos=0.05, drot_deg=0.5) -> np.ndarray:
    rng = np.random.default_rng(seed + 6)
    x = x_true.copy()
    x[0:3] += rng.uniform(-dpos, dpos, 3)
    dq = quat_from_rotvec(np.deg2rad(rng.uniform(-drot_deg, drot_deg, 3)))
    x[3:7] = quat_mul(x[3:7], dq)
    return x


def config1(n_map=2_000_000, n_scan=20_000, seed: int = SEED):
    """BASELINE.json configs[0]: Mid-360-shaped scan vs local map, one IEKF update.
    Returns dict(map, scan, x_true, x_prop, P)."""
    world = make_world(seed)
    mp = sample_map(n_map, seed, world=world)
    x_true = make_state([3.0, -2.0, 1.2], [0.01, -0.02, 0.6])
    o, Rl = lidar_pose(x_true)
    # oversample rays so ~n_scan survive range clipping
    dirs = livox_dirs(int(n_scan * 1.25), seed)
    scan = raycast(o, Rl, dirs, world, seed=seed)[:n_scan]
    return dict(map=mp, scan=np.ascontiguousarray(scan), x_true=x_true, x_prop=perturb_state(x_true, seed),
                P=init_cov(seed), world=world)


def prior_map(n_points=10_000_000, seed: int = SEED):
    """BASELINE.json configs[1]/[3]: the world tiled 2x2 with different seeds."""
    per = n_points // 4
    tiles, worlds = [], []
    for k, (ox, oy) in enumerate([(0, 0), (120, 0), (0, 80), (120, 80)]):
        w = make_world(seed + 100 * k, offset=(ox, oy, 0), beams=True)
        worlds.append(w)
        tiles.append(sample_map(per if k < 3 else n_points - 3 * per, seed + 100 * k, world=w))
    return np.concatenate(tiles, 0), worlds


def pose_vec_to_matrix(p6) -> np.ndarray:
    """(x,y,z,roll,pitch,yaw) -> 4x4 = T * Rx * Ry * Rz (ndt_omp_impl.hpp:129)."""
    cx, sx = np.cos(p6[3]), np.sin(p6[3])
    cy, sy = np.cos(p6[4]), np.sin(p6[4])
    cz, sz = np.cos(p6[5]), np.sin(p6[5])
    Rx = np.array([[1, 0, 0], [0, cx, -sx], [0, sx, cx]])
    Ry = np.array([[cy, 0, sy], [0, 1, 0], [-sy, 0, cy]])
    Rz = np.array([[cz, -sz, 0], [sz, cz, 0], [0, 0, 1]])
    M = np.eye(4)
    M[:3, :3] = Rx @ Ry @ Rz
    M[:3, 3] = p6[:3]
    return M


def config2(n_map=10_000_000, n_scan=20_000, seed: int = SEED):
    """NDT relocalization: 20k scan vs 10M prior map. Returns dict(map, scan, T_true, guess)."""
    mp, worlds = prior_map(n_map, seed)
    p_true = np.array([3.0, -2.0, 1.2, 0.0, 0.0, 0.6])
    T = pose_vec_to_matrix(p_true)
    dirs = livox_dirs(int(n_scan * 1.25), seed)
    scan = raycast(T[:3, 3], T[:3, :3], dirs, worlds[0], seed=seed)[:n_scan]
    rng = np.random.default_rng(seed + 7)
    p_guess = p_true.copy()
    p_guess[0:2] += rng.uniform(-0.5, 0.5, 2)
    p_guess[5] += np.deg2rad(rng.uniform(-3, 3))
    return dict(map=mp, scan=np.ascontiguousarray(scan), p_true=p_true, T_true=T, p_guess=p_guess,
                guess=pose_vec_to_matrix(p_guess).astype(np.float32))


def hypothesis_grid(p_center, nx=32, ny=32, nyaw=4, pitch=1.0) -> np.ndarray:
    """config 4: nx*ny*nyaw poses (float32 [h,16] column-major 4x4) around p_center."""
    out = []
    for iy in range(ny):
        for ix in range(nx):
            for k in range(nyaw):
                p = np.array(p_center, dtype=np.float64)
                p[0] += (ix - nx // 2) * pitch
                p[1] += (iy - ny // 2) * pitch
                p[5] += k * (2 * np.pi / nyaw)
                out.append(pose_vec_to_matrix(p).astype(np.float32).T.reshape(16))
    return np.ascontiguousarray(np.stack(out, 0))


def loop_pairs(P, n_src, n_tgt, seed: int = SEED, drift=(0.3, 2.0), crop_radius=35.0, map_points=None):
    """P loop-closure candidates as mapOptmization.cpp:683-693 registers them (keyframe = source, submap = target, identity
    guess).  Pair p: an anchor pose in the warehouse; the target is the seeded prior map cropped to crop_radius (m, in x/y)
    around the anchor and subsampled to n_tgt[p] points; the source is a raycast scan of n_src[p] points from the anchor,
    moved into the map frame by a drifted pose (up to drift[0] m in x/y and drift[1] degrees in yaw off the anchor).
    n_src / n_tgt are scalars or length-P sequences.  Returns dict(sources, targets, guesses, T_true): T_true[p] (4x4) is
    the correction that undoes the drift, i.e. what align() should return."""
    n_src = np.broadcast_to(np.asarray(n_src, dtype=np.int64), (P,))
    n_tgt = np.broadcast_to(np.asarray(n_tgt, dtype=np.int64), (P,))
    world = make_world(seed, beams=True)
    mp = sample_map(map_points or max(2_000_000, 12 * int(n_tgt.max())), seed, world=world)
    rng = np.random.default_rng(seed + 21)
    sources, targets, T_true = [], [], []
    for p in range(P):
        anchor = np.array([rng.uniform(-45.0, 45.0), rng.uniform(-28.0, 28.0), rng.uniform(1.0, 2.0), 0.0, 0.0, rng.uniform(-np.pi, np.pi)])
        Ta = pose_vec_to_matrix(anchor)
        near = np.flatnonzero(np.hypot(mp[:, 0] - Ta[0, 3], mp[:, 1] - Ta[1, 3]) < crop_radius)
        targets.append(np.ascontiguousarray(mp[np.sort(rng.choice(near, size=min(int(n_tgt[p]), len(near)), replace=False))]))
        dirs = livox_dirs(int(n_src[p] * 1.5) + 64, seed + 1000 + p)
        scan = raycast(Ta[:3, 3], Ta[:3, :3], dirs, world, seed=seed + 1000 + p)[: int(n_src[p])]
        r, a = drift[0] * np.sqrt(rng.uniform()), rng.uniform(-np.pi, np.pi)
        Td = Ta @ pose_vec_to_matrix([r * np.cos(a), r * np.sin(a), 0.0, 0.0, 0.0, np.deg2rad(drift[1]) * rng.uniform(-1.0, 1.0)])
        sources.append(np.ascontiguousarray((scan.astype(np.float64) @ Td[:3, :3].T + Td[:3, 3]).astype(np.float32)))
        T_true.append(Ta @ np.linalg.inv(Td))
    return dict(sources=sources, targets=targets, guesses=[np.eye(4, dtype=np.float32)] * P, T_true=np.array(T_true))


# ---- LOAM scene (jueying_slam scan-to-map): surface map + edge ("corner") map and a scan of both in the lidar frame ----
def pcl_transform(t6):
    """pcl::getTransformation(x, y, z, roll, pitch, yaw) for t6 = (roll, pitch, yaw, x, y, z): (R[3,3], t[3]) in fp64."""
    r, p, y = [float(v) for v in t6[:3]]
    A, B, Cc, D, E, F = np.cos(y), np.sin(y), np.cos(p), np.sin(p), np.cos(r), np.sin(r)
    R = np.array([[A * Cc, A * D * F - B * E, B * F + A * D * E], [B * Cc, A * E + B * D * F, B * D * E - A * F], [-D, Cc * F, Cc * E]])
    return R, np.asarray(t6[3:], dtype=np.float64)


def loam_scene(n_surf_map=60_000, seed: int = SEED, t_true=(0.01, -0.02, 0.6, 3.0, -2.0, 1.2), surf_stride=6, corner_stride=3):
    """Returns dict(corner_map, surf_map, corner, surf, t_true): the maps in the world frame, the scan features in the lidar frame."""
    world = make_world(seed, beams=True)
    _, boxes = world
    rng = np.random.default_rng(seed + 11)
    surf_map = sample_map(n_surf_map, seed, sigma=0.01, world=world)
    edges = []
    for b in boxes[:40]:
        lo, hi = b
        for x in (lo[0], hi[0]):
            for y in (lo[1], hi[1]):
                z = rng.uniform(lo[2], hi[2], 60)
                edges.append(np.stack([np.full(60, x), np.full(60, y), z], 1))
    corner_map = (np.concatenate(edges) + rng.normal(0, 0.01, (len(edges) * 60, 3))).astype(np.float32)
    t_true = np.array(t_true, np.float32)
    R, t = pcl_transform(t_true)

    def to_body(pw):
        return ((pw.astype(np.float64) - t) @ R).astype(np.float32)

    near = np.linalg.norm(surf_map - t, axis=1) < 25
    surf = to_body(surf_map[near][::surf_stride] + rng.normal(0, 0.01, (int(near.sum()), 3))[::surf_stride].astype(np.float32))
    nearc = np.linalg.norm(corner_map - t, axis=1) < 30
    corner = to_body(corner_map[nearc][::corner_stride])
    return dict(corner_map=corner_map, surf_map=surf_map, corner=np.ascontiguousarray(corner), surf=np.ascontiguousarray(surf), t_true=t_true)
