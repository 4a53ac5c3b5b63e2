"""Plain numpy restatement of the three products of csrc/voxel.cu, independent of the device and of the fp32 oracle:

- pcl::VoxelGrid's partition (the cell index floor(p * inv_leaf) in float32 exactly as PCL computes it, including the
  (float)min_b subtraction), grouped in int64, voxels in ascending leaf index, centroids as float64 means;
- construct_full_map: pose7 -> rotation in float64 narrowed to a float32 3x4, the points moved in float32 in
  pcl::transformPointCloud's order (the library is built with -fmad=false, so numpy reproduces it bit for bit), the
  float32 floor partition and float64 sums;
- ImuProcess::UndistortPcl for motions with a closed form (rest, constant velocity, constant yaw rate), in float64.

Also builds the IMU pose tables those motions need, so that the CPU and the GPU tests run the same recipes."""
import numpy as np

F32 = np.float32
U32 = 2.0 ** -24          # unit roundoff of float32
KEY_BIAS = 1 << 20        # the map builder's cells are 21-bit biased fields: [-2^20, 2^20 - 1] per axis
MAX_CELLS = 9.0e18        # the downsampler refuses grids with more leaves than this


def running_sum_bound(counts, maxabs):
    """|fp32 mean - fp64 mean| for a mean of `counts` values of magnitude <= maxabs summed left to right in float32 and
    divided in float32: (n - 1) roundings of partial sums <= n * maxabs, one of the quotient; (count + 1) * 2^-24 * maxabs."""
    return (np.asarray(counts, np.float64) + 1.0) * U32 * np.asarray(maxabs, np.float64)


def ulp32(x):
    """Spacing of float32 at |x|."""
    return np.spacing(np.abs(np.asarray(x, np.float32))).astype(np.float64)


def _records(xyzi):
    a = np.asarray(xyzi, np.float32)
    inten = a[:, 3] if a.shape[1] >= 4 else np.zeros(len(a), np.float32)
    return a[:, :3], inten


def voxel_grid(xyzi, leaf, min_points=0):
    """pcl::VoxelGrid::filter on [n, 3] or [n, >= 4] float32 records (the 4th column is the intensity).
    Returns (centroids [m, 4] float64, counts [m] int64, leaf index [m] int64) in ascending leaf index.
    Raises OverflowError where the grid has more than 9e18 leaves."""
    xyz, inten = _records(xyzi)
    ok = np.isfinite(xyz).all(1)
    p, w = xyz[ok], inten[ok]
    if len(p) == 0:
        return np.zeros((0, 4)), np.zeros(0, np.int64), np.zeros(0, np.int64)
    inv = F32(1.0) / F32(leaf)
    min_b = np.floor(p.min(0) * inv).astype(np.int64)
    div_b = np.floor(p.max(0) * inv).astype(np.int64) - min_b + 1
    if int(div_b[0]) * int(div_b[1]) * int(div_b[2]) > MAX_CELLS:
        raise OverflowError("grid of more than 9e18 leaves")
    ijk = (np.floor(p * inv) - min_b.astype(F32)).astype(np.int64)       # float32 subtraction, as (float)min_b in PCL
    idx = ijk[:, 0] + ijk[:, 1] * div_b[0] + ijk[:, 2] * div_b[0] * div_b[1]
    order = np.argsort(idx, kind="stable")
    uk, start, counts = np.unique(idx[order], return_index=True, return_counts=True)
    vals = np.concatenate([p, w[:, None]], 1).astype(np.float64)[order]
    cent = np.add.reduceat(vals, start, axis=0) / counts[:, None]
    keep = counts >= min_points
    return cent[keep], counts[keep].astype(np.int64), uk[keep]


def pose_matrix(p7):
    """x y z qw qx qy qz -> rotation in float64 narrowed to a float32 3x4 (Translation * Quaterniond, as poses.txt)."""
    x0, y0, z0, w, x, y, z = (float(v) for v in p7)
    R = np.array([[1 - 2 * (y * y + z * z), 2 * (x * y - z * w), 2 * (x * z + y * w)],
                  [2 * (x * y + z * w), 1 - 2 * (x * x + z * z), 2 * (y * z - x * w)],
                  [2 * (x * z - y * w), 2 * (y * z + x * w), 1 - 2 * (x * x + y * y)]])
    return np.concatenate([R, [[x0], [y0], [z0]]], 1).astype(F32)


def transform(xyzi, p7):
    """pcl::transformPointCloud in float32: ((m0 x + m1 y) + m2 z) + m3 per row; returns [n, 4] float32 (intensity kept)."""
    a = np.asarray(xyzi, np.float32)
    M = pose_matrix(p7)
    with np.errstate(invalid="ignore"):       # 0 * inf: a non-finite point becomes NaN and is skipped
        q = [((M[r, 0] * a[:, 0] + M[r, 1] * a[:, 1]) + M[r, 2] * a[:, 2]) + M[r, 3] for r in range(3)]
    return np.stack(q + [a[:, 3]], 1).astype(F32)


def map_build(frames, poses7, leaf):
    """construct_full_map: every keyframe moved by its pose, merged, partitioned by floor(p * inv_leaf) per axis.
    Returns dict(cells [m, 3] int64 (cx, cy, cz), counts [m], cent [m, 4] float64, out_of_range = finite points whose cell
    is outside the key range, pts = the moved finite points as float32), voxels in ascending (cz, cy, cx)."""
    moved = np.concatenate([transform(f, p) for f, p in zip(frames, poses7)])
    moved = moved[np.isfinite(moved[:, :3]).all(1)]
    inv = F32(1.0) / F32(leaf)
    cells = np.floor(moved[:, :3] * inv).astype(np.int64)
    inr = ((cells >= -KEY_BIAS) & (cells < KEY_BIAS)).all(1)
    moved, cells = moved[inr], cells[inr]
    c = cells + KEY_BIAS
    key = (c[:, 2] << 42) | (c[:, 1] << 21) | c[:, 0]
    uk, inv_idx, counts = np.unique(key, return_inverse=True, return_counts=True)
    sums = np.zeros((len(uk), 4))
    np.add.at(sums, inv_idx, moved.astype(np.float64))
    ucells = np.stack([(uk & 0x1FFFFF), (uk >> 21) & 0x1FFFFF, (uk >> 42) & 0x1FFFFF], 1) - KEY_BIAS
    return dict(cells=ucells, counts=counts.astype(np.int64), cent=sums / counts[:, None], out_of_range=int((~inr).sum()), pts=moved)


# ------------------------------------------------------------------ undistortion
def rot_z(a):
    c, s = np.cos(a), np.sin(a)
    return np.array([[c, -s, 0.0], [s, c, 0.0], [0.0, 0.0, 1.0]])


def imu_motion(times, vel=(0.0, 0.0, 0.0), yaw_rate=0.0, ext_t=(0.0, 0.0, 0.0)):
    """IMU poses (K x 22: t, acc, gyr, vel, pos, rot row-major) at the ascending `times` (s) of a motion with constant world
    velocity `vel` and constant yaw rate, and the end state (26) at T = times[-1], lidar-to-IMU rotation identity and
    translation ext_t.  Returns (poses, x_end, T).  Every segment of the reference's integration is exact for such a motion."""
    v = np.asarray(vel, np.float64)
    K = len(times)
    poses = np.zeros((K, 22))
    for k in range(K):
        t = float(times[k])
        poses[k, 0] = t
        poses[k, 4:7] = (0.0, 0.0, yaw_rate)
        poses[k, 7:10] = v
        poses[k, 10:13] = v * t
        poses[k, 13:22] = rot_z(yaw_rate * t).reshape(9)
    T = float(times[-1])
    x = np.zeros(26)
    x[0:3] = v * T
    x[3:7] = (0.0, 0.0, np.sin(yaw_rate * T / 2), np.cos(yaw_rate * T / 2))
    x[7:11] = (0.0, 0.0, 0.0, 1.0)
    x[11:14] = ext_t
    return poses, x, T


def undistort_closed_form(xyz, t, T, vel=(0.0, 0.0, 0.0), yaw_rate=0.0, ext_t=(0.0, 0.0, 0.0)):
    """The point seen at time t (s) in the lidar frame, expressed in the lidar frame at T, for the motion of imu_motion:
    p' = Rz(-w (T - t)) (p + e) - v_end (T - t) - e with v_end = Rz(-w T) v, e the lidar-to-IMU translation.  float64."""
    p = np.asarray(xyz, np.float64)
    e = np.asarray(ext_t, np.float64)
    v = np.asarray(vel, np.float64)
    dt = T - np.asarray(t, np.float64)
    a = -yaw_rate * dt
    c, s = np.cos(a), np.sin(a)
    q = p + e
    out = np.stack([c * q[:, 0] - s * q[:, 1], s * q[:, 0] + c * q[:, 1], q[:, 2]], 1)
    return out - dt[:, None] * (rot_z(-yaw_rate * T) @ v)[None, :] - e
