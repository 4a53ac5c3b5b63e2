"""CPU estimate of how many distinct leaf lines a warp of k_ndt_score_batch<7> touches per source point, for several
orderings of the scan.  No GPU involved.

k_ndt_score_batch is bound by the L1 data pipe: each (point, leaf) pair loads a 96-byte fp64 leaf with three 256-bit loads,
and one warp-wide load costs about as many wavefronts as there are distinct lines in it.  Proxy: for every warp of 32
consecutive points and every DIRECT7 slot, count the distinct target cells (occupied or not), times 3 chunks, divided by
the number of points.  Empty cells are counted too, so the absolute numbers sit above what a profiler reports; compare
the orderings with each other.

    python tools/score_order_lines.py [--poses 16] [--bins 16 32 64]

Orderings:
  sensor     Morton order of the sensor-frame voxel (Ndt::set_source's d_src: align, derivatives, fitness)
  bins=NB    Morton order of Rz(psi_b) p, psi_b the yaw bin nearest the pose's yaw (the score kernel's ordering)
  per-pose   Morton order of the exactly transformed point (a per-hypothesis sort: the bound the bins approach)
"""
import argparse
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

DIRECT7 = np.array([[0, 0, 0], [1, 0, 0], [-1, 0, 0], [0, 1, 0], [0, -1, 0], [0, 0, 1], [0, 0, -1]])


def spread10(v):
    out = np.zeros(v.shape, dtype=np.uint64)
    for b in range(10):
        out |= ((v >> b) & 1).astype(np.uint64) << np.uint64(3 * b)
    return out


def morton(x, inv_cell=1.0):
    """ndt.cu morton_key: 10 bits per axis, cell index + 512 clamped to [0, 1023], non-finite points last."""
    ok = np.isfinite(x).all(1)
    c = np.clip(np.floor(np.where(ok[:, None], x, 0) * inv_cell).astype(np.int64) + 512, 0, 1023)
    key = spread10(c[:, 0]) | (spread10(c[:, 1]) << np.uint64(1)) | (spread10(c[:, 2]) << np.uint64(2))
    return np.where(ok, key, np.uint64(0xFFFFFFFF))


def lines_per_point(cells):
    """Distinct DIRECT7 cells per (warp, slot), x 3 chunks of a 96-byte leaf, per point."""
    nb = cells[:, None, :] + DIRECT7[None]
    code = (nb[..., 0] * 8192 + nb[..., 1]) * 8192 + nb[..., 2]
    n = len(cells) // 32 * 32
    w = np.sort(code[:n].reshape(-1, 32, 7), axis=1)
    distinct = 1 + (np.diff(w, axis=1) != 0).sum(1)
    return distinct.sum() * 3 / n


def yaw_bin(M, nb):
    psi = np.arctan2(np.float32(M[1, 0]), np.float32(M[0, 0]))
    return int(np.rint(psi * nb / (2 * np.pi))) % nb


def rz(psi):
    c, s = np.cos(psi), np.sin(psi)
    return np.array([[c, -s, 0], [s, c, 0], [0, 0, 1]])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--poses", type=int, default=16, help="hypotheses sampled from the bench's 4096-pose grid")
    ap.add_argument("--bins", type=int, nargs="+", default=[16, 32, 64])
    ap.add_argument("--seed", type=int, default=1)
    ap.add_argument("--random-yaw", action="store_true", help="replace each sampled pose's yaw by a uniform random one")
    a = ap.parse_args()
    from pointcloud_slam_b200 import synth
    p_true = np.array([3.0, -2.0, 1.2, 0.0, 0.0, 0.6])      # synth.config2's scan without its 10M-point map
    T = synth.pose_vec_to_matrix(p_true)
    world = synth.make_world(synth.SEED)
    dirs = synth.livox_dirs(25000, synth.SEED)
    scan = synth.raycast(T[:3, 3], T[:3, :3], dirs, world, seed=synth.SEED)[:20000].astype(np.float32)
    scan = scan[np.argsort(morton(scan), kind="stable")]    # d_src
    poses = synth.hypothesis_grid(p_true, 32, 32, 4, 1.0)
    rng = np.random.default_rng(a.seed)
    rows = {"sensor": []} | {f"bins={nb}": [] for nb in a.bins} | {"per-pose": []}
    for h in rng.choice(len(poses), a.poses, replace=False):
        M = poses[h].reshape(4, 4).T.astype(np.float64)
        if a.random_yaw:
            M[:3, :3] = rz(rng.uniform(-np.pi, np.pi)).astype(np.float32)
        x = scan @ M[:3, :3].T + M[:3, 3]
        cells = np.floor(x).astype(np.int64)
        rows["sensor"].append(lines_per_point(cells))
        for nb in a.bins:
            o = np.argsort(morton(scan @ rz(2 * np.pi * yaw_bin(M, nb) / nb).T), kind="stable")
            rows[f"bins={nb}"].append(lines_per_point(cells[o]))
        rows["per-pose"].append(lines_per_point(cells[np.argsort(morton(x), kind="stable")]))
    base = np.mean(rows["sensor"])
    print(f"{'point order':<12} {'lines/point':>11} {'vs sensor':>9}")
    for k, v in rows.items():
        print(f"{k:<12} {np.mean(v):>11.2f} {np.mean(v) / base - 1:>+9.1%}")


if __name__ == "__main__":
    main()
