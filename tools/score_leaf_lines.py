"""CPU estimate of how many distinct 128-byte lines the leaf loads of k_ndt_score_batch<7> touch per source point, for
several layouts of the fp64 leaf data.  No GPU involved.

The kernel is bound by the L1 data pipe, and a warp-wide load costs about as many wavefronts as there are distinct lines
in it.  Proxy: the bench's map (synth.config2, 1 m leaves) and scan, the scan read in its 512-bin yaw ordering; for every
warp of 32 consecutive points, every DIRECT7 slot and every chunk load of the layout, count the distinct lines over the
lanes whose slot holds a leaf (>= 6 points), divided by the number of points.

    python tools/score_leaf_lines.py [--poses 16] [--seed 1]

Layouts (leaf ids are the engine's: occupied cells in raster order, x fastest):
  AoS 96 B            LeafD {mean[3], icov[9]}: three 32-byte chunks per leaf, leaf j at byte 96 j
  SoA 3 x 32 B        the same three chunks, each in its own array
  SoA 32 + 32 + 8 B   the score store: {mean, c00}, {s01, s02, c11, s12}, {c22} (symmetric form, off-diagonals summed)
  AoS 72 B            the symmetric record in one array (32 + 32 + 8 bytes at byte 72 j)
  SoA 32 + 32 + 8 B, 2x2x1 bricks   the score store with valid leaves renumbered brick by brick (not implemented)
"""
import argparse
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from score_order_lines import DIRECT7, morton, rz, yaw_bin  # noqa: E402


def count_lines(hit, line_of, chunks):
    """distinct lines per point over (warp, slot, chunk); hit[n, 7] = slot holds a leaf, line_of(chunk) -> line ids [n, 7]"""
    n = hit.shape[0]
    tot = 0
    for ch in chunks:
        L = np.sort(np.where(hit, line_of(ch), -1).reshape(-1, 32, 7), axis=1)
        distinct = (np.diff(L, axis=1) != 0) & (L[:, 1:] >= 0)
        tot += (distinct.sum(1) + (L[:, 0] >= 0)).sum()
    return tot / n


def brick_ids(u, valid, d):
    """valid leaves renumbered in 2 x 2 x 1-cell bricks (bricks in raster order), -1 elsewhere"""
    ux, uy, uz = u % d[0], (u // d[0]) % d[1], u // (d[0] * d[1])
    vk = np.flatnonzero(valid)
    brick = (ux[vk] // 2) + (uy[vk] // 2) * (d[0] // 2 + 1) + uz[vk] * (d[0] // 2 + 1) * (d[1] // 2 + 1)
    inner = (ux[vk] & 1) + 2 * (uy[vk] & 1)
    ids = np.full(len(u), -1)
    ids[vk[np.lexsort((inner, brick))]] = np.arange(len(vk))
    return ids


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--poses", type=int, default=16, help="hypotheses sampled from the bench's 4096-pose grid")
    ap.add_argument("--seed", type=int, default=1)
    ap.add_argument("--bins", type=int, default=512, help="yaw bins of the scan ordering")
    a = ap.parse_args()
    from pointcloud_slam_b200 import synth
    cfg = synth.config2()
    mp, scan = cfg["map"].astype(np.float32), cfg["scan"].astype(np.float32)
    cell = np.floor(mp.astype(np.float64)).astype(np.int64)
    mn = cell.min(0)
    cell -= mn
    d = cell.max(0) + 1
    lin = cell[:, 0] + cell[:, 1] * d[0] + cell[:, 2] * d[0] * d[1]
    u, cnt = np.unique(lin, return_counts=True)   # occupied cells in raster order: index = leaf id
    valid = cnt >= 6
    print(f"grid {d[0]} x {d[1]} x {d[2]} cells, {len(u)} leaves, {valid.sum()} with >= 6 points", flush=True)
    raster = np.arange(len(u))
    brick = brick_ids(u, valid, d)

    scan = scan[np.argsort(morton(scan), kind="stable")]   # d_src
    poses = synth.hypothesis_grid(cfg["p_true"], 32, 32, 4, 1.0)
    rng = np.random.default_rng(a.seed)
    rows = {}
    for h in rng.choice(len(poses), a.poses, replace=False):
        M = poses[h].reshape(4, 4).T.astype(np.float32)
        o = np.argsort(morton(scan @ rz(2 * np.pi * yaw_bin(M, a.bins) / a.bins).T), kind="stable")
        x = (scan[o] @ M[:3, :3].T + M[:3, 3]).astype(np.float32)
        c = np.floor(x.astype(np.float64)).astype(np.int64) - mn
        n = len(c) // 32 * 32
        nb = c[:n, None, :] + DIRECT7[None]
        inside = ((nb >= 0) & (nb < d)).all(-1)
        l2 = np.where(inside, nb[..., 0] + nb[..., 1] * d[0] + nb[..., 2] * d[0] * d[1], -1)
        k = np.clip(np.searchsorted(u, l2), 0, len(u) - 1)
        hit = inside & (u[k] == l2) & valid[k]
        r, b = raster[k], brick[k]
        for name, line_of, chunks in (
                ("AoS 96 B (LeafD)", lambda ch: (96 * r + 32 * ch) // 128, (0, 1, 2)),
                ("SoA 3 x 32 B", lambda ch: ch * 10**9 + r // 4, (0, 1, 2)),
                ("SoA 32 + 32 + 8 B (score store)", lambda ch: ch * 10**9 + (r // 4 if ch < 2 else r // 16), (0, 1, 2)),
                ("AoS 72 B", lambda ch: (72 * r + 32 * ch) // 128 if ch < 2 else (72 * r + 64) // 128, (0, 1, 2)),
                ("SoA 32 + 32 + 8 B, 2x2x1 bricks", lambda ch: ch * 10**9 + (b // 4 if ch < 2 else b // 16), (0, 1, 2))):
            rows.setdefault(name, []).append(count_lines(hit, line_of, chunks))
        rows.setdefault("(pairs per point)", []).append(hit.sum() / n)
    base = np.mean(rows["AoS 96 B (LeafD)"])
    print(f"{'leaf layout':<34} {'lines/point':>11} {'vs AoS 96 B':>11}")
    for name, v in rows.items():
        rel = "" if name.startswith("(") else f"{np.mean(v) / base - 1:+11.1%}"
        print(f"{name:<34} {np.mean(v):>11.2f} {rel:>11}")


if __name__ == "__main__":
    main()
