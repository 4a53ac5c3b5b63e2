"""LOAM local-map benchmark (b200_loam_set_map_from_keyframes): prints ONE JSON line.

Workload: synth.loop_session with --keyframes keyframes of about --points points each, the first fifth of every cloud taken as
its corner cloud and the rest as its surf cloud.  The session drives the 18 m circle of the synthetic warehouse enough times
that consecutive keyframes are about 1 m apart (the raycast scene ends beyond the warehouse, so the trajectory stays in it),
which makes the revisits fill the search radius.  LIO-SAM's defaults: surroundingKeyframeSearchRadius 50 m,
surroundingKeyframeDensity 2 m, corner leaf 0.2 m, surf leaf 0.4 m; time_cur = time of keyframe cur + 0.1 s.  For every cur
of a sweep over the session:

  device    ScanToMap.extractSurroundingKeyFrames: device time (CUDA events, selection to the last insert) and host wall time.
  baseline  the best a caller can do without the store: numpy selection (radius search, (d2, j) sort, key-pose VoxelGrid with
            b200_voxel_downsample, brute-force nearest keyframe, the 10 s walk, the gate) and numpy fp32 assembly, then
            b200_voxel_downsample per map, then b200_loam_set_map: host wall time of all of it, and each part.
  parity    both sides' downsampled maps are byte-equal (the device's through the b200_keyframes_surrounding_map probe).
  gpu       name and power limit, read in the same run.
The tool writes nothing into the tree.
"""
import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import numpy as np  # noqa: E402

from loop_closure_bench import gpu_info, pcl_matrix_f32  # noqa: E402

F = np.float32


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--keyframes", type=int, default=2000)
    ap.add_argument("--points", type=int, default=8000)
    ap.add_argument("--sweep", type=int, default=8)
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    from pointcloud_slam_b200 import api, synth
    prm = dict(search_radius=50.0, density=2.0, corner_leaf=0.2, surf_leaf=0.4)
    K = args.keyframes
    laps = max(2, round(K / (2 * np.pi * 18.0)))
    t0 = time.perf_counter()
    s = synth.loop_session(K=K, n_points=args.points, laps=laps, workers=min(32, os.cpu_count() or 1))
    clouds = [np.asarray(c, F) for c in s["clouds"]]
    ncor = [len(c) // 5 for c in clouds]
    P, times = s["poses"], s["times"]
    out = dict(workload=dict(keyframes=K, points=args.points, laps=laps, spacing_m=round(2 * np.pi * 18.0 * laps / K, 3), **prm,
                             synth_s=round(time.perf_counter() - t0, 1)), gpu=gpu_info())
    st = api.KeyframeStore()
    for k, c in enumerate(clouds):
        st.add_features(c[: ncor[k]], c[ncor[k]:], P[k], times[k])
    dev = api.ScanToMap(max_map_points=4_000_000)
    host = api.ScanToMap(max_map_points=4_000_000)
    vg = api.VoxelGrid()
    mats = [pcl_matrix_f32(p) for p in P]
    pos = np.ascontiguousarray(P[:, :3], F)

    def sqd(a, b):
        d = (a - b).astype(F)
        return (d[..., 0] * d[..., 0] + d[..., 1] * d[..., 1]) + d[..., 2] * d[..., 2]

    def baseline(cur, tc):
        tm = {}
        t = time.perf_counter()
        q = pos[cur]
        d2 = sqd(pos[: cur + 1], q[None, :])
        hits = np.flatnonzero(d2 < F(np.float64(prm["search_radius"]) ** 2))
        hits = hits[np.lexsort((hits, d2[hits]))]
        vg.setLeafSize(prm["density"])
        vg.setInputCloud(np.concatenate([pos[hits], np.zeros((len(hits), 1), F)], 1))
        cent, _ = vg.filter()
        ent = [(int(np.argmin(sqd(pos[: cur + 1], c[None, :3]))), c[:3]) for c in cent]
        for j in range(cur, -1, -1):
            if not (tc - times[j] < 10.0):
                break
            ent.append((j, pos[j]))
        keys = [k for k, p in ent if not (np.sqrt(sqd(p, q)) > F(prm["search_radius"]))]
        tm["select_ms"] = 1e3 * (time.perf_counter() - t)
        t = time.perf_counter()
        cs, ss = [], []
        for k in keys:
            T, c = mats[k], clouds[k]
            xyz = [((T[i, 0] * c[:, 0] + T[i, 1] * c[:, 1]) + T[i, 2] * c[:, 2]) + T[i, 3] for i in range(3)]
            m = np.stack(xyz + [c[:, 3]], 1)
            cs.append(m[: ncor[k]]); ss.append(m[ncor[k]:])
        raw_c, raw_s = np.concatenate(cs, 0), np.concatenate(ss, 0)
        tm["assemble_ms"] = 1e3 * (time.perf_counter() - t)
        t = time.perf_counter()
        vg.setLeafSize(prm["corner_leaf"]); vg.setInputCloud(raw_c); dc, _ = vg.filter()
        vg.setLeafSize(prm["surf_leaf"]); vg.setInputCloud(raw_s); ds, _ = vg.filter()
        tm["downsample_ms"] = 1e3 * (time.perf_counter() - t)
        t = time.perf_counter()
        host.setInputCloud(dc[:, :3], ds[:, :3])
        tm["set_map_ms"] = 1e3 * (time.perf_counter() - t)
        return dc, ds, len(raw_c), len(raw_s), tm

    curs = np.unique(np.linspace(K // 4, K - 1, args.sweep).astype(np.int64))
    rows, parity = [], True
    for cur in curs:
        tc = float(times[cur]) + 0.1
        dev.extractSurroundingKeyFrames(st, int(cur), tc, **prm)   # warm-up: grows the buffers, loads the modules
        walls, devs = [], []
        for _ in range(args.reps):
            t = time.perf_counter()
            info = dev.extractSurroundingKeyFrames(st, int(cur), tc, **prm)
            walls.append(time.perf_counter() - t)
            devs.append(info.gpu_ms)
        baseline(int(cur), tc)
        best = None
        for _ in range(args.reps):
            t = time.perf_counter()
            dc, ds, nrc, nrs, tm = baseline(int(cur), tc)
            w = time.perf_counter() - t
            if best is None or w < best[0]:
                best = (w, tm)
        gc, gs = st.surrounding_map(int(cur), tc, **prm)
        same = gc.tobytes() == np.ascontiguousarray(dc, F).tobytes() and gs.tobytes() == np.ascontiguousarray(ds, F).tobytes()
        parity &= same
        rows.append(dict(cur=int(cur), n_list=info.n_list, n_kept=info.n_kept, raw=[info.n_corner_raw, info.n_surf_raw], ds=[info.n_corner, info.n_surf],
                         device_ms=round(min(devs), 3), device_wall_ms=round(1e3 * min(walls), 3), host_wall_ms=round(1e3 * best[0], 3),
                         **{k: round(v, 2) for k, v in best[1].items()}, speedup_wall=round(best[0] / min(walls), 2), maps_equal=same))
    out["sweep"] = rows
    out["parity"] = dict(maps_identical=bool(parity))
    print(json.dumps(out))


if __name__ == "__main__":
    main()
