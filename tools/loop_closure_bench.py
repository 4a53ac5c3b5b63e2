"""Loop-closure benchmark (b200_loop_close): prints ONE JSON line.

Workload: synth.loop_session with --keyframes keyframes of about --points points (a circle driven twice, drift 0.3 m and 1
degree per lap), --queries query keyframes spread over the second lap, historyKeyframeSearchRadius 15 m, time gap 30 s,
historyKeyframeSearchNum 25, ICP leaf 0.4 m, size gates 300 / 1000, NDT resolution 1.0 m, DIRECT7, transformation epsilon
0.01, identity guesses.

  device    b200_loop_close with detection on the device: device time of the call (CUDA events), host wall time of the call
            and pairs/s of the registered queries.  Host synchronisations per call: one read-back of the partners, then per
            chunk the min / max and run-count read-backs of the submap downsample and those of b200_ndt_pairs_align (its
            target min / max, the done polls of the alignment loop, the final copy); "chunks" is their number.
  baseline  the best a caller can do without the store: numpy detection and assembly (fp32 transformPointCloud of every
            keyframe of every submap, concatenated), b200_voxel_downsample per submap and per source, the size gates, then one
            b200_ndt_pairs_align of the survivors: host wall time of all of it, and each part.
  parity    the registered queries' records are byte-equal between the two (gpu_ms zeroed).
  gpu       name and power limit, read in the same run.
The tool writes nothing into the tree.
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True, timeout=60).stdout
        name, power = out.strip().splitlines()[0].split(", ")
        return dict(name=name, power_limit=power)
    except Exception as e:  # noqa: BLE001
        return dict(error=str(e))


def pcl_matrix_f32(p6):
    f = np.float32
    cs = lambda a: (f(np.cos(np.float64(a))), f(np.sin(np.float64(a))))
    (A, B), (C, D), (E, F) = cs(p6[5]), cs(p6[4]), cs(p6[3])
    DE, DF = D * E, D * F
    return np.array([[A * C, A * DF - B * E, B * F + A * DE, f(p6[0])], [B * C, A * E + B * DF, B * DE - A * F, f(p6[1])],
                     [-D, C * F, C * E, f(p6[2])]], np.float32)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--keyframes", type=int, default=4000)
    ap.add_argument("--points", type=int, default=8000)
    ap.add_argument("--queries", type=int, default=512)
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    from pointcloud_slam_b200 import api, synth
    loop = dict(search_radius=15.0, time_gap=30.0, search_num=25, leaf=0.4, min_source_points=300, min_target_points=1000)
    ndt = dict(resolution=1.0, search=7, trans_eps=0.01)
    t0 = time.perf_counter()
    s = synth.loop_session(K=args.keyframes, n_points=args.points, laps=2, workers=min(32, os.cpu_count() or 1))
    gen_s = time.perf_counter() - t0
    K = args.keyframes
    cur = np.unique(np.linspace(K // 2 + 40, K - 1, args.queries).astype(np.int64))
    Q = len(cur)
    out = dict(workload=dict(keyframes=K, points=args.points, queries=Q, **loop, resolution=1.0, search="DIRECT7", trans_eps=0.01,
                             synth_s=round(gen_s, 1)), gpu=gpu_info())
    t0 = time.perf_counter()
    st = api.KeyframeStore()
    for k, c in enumerate(s["clouds"]):
        st.add(c, s["poses"][k], s["times"][k])
    out["store_add_s"] = round(time.perf_counter() - t0, 3)
    b = api.NdtPairBatch(**ndt)
    b.close_loops(st, cur, **loop)   # warm-up: grows every buffer, loads the modules
    walls, devs = [], []
    for _ in range(args.reps):
        t = time.perf_counter()
        r = b.close_loops(st, cur, **loop)
        walls.append(time.perf_counter() - t)
        devs.append(r["gpu_ms"] / 1e3)
    reg = np.flatnonzero(r["status"] != 1)
    out["device"] = dict(wall_ms=1e3 * min(walls), device_ms=1e3 * min(devs), registered=int(len(reg)), with_partner=int((r["pre"] >= 0).sum()),
                         pairs_per_s_wall=len(reg) / min(walls), pairs_per_s_device=len(reg) / min(devs),
                         statuses={str(k): int(v) for k, v in zip(*np.unique(r["status"], return_counts=True))})
    # baseline: numpy detection and assembly, one downsample per cloud, one pair call
    vg = api.VoxelGrid()
    vg.setLeafSize(loop["leaf"])
    pb = api.NdtPairBatch(**ndt)
    mats = [pcl_matrix_f32(p) for p in s["poses"]]

    def assemble(key, num):
        parts = []
        for k in range(max(0, key - num), min(K - 1, key + num) + 1):
            T, p = mats[k], s["clouds"][k]
            xyz = [((T[i, 0] * p[:, 0] + T[i, 1] * p[:, 1]) + T[i, 2] * p[:, 2]) + T[i, 3] for i in range(3)]
            parts.append(np.stack(xyz + [p[:, 3]], 1))
        return np.concatenate(parts, 0)

    def baseline():
        tm = {}
        t = time.perf_counter()
        P = s["poses"]
        r2 = np.float32(np.float64(loop["search_radius"]) ** 2)
        pre = np.full(Q, -1, np.int64)
        for i, c in enumerate(cur):
            d = P[c, :3][None, :] - P[:c, :3]
            d2 = (d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1]) + d[:, 2] * d[:, 2]
            ok = np.flatnonzero((d2 < r2) & (np.abs(s["times"][:c] - s["times"][c]) > loop["time_gap"]))
            if len(ok):
                pre[i] = ok[np.argmin(d2[ok])]
        tm["detect_ms"] = 1e3 * (time.perf_counter() - t)
        t = time.perf_counter()
        raws = [(assemble(int(pre[i]), loop["search_num"]), assemble(int(cur[i]), 0)) if pre[i] >= 0 else None for i in range(Q)]
        tm["assemble_ms"] = 1e3 * (time.perf_counter() - t)
        t = time.perf_counter()
        srcs, tgts, ids = [], [], []
        for i, rw in enumerate(raws):
            if rw is None:
                continue
            vg.setInputCloud(rw[0]); tg, _ = vg.filter()
            vg.setInputCloud(rw[1]); sc, _ = vg.filter()
            if len(sc) >= loop["min_source_points"] and len(tg) >= loop["min_target_points"]:
                srcs.append(sc[:, :3]); tgts.append(tg[:, :3]); ids.append(i)
        tm["downsample_ms"] = 1e3 * (time.perf_counter() - t)
        t = time.perf_counter()
        rp = pb.align(srcs, tgts)
        tm["align_ms"] = 1e3 * (time.perf_counter() - t)
        return pre, ids, rp, tm

    baseline()   # warm-up
    best = None
    for _ in range(args.reps):
        t = time.perf_counter()
        pre, ids, rp, tm = baseline()
        w = time.perf_counter() - t
        if best is None or w < best[0]:
            best = (w, tm)
    out["baseline"] = dict(wall_ms=1e3 * best[0], registered=len(ids), pairs_per_s_wall=len(ids) / best[0],
                           **{k: round(v, 2) for k, v in best[1].items()})
    out["speedup_wall"] = best[0] / min(walls)

    def rb(x):
        y = type(x).from_buffer_copy(x)
        y.ndt.gpu_ms = 0.0
        return bytes(memoryview(y).cast("B"))
    out["parity"] = dict(same_partners=bool((pre == r["pre"]).all()), same_registered=ids == reg.tolist(),
                         records_identical=bool(ids == reg.tolist() and all(rb(r["loop_records"][i].reg) == rb(rp["records"][k]) for k, i in enumerate(ids))))
    print(json.dumps(out))


if __name__ == "__main__":
    main()
