"""Measures the LOAM front end on the device (b200_features_extract) against its host baseline.

Prints one JSON line:
  gpu       name and power limit, read in the same run;
  extract   per image size (16x1800, 32x1800, 64x1800, 128x2048; synth.spinning_scan of the warehouse world): device time
            (events) and wall time of b200_features_extract, median over --reps calls after --warmup, and the oracle
            (oracle/feature_oracle.cpp, one thread, as the single-threaded LIO-SAM nodes run it) on the same scan;
  chain     raw scan -> b200_features_extract -> b200_loam_optimize_device -> b200_keyframes_add_features_device against
            oracle features -> b200_loam_optimize -> b200_keyframes_add_features, each end to end (wall, median), with the
            parity of the two chains (DS clouds and t6 bits).
The tool writes nothing into the tree.
"""
import argparse
import json
import os
import subprocess
import sys
import time

os.environ.setdefault("OMP_NUM_THREADS", "1")
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

from oracle import feature_binding as fb  # noqa: E402
from pointcloud_slam_b200 import api, synth  # noqa: E402

SIZES = ((16, 1800), (32, 1800), (64, 1800), (128, 2048))


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True, check=True)
    name, power = out.stdout.strip().splitlines()[0].split(", ")
    return {"name": name, "power_limit": power}


def scan(n_scan, horizon, seed=0):
    xyz, ring, inten = synth.spinning_scan(n_scan, horizon, seed=seed, dup=0.02)
    rec, stride, io, ro, rb = fb.records(xyz, inten, ring)
    return rec, stride, io, ro, rb, fb.FeatureParams(n_scan=n_scan, horizon_scan=horizon)


def median_ms(fn, reps, warmup):
    for _ in range(warmup):
        fn()
    t = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        t.append((time.perf_counter() - t0) * 1e3)
    return float(np.median(t)), t


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--oracle-reps", type=int, default=5)
    a = ap.parse_args()
    fb.build()
    res = {"tool": "loam_features_bench", "gpu": gpu_info(), "extract": [], "chain": []}
    for n_scan, horizon in SIZES:
        rec, stride, io, ro, rb, prm = scan(n_scan, horizon)
        fx = api.FeatureExtraction(**prm.__dict__)
        dev = []

        def run():
            fx.extract(rec, stride, io, ro, rb)
            dev.append(fx.info.gpu_ms)

        wall, _ = median_ms(run, a.reps, a.warmup)
        orc, _ = median_ms(lambda: fb.features(rec, stride, io, ro, rb, prm), a.oracle_reps, 1)
        want = fb.features(rec, stride, io, ro, rb, prm)
        same = all(fx.cloud(w).tobytes() == want[k].tobytes() for w, k in ((0, "corner"), (1, "surface"), (2, "corner_ds"), (3, "surf_ds")))
        res["extract"].append({"n_scan": n_scan, "horizon": horizon, "points": len(rec), "extracted": int(fx.info.n_extracted),
                               "corner_ds": int(fx.info.n_corner_ds), "surf_ds": int(fx.info.n_surf_ds),
                               "device_ms": float(np.median(dev[a.warmup:])), "wall_ms": wall, "oracle_1t_ms": orc, "parity": bool(same)})
        # the chains, with a map made of this scan's own DS clouds
        cds, sds = fx.cloud(2), fx.cloud(3)
        s2m = api.ScanToMap(max_map_points=1_000_000)
        s2m.setInputCloud(cds[:, :3], sds[:, :3])
        t0 = np.array([0.005, -0.004, 0.01, 0.05, -0.03, 0.02], np.float32)
        pose = np.zeros(6, np.float32)
        st_d, st_h = api.KeyframeStore(), api.KeyframeStore()
        out = {}

        def dev_chain():
            fx.extract(rec, stride, io, ro, rb)
            t, _ = s2m.scan2MapOptimization_device(fx.device_cloud(2), fx.device_cloud(3), t0, 30)
            st_d.add_features_device(fx.device_cloud(2), fx.device_cloud(3), pose, 0.0)
            out["dev"] = t

        def host_chain():
            f = fb.features(rec, stride, io, ro, rb, prm)
            t, _ = s2m.scan2MapOptimization(f["corner_ds"], f["surf_ds"], t0, 30)
            st_h.add_features(f["corner_ds"], f["surf_ds"], pose, 0.0)
            out["host"] = t

        wd, _ = median_ms(dev_chain, a.reps, a.warmup)
        wh, _ = median_ms(host_chain, a.oracle_reps, 1)
        res["chain"].append({"n_scan": n_scan, "horizon": horizon, "device_chain_ms": wd, "host_chain_ms": wh,
                             "parity_t6": out["dev"].tobytes() == out["host"].tobytes(), "parity_ds": bool(same)})
        for h in (fx, s2m, st_d, st_h):
            h.close()
    print(json.dumps(res))


if __name__ == "__main__":
    main()
