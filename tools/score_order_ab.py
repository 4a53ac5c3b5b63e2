"""A/B timing of the relocalization headline (configs[3]: 4096 hypotheses against the 10M-point prior map) for two or more
builds of libb200reg.so, alternated round by round in ONE process on one GPU, so clocks, temperature and neighbours are
shared by every build.

    python tools/score_order_ab.py --lib parent=build/parent/libb200reg.so --lib this=pointcloud-slam_b200/libb200reg.so

Each build gets its own engine (same map, same scan, same poses).  A round runs `--steps` timed steps per build, each step
preceded by an untimed L2 flush, as bench.py does.  Printed per round and build: mean step ms (device time of the
relocalize call, what bench.py's value is made of) and mean k_ndt_score_batch ms.  At the end: medians over rounds, the
speed-up of every build against the first, card name and power limit read in the same run, and the largest relative
score difference between builds over all 4096 hypotheses.

Per-source cost (`--fresh` scans per build): a new scan (the bench scan jittered by 1 cm, so every source is new) is set
with setInputSource, then relocalized twice; reported are the wall ms of setInputSource, of the first relocalize (which
builds the orderings that batch needs) and of the second (which completes them), and the first call's device ms.

`--random-yaw` also times the 4096 grid poses with uniformly random yaws (same rounds / steps), so the measured gain is
not tied to the bench's four yaws.
"""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card_info(dev):
    try:
        out = subprocess.run(["nvidia-smi", f"--id={dev}", "--query-gpu=name,power.limit,power.max_limit,clocks.max.sm",
                              "--format=csv,noheader"], capture_output=True, text=True, timeout=20).stdout.strip()
        name, pl, pmax, smax = [x.strip() for x in out.split(",")]
        return {"name": name, "power_limit": pl, "power_max_limit": pmax, "sm_clock_max": smax}
    except Exception as e:  # noqa: BLE001 - informational only
        return {"error": repr(e)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--lib", action="append", required=True, metavar="LABEL=PATH", help="a build to time (first = baseline)")
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--device", type=int, default=0)
    ap.add_argument("--json", metavar="FILE", help="also write the result as JSON")
    ap.add_argument("--fresh", type=int, default=5, help="fresh scans per build for the per-source cost")
    ap.add_argument("--random-yaw", action="store_true")
    a = ap.parse_args()
    from pointcloud_slam_b200 import api, synth

    builds = []
    for spec in a.lib:
        label, path = spec.split("=", 1)
        os.environ["B200REG_LIB"] = os.path.abspath(path)
        api._LIB = None
        builds.append({"label": label, "path": path, "lib": api.lib()})
    os.environ.pop("B200REG_LIB", None)

    cfg = synth.config2()
    poses = synth.hypothesis_grid(cfg["p_true"], 32, 32, 4, 1.0)
    for b in builds:
        api._LIB = b["lib"]
        g = api.NormalDistributionsTransform(device=a.device)
        g.setTransformationEpsilon(0.01)
        g.setInputTarget(cfg["map"])
        g._handle()
        g.setInputSource(cfg["scan"])
        b["engine"] = g
        b["scores"] = g.calculateScore(poses)
        for _ in range(a.warmup):
            api.flush_l2(a.device)
            api.relocalize(g, poses)
        b["rounds"] = []

    info = card_info(a.device)
    print(json.dumps({"card": info}), flush=True)
    for r in range(a.rounds):
        row = {"round": r}
        for b in builds:
            api._LIB = b["lib"]
            g = b["engine"]
            for _ in range(2):
                api.flush_l2(a.device)
                api.relocalize(g, poses)
            dev, kern = [], []
            for _ in range(a.steps):
                api.flush_l2(a.device)
                best, score, ms = api.relocalize(g, poses)
                dev.append(ms)
                kern.append(g.last_score_kernel_ms())
            b["rounds"].append((statistics.mean(dev), statistics.mean(kern)))
            b["best"], b["best_score"] = best, score
            row[b["label"]] = {"step_ms": round(statistics.mean(dev), 4), "kernel_ms": round(statistics.mean(kern), 4)}
        print(json.dumps(row), flush=True)

    rng = np.random.default_rng(5)
    for b in builds:   # per-source cost: setInputSource + first / second relocalize of a scan the engine has not seen
        api._LIB = b["lib"]
        g = b["engine"]
        rows = []
        for t in range(a.fresh):
            scan = np.ascontiguousarray(cfg["scan"] + rng.normal(0, 0.01, cfg["scan"].shape).astype(np.float32))
            api.flush_l2(a.device)
            t0 = time.perf_counter()
            g.setInputSource(scan)
            t1 = time.perf_counter()
            _, _, ms1 = api.relocalize(g, poses)
            t2 = time.perf_counter()
            api.relocalize(g, poses)
            t3 = time.perf_counter()
            rows.append(((t1 - t0) * 1e3, (t2 - t1) * 1e3, ms1, (t3 - t2) * 1e3))
        b["fresh"] = {k: statistics.median(r[i] for r in rows) for i, k in
                      enumerate(("set_source_wall_ms", "first_relocalize_wall_ms", "first_relocalize_device_ms", "second_relocalize_wall_ms"))}
        b["fresh"]["set_source_plus_first_relocalize_wall_ms"] = statistics.median(r[0] + r[1] for r in rows)
        g.setInputSource(cfg["scan"])
        print(json.dumps({"fresh": b["label"], **b["fresh"]}), flush=True)
    if a.random_yaw:
        ryaw = poses.copy()
        for i in range(len(ryaw)):
            M = ryaw[i].reshape(4, 4).T.astype(np.float64)
            psi = rng.uniform(-np.pi, np.pi)
            c, s_ = np.cos(psi), np.sin(psi)
            M[:3, :3] = np.array([[c, -s_, 0], [s_, c, 0], [0, 0, 1]])
            ryaw[i] = M.astype(np.float32).T.reshape(16)
        for b in builds:
            b["ryaw"] = []
        for r in range(a.rounds):
            for b in builds:
                api._LIB = b["lib"]
                g = b["engine"]
                for _ in range(2):
                    api.relocalize(g, ryaw)
                dev = []
                for _ in range(a.steps):
                    api.flush_l2(a.device)
                    dev.append(api.relocalize(g, ryaw)[2])
                b["ryaw"].append((statistics.mean(dev), g.last_score_kernel_ms()))
            print(json.dumps({"random_yaw_round": r, **{b["label"]: round(b["ryaw"][-1][0], 4) for b in builds}}), flush=True)

    base = builds[0]
    res = {"card": info, "rounds": a.rounds, "steps": a.steps, "hypotheses": len(poses), "builds": {}}
    for b in builds:
        step = statistics.median(x[0] for x in b["rounds"])
        kern = statistics.median(x[1] for x in b["rounds"])
        rel = np.abs(b["scores"] - base["scores"]) / np.maximum(np.abs(base["scores"]), 1e-300)
        res["builds"][b["label"]] = {
            "path": b["path"], "step_ms_median": step, "kernel_ms_median": kern,
            "step_ms_range": [min(x[0] for x in b["rounds"]), max(x[0] for x in b["rounds"])],
            "kernel_ms_range": [min(x[1] for x in b["rounds"]), max(x[1] for x in b["rounds"])],
            "hyp_per_s": len(poses) / (step * 1e-3), "speedup_vs_" + base["label"]: statistics.median(x[0] for x in base["rounds"]) / step,
            "fresh_source": b["fresh"], "best": int(b["best"]), "best_score": float(b["best_score"]),
            "max_rel_score_diff_vs_" + base["label"]: float(rel.max()),
        }
        if a.random_yaw:
            res["builds"][b["label"]]["random_yaw_step_ms_median"] = statistics.median(x[0] for x in b["ryaw"])
            res["builds"][b["label"]]["random_yaw_speedup_vs_" + base["label"]] = (
                statistics.median(x[0] for x in base["ryaw"]) / statistics.median(x[0] for x in b["ryaw"]))
    print(json.dumps(res, indent=1), flush=True)
    if a.json:
        with open(a.json, "w") as f:
            json.dump(res, f, indent=1)
    for b in builds:   # every engine is destroyed by the build that created it
        api._LIB = b["lib"]
        b.pop("engine").close()
    api._LIB = None


if __name__ == "__main__":
    main()
