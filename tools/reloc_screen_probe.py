"""Relocalization screen probe on the bench workload (configs[3]: 4096 hypotheses against the 10M-point prior map):
survivor counts and interval widths on the bench grid and with random yaws, then a torch.profiler table of the kernels
of 20 relocalization steps (L2 flushed before each), and the set_target device time.

    python tools/reloc_screen_probe.py
"""
import json, sys, os
import numpy as np
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from pointcloud_slam_b200 import api, synth
import torch
from torch.profiler import profile, ProfilerActivity
cfg = synth.config2()
poses = synth.hypothesis_grid(cfg["p_true"], 32, 32, 4, 1.0)
g = api.NormalDistributionsTransform(device=0)
g.setTransformationEpsilon(0.01)
g.setInputTarget(cfg["map"])
print("set_target device ms", g.last_ms())
g.setInputSource(cfg["scan"])
lo, hi = g.screenScore(poses)
s = g.calculateScore(poses)
print(json.dumps({"survivors": int((hi >= lo.max()).sum()), "contained": bool(((lo <= s) & (s <= hi)).all()),
                  "max_rel_width": float(((hi - lo) / np.abs(s)).max()), "median_rel_width": float(np.median((hi - lo) / np.abs(s)))}))
rng = np.random.default_rng(5)
ryaw = poses.copy()
for i in range(len(ryaw)):
    M = ryaw[i].reshape(4, 4).T.astype(np.float64)
    psi = rng.uniform(-np.pi, np.pi); c, s_ = np.cos(psi), np.sin(psi)
    M[:3, :3] = np.array([[c, -s_, 0], [s_, c, 0], [0, 0, 1]])
    ryaw[i] = M.astype(np.float32).T.reshape(16)
lo2, hi2 = g.screenScore(ryaw)
print(json.dumps({"random_yaw_survivors": int((hi2 >= lo2.max()).sum())}))
for _ in range(5): api.relocalize(g, poses)
with profile(activities=[ProfilerActivity.CUDA]) as prof:
    for _ in range(20):
        api.flush_l2(0)
        api.relocalize(g, poses)
    torch.cuda.synchronize()
print(prof.key_averages().table(sort_by="cuda_time_total", row_limit=14))
for _ in range(3):   # set_target device time
    g.setInputTarget(cfg["map"]); print("set_target device ms", g.last_ms())
