#!/usr/bin/env python
"""bench.py — scan-to-map registration hot path on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Headline (every N, so that the driver's 1 -> 8 scaling is computed on ONE metric): BASELINE.json's sharded metric,
"reloc hypotheses/sec at 1/2/4/8 B200" = configs[3]: 4096 initial-pose hypotheses (32 x 32 xy grid at 1 m, 4 yaws) scored
with pclomp's calculateScore against a 10M-point prior map (1.0 m voxels, DIRECT7).  The map is replicated on every rank
(rank 0 uploads it once, ncclBroadcast over NVLink), hypothesis h lives on rank h mod N, every rank scores its slice and
ONE ncclAllGather of 16 bytes per rank carries the local winners (allreduce-argmin).  Strong scaling: 4096 hypotheses in
total at every N.  A step = one such batch.

value      hypotheses/s = 4096 / (device time per step, CUDA events on the engine's stream around score kernels + local
           argmin + collective, L2 flushed (untimed) and the ranks aligned by a device-side rendezvous before each step;
           mean over the K timed steps, MAX over ranks).
e2e        same metric through the C-ABI call (b200_reloc_argmin_strided) with the slice's poses in HOST memory: H2D of
           the poses + kernels + collective + D2H of the winners, wall clock per call, max over ranks.
roofline   dominant kernel k_ndt_score_batch: algorithmic bytes per launch (DESIGN.md 7) / its CUDA-event duration.
cpu_baseline / --impl reference
           the CPU oracle port of calculateScore (oracle/), all host threads, on a bounded sample of the 4096 hypotheses.
parity     argmin index and score equal to the single-GPU result over all 4096 hypotheses and to the oracle's on a sample.

Objects that ride on the same JSON line (the other workloads BASELINE.json's metric and configs name):
iekf       configs[0] ("registered points/sec and ms per IEKF update"): one jueying_lio point-to-plane IEKF update of a
           20k-point Mid-360-shaped scan against a 2M-point local map: device value, e2e through b200_iekf_update with
           host buffers, roofline of the k-NN gather (k_search), k_obs latency line, cpu_baseline, parity.  The single-scan
           update does not shard (SURVEY.md 8e): at N > 1 every rank runs a replica ("iekf_replicas", no collective).
ndt        configs[1] (N = 1): setInputTarget / computeDerivatives / align of the scan against the 10M-point map.
sequence   configs[2] (N = 1): sliding-map odometry over --seq-scans scans (default 1000 = full size), update +
           MapIncremental per scan, oracle parity over the first --seq-parity scans.
fullmap    configs[4]: construct_full_map over --fullmap-frames keyframes x 100k points (default 10000 = full size), keyframes
           cut into one block per rank, partial voxel sums exchanged over NCCL (strong scaling).
scan2map   jueying_slam's LOAM-style scan2MapOptimization for one scan (N = 1).
gicp       pclomp GICP align of a 20k-point scan against a 1M-point map (N = 1).
summary    the headline numbers of every leg once more, last on the line.

--dump-outputs DIR writes what the headline path returned to its caller in the last timed step, the global winner's index
and score, as DIR/reloc_best_index.npy and DIR/reloc_best_score.npy (float64).  The inputs are seeded, so two builds run
with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True   # the benchmark leaves the tree as it found it (it may be read-only)

PARAMS = {
    # jueying_lio/config/livox.yaml:19,41-48 and config/horizon.yaml:18,37-42
    "livox": dict(resolution=0.2, nearby=26, ext=False, stencil=27),
    "horizon": dict(resolution=0.5, nearby=18, ext=True, stencil=19),
}
N_MAP, N_SCAN = 2_000_000, 20_000
N_PRIOR, N_HYP = 10_000_000, 4096
NDT_KW = dict(resolution=1.0, step_size=0.1, outlier_ratio=0.55, trans_eps=0.01, max_iter=35, search=7)
L2_NOTE = "GPU arm: L2 flushed between timed steps (256 MiB streaming write, untimed); CPU arm: not applicable"


def headline_config():
    """The `config` object - identical in the GPU arm and in --impl reference."""
    return {"workload": "configs[3]: global relocalization - 4096 initial-pose hypotheses (32x32 xy grid at 1 m x 4 yaws) scored with "
                        "calculateScore against a 10M-point prior map (1.0 m voxels, DIRECT7), 20k-point scan; hypotheses sharded over "
                        "the ranks (h mod N), map replicated, NCCL argmin",
            "hypotheses": N_HYP, "n_map": N_PRIOR, "n_scan": N_SCAN, "resolution": NDT_KW["resolution"], "search": "DIRECT7", "l2": L2_NOTE}


def host_threads():
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


class ClockSampler(threading.Thread):
    """SM clock and throttle reasons DURING the timed region (NVML, 5 ms period; nvidia-smi as a fallback)."""

    def __init__(self, gpu_index):
        super().__init__(daemon=True)
        self.gpu = gpu_index
        self.stop_flag = threading.Event()
        self.sm, self.reasons, self.sm_max = [], set(), None

    def run(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByIndex(self.gpu)
            self.sm_max = float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM))
            bits = {"hw_slowdown": 0x8, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20, "sw_power_cap": 0x4}
            while not self.stop_flag.is_set():
                self.sm.append(float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                for name, b in bits.items():
                    if r & b:
                        self.reasons.add(name)
                self.stop_flag.wait(0.005)
            return
        except Exception:
            pass
        q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
            "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        while not self.stop_flag.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={q}", "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                c = [v.strip() for v in out.split(",")]
                self.sm.append(float(c[0]))
                self.sm_max = float(c[1])
                for i, nme in enumerate(names):
                    if c[2 + i].lower().startswith("active"):
                        self.reasons.add(nme)
            except Exception:
                pass
            self.stop_flag.wait(0.05)

    def summary(self):
        self.stop_flag.set()
        self.join(timeout=6)
        sm = sorted(self.sm)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": self.sm_max, "reasons": sorted(self.reasons),
                "samples": len(sm)}


def dist_env():
    return int(os.environ.get("RANK", 0)), int(os.environ.get("LOCAL_RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))


def measured_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_traffic(kernel):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of `kernel` from the committed ncu --set full capture
    (profiles/traffic.json, written by tools/ncu_traffic.py with the commit it was taken at); None when not captured."""
    path = os.path.join(ROOT, "profiles", "traffic.json")
    try:
        t = json.load(open(path))
        e = t["kernels"].get(kernel)
        return (int(e["dram_bytes_per_launch"]), f"profiles/traffic.json ({e.get('capture', '?')}, commit {t.get('commit', '?')})") if e else (None, None)
    except Exception:
        return None, None


def mean(v):
    return float(np.mean(v)) if len(v) else float("nan")


def dump_outputs(path, arrays):
    """Writes each array as <path>/<name>.npy in float64, so that two builds run with the same arguments (hence the same
    seeded inputs) can be compared output for output."""
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, f"{name}.npy"), np.atleast_1d(np.asarray(a, dtype=np.float64)))


# =============================================================================================== CPU oracle legs
def cpu_reloc_sample(o, poses, n_s):
    """calculateScore on every (4096 / n_s)-th hypothesis, one hypothesis per thread (all host threads)."""
    sel = np.arange(0, len(poses), max(1, len(poses) // n_s))[:n_s]
    t0 = time.perf_counter()
    sc = o.score_batch(poses[sel])
    return sel, sc, time.perf_counter() - t0


def cpu_oracle_iekf(data, prm, steps, warmup, budget_s=25.0):
    """The reference IEKF path's CPU port (oracle/), all host threads."""
    from oracle import binding as ob
    lio = ob.OracleLio(resolution=prm["resolution"], nearby=prm["nearby"], extrinsic_est_en=prm["ext"], num_threads=host_threads())
    t0 = time.perf_counter()
    lio.insert(data["map"])
    t_insert = time.perf_counter() - t0
    ms, out = [], None
    t_start = time.perf_counter()
    for k in range(warmup + steps):
        t0 = time.perf_counter()
        out = lio.update(data["scan"], data["x_prop"], data["P"])
        dt = (time.perf_counter() - t0) * 1e3
        if k >= warmup:
            ms.append(dt)
        if time.perf_counter() - t_start > budget_s and len(ms) >= 3:
            break
    return ms, t_insert, out


def ndt_cpu(cfg, want_align=True):
    """NDT legs on the CPU oracle (OpenMP derivatives as pclomp does; serial voxel build as the reference)."""
    from oracle import binding as ob
    o = ob.OracleNdt(**NDT_KW, num_threads=host_threads())
    t0 = time.perf_counter()
    o.set_target(cfg["map"])
    t_build = time.perf_counter() - t0
    o.set_source(cfg["scan"])
    out = dict(oracle=o, build_s=t_build)
    if want_align:
        t0 = time.perf_counter()
        for _ in range(3):
            s, g, H = o.derivatives(cfg["p_guess"])
        out["deriv_ms"] = (time.perf_counter() - t0) / 3 * 1e3
        t0 = time.perf_counter()
        out["align"] = o.align(cfg["guess"])
        out["align_ms"] = (time.perf_counter() - t0) * 1e3
        out["deriv"] = (s, g, H)
    return out


# =============================================================================================== headline: relocalization
def reloc_leg(args, rank, local_rank, world, api, synth, torch, comm, cfg):
    dist = torch.distributed if world > 1 else None
    g = api.NormalDistributionsTransform(device=local_rank)
    g.setTransformationEpsilon(NDT_KW["trans_eps"])
    build_wall, build_dev = [], []
    for k in range(3 if world == 1 else 1):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        if world > 1:
            g.setInputTargetReplicated(comm, cfg.get("map") if rank == 0 else None, N_PRIOR)
        else:
            g.setInputTarget(cfg["map"])
            g._handle()
        build_wall.append((time.perf_counter() - t0) * 1e3)
        build_dev.append(g.last_ms())
    pin_wall = []
    if world == 1:   # the same cloud in page-locked caller memory (b200_host_alloc): raw records cross PCIe, unpacked on the device
        pinned = api.PinnedCloud(N_PRIOR, 3)
        pinned.array[:] = cfg["map"]
        for k in range(3):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            g.setInputTarget(pinned.array)
            pin_wall.append((time.perf_counter() - t0) * 1e3)
        pinned.close()
    g.setInputSource(cfg["scan"])
    g._handle()
    poses = synth.hypothesis_grid(cfg["p_true"], 32, 32, 4, 1.0)
    assert len(poses) == N_HYP
    mine = np.ascontiguousarray(poses[rank::world])   # interleaved slices: neighbouring, similarly expensive hypotheses spread over the ranks
    steps, warmup = args.steps, max(args.warmup, 3)

    def step(aligned):
        api.flush_l2(local_rank)                      # untimed: evict the 126 MB L2
        if world > 1:
            if aligned:
                g.stream_barrier(comm)                # device-side rendezvous on the engine's stream, before its start event
            else:
                dist.barrier()
        t0 = time.perf_counter()
        best, score, ms = api.relocalize(g, mine, comm, h_begin=rank, h_stride=world)
        return best, score, ms, (time.perf_counter() - t0) * 1e3, g.last_score_kernel_ms()

    for _ in range(warmup):
        step(True)
    sampler = ClockSampler(local_rank)
    sampler.start()
    t_wait = time.perf_counter()
    while not sampler.sm and time.perf_counter() - t_wait < 3.0:   # NVML start-up must not eat the (short) timed region.  Rank-local
        time.sleep(0.002)                                          # wait only: a step is a collective, every rank must run the same number
    for _ in range(2):
        step(True)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    launches0 = api.kernel_launches()
    t_wall0 = time.perf_counter()
    dev, kern = [], []
    for _ in range(steps):
        best, score, ms, _, kms = step(True)
        dev.append(ms)
        kern.append(kms)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    wall_s = time.perf_counter() - t_wall0
    launches = api.kernel_launches() - launches0
    clocks = sampler.summary()
    wall = []
    for _ in range(steps):                            # e2e: host poses in, winners out, wall clock around the C-ABI call
        wall.append(step(False)[3])
    t = torch.tensor([mean(dev), mean(wall), mean(kern)], device="cuda", dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dev_ms, wall_ms, kern_ms = float(t[0]), float(t[1]), float(t[2])

    # roofline of the score kernel on this rank's launch: per hypothesis N*16 (scan point) + N*32 (one nbr7 record: the seven
    # DIRECT7 leaf slots of the point's cell + count) + 96 B per (point, occupied voxel) pair (fp64 mean + inverse covariance)
    pairs = g.score_pairs(mine)
    algo = len(mine) * (N_SCAN * 16 + N_SCAN * 32) + 96 * pairs
    peak, peak_src = measured_peak()
    traffic, traffic_src = ncu_traffic("k_ndt_score_batch")
    roofline = {"bound": "hbm", "kernel": "k_ndt_score_batch<7> (one launch per step and rank)", "achieved": algo / (kern_ms * 1e-3) / 1e9,
                "peak": peak, "unit": "GB/s", "frac": algo / (kern_ms * 1e-3) / 1e9 / peak, "peak_source": peak_src,
                "traffic": traffic, "traffic_source": traffic_src, "algorithmic_bytes": int(algo), "kernel_ms": kern_ms,
                "pairs_per_hypothesis": pairs / max(len(mine), 1), "hypotheses_per_launch": len(mine), "share_of_step": kern_ms / dev_ms,
                "note": "every hypothesis re-reads the same few MB of voxel Gaussians, so the algorithmic bytes are served by L1/L2, not "
                        "by DRAM (compare traffic): the kernel is bound by the L1 data pipe (96-byte fp64 leaf per pair) and fp64 exp, "
                        "which is why achieved can exceed the DRAM peak"}

    out = {"value": N_HYP / (dev_ms * 1e-3), "ms_per_step": dev_ms, "per_rank": len(mine),
           "e2e": {"value": N_HYP / (wall_ms * 1e-3), "unit": "hypotheses/s", "ms_per_step": wall_ms,
                   "h2d_bytes_per_step": int(mine.nbytes), "d2h_bytes_per_step": 16 * world},
           "gpu_launches": int(launches), "clocks": clocks, "roofline": roofline, "wall_s_timed_region_incl_flush": wall_s,
           "best": int(best), "best_score": float(score), "true_index": (16 * 32 + 16) * 4,
           "collective": "one ncclAllGather of 16 B per rank ((score key, index) winners), reduced identically on every rank" if world > 1 else "none (single GPU)",
           "set_target_ms": {"device": float(np.min(build_dev)), "e2e_wall": float(np.min(pin_wall)) if pin_wall else float(np.min(build_wall)),
                             "e2e_wall_pageable": float(np.min(build_wall)), "h2d_bytes": N_PRIOR * 12 if pin_wall else N_PRIOR * 16,
                             "input": "10M x 12-byte records in page-locked host memory (b200_host_alloc), unpacked on the device" if pin_wall else "pageable host cloud, packed through the pinned stage",
                             "voxels": int(g.numVoxels()),
                             "how": "rank 0 uploads, ncclBroadcast of the packed points, every rank builds identical leaves" if world > 1 else "host cloud -> device build"}}
    # parity: the sharded winner against the single-GPU result over all 4096 hypotheses (rank 0), and against the oracle on a sample
    if rank == 0:
        s_all = g.calculateScore(poses)
        b1 = int(np.argmax(s_all))
        out["parity"] = {"argmin_equal_single_gpu": bool(b1 == best), "score_equal_single_gpu": bool(s_all[b1] == score),
                         "winner_is_true_pose_cell": bool(best == out["true_index"])}
        if not args.no_cpu:
            c = ndt_cpu(cfg, want_align=False)
            n_s = 256 if world == 1 else 64
            sel, sc, t_sc = cpu_reloc_sample(c["oracle"], poses, n_s)
            if best not in sel:
                sel = np.concatenate([sel, [best]])
                sc = np.concatenate([sc, c["oracle"].score_batch(poses[[best]])])
            out["parity"].update({"oracle_sample": len(sel), "scores_rel_vs_oracle": float(np.abs(s_all[sel] - sc).max() / np.abs(sc).max()),
                                  "argmin_equal_oracle_on_sample": bool(int(sel[np.argmax(sc)]) == int(sel[np.argmax(s_all[sel])])),
                                  "oracle_argmin_on_sample": int(sel[np.argmax(sc)])})
            if world == 1:
                out["cpu_baseline"] = {"value": n_s / t_sc, "unit": "hypotheses/s", "cores": host_threads(), "kind": "port",
                                       "sample": f"{n_s} of the 4096 hypotheses (every {N_HYP // n_s}th), one hypothesis per thread, {t_sc:.2f} s; "
                                                 f"serial 10M-pt voxel build {c['build_s']:.1f} s not included"}
            out["_oracle_ndt"] = c
    return g, poses, out


# =============================================================================================== configs[1]: NDT align (N = 1)
def ndt_leg(args, local_rank, api, g, cfg, c):
    der_dev, der_wall = [], []
    for k in range(args.steps + 3):
        api.flush_l2(local_rank)
        t0 = time.perf_counter()
        s, gr, H = g.computeDerivatives(cfg["p_guess"])
        if k >= 3:
            der_wall.append((time.perf_counter() - t0) * 1e3)
            der_dev.append(g.last_ms())
    al_dev, al_wall = [], []
    for k in range(args.steps + 3):
        api.flush_l2(local_rank)
        t0 = time.perf_counter()
        g.align(cfg["guess"])
        if k >= 3:
            al_wall.append((time.perf_counter() - t0) * 1e3)
            al_dev.append(g.result.gpu_ms)
    r = g.result
    pairs = g.nbhd_total(cfg["p_guess"])
    peak, _ = measured_peak()
    # algorithmic bytes of one derivative evaluation: N*16 (source point) + N*7*4 (one 4-byte cell-table probe per neighbourhood
    # cell) + 64 B per (point, voxel) pair (float-path leaf record)
    der_bytes = N_SCAN * 16 + N_SCAN * 7 * 4 + 64 * pairs
    der_ms = mean(der_dev)
    traffic, traffic_src = ncu_traffic("k_ndt_eval")
    out = {"workload": "configs[1]: 20k-pt scan vs 10M-pt prior map, 1.0 m voxels, DIRECT7, eps 0.01, step 0.1",
           "derivatives_ms": {"device": der_ms, "e2e_wall": mean(der_wall), "pairs": int(pairs)},
           "align_ms": {"device": mean(al_dev), "e2e_wall": mean(al_wall), "iters": r.iters, "evals": r.evals,
                        "hess_evals": r.hess_evals, "launches": g.last_launches(), "converged": bool(r.converged),
                        "points_per_s": N_SCAN / (mean(al_dev) * 1e-3)},
           "roofline": {"bound": "hbm", "kernel": "k_ndt_eval (one init + one evaluation launch, CUDA events around both)",
                        "achieved": der_bytes / (der_ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                        "frac": der_bytes / (der_ms * 1e-3) / 1e9 / peak, "algorithmic_bytes": int(der_bytes),
                        "traffic": traffic, "traffic_source": traffic_src}}
    if c is not None:
        rc0, T0, r0 = c["align"]
        s0, g0, H0 = c["deriv"]
        out["cpu_baseline"] = {"kind": "port", "cores": host_threads(), "set_target_s": c["build_s"], "derivatives_ms": c["deriv_ms"],
                               "align_ms": c["align_ms"], "sample": "full size: 10M-pt voxel build (serial, as the reference), "
                               "3 derivative evaluations and 1 align on all threads"}
        out["parity"] = {"align_dpos_m": float(np.abs(np.array(r.p_final)[:3] - np.array(r0.p_final)[:3]).max()),
                         "align_drot_rad": float(np.abs(np.array(r.p_final)[3:] - np.array(r0.p_final)[3:]).max()),
                         "iters_equal": bool(r.iters == r0.iters and r.evals == r0.evals),
                         "score_rel": float(abs(s - s0) / abs(s0)),
                         "g_rel": float(np.abs(gr - g0).max() / np.abs(g0).max()),
                         "H_rel": float(np.abs(H - H0).max() / np.abs(H0).max())}
    return out


# =============================================================================================== configs[0]: IEKF update
def iekf_leg(args, rank, local_rank, world, api, synth, torch, full):
    """One IEKF update per step on configs[0].  full = all the trimmings (N = 1); otherwise the replica figure only."""
    prm = PARAMS[args.params]
    data = synth.config1(N_MAP, N_SCAN)
    scan = data["scan"]
    n = len(scan)
    ivox = api.IVox(resolution=prm["resolution"], nearby=prm["nearby"], device=local_rank)
    ivox.AddPoints(data["map"])
    kf = api.Esekf(ivox, extrinsic_est_en=prm["ext"])
    scan4 = np.zeros((n, 4), np.float32)
    scan4[:, :3] = scan
    d_scan = torch.from_numpy(scan4).cuda()
    torch.cuda.synchronize()
    steps = args.steps

    def step_device():
        kf.change_x(data["x_prop"])
        kf.change_P(data["P"])
        kf.update_device(d_scan.data_ptr(), n)
        return kf.stats.gpu_ms

    for _ in range(max(args.warmup, 3)):
        api.flush_l2(local_rank)
        step_device()
    launches0 = api.kernel_launches()
    dev_ms = []
    for _ in range(steps):
        api.flush_l2(local_rank)          # untimed: evict the 126 MB L2 between steps
        dev_ms.append(step_device())      # timed on the device: CUDA events on the engine's stream
    launches = api.kernel_launches() - launches0
    passes, knn_passes = kf.stats.passes, kf.stats.knn_passes
    n_eff = list(kf.stats.n_eff)[:passes]
    ms_step = mean(dev_ms)
    if world > 1:
        t = torch.tensor([ms_step], device="cuda", dtype=torch.float64)
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
        ms_step = float(t[0])
    out = {"workload": "configs[0]: 20k-pt Mid-360-shaped scan vs 2M-pt local map, one IEKF update per step",
           "metric": "registered points/sec (IEKF update)", "value": world * n / (ms_step * 1e-3), "unit": "points/s", "ms_per_update": ms_step,
           "params": args.params, "passes": passes, "knn_passes": knn_passes, "n_eff": n_eff, "gpu_launches": int(launches),
           "parallelism": f"{world} independent replicas, no collective" if world > 1 else "single GPU"}
    if not full:
        return out
    warm_ms = [step_device() for _ in range(steps)]   # warm-L2 variant (the map stays L2-resident between scans in real operation)
    out["ms_per_update_warm_l2"] = mean(warm_ms)
    # e2e: the C-ABI call with host buffers (H2D + kernels + D2H), wall clock per call.  Headline: the scan sits in page-locked
    # host memory (b200_host_alloc); second figure: a pageable buffer (what a PCL cloud is), packed through the handle's pinned stage
    pinned = api.PinnedCloud(n, 3)
    pinned.array[:] = scan
    e2e_ms, e2e_pageable_ms = [], []
    for src, dst in ((pinned.array, e2e_ms), (scan, e2e_pageable_ms)):
        for k in range(steps + 3):
            api.flush_l2(local_rank)
            kf.change_x(data["x_prop"])
            kf.change_P(data["P"])
            t0 = time.perf_counter()
            kf.update_iterated_dyn_share_modified(src)
            dt = (time.perf_counter() - t0) * 1e3
            if k >= 3:
                dst.append(dt)
    h2d, d2h = kf.io_bytes(n)
    h2d = h2d - n * 16 + n * 12   # the pinned path ships the caller's 12-byte records
    out["e2e"] = {"value": n / (mean(e2e_ms) * 1e-3), "unit": "points/s", "ms_per_update": mean(e2e_ms),
                  "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                  "input": "scan in page-locked host memory (b200_host_alloc), unpacked on the device",
                  "pageable_input_ms_per_update": mean(e2e_pageable_ms)}
    # per-kernel durations by CUDA events (profiling mode launches kernel by kernel)
    kf.set_profiling(True)
    search_ms, obs_s_ms, obs_n_ms, init_ms, prof_totals = [], [], [], [], []
    for k in range(steps + 2):
        api.flush_l2(local_rank)
        step_device()
        if k >= 2:
            t = kf.kernel_times_ms()
            prof_totals.append(sum(t[:1 + 2 * passes]))
            init_ms.append(t[0])
            for p in range(passes):
                if kf.stats.knn[p]:
                    search_ms.append(t[1 + 2 * p])
                    obs_s_ms.append(t[2 + 2 * p])
                else:
                    obs_n_ms.append(t[2 + 2 * p])
    kf.set_profiling(False)
    # roofline of the k-NN search kernel: algorithmic bytes per launch (SURVEY.md 8d / DESIGN.md):
    #   N*16 (scan point) + N*S*8 (one table probe per stencil cell) + 16*sum(C_i) (gathered map points) + N*20 (5 indices out)
    o_l, Rl = synth.lidar_pose(data["x_prop"])
    qw = (scan.astype(np.float64) @ Rl.T + o_l).astype(np.float32)
    sum_c, cells = ivox.stencil_points(qw)
    algo_bytes = n * 16 + n * prm["stencil"] * 8 + 16 * sum_c + n * 20
    peak, peak_src = measured_peak()
    k_ms = mean(search_ms)
    tot = mean(prof_totals)
    traffic, traffic_src = ncu_traffic("k_search")
    out["roofline"] = {"bound": "hbm", "kernel": "k_search (stencil k-NN gather)", "achieved": algo_bytes / (k_ms * 1e-3) / 1e9, "peak": peak,
                       "unit": "GB/s", "frac": algo_bytes / (k_ms * 1e-3) / 1e9 / peak, "peak_source": peak_src, "traffic": traffic,
                       "traffic_source": traffic_src, "algorithmic_bytes": int(algo_bytes), "kernel_ms": k_ms,
                       "candidates_per_query": sum_c / n, "occupied_cells_per_query": cells / n, "share_of_step": knn_passes * k_ms / tot}
    # the same search body with enough parallelism to leave the launch-latency regime: 50 scans' worth of queries in one call
    rng = np.random.default_rng(1)
    qbig = np.ascontiguousarray(np.concatenate([qw + rng.normal(0, 0.05, qw.shape).astype(np.float32) for _ in range(50)], 0))
    ivox.GetClosestPoint(qbig)
    big_ms = []
    for _ in range(5):
        api.flush_l2(local_rank)
        ivox.GetClosestPoint(qbig)
        big_ms.append(ivox.last_knn_ms())
    sum_cb, _ = ivox.stencil_points(qbig)
    nb_ = len(qbig)
    big_bytes = nb_ * 16 + nb_ * prm["stencil"] * 8 + 16 * sum_cb + nb_ * 20 + nb_ * 24   # + sqdist (20 B) and count (4 B) out
    out["roofline"]["batched"] = {"queries": nb_, "kernel": "k_knn5 (same search body, 1M queries per launch)", "kernel_ms": mean(big_ms),
                                  "algorithmic_bytes": int(big_bytes), "achieved": big_bytes / (mean(big_ms) * 1e-3) / 1e9,
                                  "frac": big_bytes / (mean(big_ms) * 1e-3) / 1e9 / peak, "queries_per_s": nb_ / (mean(big_ms) * 1e-3)}
    # k_obs: latency line + bytes (SURVEY 8d: N*41 B on a pass that reuses the planes, N*126 B on a search pass = + N*85 B hand-off)
    obs_ms = obs_s_ms + obs_n_ms
    obs_bytes_s, obs_bytes_n = n * 126, n * 41
    out["kernels"] = {
        "k_iekf_init_ms": mean(init_ms), "k_search_ms": k_ms, "k_obs_ms": mean(obs_ms),
        "per_update": f"1 init + {passes} x (k_search, k_obs); k_search is a no-op on non-search passes",
        "share_of_step": {"k_search": knn_passes * k_ms / tot, "k_obs": passes * mean(obs_ms) / tot},
        "k_obs": {"bound": "latency (serial fp64 filter chain + per-point QR), not bytes",
                  "search_pass": {"ms": mean(obs_s_ms), "algorithmic_bytes": obs_bytes_s,
                                  "achieved_gbs": obs_bytes_s / (mean(obs_s_ms) * 1e-3) / 1e9 if obs_s_ms else None,
                                  "frac": obs_bytes_s / (mean(obs_s_ms) * 1e-3) / 1e9 / peak if obs_s_ms else None},
                  "reuse_pass": {"ms": mean(obs_n_ms), "algorithmic_bytes": obs_bytes_n,
                                 "achieved_gbs": obs_bytes_n / (mean(obs_n_ms) * 1e-3) / 1e9 if obs_n_ms else None,
                                 "frac": obs_bytes_n / (mean(obs_n_ms) * 1e-3) / 1e9 / peak if obs_n_ms else None}},
        "note": "event-to-event per kernel with plain launches (each interval carries ~3-4 us of launch / event gap that the graph replay of the timed steps does not pay)"}
    if not args.no_cpu:
        ms, t_insert, res = cpu_oracle_iekf(data, prm, 20, 3, budget_s=25.0)
        cpu_ms = float(np.median(ms))
        out["cpu_baseline"] = {"value": n / (cpu_ms * 1e-3), "unit": "points/s", "cores": host_threads(), "kind": "port", "ms_per_update": cpu_ms,
                               "sample": f"{len(ms)} full-size updates on the same inputs (median); map insert {t_insert:.2f} s excluded"}
        rc, x_o, P_o, st_o = res
        step_device()
        from oracle import binding as ob
        d = ob.boxminus(kf.get_x(), x_o)
        out["parity"] = {"pos_m": float(np.abs(d[:3]).max()), "rot_rad": float(np.abs(d[3:6]).max()),
                         "passes_equal": bool(st_o.passes == kf.stats.passes),
                         "n_eff_equal": bool(list(st_o.n_eff)[:passes] == list(kf.stats.n_eff)[:passes])}
    kf.close()
    ivox.close()
    return out


# =============================================================================================== configs[2]: sliding-map sequence
def sequence_leg(args, local_rank, api, synth, n_scans, n_parity):
    """configs[2]: sliding-map odometry over a synthetic scan sequence.  The map starts from the first scan and grows by
    MapIncremental (downsample-on-insert); the prior of scan k is the posterior of scan k-1 moved by the true relative
    motion plus a seeded perturbation (stand-in for the IMU propagation)."""
    from concurrent.futures import ThreadPoolExecutor
    prm = PARAMS["horizon"]
    world = synth.make_world(synth.SEED)
    rng = np.random.default_rng(synth.SEED + 31)
    per_lap = 290

    def true_state(k):
        a = 2 * np.pi * k / per_lap
        pos = np.array([30.0 * np.cos(a), 15.0 * np.sin(a), 1.2])
        yaw = np.arctan2(15.0 * np.cos(a), -30.0 * np.sin(a))
        return synth.make_state(pos, [0.0, 0.0, yaw])

    def scan_of(k):
        o, Rl = synth.lidar_pose(true_state(k))
        return np.ascontiguousarray(synth.raycast(o, Rl, synth.livox_dirs(25_000, seed=synth.SEED + k), world, seed=synth.SEED + 7 * k)[:N_SCAN])

    def move(x_post, k):  # posterior of k-1 -> prior of k by the true relative motion + noise
        a, b = true_state(k - 1), true_state(k)
        Ra, Rp = synth.quat_to_R(a[3:7]), synth.quat_to_R(x_post[3:7])
        x = x_post.copy()
        x[0:3] = x_post[0:3] + Rp @ (Ra.T @ (b[0:3] - a[0:3])) + rng.uniform(-0.02, 0.02, 3)
        qa_inv = a[3:7] * np.array([-1, -1, -1, 1.0])
        dq = synth.quat_mul(qa_inv, b[3:7])
        q = synth.quat_mul(synth.quat_mul(x_post[3:7], dq), synth.quat_from_rotvec(np.deg2rad(rng.uniform(-0.2, 0.2, 3))))
        x[3:7] = q / np.linalg.norm(q)
        return x

    t_gen = time.perf_counter()
    with ThreadPoolExecutor(min(16, host_threads())) as ex:   # host-side ray casting of the whole sequence (synthetic data, untimed)
        scans = list(ex.map(scan_of, range(n_scans)))
    t_gen = time.perf_counter() - t_gen
    ivox = api.IVox(resolution=prm["resolution"], nearby=prm["nearby"], device=local_rank)
    kf = api.Esekf(ivox, extrinsic_est_en=False, filter_size_map=0.5)
    oracle_on = n_parity > 0 and not args.no_cpu
    if oracle_on:
        from oracle import binding as ob
        orc = ob.OracleLio(resolution=prm["resolution"], nearby=prm["nearby"], extrinsic_est_en=False, filter_size_map=0.5, num_threads=host_threads())
    P0 = synth.init_cov() * 0.01
    x_g = true_state(0)
    ol, Rl = synth.lidar_pose(x_g)
    w0 = (scans[0].astype(np.float64) @ Rl.T + ol).astype(np.float32)
    ivox.AddPoints(w0)                      # first frame: every point goes in (laser_mapping.cc:314-319)
    if oracle_on:
        orc.insert(w0)
    ms_update, ms_incr, ms_wall, voxels, points, par, passes, knn_passes, neff, add_par = [], [], [], [], [], [], [], [], [], []
    cpu_ms = []
    for k in range(1, n_scans):
        scan = scans[k]
        prior = move(x_g, k)
        kf.change_x(prior)
        kf.change_P(P0)
        t0 = time.perf_counter()
        kf.update_iterated_dyn_share_modified(scan)
        t1 = time.perf_counter()
        na, nd = kf.MapIncremental(kf.get_x(), True)
        t2 = time.perf_counter()
        x_g = kf.get_x().copy()
        ms_update.append(kf.stats.gpu_ms)
        passes.append(kf.stats.passes)
        knn_passes.append(kf.stats.knn_passes)
        neff.append(kf.stats.n_eff[max(kf.stats.passes - 1, 0)])
        ms_wall.append((t2 - t0) * 1e3)
        ms_incr.append((t2 - t1) * 1e3)
        if k % 100 == 0 or k == n_scans - 1:
            voxels.append(ivox.NumValidGrids())
            points.append(ivox.NumPoints())
        if oracle_on and k <= n_parity:      # the oracle is fed the same prior and grows its own map from its own posterior
            t0 = time.perf_counter()
            rco, x_o, P_o, st_o = orc.update(scan, prior, P0)
            _, na_o, nd_o = orc.map_incremental(scan, x_o, True)
            cpu_ms.append((time.perf_counter() - t0) * 1e3)
            d = ob.boxminus(x_g, x_o)
            par.append(float(np.abs(d[:6]).max()))
            add_par.append((na, nd) == (na_o, nd_o))
    xt = true_state(n_scans - 1)
    drift = float(np.linalg.norm(x_g[0:3] - xt[0:3]))
    out = {"workload": f"configs[2]: {n_scans}-scan closed-loop sequence (0.5 m / 1.2 deg steps), 20k-pt scans, P-horizon map "
                       "(0.5 m voxels, NEARBY18), update + MapIncremental (filter_size_map 0.5) per scan",
           "scans": n_scans, "ms_update_device": {"mean": mean(ms_update), "median": float(np.median(ms_update)), "p95": float(np.percentile(ms_update, 95))},
           "ms_per_scan_e2e": {"mean": mean(ms_wall), "p95": float(np.percentile(ms_wall, 95)), "map_incremental_mean": mean(ms_incr)},
           "scans_per_s_e2e": 1e3 / mean(ms_wall), "points_per_s_e2e": N_SCAN * 1e3 / mean(ms_wall),
           "passes_mean": mean(passes), "knn_passes_mean": mean(knn_passes), "n_eff_mean": mean(neff),
           "launch_modes": dict(zip(("graph_captures", "graph_replays", "plain"), kf.launch_modes())),
           "map_voxels": voxels, "map_points": points, "final_position_error_m": drift, "scan_generation_s_untimed": t_gen,
           "parity_vs_oracle": {"scans": len(par), "max_state_diff": max(par) if par else None, "map_incremental_counts_equal": bool(all(add_par)) if add_par else None,
                                "note": "both filters fed the same priors; each grows its own map from its own posterior"}}
    if cpu_ms:
        out["cpu_baseline"] = {"value": 1e3 / mean(cpu_ms), "unit": "scans/s", "ms_per_scan": mean(cpu_ms), "cores": host_threads(), "kind": "port",
                               "sample": f"the first {len(cpu_ms)} scans of the sequence (update on all threads + serial MapIncremental)"}
    if os.environ.get("B200_SEQ_TRACE"):
        out["trace_ms_update_device"] = [round(v, 4) for v in ms_update]
        out["trace_ms_map_incremental"] = [round(v, 4) for v in ms_incr]
    kf.close()
    ivox.close()
    return out


# =============================================================================================== configs[4]: construct_full_map
def fullmap_leg(args, rank, local_rank, world, api, synth, torch, comm):
    """configs[4]: construct_full_map - keyframes (Avia-shaped, 100k points) moved by their poses and merged into a 0.1 m
    voxel-grid map.  A pool of ray-cast keyframes along a loop in the synthetic hall is replayed on a grid of tiles
    (copies of the hall side by side), so the map keeps growing; the keyframe list is cut into contiguous blocks, one per
    rank; the total is fixed = strong scaling."""
    n_frames, n_pool, n_pts = args.fullmap_frames, args.fullmap_pool, 100_000
    world_geo = synth.make_world(synth.SEED, beams=True)
    pool, pool_pose = [], []
    for k in range(n_pool):
        a = 2 * np.pi * k / n_pool
        pos = np.array([30.0 * np.cos(a), 15.0 * np.sin(a), 1.2])
        q = synth.quat_from_rotvec([0.0, 0.0, a + np.pi / 2])
        pts = synth.raycast(pos, synth.quat_to_R(q), synth.avia_dirs(int(n_pts * 1.15), seed=900 + k), world_geo, seed=950 + k)[:n_pts]
        inten = np.full((len(pts), 1), float(k), np.float32)
        pool.append(np.ascontiguousarray(np.concatenate([pts, inten], 1)))
        pool_pose.append(np.array([pos[0], pos[1], pos[2], q[3], q[0], q[1], q[2]]))
    reuse = args.fullmap_reuse   # keyframes per tile = pool x reuse: ~20 points per voxel, the density BASELINE.json quotes (1e9 pts -> 50M)

    def pose_of(i):
        t = i // (n_pool * reuse)
        p = pool_pose[i % n_pool].copy()
        p[0] += (t % 16) * 125.0
        p[1] += (t // 16) * 85.0
        return p

    fb, fe = api.shard_range(n_frames, world, rank)
    frame_poses = np.stack([pose_of(i) for i in range(n_frames)])   # poses.txt of the job, read once
    d_pool = [torch.from_numpy(f).cuda() for f in pool]
    tiles = -(-n_frames // (n_pool * reuse))
    cap = int(min(1 << 29, max(4_000_000, 1.6e6 * (-(-tiles // world) + 2))))
    times, times_e2e, exch, vox_local = [], [], [], 0
    n_host = min(fe - fb, max(1, args.fullmap_host_frames // world))   # e2e (host buffers) on a bounded block of this rank's keyframes
    for rep in range(3):
        for mode in ("device", "host"):
            if mode == "host" and rep > 0:
                continue
            b = api.FullMapBuilder(leaf=0.1, capacity_voxels=cap, device=local_rank)
            torch.cuda.synchronize()
            if world > 1:
                torch.distributed.barrier()
            t0 = time.perf_counter()
            if mode == "device":   # batched entry point: keyframes are accumulated several per launch
                BATCH = 96
                for i0 in range(fb, fe, BATCH):
                    idx = range(i0, min(fe, i0 + BATCH))
                    b.add_keyframes_device([d_pool[i % n_pool].data_ptr() for i in idx], [len(pool[i % n_pool]) for i in idx],
                                           frame_poses[i0:idx[-1] + 1])
            else:
                for i in range(fb, fb + n_host):
                    b.add_keyframe(pool[i % n_pool], frame_poses[i])
            b.merge(comm)
            nv = b.num_voxels()
            dt = time.perf_counter() - t0
            (times if mode == "device" else times_e2e).append(dt)
            if mode == "device":
                exch.append(b.exchange_ms())
                vox_local = nv
            b.close()
    t = torch.tensor([min(times), min(times_e2e), float(vox_local)], device="cuda", dtype=torch.float64)
    if world > 1:
        tm = t.clone()
        torch.distributed.all_reduce(tm, op=torch.distributed.ReduceOp.MAX)
        ts = t.clone()
        torch.distributed.all_reduce(ts, op=torch.distributed.ReduceOp.SUM)
        t_dev, t_e2e, vox_total = float(tm[0]), float(tm[1]), int(ts[2])
    else:
        t_dev, t_e2e, vox_total = float(t[0]), float(t[1]), int(t[2])
    out = {"workload": f"configs[4]: construct_full_map, {n_frames} keyframes x {n_pts} pts (pool of {n_pool} ray-cast Avia keyframes replayed {reuse}x per "
                       f"tile, {tiles} tiles side by side), leaf 0.1 m" + ("" if n_frames >= 10000 else " - REDUCED SIZE (10000 keyframes = full)"),
           "metric": "keyframes/s", "value": n_frames / t_dev, "unit": "keyframes/s", "points_per_s": n_frames * n_pts / t_dev, "n_gpus": world,
           "scaling": "strong", "seconds": t_dev, "map_voxels": vox_total, "exchange_ms": float(np.min(exch)) if exch else 0.0,
           "timing": "wall clock around b200_mapbuild_add_keyframes_device (batches of 96 keyframes) + merge (NCCL exchange) + final sync, keyframes resident in HBM; max over ranks, best of 3",
           "e2e": {"value": n_host * world / t_e2e, "unit": "keyframes/s", "seconds": t_e2e, "keyframes": n_host * world, "h2d_bytes_per_keyframe": n_pts * 16,
                   "note": "b200_mapbuild_add_keyframe with host buffers (pack + H2D per keyframe) on a bounded block of keyframes + merge"}}
    if rank == 0 and not args.no_cpu:
        from oracle import binding as ob
        ns = min(64, n_frames)
        t0 = time.perf_counter()
        c0, n0 = ob.full_map([pool[i % n_pool] for i in range(ns)], np.array([pose_of(i) for i in range(ns)]), 0.1)
        dt = time.perf_counter() - t0
        b = api.FullMapBuilder(leaf=0.1, capacity_voxels=8_000_000, device=local_rank)
        for i in range(ns):
            b.add_keyframe(pool[i % n_pool], pose_of(i))
        c1, n1 = b.extract()
        out["cpu_baseline"] = {"value": ns / dt, "unit": "keyframes/s", "cores": 1, "kind": "port", "sample": f"first {ns} keyframes (single thread, as pcl::VoxelGrid)"}
        out["parity"] = {"keyframes": ns, "voxels_equal": bool(len(c0) == len(c1) and np.array_equal(n0, n1)),
                         "max_centroid_diff_m": float(np.abs(c0 - c1).max()) if len(c0) == len(c1) else None}
        b.close()
    return out


def loam_leg(args, local_rank, api, synth):
    """SURVEY 8f rank 3: jueying_slam's scan2MapOptimization (corner + surf features, 6x6 LM) for one scan."""
    sc = synth.loam_scene(n_surf_map=400_000, surf_stride=4, corner_stride=2)
    g = api.ScanToMap(max_map_points=1_000_000, device=local_rank)
    t_set = []
    for _ in range(3):
        t0 = time.perf_counter()
        g.setInputCloud(sc["corner_map"], sc["surf_map"])
        t_set.append((time.perf_counter() - t0) * 1e3)
    guess = sc["t_true"] + np.array([0.01, -0.01, 0.02, 0.15, -0.1, 0.05], np.float32)
    dev, wall = [], []
    for k in range(args.steps + 3):
        api.flush_l2(local_rank)
        t0 = time.perf_counter()
        t, rc = g.scan2MapOptimization(sc["corner"], sc["surf"], guess)
        if k >= 3:
            wall.append((time.perf_counter() - t0) * 1e3)
            dev.append(g.stats.gpu_ms)
    out = {"workload": f"jueying_slam scan2MapOptimization: {len(sc['corner'])} corner + {len(sc['surf'])} surf features vs "
                       f"{len(sc['corner_map'])} / {len(sc['surf_map'])}-point feature maps, 0.18 m / 1 deg initial error",
           "set_map_ms_e2e": float(np.min(t_set)), "optimize_ms": {"device": mean(dev), "e2e_wall": mean(wall)},
           "iters": g.stats.iters, "n_sel": g.stats.n_sel, "converged": bool(g.stats.converged),
           "pose_error": {"trans_m": float(np.abs(t[3:] - sc["t_true"][3:]).max()), "rot_rad": float(np.abs(t[:3] - sc["t_true"][:3]).max())}}
    if not args.no_cpu:
        from oracle import binding as ob
        o = ob.OracleLoam(num_threads=host_threads())
        o.set_map(sc["corner_map"], sc["surf_map"])
        t0 = time.perf_counter()
        t_o, st = o.optimize(sc["corner"], sc["surf"], guess)
        out["cpu_baseline"] = {"optimize_ms": (time.perf_counter() - t0) * 1e3, "cores": host_threads(), "kind": "port",
                               "sample": "one full optimisation; the port finds neighbours by brute force (exact, like the kd-tree, but slower than one)"}
        out["parity"] = {"iters_equal": bool(st["iters"] == g.stats.iters), "max_transform_diff": float(np.abs(t_o - t).max())}
    g.close()
    return out


def gicp_leg(args, local_rank, api, synth):
    """SURVEY 8a-14: pclomp GICP ("GICP_OMP" in localization.cpp) - 20k-point scan against a 1M-point local map, constructor defaults."""
    world = synth.make_world(synth.SEED, beams=True)
    mp = synth.sample_map(100_000 if args.small else 1_000_000, synth.SEED, world=world)
    p_true = np.array([3.0, -2.0, 1.2, 0.0, 0.0, 0.6])
    T = synth.pose_vec_to_matrix(p_true)
    scan = np.ascontiguousarray(synth.raycast(T[:3, 3], T[:3, :3], synth.livox_dirs(24000, synth.SEED), world, seed=synth.SEED)[:20000])
    guess = synth.pose_vec_to_matrix(p_true + np.array([0.15, -0.1, 0.05, 0.01, -0.01, 0.03]))
    g = api.GeneralizedIterativeClosestPoint(device=local_rank)
    t0 = time.perf_counter()
    g.setInputTarget(mp)
    g.setInputSource(scan)
    g.covariances("target")                       # the reference computes them inside the first align (gicp_omp_impl.hpp:383-394)
    t_first = (time.perf_counter() - t0) * 1e3
    dev, wall = [], []
    for k in range(args.steps + 3):
        api.flush_l2(local_rank)
        t0 = time.perf_counter()
        rc = g.align(guess)
        if k >= 3:
            wall.append((time.perf_counter() - t0) * 1e3)
            dev.append(g.result.gpu_ms)
    fin, r = g.getFinalTransformation(), g.result
    out = {"workload": f"pclomp GICP (k = 20, BFGS): {len(scan)}-pt scan vs {len(mp)}-pt map, 0.19 m / 2 deg initial error, constructor defaults",
           "index_and_target_covariances_ms_e2e": t_first, "align_ms": {"device": mean(dev), "e2e_wall": mean(wall)},
           "outer_iterations": int(r.iterations), "bfgs_steps": int(r.inner_total), "functor_calls": [int(r.n_f), int(r.n_df), int(r.n_fdf)],
           "matches": int(r.last_m), "converged": bool(r.converged), "index": g.index_info("target"),
           "pose_error": {"trans_m": float(np.abs(fin[:3, 3] - T[:3, 3]).max()), "rot": float(np.abs(fin[:3, :3] - T[:3, :3]).max())}}
    if not args.no_cpu:
        from oracle import binding as ob
        o = ob.OracleGicp(num_threads=host_threads())
        o.set_target(mp)
        o.set_source(scan)
        t0 = time.perf_counter()
        o.covariances("target")
        t_cov = (time.perf_counter() - t0) * 1e3
        t0 = time.perf_counter()
        rc0, fin0, r0 = o.align(guess)
        out["cpu_baseline"] = {"align_ms": (time.perf_counter() - t0) * 1e3, "covariances_ms": t_cov, "cores": host_threads(), "kind": "port",
                               "sample": "one full align; the port's exact neighbour search is a uniform grid, not PCL's kd-tree"}
        out["parity"] = {"outer_iterations_equal": bool(r0.iterations == r.iterations), "matches_equal": bool(r0.last_m == r.last_m),
                         "max_transform_diff": float(np.abs(fin0 - fin).max())}
    g.close()
    return out


# =============================================================================================== arms
def run_reference(args, rank, world):
    """--impl reference: the reference's own CPU implementation of the path = its restatement in oracle/
    (the reference cannot be compiled here: no PCL/Eigen-Core/Boost/TBB, SURVEY.md F5), all host threads (set explicitly:
    torchrun exports OMP_NUM_THREADS=1).  A step = calculateScore on a bounded sample of the 4096 hypotheses."""
    if rank != 0:
        return
    from pointcloud_slam_b200 import synth
    threads = host_threads()
    cfg = synth.config2(N_PRIOR, N_SCAN)
    poses = synth.hypothesis_grid(cfg["p_true"], 32, 32, 4, 1.0)
    c = ndt_cpu(cfg, want_align=(world == 1 and not args.no_ndt))
    n_s = args.ref_sample
    steps, warmup = args.steps, args.warmup
    ms = []
    t_start = time.perf_counter()
    for k in range(warmup + steps):
        sel, sc, t_sc = cpu_reloc_sample(c["oracle"], poses, n_s)
        if k >= warmup:
            ms.append(t_sc * 1e3)
        if time.perf_counter() - t_start > 150.0 and len(ms) >= 3:
            break
    ms_step = mean(ms)
    value = n_s / (ms_step * 1e-3)
    sample = f"each step scores {n_s} of the 4096 hypotheses (every {N_HYP // n_s}th), one hypothesis per thread; serial 10M-pt voxel build {c['build_s']:.1f} s not included"
    line = {
        "impl": "reference", "metric": "relocalization hypotheses/sec", "value": value, "unit": "hypotheses/s",
        "n_gpus": args.gpus, "steps": len(ms), "warmup": warmup, "ms_per_step": ms_step, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": headline_config(),
        "cpu_baseline": {"value": value, "unit": "hypotheses/s", "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "hypotheses/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    if world == 1:
        if not args.no_ndt:
            rc0, T0, r0 = c["align"]
            line["ndt"] = {"workload": "configs[1]: 20k-pt scan vs 10M-pt prior map, 1.0 m voxels, DIRECT7, eps 0.01, step 0.1",
                           "set_target_ms": {"e2e_wall": c["build_s"] * 1e3}, "derivatives_ms": {"e2e_wall": c["deriv_ms"]},
                           "align_ms": {"e2e_wall": c["align_ms"], "iters": r0.iters, "evals": r0.evals, "hess_evals": r0.hess_evals,
                                        "points_per_s": N_SCAN / (c["align_ms"] * 1e-3)}}
        if not args.no_iekf:
            data = synth.config1(N_MAP, N_SCAN)
            ims, t_insert, _ = cpu_oracle_iekf(data, PARAMS[args.params], 20, 3, budget_s=30.0)
            line["iekf"] = {"workload": "configs[0]: 20k-pt Mid-360-shaped scan vs 2M-pt local map, one IEKF update per step",
                            "metric": "registered points/sec (IEKF update)", "value": N_SCAN / (float(np.median(ims)) * 1e-3), "unit": "points/s",
                            "ms_per_update": float(np.median(ims)), "cores": threads, "sample": f"{len(ims)} full-size updates (median)"}
    print(json.dumps(line), flush=True)


def run_b200(args, rank, local_rank, world):
    import torch
    from pointcloud_slam_b200 import api, synth

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the engine has no CPU path (use --impl reference for the CPU baseline)")
    torch.cuda.set_device(local_rank)
    comm = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        ident = [api.Communicator.unique_id() if rank == 0 else None]
        dist.broadcast_object_list(ident, src=0)
        comm = api.Communicator(world, rank, ident[0], device=local_rank)

    # ---- headline: configs[3] on all ranks
    cfg = synth.config2(N_PRIOR, N_SCAN) if rank == 0 else None
    if world > 1:
        small = [dict(scan=cfg["scan"], p_true=cfg["p_true"], p_guess=cfg["p_guess"], guess=cfg["guess"]) if rank == 0 else None]
        torch.distributed.broadcast_object_list(small, src=0)
        if rank != 0:
            cfg = small[0]
    g, poses, rel = reloc_leg(args, rank, local_rank, world, api, synth, torch, comm, cfg)
    oracle_ndt = rel.pop("_oracle_ndt", None)
    extra = {}
    if rank == 0 and world == 1 and not args.no_ndt:
        c = None
        if oracle_ndt is not None:
            o = oracle_ndt["oracle"]
            t0 = time.perf_counter()
            for _ in range(3):
                s, gg, H = o.derivatives(cfg["p_guess"])
            oracle_ndt["deriv_ms"] = (time.perf_counter() - t0) / 3 * 1e3
            t0 = time.perf_counter()
            oracle_ndt["align"] = o.align(cfg["guess"])
            oracle_ndt["align_ms"] = (time.perf_counter() - t0) * 1e3
            oracle_ndt["deriv"] = (s, gg, H)
            c = oracle_ndt
        extra["ndt"] = ndt_leg(args, local_rank, api, g, cfg, c)
        extra["ndt"]["set_target_ms"] = rel["set_target_ms"]
    g.close()
    del oracle_ndt
    if cfg is not None:
        cfg.pop("map", None)

    # ---- the other workloads
    if not args.no_iekf:
        extra["iekf" if world == 1 else "iekf_replicas"] = iekf_leg(args, rank, local_rank, world, api, synth, torch, full=(world == 1))
    if args.fullmap_frames > 0:
        extra["fullmap"] = fullmap_leg(args, rank, local_rank, world, api, synth, torch, comm)
    if comm is not None:
        comm.close()
    if world == 1:
        if args.seq_scans > 1:
            extra["sequence"] = sequence_leg(args, local_rank, api, synth, args.seq_scans, args.seq_parity)
        if not args.no_ndt:
            extra["scan2map"] = loam_leg(args, local_rank, api, synth)
            try:
                extra["gicp"] = gicp_leg(args, local_rank, api, synth)
            except Exception as e:  # the newest leg must not take the headline down with it
                extra["gicp"] = {"error": f"{type(e).__name__}: {e}"}
    if rank != 0:
        if world > 1:
            torch.distributed.barrier()
            torch.distributed.destroy_process_group()
        return

    line = {
        "metric": "relocalization hypotheses/sec", "value": rel["value"], "unit": "hypotheses/s",
        "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": rel["ms_per_step"], "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": headline_config(),
        "e2e": rel["e2e"], "gpu_launches": rel["gpu_launches"], "clocks": rel["clocks"], "roofline": rel["roofline"],
        "cpu_baseline": rel.get("cpu_baseline"), "parity": rel.get("parity"),
        "reloc": {k: rel[k] for k in ("per_rank", "best", "best_score", "true_index", "collective", "set_target_ms", "wall_s_timed_region_incl_flush")},
    }
    line.update(extra)
    # the headline numbers of every leg once more, last on the line (stored tails keep the end of the line)
    summ = {"reloc_hyp_per_s": rel["value"], "reloc_ms_per_4096": rel["ms_per_step"], "reloc_e2e_hyp_per_s": rel["e2e"]["value"], "n_gpus": world,
            "reloc_parity": rel.get("parity"), "reloc_roofline_frac": rel["roofline"]["frac"]}
    ie = extra.get("iekf") or extra.get("iekf_replicas")
    if ie:
        summ.update({"iekf_points_per_s": ie["value"], "iekf_ms_per_update": ie["ms_per_update"]})
        if "e2e" in ie:
            summ.update({"iekf_e2e_ms_per_update": ie["e2e"]["ms_per_update"], "knn_roofline_frac": ie["roofline"]["frac"],
                         "knn_roofline_frac_1M_queries": ie["roofline"]["batched"]["frac"], "iekf_cpu_ms_per_update": (ie.get("cpu_baseline") or {}).get("ms_per_update"),
                         "iekf_parity": ie.get("parity")})
    if "ndt" in extra:
        summ.update({"ndt_align_ms": extra["ndt"]["align_ms"]["device"], "ndt_set_target_ms_device": extra["ndt"]["set_target_ms"]["device"],
                     "ndt_set_target_ms_e2e": extra["ndt"]["set_target_ms"]["e2e_wall"], "ndt_parity": extra["ndt"].get("parity")})
    if "sequence" in extra:
        sq = extra["sequence"]
        summ.update({"seq_scans": sq["scans"], "seq_ms_per_scan_e2e": sq["ms_per_scan_e2e"]["mean"], "seq_map_incremental_ms": sq["ms_per_scan_e2e"]["map_incremental_mean"],
                     "seq_ms_update_device": sq["ms_update_device"]["mean"], "seq_parity": sq["parity_vs_oracle"]})
    if "fullmap" in extra:
        fm = extra["fullmap"]
        summ.update({"fullmap_keyframes": args.fullmap_frames, "fullmap_keyframes_per_s": fm["value"], "fullmap_seconds": fm["seconds"],
                     "fullmap_exchange_ms": fm["exchange_ms"], "fullmap_parity": fm.get("parity")})
    if "gicp" in extra and "align_ms" in extra["gicp"]:
        gi = extra["gicp"]
        summ.update({"gicp_align_ms": gi["align_ms"]["device"], "gicp_cpu_align_ms": (gi.get("cpu_baseline") or {}).get("align_ms"), "gicp_parity": gi.get("parity")})
    line["summary"] = summ
    if args.dump_outputs:   # what the caller of the headline path received in the last timed step
        dump_outputs(args.dump_outputs, {"reloc_best_index": rel["best"], "reloc_best_score": rel["best_score"]})
    print(json.dumps(line), flush=True)
    if world > 1:
        torch.distributed.barrier()
        torch.distributed.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--params", default="livox", choices=list(PARAMS), help="configs[0] parameter set (livox.yaml / horizon.yaml)")
    ap.add_argument("--no-ndt", action="store_true", help="skip the configs[1] and scan2map legs")
    ap.add_argument("--no-iekf", action="store_true", help="skip the configs[0] leg")
    ap.add_argument("--no-cpu", action="store_true", help="skip the CPU baseline / oracle parity legs")
    ap.add_argument("--seq-scans", type=int, default=1000, help="configs[2] leg: scans in the sliding-map sequence (1000 = full size; 0 = skip)")
    ap.add_argument("--seq-parity", type=int, default=120, help="configs[2] leg: scans checked against the CPU oracle")
    ap.add_argument("--fullmap-frames", type=int, default=10000, help="configs[4] leg: keyframes to merge (10000 = full size; 0 = skip)")
    ap.add_argument("--fullmap-pool", type=int, default=32, help="distinct ray-cast keyframes in the replay pool")
    ap.add_argument("--fullmap-reuse", type=int, default=5, help="times the pool is replayed on one tile before moving to the next")
    ap.add_argument("--fullmap-host-frames", type=int, default=800, help="keyframes of the host-buffer (e2e) pass of the configs[4] leg")
    ap.add_argument("--ref-sample", type=int, default=256, help="--impl reference: hypotheses scored per step")
    ap.add_argument("--small", action="store_true", help="DEV ONLY: shrink the maps 10x (not a valid bench number)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write the headline's result of the last timed step "
                                                         "(winning hypothesis index and score) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs applies to --impl b200")
    rank, local_rank, world = dist_env()
    if args.small:
        global N_MAP, N_PRIOR
        N_MAP, N_PRIOR = N_MAP // 10, N_PRIOR // 10
    if args.impl == "reference":
        run_reference(args, rank, world)
    else:
        run_b200(args, rank, local_rank, world)


if __name__ == "__main__":
    main()
