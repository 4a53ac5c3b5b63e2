"""Batched loop-closure registration benchmark: prints ONE JSON line.

Workload (the loop-closure call of mapOptmization.cpp:683-693): P = 512 pairs from synth.loop_pairs, 10k-point keyframe
sources, 100k-point submap targets, resolution 1.0 m, DIRECT7, transformation epsilon 0.01, identity guesses.

  batched   b200_ndt_pairs_align on all P pairs: pairs/s from the call's device time (CUDA events) and from the host wall
            time of the call including the host-to-device copies (clouds already packed in the offset layout)
  loop      the same pairs through the existing per-pair calls (set_target, set_source, align, fitness_score), wall time
  oracle    the CPU oracle (OpenMP over all cores) on a sample of pairs, with the core count
  parity    batched vs per-pair loop (iterations / evaluations / fitness bits / finals) and vs the oracle on the sample
  gpu       name and power limit, read in the same run

Under torchrun (python -m torch.distributed.run --nproc-per-node N tools/ndt_pairs_bench.py --gpus N) every rank takes part
in the sharded call; rank 0 also times the single-GPU call in the same process and reports the scaling efficiency.
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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--pairs", type=int, default=512)
    ap.add_argument("--n-src", type=int, default=10_000)
    ap.add_argument("--n-tgt", type=int, default=100_000)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--oracle-sample", type=int, default=8)
    ap.add_argument("--loop-pairs", type=int, default=0, help="pairs timed through the per-pair loop (0 = all)")
    ap.add_argument("--gpus", type=int, default=1)
    args = ap.parse_args()
    from pointcloud_slam_b200 import api, synth
    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    P = args.pairs
    settings = dict(resolution=1.0, search=7, trans_eps=0.01)
    t0 = time.perf_counter()
    d = synth.loop_pairs(P, args.n_src, args.n_tgt)
    gen_s = time.perf_counter() - t0
    src, soff = api.NdtPairBatch.pack(d["sources"])
    tgt, toff = api.NdtPairBatch.pack(d["targets"])
    out = dict(workload=dict(pairs=P, n_src=args.n_src, n_tgt=args.n_tgt, resolution=1.0, search="DIRECT7", trans_eps=0.01, guess="identity",
                             synth_s=round(gen_s, 1)))
    comm = None
    if world > 1:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        ident = [api.Communicator.unique_id() if rank == 0 else None]
        dist.broadcast_object_list(ident, src=0)
        comm = api.Communicator(world, rank, ident[0], device=local)
    b = api.NdtPairBatch(device=local, **settings)

    def timed(c):
        b.align_packed(src, soff, tgt, toff, P, comm=c)   # warm-up: grows every buffer, loads the modules
        walls, devs = [], []
        for _ in range(args.reps):
            if c is not None:
                import torch.distributed as dist
                dist.barrier()
            t = time.perf_counter()
            r = b.align_packed(src, soff, tgt, toff, P, comm=c)
            walls.append(time.perf_counter() - t)
            devs.append(r["gpu_ms"] / 1e3)
        return r, min(walls), min(devs)

    if world > 1:
        r, wall, dev = timed(comm)
        out[f"gpus_{world}"] = dict(pairs_per_s_wall=P / wall, pairs_per_s_device=P / dev, wall_s=wall, device_s=dev)
    r1, wall1, dev1 = timed(None) if rank == 0 else (None, None, None)
    if rank == 0:
        out["batched"] = dict(pairs_per_s_wall=P / wall1, pairs_per_s_device=P / dev1, wall_s=wall1, device_s=dev1,
                              statuses={str(k): int(v) for k, v in zip(*np.unique(r1["status"], return_counts=True))})
        if world > 1:
            g = out[f"gpus_{world}"]
            g["efficiency_wall"] = g["pairs_per_s_wall"] / (world * out["batched"]["pairs_per_s_wall"])
            g["same_results_as_1_gpu"] = bool(all(bytes(memoryview(x).cast("B"))[:8] == bytes(memoryview(y).cast("B"))[:8]
                                                  and x.fitness == y.fitness and list(x.final16) == list(y.final16)
                                                  for x, y in zip(r["records"][:P], r1["records"][:P])))
        else:
            # the existing per-pair loop on the same pairs
            nl = args.loop_pairs or P
            g = api.NormalDistributionsTransform(device=local)
            g.setResolution(1.0)
            g.setTransformationEpsilon(0.01)
            g.setInputTarget(d["targets"][0])
            g.setInputSource(d["sources"][0])
            g.align(None)
            g.getFitnessScore()
            it_eq = fit_eq = 0
            dmax = 0.0
            t = time.perf_counter()
            for p in range(nl):
                g.setInputTarget(d["targets"][p])
                g.setInputSource(d["sources"][p])
                g.align(None)
                f = g.getFitnessScore()
                it_eq += int((g.result.iters, g.result.evals, g.result.converged) == (r1["iters"][p], r1["evals"][p], r1["converged"][p]))
                fit_eq += int(f == r1["fitness"][p])
                dmax = max(dmax, float(np.abs(g.getFinalTransformation() - r1["final"][p]).max()))
            loop_s = time.perf_counter() - t
            out["loop"] = dict(pairs=nl, pairs_per_s_wall=nl / loop_s, wall_s=loop_s)
            out["speedup_wall"] = out["batched"]["pairs_per_s_wall"] / out["loop"]["pairs_per_s_wall"]
            # the CPU oracle on a sample
            from oracle import binding as ob
            sample = list(range(0, P, max(1, P // args.oracle_sample)))[: args.oracle_sample]
            o_it = 0
            o_dp = 0.0
            t = time.perf_counter()
            for p in sample:
                o = ob.OracleNdt(resolution=1.0, trans_eps=0.01, search=7)
                o.set_target(d["targets"][p])
                o.set_source(d["sources"][p])
                rc0, T0, r0 = o.align(np.eye(4, dtype=np.float32))
                o.fitness(T0)
                o_it += int((r0.iters, r0.evals, r0.converged) == (r1["iters"][p], r1["evals"][p], r1["converged"][p]))
                o_dp = max(o_dp, float(np.abs(np.array(r0.p_final) - r1["p_final"][p]).max()))
            o_s = time.perf_counter() - t
            out["oracle"] = dict(pairs=len(sample), cores=os.cpu_count(), pairs_per_s=len(sample) / o_s)
            out["parity"] = dict(loop_iters_evals_converged_equal=f"{it_eq}/{nl}", loop_fitness_bit_equal=f"{fit_eq}/{nl}", loop_final_max_abs_diff=dmax,
                                 oracle_iters_evals_converged_equal=f"{o_it}/{len(sample)}", oracle_p_final_max_abs_diff=o_dp)
        out["gpu"] = gpu_info()
        out["gpus"] = world
        print(json.dumps(out), flush=True)
    if comm is not None:
        import torch.distributed as dist
        comm.close()
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
