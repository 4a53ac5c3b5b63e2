"""Relocalization with NDT refinement (b200_reloc_refine) benchmark: prints one JSON line per top_k.

Workload: configs[3]'s inputs (bench.py: synth.config2 with a 10M-point prior map, 20k-point scan, 1.0 m voxels, DIRECT7,
transformation epsilon 0.01; 4096 hypotheses = 32 x 32 xy grid at 1 m x 4 yaws), hypotheses interleaved over the ranks
(h mod N), map replicated.  For each top_k the same step is timed in full-align mode (b200_reloc_refine) and in score-only
mode (b200_reloc_argmin); the L2 is flushed (untimed) before every step and the ranks meet on the engine's stream before it,
as bench.py does.  Per line: device ms (CUDA events on the engine stream, median over the steps), hypotheses/s, ms per
refined candidate, kernel launches and host synchronisations per step, the GPU's name and power limit.

  python tools/reloc_refine_bench.py [--steps 5] [--top-k 16 64 256 4096]
  python -m torch.distributed.run --nproc-per-node N tools/reloc_refine_bench.py
The tool writes nothing into the tree.
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

from tools.ndt_pairs_bench import gpu_info  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--top-k", type=int, nargs="+", default=[16, 64, 256, 4096])
    ap.add_argument("--n-map", type=int, default=10_000_000)
    args = ap.parse_args()
    from pointcloud_slam_b200 import api, synth
    import torch
    rank, world, local = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1)), int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    comm, dist = None, None
    cfg = synth.config2(args.n_map, 20_000) if rank == 0 else None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        small = [dict(scan=cfg["scan"], p_true=cfg["p_true"]) if rank == 0 else None]
        dist.broadcast_object_list(small, src=0)
        ident = [api.Communicator.unique_id() if rank == 0 else None]
        dist.broadcast_object_list(ident, src=0)
        comm = api.Communicator(world, rank, ident[0], device=local)
        if rank != 0:
            cfg = small[0]
    g = api.NormalDistributionsTransform(device=local)
    g.setTransformationEpsilon(0.01)
    if world > 1:
        g.setInputTargetReplicated(comm, cfg["map"] if rank == 0 else None, args.n_map)
    else:
        g.setInputTarget(cfg["map"])
    g.setInputSource(cfg["scan"])
    g._handle()
    poses = synth.hypothesis_grid(cfg["p_true"], 32, 32, 4, 1.0)
    mine = np.ascontiguousarray(poses[rank::world])
    H = len(poses)

    def step(fn):
        api.flush_l2(local)
        g.stream_barrier(comm)
        l0 = api.kernel_launches()
        out = fn()
        return out, api.kernel_launches() - l0

    refine = lambda k: step(lambda: api.relocalize_refine(g, mine, comm, h_begin=rank, h_stride=world, top_k=k))
    score = lambda: step(lambda: api.relocalize(g, mine, comm, h_begin=rank, h_stride=world))
    for k in args.top_k:
        for _ in range(args.warmup):
            refine(k)
            score()
        ref_ms, sc_ms, launches, polls = [], [], [], []
        for _ in range(args.steps):
            (best, cands, ms), nl = refine(k)
            ref_ms.append(ms)
            launches.append(nl)
            polls.append(int(api.lib().b200_ndt_last_polls(g._handle())))
            (arg, _, ms_s), _ = score()
            sc_ms.append(ms_s)
        ms, ms_s = float(np.median(ref_ms)), float(np.median(sc_ms))
        if rank == 0:
            line = dict(workload=dict(hypotheses=H, n_map=args.n_map, n_scan=20_000, resolution=1.0, search="DIRECT7", trans_eps=0.01,
                                      slices="interleaved", l2="flushed before every step (untimed)"),
                        gpus=world, top_k=k, n_cands=len(cands), best=int(best), status=int(cands.status),
                        converged=int(sum(c.refined.status == 0 for c in cands)), score_only_best=int(arg),
                        full_align=dict(device_ms=ms, hypotheses_per_s=H / (ms / 1e3), ms_per_candidate=ms / max(len(cands), 1),
                                        launches=int(np.median(launches)), host_polls=int(np.median(polls))),
                        score_only=dict(device_ms=ms_s, hypotheses_per_s=H / (ms_s / 1e3)), steps=args.steps, gpu=gpu_info())
            print(json.dumps(line), flush=True)
    if comm is not None:
        comm.close()
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
