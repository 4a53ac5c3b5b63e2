"""Worker for the multi-rank relocalization-with-refinement tests (launched with torch.distributed.run).

mode "gloo": CPU only - the oracle scores each rank's slice and aligns the candidates dealt to it, and the two exchanges of
             b200_reloc_refine run over gloo through api.reloc_refine_protocol_host.
mode "nccl": the product path - map replicated with b200_ndt_set_target_bcast, b200_reloc_refine over NCCL, compared with the
             one-GPU call over the whole grid.
Every rank writes its JSON result to <argv[2]>.<rank>.
"""
import ctypes
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

import numpy as np
import torch
import torch.distributed as dist

TOP_K = 8


def scene():
    from pointcloud_slam_b200 import synth
    world_geo = synth.make_world(synth.SEED, beams=True)
    mp = synth.sample_map(150_000, synth.SEED, world=world_geo)
    p_true = np.array([3.0, -2.0, 1.2, 0.0, 0.0, 0.6])
    T = synth.pose_vec_to_matrix(p_true)
    scan = np.ascontiguousarray(synth.raycast(T[:3, 3], T[:3, :3], synth.livox_dirs(3000, synth.SEED), world_geo, seed=synth.SEED)[:2000])
    poses = synth.hypothesis_grid(p_true, nx=5, ny=5, nyaw=3, pitch=1.0)   # 75 hypotheses: ragged over 2 ranks
    return mp, scan, poses


def slices(api, h, world, rank):
    """(name, local indices, h_begin, h_stride): contiguous, interleaved, and everything on rank 0 (rank 1 empty)."""
    b, e = api.shard_range(h, world, rank)
    yield "contiguous", np.arange(b, e), b, 1
    yield "interleaved", np.arange(rank, h, world), rank, world
    yield "empty", np.arange(h) if rank == 0 else np.arange(0), 0, 1


def gather_fn(world):
    def gather(t):
        out = [torch.zeros_like(t) for _ in range(world)]
        dist.all_gather(out, t)
        return torch.stack(out)
    return gather


def run_gloo(rank, world):
    from oracle import binding as ob
    from pointcloud_slam_b200 import api
    dist.init_process_group("gloo")
    mp, scan, poses = scene()
    o = ob.OracleNdt(resolution=1.0)
    o.set_target(mp)
    o.set_source(scan)

    def refine(pose16):
        rc, T, r = o.align(np.asarray(pose16, np.float32).reshape(4, 4).T)
        return rc, r.trans_probability, o.fitness(T)[0]

    full = o.score_batch(poses)
    res = dict(world=world, runs={})
    for name, idx, hb, hs in slices(api, len(poses), world, rank):
        out = api.reloc_refine_protocol_host(full[idx], poses[idx], hb, hs, TOP_K, world, rank, gather_fn(world), refine)
        res["runs"][name] = dict(out, n_local=int(len(idx)))
    # the single-process statement: every score, sorted by (score desc, index asc), the first TOP_K aligned in order
    keys = [api.score_key(float(s)) for s in full]
    order = sorted(range(len(full)), key=lambda i: (-keys[i], i))[:TOP_K]
    ref = [(i,) + tuple(refine(poses[i])) for i in order]
    ok = [r for r in ref if r[1] == 0]
    pick = min(ok or ref, key=lambda r: (-api.score_key(r[2]), r[0]))
    res["single"] = dict(candidates=[(i, keys[i]) for i in order], refined=[(i, int(st), float(tp), float(f)) for i, st, tp, f in ref],
                         best=int(pick[0]), status=0 if ok else 2)
    # a rank that fails locally: every rank reports its error
    out = api.reloc_refine_protocol_host(full[:3], poses[:3], 0, 1, TOP_K, world, rank, gather_fn(world), refine, status=-1 if rank == 1 else 0)
    res["failing_rank"] = dict(status=out["status"], best=out["best"])
    return res


def run_nccl(rank, world, local):
    from pointcloud_slam_b200 import api
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    mp, scan, poses = scene()
    ident = [api.Communicator.unique_id() if rank == 0 else None]
    dist.broadcast_object_list(ident, src=0)
    comm = api.Communicator(world, rank, ident[0], device=local)
    g = api.NormalDistributionsTransform(device=local)
    g.setTransformationEpsilon(0.01)
    g.setInputTargetReplicated(comm, mp if rank == 0 else None, len(mp))
    g.setInputSource(scan)
    raw = lambda cands: [bytes(c) for c in cands.records]
    best1, c1, _ = api.relocalize_refine(g, poses, None, top_k=TOP_K)
    res = dict(world=world, single=dict(best=best1, status=c1.status, n=len(c1), records=[r.hex() for r in raw(c1)]), runs={})
    for name, idx, hb, hs in slices(api, len(poses), world, rank):
        best, c, _ = api.relocalize_refine(g, poses[idx], comm, h_begin=hb, h_stride=hs, top_k=TOP_K)
        res["runs"][name] = dict(best=best, status=c.status, n=len(c), records=[r.hex() for r in raw(c)])
    # rank 1 passes h > 0 with a NULL pose pointer: every rank returns B200_ERR_ARG
    out = (api.RelocCandidate * TOP_K)()
    best, nc, ms = ctypes.c_int64(0), ctypes.c_int64(0), ctypes.c_float(0)
    idx = np.arange(rank, len(poses), world)
    p = np.ascontiguousarray(poses[idx])
    rc = api.lib().b200_reloc_refine(comm.h, g._handle(), None if rank == 1 else api._p(p), len(idx), rank, world, TOP_K,
                                     1.7976931348623157e308, ctypes.byref(best), out, ctypes.byref(nc), ctypes.byref(ms))
    res["null_poses"] = dict(rc=int(rc), best=int(best.value), error=api.lib().b200_last_error().decode())
    # and the argmin is what it was
    res["argmin"] = list(api.relocalize(g, poses)[:2])
    comm.close()
    return res


def main():
    mode, out_path = sys.argv[1], sys.argv[2]
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ.get("LOCAL_RANK", 0))
    res = run_gloo(rank, world) if mode == "gloo" else run_nccl(rank, world, local)
    json.dump(res, open(f"{out_path}.{rank}", "w"))
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
