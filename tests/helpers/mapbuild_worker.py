"""Worker for the multi-rank full-map test (launched with torch.distributed.run, one process per GPU; on one rank both
merges are local).  Each worker writes its pid next to the result so that the test can kill it if the launch is stuck.

Phase 1: the hall's keyframes 2 km from the origin, all on rank 0 (rank 1 has none), then a merge.  Phase 2: the same
keyframes 100 km away, split in contiguous blocks over the ranks, then a second merge.  Each rank must then hold exactly
the fp64 reference's voxels that hash to it (owner = hash of the key), with their full counts and centroids.
Rank 0 writes a JSON result to argv[1]."""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np
import torch
import torch.distributed as dist


def main():
    out_path = sys.argv[1]
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ.get("LOCAL_RANK", 0))
    with open(os.path.join(os.path.dirname(out_path), f"worker{rank}.pid"), "w") as f:   # lets the test kill a stuck worker
        f.write(str(os.getpid()))
    from pointcloud_slam_b200 import api, synth
    import voxel_ref as vr
    from test_gpu_voxel import make_frames
    from test_gpu_voxel_more import assert_map_matches_ref
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    ident = [api.Communicator.unique_id() if rank == 0 else None]
    dist.broadcast_object_list(ident, src=0)
    comm = api.Communicator(world, rank, ident[0], device=local)

    frames, poses = make_frames(synth, k=8, n=4000)
    near, far = poses.copy(), poses.copy()
    near[:, :3] += (2000.0, 300.0, 0.0)
    far[:, :3] += (100000.0, 0.0, 0.0)
    b = api.FullMapBuilder(leaf=0.1, capacity_voxels=400_000, device=local)
    if rank == 0:
        for f, p in zip(frames, near):
            b.add_keyframe(f, p)
    b.merge(comm)
    n_after_first = b.num_voxels()
    fb, fe = api.shard_range(len(frames), world, rank)
    for f, p in zip(frames[fb:fe], far[fb:fe]):
        b.add_keyframe(f, p)
    b.merge(comm)
    c, n = b.extract()

    ref = vr.map_build(frames + frames, np.concatenate([near, far]), 0.1)
    mine = api.voxel_owner(api.voxel_key(ref["cells"]), world) == rank
    sub = {k: ref[k][mine] for k in ("cells", "counts", "cent")}
    err = ""
    try:
        assert len(n) == mine.sum(), f"rank {rank}: {len(n)} voxels, the reference gives it {mine.sum()}"
        assert_map_matches_ref(c, n, sub, 0.1, 100.0)
    except AssertionError as e:
        err = str(e)[:500] or "mismatch"
    errs = [None] * world
    dist.all_gather_object(errs, err)
    counts = [None] * world
    dist.all_gather_object(counts, (int(n_after_first), int(len(n)), int(n.sum())))
    if rank == 0:
        ok = not any(errs) and sum(x[1] for x in counts) == len(ref["counts"]) and sum(x[2] for x in counts) == int(ref["counts"].sum())
        json.dump(dict(ok=bool(ok), world=world, errors=errs, per_rank=counts, ref_voxels=int(len(ref["counts"]))), open(out_path, "w"))
    comm.close()
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
