"""Worker for the 2-GPU loop-closure test (launched with torch.distributed.run).

Every rank builds the same keyframe store and calls b200_loop_close with an NCCL communicator on the same queries; rank r
assembles and registers the queries q = r (mod N).  Rank 0 writes the gathered records of every rank and of a single-GPU
call to argv[1] as JSON (hex, gpu_ms zeroed).
"""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

import numpy as np
import torch
import torch.distributed as dist

NDT = dict(resolution=1.0, trans_eps=0.01, step_size=0.1, max_iter=35)
LOOP = dict(search_radius=5.0, time_gap=30.0, search_num=25, leaf=0.4, min_source_points=100, min_target_points=1000)


def records_hex(r, Q):
    out = []
    for q in range(Q):
        x = type(r["loop_records"][q]).from_buffer_copy(r["loop_records"][q])
        x.reg.ndt.gpu_ms = 0.0
        out.append(bytes(memoryview(x).cast("B")).hex())
    return out


def main():
    out_path = sys.argv[1]
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ.get("LOCAL_RANK", 0))
    from pointcloud_slam_b200 import api, synth
    s = synth.loop_session(K=600, n_points=500, laps=2)
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    ident = [api.Communicator.unique_id() if rank == 0 else None]
    dist.broadcast_object_list(ident, src=0)
    comm = api.Communicator(world, rank, ident[0], device=local)
    st = api.KeyframeStore(device=local)
    for k, c in enumerate(s["clouds"]):
        st.add(c, s["poses"][k], s["times"][k])
    cur = np.arange(320, 600, 9)[:31]   # an odd Q: the ranks' slices differ in length
    Q = len(cur)
    sharded = records_hex(api.NdtPairBatch(device=local, **NDT).close_loops(st, cur, comm=comm, **LOOP), Q)
    single = records_hex(api.NdtPairBatch(device=local, **NDT).close_loops(st, cur, **LOOP), Q)
    gathered = [None] * world
    dist.all_gather_object(gathered, dict(sharded=sharded, single=single))
    if rank == 0:
        json.dump(dict(world=world, ranks=gathered), open(out_path, "w"))
    comm.close()
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
