"""Worker for the 2-GPU batched pair registration test (launched with torch.distributed.run).

Every rank passes the same P = 37 pairs (ragged over the ranks) to b200_ndt_pairs_align with an NCCL communicator; rank r
registers pairs p = r (mod N).  Then once more with a pair that only its owning rank finds broken (an empty source).
Rank 0 writes the gathered result records of every rank and of a single-GPU call to argv[1] as JSON (hex).
"""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

import numpy as np
import torch
import torch.distributed as dist


def records_hex(r, P):
    out = []
    for p in range(P):
        rec = type(r["records"][0]).from_buffer_copy(r["records"][p])
        rec.ndt.gpu_ms = 0.0
        out.append(bytes(memoryview(rec).cast("B")).hex())
    return out


def main():
    out_path = sys.argv[1]
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ.get("LOCAL_RANK", 0))
    from pointcloud_slam_b200 import api, synth
    P = 37
    rng = np.random.default_rng(5)
    d = synth.loop_pairs(P, rng.integers(500, 6000, P), rng.integers(20_000, 60_000, P))
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    ident = [api.Communicator.unique_id() if rank == 0 else None]
    dist.broadcast_object_list(ident, src=0)
    comm = api.Communicator(world, rank, ident[0], device=local)
    b = api.NdtPairBatch(device=local, trans_eps=0.01)
    sharded = records_hex(b.align(d["sources"], d["targets"], comm=comm), P)
    single = records_hex(api.NdtPairBatch(device=local, trans_eps=0.01).align(d["sources"], d["targets"]), P)
    bad_src = list(d["sources"])
    bad_src[3] = np.zeros((0, 3), np.float32)   # pair 3 belongs to rank 1 of 2
    rb = b.align(bad_src, d["targets"], comm=comm)
    bad = dict(status=rb["status"].tolist(), records=records_hex(rb, P))
    gathered = [None] * world
    dist.all_gather_object(gathered, dict(sharded=sharded, single=single, bad=bad))
    if rank == 0:
        json.dump(dict(world=world, ranks=gathered), open(out_path, "w"))
    comm.close()
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
