"""torchrun worker (one process per GPU, NCCL): sharding.shard_from_reads + hot_path_step with the library's communicator; the
ranks' records and events, gathered in rank order, must equal e2s_pipeline_reads on the whole index.  Prints "OK <world>" on rank 0."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from ebwt2snp_b200 import api, sharding  # noqa: E402
from tests.test_from_reads_gpu import case_reads, pipeline_outputs  # noqa: E402


def main():
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    dev = torch.device("cuda", rank)
    torch.cuda.set_device(dev)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    bases, off = case_reads("genome")
    p = api.default_params((len(off) - 1) // 2)
    ctx = api.Context(rank)
    sh = sharding.shard_from_reads(ctx, bases, off, 1, 4, 1, dev)
    comm = sharding.make_comm(ctx, dev)
    mg, st, cnt, ids = sharding.hot_path_step(sh, p, 16, 2, dev, comm=comm)
    first_id, _ = ids.resolve()
    mine = (sh.cluster_fetch_packed(), [bytes(e) for e in sh.events()], first_id)
    got = [None] * world
    dist.all_gather_object(got, mine)
    if rank == 0:
        n = int(off[-1]) + len(off) - 1
        rc, whole = pipeline_outputs(ctx, lambda r, e: ctx.pipeline_reads(bases, off, p, 16, 2, 1, 4, 1, rec10=r, events=e), n)[:2]
        assert rc == 0, whole
        assert b"".join(g[0] for g in got) == whole[1]
        assert sum((g[1] for g in got), []) == whole[2]
        assert [g[2] for g in got] == list(np.cumsum([1] + [len(g[1]) for g in got[:-1]]))
        print(f"OK {world}", flush=True)
    comm.close()
    sh.close()
    ctx.close()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
