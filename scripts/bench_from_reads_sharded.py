"""Reads to SNPs over N shards, one process per rank (torchrun; plain python = one rank): each rank stages all the reads, computes the
key cuts, builds its own key range into its resident shard, exchanges the halo rows (one all-gather), applies them, seals and runs
the first hot-path step.

    torchrun --nproc-per-node N scripts/bench_from_reads_sharded.py --config C3 --reps 3 --out profiles/X.json
    python scripts/bench_from_reads_sharded.py --config C2 --cli 1 2 4 --out profiles/Y.json

Per rank, one warm-up and `reps` timed repetitions of each phase (host clock around work that ends in a device synchronise):
  stage       the reads to the device (H2D)
  cuts        e2s_reads_key_cuts
  build       shard creation + e2s_shard_build_egsa_range
  halo        e2s_shard_halo_row + the all-gather of the rows + e2s_shard_halo_apply + seal
  first_step  sharding.hot_path_step on the sealed shard (with the library's NCCL communicator when N > 1)
  whole       sharding.shard_from_reads + hot_path_step from host reads (all of the above in one go)
With one rank, e2s_pipeline_reads on the same reads is timed in the same run (the one-GPU path this generalises) and the records
and events of both are compared.  Peak device memory per rank is sampled during `whole`.  --cli: the ebwt2snp CLI at each -G on
this box's GPUs (shards share a device when -G exceeds them), files compared across -G.  Rank 0 writes one JSON line with the
card's name and power limit read in the same run."""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--config", default="C3")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--cli", nargs="*", type=int, default=[])
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench_from_reads_sharded: needs a CUDA device")
    from bench_from_reads import PeakMemory, gpu_info
    from ebwt2snp_b200 import api, sharding, synth

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    dev = torch.device("cuda", rank % torch.cuda.device_count())
    torch.cuda.set_device(dev)
    if world > 1:
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    rs = synth.make_config(args.config, seed=1)
    R, L = rs.reads.shape
    bases = torch.from_numpy(np.ascontiguousarray(rs.reads).reshape(-1)).pin_memory().numpy()  # (pinned, as bench_from_reads.py stages them)
    off = np.arange(R + 1, dtype=np.uint64) * np.uint64(L)
    p = api.default_params(rs.nreads1)
    ctx = api.Context(dev.index)
    comm = sharding.make_comm(ctx, dev) if world > 1 else None

    def timed(fn):
        fn()
        torch.cuda.synchronize(dev)
        ts = []
        for _ in range(args.reps):
            t0 = time.perf_counter()
            fn()
            torch.cuda.synchronize(dev)
            ts.append(time.perf_counter() - t0)
        return ts

    state = {}

    def build():
        key_lo, pos = state["cuts"]
        if "sh" in state:
            state.pop("sh").close()
        sh = ctx.shard(int(pos[rank + 1]) - int(pos[rank]), int(pos[rank]), int(pos[world]))
        sh.build_egsa_range(off, int(key_lo[rank]), int(key_lo[rank + 1]) if rank + 1 < world else 0, 4, 4, 4)
        state["sh"] = sh

    def halo():
        rows = sharding.all_gather_words(state["sh"].halo_row(), dev)
        state["sh"].halo_apply(rows, rank)
        state["sh"].seal()

    def whole():
        if "sh" in state:
            state.pop("sh").close()
        sh = sharding.shard_from_reads(ctx, bases, off, 4, 4, 4, dev)
        state["step"] = sharding.hot_path_step(sh, p, 16, 2, dev, comm=comm)
        state["sh"] = sh

    out = {"config": args.config, "ranks": world, "rank": rank, "positions": int(bases.size + R)}
    out["stage_s"] = timed(lambda: ctx.stage_reads(bases, off))
    out["cuts_s"] = timed(lambda: state.__setitem__("cuts", ctx.key_cuts(off, world)))
    out["shard_positions"] = int(state["cuts"][1][rank + 1] - state["cuts"][1][rank])
    out["build_s"] = timed(build)
    out["halo_s"] = timed(halo)
    out["first_step_s"] = timed(lambda: sharding.hot_path_step(state["sh"], p, 16, 2, dev, comm=comm))
    with PeakMemory(torch, dev) as pk:
        out["whole_s"] = timed(whole)
    out["peak_device_bytes_whole"] = int(pk.peak)
    sh = state.pop("sh")
    recs, evs = sh.cluster_fetch_packed(), b"".join(bytes(e) for e in sh.events())
    sh.close()
    if world == 1:  # the one-GPU call on the same reads, in the same run
        n = int(bases.size + R)
        rec10 = torch.empty((n // 2 + 64) * 10, dtype=torch.uint8, pin_memory=True).numpy()
        evbuf = (api.Event * (n // 2000 + 100_000))()
        res = {}
        out["pipeline_reads_s"] = timed(lambda: res.__setitem__("r", ctx.pipeline_reads(bases, off, p, 16, 2, 4, 4, 4, rec10=rec10, events=evbuf)))
        r = res["r"]
        out["same_outputs_as_pipeline_reads"] = (rec10[: int(r.n_written) * 10].tobytes() == recs and
                                                 b"".join(bytes(e) for e in list(evbuf)[: int(r.snp.n_variants)]) == evs)
    if comm is not None:
        comm.close()
    ctx.close()
    rows = [out]
    if world > 1:
        rows = [None] * world
        dist.all_gather_object(rows, out)
        dist.destroy_process_group()
    if rank != 0:
        return
    result = {"bench": "from_reads_sharded", "gpu": gpu_info(), "ranks": rows}
    if args.cli:
        result["cli"] = cli_times(rs, args.cli, args.reps)
    line = json.dumps(result)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


def cli_times(rs, shard_counts, reps):
    """ebwt2snp -G g on this box, each run timed whole (process start, contexts, files); the files must not depend on g"""
    from ebwt2snp_b200 import synth
    exe = os.path.join(ROOT, "ebwt2snp_b200", "bin", "ebwt2snp")
    with tempfile.TemporaryDirectory(prefix="e2s_sharded_") as d:
        fa = os.path.join(d, "ALL.fasta")
        synth.write_fasta(fa, rs.reads)
        res, files = {}, set()
        for _ in range(reps):  # the shard counts alternated
            for g in shard_counts:
                t0 = time.perf_counter()
                r = subprocess.run([exe, "-i", fa, "-n", str(rs.nreads1), "-G", str(g)], capture_output=True, text=True, timeout=3600)
                res.setdefault(f"G{g}_s", []).append(time.perf_counter() - t0)
                if r.returncode != 0:
                    raise RuntimeError(f"ebwt2snp -G {g}: {r.stdout[-2000:]} {r.stderr[-2000:]}")
                files.add((open(fa + ".clusters", "rb").read(), open(os.path.join(d, "ALL.snp"), "rb").read()))
        res["same_files"] = len(files) == 1
        return res


if __name__ == "__main__":
    main()
