"""Reads to SNPs on one GPU: e2s_pipeline_reads (the index built into the resident shard that scans it) against e2s_pipeline_host
on the host records of the same index, and the ebwt2snp CLI against build_gesa -> ebwt2clust -> clust2snp.

    python scripts/bench_from_reads.py --configs C2 C3 --reps 3 --cli C2 [--out FILE]

Per config, with one warm-up call and `reps` timed calls each (host clock around calls that end in a synchronise):
  reads_call   e2s_pipeline_reads from pinned host reads (H2D of the reads, build, seal, step, records + events out)
  build        e2s_shard_build_egsa alone on the staged reads (+ seal), and which path it took (whole or key ranges)
  step         e2s_pipeline_resident alone on the built shard
  host_call    e2s_pipeline_host on the 13-byte records of the same index (pinned)
The outputs of the two calls (counts, .clusters records, events) are compared.  Peak device memory is sampled with
cudaMemGetInfo during the reads call.  Prints one JSON line with the card's name and power limit."""
import argparse
import json
import os
import shutil
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True,
                             timeout=30).stdout.strip().splitlines()[0]
        name, power = (s.strip() for s in out.split(","))
        return {"name": name, "power_limit": power}
    except Exception as e:  # noqa: BLE001
        return {"name": None, "power_limit": None, "error": str(e)}


class PeakMemory:
    """device memory in use (total - free), sampled every 2 ms while running"""

    def __init__(self, torch, dev):
        self.torch, self.dev, self.peak, self.stop = torch, dev, 0, threading.Event()

    def __enter__(self):
        def run():
            while not self.stop.is_set():
                free, total = self.torch.cuda.mem_get_info(self.dev)
                self.peak = max(self.peak, total - free)
                time.sleep(0.002)
        self.th = threading.Thread(target=run, daemon=True)
        self.th.start()
        return self

    def __exit__(self, *a):
        self.stop.set()
        self.th.join()


def timed(fn, reps, torch):
    fn()  # warm-up
    torch.cuda.synchronize()
    ts, out = [], None
    for _ in range(reps):
        t0 = time.perf_counter()
        out = fn()
        torch.cuda.synchronize()
        ts.append(time.perf_counter() - t0)
    return out, ts


def outputs(res, rec10, evbuf):
    m = int(res.n_written)
    return ((m, int(res.n_clust_out), int(res.max_clust_length), bytes(res.snp)), rec10[: m * 10].tobytes(),
            b"".join(bytes(e) for e in list(evbuf)[: int(res.snp.n_variants)]))


def bench_config(name, reps, torch, api, bench):
    dev = torch.device("cuda", 0)
    rs, eg = bench.make_dataset(name, 1, 1.0, "cuda:0", builder="native")
    n = int(eg["n"])
    R, L = rs.reads.shape
    host_rec = bench.aos_records_pinned(eg, torch)
    m_bound = n // 2 + 64
    del eg
    torch.cuda.empty_cache()
    reads_pin = torch.from_numpy(rs.reads).view(-1).pin_memory()
    off_np = np.arange(R + 1, dtype=np.uint64) * np.uint64(L)
    off_pin = torch.from_numpy(off_np.view(np.int64)).pin_memory()
    params = api.default_params(rs.nreads1)
    ctx = api.Context(0)
    out = {"config": name, "positions": n, "reads": int(R), "read_length": int(L)}
    try:
        rec10 = torch.empty(m_bound * 10, dtype=torch.uint8, pin_memory=True).numpy()
        evbuf = (api.Event * (n // 2000 + 100_000))()
        host_res, t_host = timed(lambda: ctx.pipeline_host(host_rec, n, reads_pin, off_pin, params, 16, 2, 4, 4, 4, rec10=rec10, events=evbuf),
                                 reps, torch)
        want = outputs(host_res, rec10, evbuf)
        del host_rec
        torch.cuda.empty_cache()
        with PeakMemory(torch, dev) as pk:
            reads_res, t_reads = timed(lambda: ctx.pipeline_reads(reads_pin.numpy(), off_np, params, 16, 2, 4, 4, 4, rec10=rec10, events=evbuf),
                                       reps, torch)
        got = outputs(reads_res, rec10, evbuf)
        out.update(host_call_s=t_host, reads_call_s=t_reads, peak_device_bytes_reads_call=pk.peak,
                   same_outputs=got == want, same_counts=got[0] == want[0], n_written=want[0][0], n_clust_out=want[0][1],
                   n_candidates=int(host_res.snp.n_candidates), n_variants=int(host_res.snp.n_variants),
                   reads_h2d_bytes=int(reads_res.h2d_bytes), host_h2d_bytes=int(host_res.h2d_bytes))
        # the build alone and the step alone, on a shard of our own (the context's cached one is released first)
        ctx.close()
        torch.cuda.empty_cache()
        ctx = api.Context(0)
        ctx.stage_reads(reads_pin.numpy(), off_np)
        sh = ctx.shard(n)
        free_before, _ = torch.cuda.mem_get_info(dev)
        whole_need = n * (33 if os.environ.get("E2S_BUILD_IDS64") else 25) + rs.reads.size / 2
        builds = []

        def build():
            l0 = ctx.launches
            sh.build_egsa(off_np, 4, 4, 4)
            sh.seal()
            builds.append(ctx.launches - l0)
        _, t_build = timed(build, reps, torch)
        _, t_step = timed(lambda: sh.pipeline_resident(params, 16, 2), reps, torch)
        out.update(build_s=t_build, step_s=t_step, build_launches=builds[-1], free_bytes_before_build=int(free_before),
                   whole_build_scratch_bytes=int(whole_need), build_path="whole" if whole_need <= 0.92 * free_before else "key ranges")
        sh.close()
    finally:
        ctx.close()
        torch.cuda.empty_cache()
    return out, rs


def cli_times(rs, reps):
    from ebwt2snp_b200 import synth
    bin_dir = os.path.join(ROOT, "ebwt2snp_b200", "bin")
    d = tempfile.mkdtemp(prefix="e2s_from_reads_")
    try:
        fa = os.path.join(d, "ALL.fasta")
        synth.write_fasta(fa, rs.reads)

        def run(*cmd):
            r = subprocess.run([os.path.join(bin_dir, cmd[0]), *[str(c) for c in cmd[1:]]], capture_output=True, text=True, timeout=3600)
            if r.returncode != 0:
                raise RuntimeError(f"{cmd[0]}: {r.stdout[-2000:]} {r.stderr[-2000:]}")

        def one():
            run("ebwt2snp", "-i", fa, "-n", rs.nreads1)
            return open(fa + ".clusters", "rb").read(), open(os.path.join(d, "ALL.snp"), "rb").read()

        def chain():
            run("build_gesa", "-i", fa)
            run("ebwt2clust", "-i", fa)
            run("clust2snp", "-i", fa, "-n", rs.nreads1)
            os.remove(fa + ".gesa")
            return open(fa + ".clusters", "rb").read(), open(os.path.join(d, "ALL.snp"), "rb").read()

        t1, t3 = [], []
        a = b = None
        for _ in range(reps):  # alternated, each timed whole (process start, context, files)
            t0 = time.perf_counter()
            a = one()
            t1.append(time.perf_counter() - t0)
            t0 = time.perf_counter()
            b = chain()
            t3.append(time.perf_counter() - t0)
        return {"ebwt2snp_s": t1, "three_tools_s": t3, "same_files": a == b}
    finally:
        shutil.rmtree(d, ignore_errors=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", nargs="+", default=["C2", "C3"])
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--cli", nargs="*", default=["C2"])
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_from_reads: needs a CUDA device")
    import bench
    from ebwt2snp_b200 import api
    result = {"bench": "from_reads", "gpu": gpu_info(), "configs": []}
    for name in args.configs:
        r, rs = bench_config(name, args.reps, torch, api, bench)
        if name in args.cli:
            r["cli"] = cli_times(rs, args.reps)
        result["configs"].append(r)
        print(json.dumps(r), file=sys.stderr, flush=True)
    line = json.dumps(result)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
