#!/usr/bin/env python
"""bench.py -- eBWT positions/s of the ebwt2clust + clust2snp hot path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--workload C2] [--dump-outputs DIR]

One "step" = one full pass of the hot path (cluster scan -> merge -> statistics -> per-cluster
SNP calling) over the shard(s) resident in HBM.  `value` is device-resident throughput (CUDA
events on the launch stream, max over ranks); `e2e` is the same metric through the C-ABI call a
CLI makes (e2s_pipeline_host) from pinned HOST buffers, H2D + D2H inside the timed region.
`--impl reference` times the unmodified reference binaries (oracle/_ref, single-threaded like
the reference) on a bounded sample of the same workload.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import shutil
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "ebwt_positions_per_s"
UNIT = "positions/s"
K_DEF, M_DEF = 16, 2  # ebwt2clust defaults (ref:ebwt2clust.cpp:18-19)
KERNELS = {0: "k_lcp_flags", 1: "k_cluster_emit", 2: "k_code_scan", 3: "k_cluster_exact", 4: "k_cluster_scan",
           5: "k_chunk_resolve", 6: "k_candidates", 7: "k_events", 8: "exchange (k_pack_exchange [+ ncclAllGather] + k_merge_stats)"}


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def hbm_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.index)], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for nm, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def bind_to_gpu_numa(local, torch):
    """Host staging buffers should live on the GPU's NUMA node: a pinned buffer on the far socket costs 2-4x of the
    PCIe rate (seen as 12-21 GB/s instead of 54 GB/s on some boxes).  Prefer that node for this process' memory
    (set_mempolicy MPOL_PREFERRED) and, when the container allows it, run on its CPUs."""
    info = {"gpu_node": None, "cpus_bound": False, "mempolicy": False}
    try:
        pr = torch.cuda.get_device_properties(local)
        bdf = "%04x:%02x:%02x.0" % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)
        node = int(open(f"/sys/bus/pci/devices/{bdf}/numa_node").read())
        info["gpu_node"] = node
        if node < 0:
            return info
        try:
            cpus = set()
            for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
                a, _, b = part.partition("-")
                cpus |= set(range(int(a), int(b or a) + 1))
            cpus &= os.sched_getaffinity(0)
            if cpus:
                os.sched_setaffinity(0, cpus)
                info["cpus_bound"] = True
        except Exception:
            pass
        try:
            libc = C.CDLL(None, use_errno=True)
            mask = C.c_ulong(1 << node)
            rc = libc.syscall(238, 1, C.byref(mask), C.c_ulong(64))  # set_mempolicy(MPOL_PREFERRED, {node})
            info["mempolicy"] = rc == 0
        except Exception:
            pass
    except Exception:
        pass
    return info


def h2d_probe(torch, dev, mb=1024):
    """pinned host -> device copy rate of this box right now (GB/s), for reading the e2e number"""
    a = torch.empty(mb << 20, dtype=torch.uint8, pin_memory=True)
    b = torch.empty(mb << 20, dtype=torch.uint8, device=dev)
    b.copy_(a, non_blocking=True)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(2):
        b.copy_(a, non_blocking=True)
    torch.cuda.synchronize()
    return 2 * a.numel() / (time.perf_counter() - t0) / 1e9


# --------------------------------------------------------------------------------------------
# data
# --------------------------------------------------------------------------------------------

def make_dataset(workload, seed, scale, device, builder="torch"):
    """builder: "torch" = synth.build_egsa (plain torch sorts, the independent check of the library's builder, needs
    ~65 B of device memory per suffix); "native" = the library's e2s_build_egsa_dev (37 B per suffix incl. its outputs:
    what makes a C3-size index, 3.9e9 suffixes, fit one GPU)."""
    import torch
    from ebwt2snp_b200 import synth
    t0 = time.time()
    rs = synth.make_config(workload, seed=seed, scale=scale)
    t1 = time.time()
    if builder == "native":
        from ebwt2snp_b200 import api
        torch.cuda.empty_cache()
        bctx = api.Context(torch.device(device).index or 0)
        try:
            eg = bctx.build_egsa(rs.reads)
        finally:
            bctx.close()
    else:
        eg = synth.build_egsa(rs.reads, device=device)
    eg["build_seconds"] = time.time() - t1
    log(f"[data] {workload} scale={scale} seed={seed}: reads={rs.reads.shape} in {t1 - t0:.1f}s, n={eg['n']} built on {device} "
        f"by the {builder} builder in {eg['build_seconds']:.1f}s")
    return rs, eg


def check_egsa_sample(rs, eg, samples=200000, seed=7):
    """Size-independent property check of an index nobody else can build at this size: for sampled i, record i-1 sorts
    before record i (`$` < A < C < G < T, equal suffixes by read id), lcp[i] is their common prefix (capped at the shorter
    suffix) and bwt / text / suff agree with the reads.  Host-side numpy on the sample; -> (ok, records checked)."""
    import torch
    n, L = int(eg["n"]), int(eg["L"])
    rng = np.random.default_rng(seed)
    idx = np.unique(np.concatenate([rng.integers(1, n, size=samples), np.arange(1, min(n, 2000)), np.arange(max(1, n - 2000), n)]))
    it = torch.from_numpy(idx).to(eg["text"].device)

    def pick(k, off):
        return eg[k][it - off].cpu().numpy().astype(np.int64) & 0xFFFFFFFF

    t1, s1, t0, s0, lcp = pick("text", 0), pick("suff", 0), pick("text", 1), pick("suff", 1), pick("lcp", 0)
    bwt = eg["bwt"][it].cpu().numpy()
    reads = rs.reads
    cols = np.arange(L + 1)[None, :]

    def suffixes(t, sf):  # suffix strings, 0-padded (0 = the terminator, smaller than every base)
        out = np.zeros((len(t), L + 1), dtype=np.uint8)
        pos = sf[:, None] + cols
        valid = pos < L
        out[valid] = reads[np.broadcast_to(t[:, None], pos.shape)[valid], pos[valid]]
        return out

    a, b = suffixes(t0, s0), suffixes(t1, s1)
    diff = a != b
    differs = diff.any(axis=1)
    first = np.where(differs, diff.argmax(axis=1), L + 1)
    ok = bool(np.array_equal(np.minimum(first, np.minimum(L - s0, L - s1)), lcp))
    rows, at = np.arange(len(idx)), np.minimum(first, L)
    ok &= bool(np.where(differs, a[rows, at] < b[rows, at], t0 < t1).all())
    ok &= bool(np.array_equal(np.where(s1 > 0, reads[t1, np.maximum(s1, 1) - 1], ord("$")).astype(np.uint8), bwt))
    ok &= bool((s1 <= L).all() and (t1 < reads.shape[0]).all())
    return ok, len(idx)


def aos_records_pinned(eg, torch, lo=0, hi=None, chunk=1 << 26):
    """13-byte .gesa records (text suff lcp bwt) of positions [lo, hi) in pinned host memory, interleaved on the device
    in bounded chunks (a C3-size index is 50 GB of records)."""
    hi = int(eg["n"]) if hi is None else hi
    n = hi - lo
    dev = eg["lcp"].device
    host = torch.empty(n * 13, dtype=torch.uint8, pin_memory=True)
    rec = torch.empty((min(chunk, n), 13), dtype=torch.uint8, device=dev)
    for a in range(lo, hi, chunk):
        b = min(hi, a + chunk)
        r = rec[: b - a]
        r[:, 0:4] = eg["text"][a:b].view(torch.uint8).view(b - a, 4)
        r[:, 4:8] = eg["suff"][a:b].view(torch.uint8).view(b - a, 4)
        r[:, 8:12] = eg["lcp"][a:b].view(torch.uint8).view(b - a, 4)
        r[:, 12] = eg["bwt"][a:b]
        host[(a - lo) * 13:(b - lo) * 13].copy_(r.view(-1))
    del rec
    return host


def lcp_fits_byte(eg, torch):
    return int(eg["lcp"].max().item()) <= 127 if int(eg["n"]) else False


def soa_triple_host(eg, torch, chunk=1 << 26):
    """the index as the BCR triple: (lcp u8 pinned, bwt u8 pinned, pairSA bytes = suff(1) text(4) per position, pageable)"""
    n = int(eg["n"])
    dev = eg["lcp"].device
    lcp = torch.empty(n, dtype=torch.uint8, pin_memory=True)
    bwt = torch.empty(n, dtype=torch.uint8, pin_memory=True)
    pair = torch.empty(n * 5, dtype=torch.uint8)
    rec = torch.empty((min(chunk, n), 5), dtype=torch.uint8, device=dev)
    for a in range(0, n, chunk):
        b = min(n, a + chunk)
        r = rec[: b - a]
        r[:, 0] = eg["suff"][a:b].to(torch.uint8)
        r[:, 1:5] = eg["text"][a:b].view(torch.uint8).view(b - a, 4)
        pair[a * 5:b * 5].copy_(r.view(-1))
        lcp[a:b].copy_(eg["lcp"][a:b].to(torch.uint8))
        bwt[a:b].copy_(eg["bwt"][a:b])
    del rec
    return lcp, bwt, pair


# --------------------------------------------------------------------------------------------
# the reference arm / CPU baseline: oracle/_ref binaries on a bounded sample
# --------------------------------------------------------------------------------------------

def reference_sample(workload, seed, target_positions, device):
    """Writes a scaled-down instance of the workload (same coverage / read length) to a tmp dir."""
    from ebwt2snp_b200 import synth
    full = synth.CONFIGS[workload]
    n_full = full["reads_per_sample"] * 2 * (2 if full["rc"] else 1) * (full["L"] + 1)
    scale = min(1.0, target_positions / n_full)
    rs, eg = make_dataset(workload, seed, scale, device)
    d = tempfile.mkdtemp(prefix="e2s_ref_", dir="/dev/shm" if os.path.isdir("/dev/shm") else None)
    fasta = synth.write_dataset(d, rs, eg, fixed_headers=True)
    return d, fasta, rs, eg, scale


def run_reference_once(fasta, nreads1):
    from oracle import oracle as O
    t0 = time.perf_counter()
    r1, ncl = O.ref_ebwt2clust(fasta)  # defaults -k 16 -m 2, -x 4 -y 4 -z 4
    t1 = time.perf_counter()
    r2, info = O.ref_clust2snp(fasta, nreads1)
    t2 = time.perf_counter()
    if r1.returncode != 0 or info["returncode"] != 0:
        raise RuntimeError(f"reference failed: {r1.returncode} {info}")
    return t1 - t0, t2 - t1, ncl, info


def cpu_baseline_leg(args, device, check_ctx=None):
    """Times the reference on a bounded sample; optionally checks the CUDA path on the same files."""
    from oracle import oracle as O
    if not O.ref_available():
        return {"value": None, "unit": UNIT, "cores": 0, "kind": "reference", "sample": "oracle/_ref missing"}
    d, fasta, rs, eg, scale = reference_sample(args.workload, args.seed + 1000, args.cpu_positions or 1.2e8, device)
    try:
        n = int(eg["n"])
        tc, ts, ncl, info = run_reference_once(fasta, rs.nreads1)
        out = {"value": n / (tc + ts), "unit": UNIT, "cores": 1, "kind": "reference",
               "host_cores_total": os.cpu_count(),
               "sample": f"{args.workload} scaled x{scale:.4f}: n={n} positions, ebwt2clust {tc:.2f}s + clust2snp {ts:.2f}s "
                         f"(oracle/_ref, 1 thread: the reference is single-threaded)",
               "ebwt2clust_positions_per_s": n / tc, "clust2snp_positions_per_s": n / ts}
        if check_ctx is not None:
            from ebwt2snp_b200 import api
            sh = check_ctx.shard(n)
            sh.load_soa(eg["lcp"], eg["text"], eg["suff"], eg["bwt"], device=True)
            sh.seal()
            sh.cluster_lm(K_DEF, M_DEF)
            same_cl = sh.cluster_fetch_packed() == open(fasta + ".clusters", "rb").read()
            p = api.default_params(rs.nreads1)
            st = sh.statistics(p.mcov_out, p.pval)
            check_ctx.stage_reads(rs.reads, O.uniform_read_offsets(*rs.reads.shape))
            sh.find_events(p, st.max_clust_length)
            snp = api.events_format(sh.events(), p)
            same_snp = snp == open(os.path.join(d, "ALL.snp"), "rb").read()
            out["parity_vs_reference_on_sample"] = bool(same_cl and same_snp)
            sh.close()
        out["cli"] = cli_leg(fasta, d, rs.nreads1, n, tc, ts)
        return out
    finally:
        shutil.rmtree(d, ignore_errors=True)


def cli_leg(fasta, d, nreads1, n, ref_tc, ref_ts):
    """The drop-in boundary itself (SURVEY.md 8(b)): this repository's ebwt2clust + clust2snp as processes on the files the
    reference just ran on (in /dev/shm), wall clock incl. process start and CUDA context creation; outputs compared."""
    bin_dir = os.path.join(ROOT, "ebwt2snp_b200", "bin")
    if not all(os.access(os.path.join(bin_dir, t), os.X_OK) for t in ("ebwt2clust", "clust2snp")):
        return None
    snp = os.path.join(d, "ALL.snp")
    ref_cl, ref_snp = open(fasta + ".clusters", "rb").read(), open(snp, "rb").read()
    runs, same = [], True
    for _ in range(3):  # context creation in a fresh process is noisy (0.24 - 1.2 s on the same box): best of three, all reported
        os.remove(fasta + ".clusters")
        os.remove(snp)
        t0 = time.perf_counter()
        r1 = subprocess.run([os.path.join(bin_dir, "ebwt2clust"), "-i", fasta, "-x", "4", "-y", "4", "-z", "4"], capture_output=True)
        t1 = time.perf_counter()
        r2 = subprocess.run([os.path.join(bin_dir, "clust2snp"), "-i", fasta, "-n", str(nreads1), "-x", "4", "-y", "4", "-z", "4"], capture_output=True)
        t2 = time.perf_counter()
        same = same and (r1.returncode == 0 and r2.returncode == 0 and open(fasta + ".clusters", "rb").read() == ref_cl and
                         open(snp, "rb").read() == ref_snp)
        runs.append((t1 - t0, t2 - t1))
        if not same:
            break
    tc, ts = min(runs, key=lambda r: r[0] + r[1])
    return {"positions": n, "ebwt2clust_s": tc, "clust2snp_s": ts, "positions_per_s": n / (tc + ts),
            "runs_s": [[round(a, 3), round(b, 3)] for a, b in runs],
            "reference_ebwt2clust_s": ref_tc, "reference_clust2snp_s": ref_ts, "speedup_vs_reference": (ref_tc + ref_ts) / (tc + ts),
            "outputs_identical": bool(same),
            "note": "wall clock of the two processes (best of 3 runs, all listed), files in /dev/shm, process start + CUDA context creation "
                    "(0.24 - 1.2 s per process on this pool) included; the index is read from the file through a pinned ring (e2s_shard_load_gesa_fd)"}


def reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import oracle as O
    if not O.ref_available():
        print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref binaries missing"}))
        return
    device = "cpu"  # the reference arm needs no GPU: its sample index is built by the torch sorts on the host
    d, fasta, rs, eg, scale = reference_sample(args.workload, args.seed + 1000, args.cpu_positions or 3e7, device)
    try:
        n = int(eg["n"])
        for _ in range(args.warmup):
            run_reference_once(fasta, rs.nreads1)
        t0 = time.perf_counter()
        tcs = tss = 0.0
        for _ in range(args.steps):
            tc, ts, _, _ = run_reference_once(fasta, rs.nreads1)
            tcs += tc
            tss += ts
        dt = time.perf_counter() - t0
        v = n * args.steps / dt
        sample = (f"{args.workload} scaled x{scale:.4f}: n={n} positions per step, ebwt2clust {tcs / args.steps:.2f}s + "
                  f"clust2snp {tss / args.steps:.2f}s per step (oracle/_ref, 1 thread: the reference is single-threaded)")
        print(json.dumps({
            "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u32", "data": "synthetic",
            "config": {"workload": workload_name(args), "sample_positions": n},
            "cpu_baseline": {"value": v, "unit": UNIT, "cores": 1, "kind": "reference", "sample": sample,
                             "host_cores_total": os.cpu_count()},
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        }))
    finally:
        shutil.rmtree(d, ignore_errors=True)


def workload_name(args):
    from ebwt2snp_b200 import synth
    c = synth.CONFIGS[args.workload]
    return (f"{args.workload}: synthetic {c['G']} bp genome, 2 samples x {c['reads_per_sample']} reads of {c['L']} bp"
            f"{' + reverse complements' if c['rc'] else ''}, {c['n_snps']} SNPs, {c['n_indels']} indels; "
            f"ebwt2clust -k 16 -m 2, clust2snp defaults, -x 4 -y 4 -z 4")


# --------------------------------------------------------------------------------------------
# the B200 arm
# --------------------------------------------------------------------------------------------

def bench_c4_streamed(args, torch, dist, api, sharding, rank, world, local, dev):
    """BASELINE config 4 (1.21e11 positions: more than the HBM of the box holds as records) in the mode built for it: every
    GPU STREAMS its contiguous range through a chunked shard -- a chunk is a shard in time -- and the ranks exchange their
    summaries once at the end.  The eBWT is the C2 index tiled with shifted read ids (SURVEY.md section 7); chunks are
    produced on the device just before they are loaded (outside the timed regions: the 1.58 TB of records exist nowhere),
    so the line measures the streaming machinery itself: chunk load (13 B/position copied + narrow copies derived), scan
    with carried state, capture of the survivors, exchange, phase 2."""
    rs, eg = make_dataset("C2", args.seed, args.scale, dev)
    n_tile, R0 = int(eg["n"]), rs.reads.shape[0]
    full = synth_positions("C4")
    T_total = max(world, int(round(full * args.scale / n_tile))) if args.tiles <= 1 else args.tiles * world
    n_global = T_total * n_tile
    cuts = sharding.shard_cuts(n_global, world)
    lo, hi = cuts[rank], cuts[rank + 1]
    stream = torch.cuda.Stream(device=dev)
    ctx = api.Context(local, stream.cuda_stream)
    chunk_positions = int(os.environ.get("E2S_CHUNK_POSITIONS", 1 << 27))
    params = api.default_params(rs.nreads1)
    reads_dev = torch.from_numpy(rs.reads).to(dev).contiguous().view(-1)  # only tile 0 holds reads of sample 1: candidates come from it
    L = rs.reads.shape[1]
    off_dev = torch.arange(R0 + 1, dtype=torch.int64, device=dev) * L
    ctx.stage_reads(reads_dev, off_dev, device=True, n_bases=R0 * L)
    comm = sharding.make_comm(ctx, dev) if world > 1 else None
    # what the totals must be: tiles repeat, so written(T) is linear in T -- from two small resident runs (rank 0's GPU)
    expect = None
    if rank == 0:
        w = {}
        for T in (2, 3):
            s2 = ctx.shard(T * n_tile)
            for t in range(T):
                s2.load_soa(eg["lcp"], eg["text"] + t * R0 if t else eg["text"], eg["suff"], eg["bwt"], first=t * n_tile, device=True)
            s2.seal()
            w[T] = s2.cluster_lm(K_DEF, M_DEF)
            s2.close()
        expect = tuple(w[2][i] + (T_total - 2) * (w[3][i] - w[2][i]) for i in range(2))
        torch.cuda.empty_cache()

    def gen(a, b):
        idx = torch.arange(a, b, dtype=torch.int64, device=dev)
        t = idx // n_tile
        i = idx - t * n_tile
        text = (eg["text"][i].to(torch.int64) + t * R0).to(torch.int32)
        return eg["lcp"][i], text, eg["suff"][i], eg["bwt"][i]

    sh = ctx.shard(hi - lo, lo, n_global, chunk_positions=chunk_positions)

    def one_pass():
        """-> (device ms inside the library calls, merged, stats, counts)"""
        sh.chunked_reset()
        ms = 0.0
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        for clo, cn in sh.chunks():
            a, b = max(0, clo - 176), min(n_global, clo + cn + 152)
            arrs = gen(a, b)
            torch.cuda.synchronize()
            e0.record(stream)
            sh.chunk_begin(clo, cn)
            sh.load_soa(*arrs, first=a, device=True)
            sh.chunk_scan(K_DEF, M_DEF, params.mcov_out)
            e1.record(stream)
            torch.cuda.synchronize()
            ms += e0.elapsed_time(e1)
            del arrs
        e0.record(stream)
        if comm is not None:
            mg, st = sh.chunked_exchange(comm, K_DEF, M_DEF, params.mcov_out, params.pval)
        else:
            sm = sh.chunked_finish(K_DEF, M_DEF)
            mg = api.cluster_merge([sm], 0)
            sh.cluster_finalize(mg)
            st = sh.statistics(params.mcov_out, params.pval)
        cnt = sh.find_events(params, st.max_clust_length)
        e1.record(stream)
        torch.cuda.synchronize()
        ms += e0.elapsed_time(e1)
        return ms, mg, st, cnt

    with torch.cuda.stream(stream):
        for _ in range(max(1, min(args.warmup, 1))):
            one_pass()
        if world > 1:
            dist.barrier()
        sampler = ClockSampler(local)
        sampler.start()
        launches0 = ctx.launches
        t_wall = time.perf_counter()
        tot_ms = 0.0
        for _ in range(args.steps):
            ms, mg, st, cnt = one_pass()
            tot_ms += ms
        wall = time.perf_counter() - t_wall
        clocks = sampler.stop()
    launches = ctx.launches - launches0
    ncand = int(cnt.n_candidates)
    if world > 1:
        t = torch.tensor([tot_ms, float(ncand)], dtype=torch.float64, device=dev)
        tm = t.clone()
        dist.all_reduce(tm, op=dist.ReduceOp.MAX)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        tot_ms, ncand = float(tm[0].item()), int(t[1].item())
    if rank == 0:
        peak, peak_src = hbm_peak()
        per_step = tot_ms / args.steps
        ok = expect is not None and (int(mg.total_written), int(mg.n_clust_out)) == expect
        print(json.dumps({
            "metric": METRIC, "value": n_global / (per_step * 1e-3), "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": 1, "ms_per_step": per_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "u32",
            "data": "synthetic",
            "config": {"workload": workload_name_of("C4") + f"; STREAMED as {T_total} tiles of the C2 index ({n_tile} positions each, read ids shifted) "
                                   f"through chunked shards of {sh.chunk_positions} positions",
                       "positions_total": n_global, "positions_per_gpu": hi - lo, "chunk_positions": sh.chunk_positions,
                       "resident_bytes_per_gpu": int(sh.chunk_positions * 14.6),
                       "timed": "CUDA events around the library calls of every chunk (begin, device-to-device load + narrow copies, scan, capture) "
                                "and around the exchange + phase 2; producing the tile arrays on the device is outside (the 1.58 TB of records exist nowhere)",
                       "wall_s_per_step_incl_tile_production": wall / args.steps,
                       "l2": "every chunk (>= 1.9 GB of resident arrays) exceeds the 126 MB L2"},
            "clocks": clocks, "e2e": None, "gpu_launches": int(launches),
            "roofline": {"bound": "hbm", "kernel": "chunk load + k_cluster_scan", "achieved": n_global / world * (2 * 13 + 1.375 + 1.25) / (per_step * 1e-3) / 1e9,
                         "peak": peak, "unit": "GB/s", "frac": n_global / world * (2 * 13 + 1.375 + 1.25) / (per_step * 1e-3) / 1e9 / peak, "traffic": None,
                         "peak_source": peak_src,
                         "note": "per position: 13 B copied device to device (read + write) + 5 B re-read and 1.375 B written by k_derive "
                                 "(counted as 1.375 here) + 1.25 B read by the scan"},
            "cpu_baseline": None,
            "results": {"n_written": int(mg.total_written), "n_clust_out": int(mg.n_clust_out), "max_clust_length": int(st.max_clust_length),
                        "n_candidates": ncand, "totals_match_linear_extrapolation_of_resident_runs": bool(ok), "expected": expect},
        }))
    sh.close()
    if world > 1:
        dist.destroy_process_group()


DUMP_CLUSTER_SAMPLE = 1 << 20   # cluster records kept by --dump-outputs (20 B each as float64 index / start + float32 length)
DUMP_EVENT_BYTES = 40 << 20     # budget of the events' arrays


def dump_outputs(out_dir, counts, start, ln, events, event_type, seed=0):
    """--dump-outputs: what one step of the timed path hands its caller, as float .npy files in out_dir (under 63 MB).
    counts: {name: int} of the step's result; start / ln: the .clusters records; events: event_type (api.Event) list in
    .snp order.
    Larger outputs are cut to a sample that depends only on their size (seeded), so two builds of the project that compute
    the same outputs dump the same files."""
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"counts": np.array([counts[k] for k in sorted(counts)], dtype=np.float64)}  # in the order of the names
    m = len(ln)
    idx = np.arange(m, dtype=np.int64)
    if m > DUMP_CLUSTER_SAMPLE:
        idx = np.sort(np.random.default_rng(seed).choice(m, size=DUMP_CLUSTER_SAMPLE, replace=False))
    arrays["cluster_index"] = idx.astype(np.float64)
    arrays["cluster_start"] = np.asarray(start, dtype=np.uint64)[idx].astype(np.float64)
    arrays["cluster_len"] = np.asarray(ln)[idx].astype(np.float32)
    n_ev = len(events)
    ev = {f: np.array([getattr(e, f) for e in events], dtype=np.int64) for f in
          ("cluster_start", "D", "gap", "supp0", "supp1", "right_len", "keep")}
    raw = np.frombuffer(b"".join(bytes(e) for e in events), dtype=np.uint8).reshape(n_ev, C.sizeof(event_type))
    ctx = {f: raw[:, getattr(event_type, f).offset:getattr(event_type, f).offset + getattr(event_type, f).size]
           for f in ("left0", "left1", "right")}
    width = max(int(np.flatnonzero(c.any(axis=0)).max()) + 1 if c.any() else 0 for c in ctx.values())  # the rest is 0
    keep = np.arange(n_ev)
    per_event = 2 * 8 + 6 * 4 + 3 * 4 * width
    if n_ev * per_event > DUMP_EVENT_BYTES:
        keep = np.sort(np.random.default_rng(seed + 1).choice(n_ev, size=DUMP_EVENT_BYTES // per_event, replace=False))
    arrays["event_index"] = keep.astype(np.float64)
    arrays["event_cluster_start"] = ev["cluster_start"][keep].astype(np.float64)
    arrays["event_fields"] = np.stack([ev[f][keep] for f in ("D", "gap", "supp0", "supp1", "right_len", "keep")], axis=1).astype(np.float32).reshape(-1, 6)
    for f, c in ctx.items():
        arrays[f"event_{f}"] = c[keep, :width].astype(np.float32)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)
    return arrays


def synth_positions(name):
    from ebwt2snp_b200 import synth
    c = synth.CONFIGS[name]
    return c["reads_per_sample"] * 2 * (2 if c["rc"] else 1) * (c["L"] + 1)


def workload_name_of(name):
    from ebwt2snp_b200 import synth
    c = synth.CONFIGS[name]
    return (f"{name}: synthetic {c['G']} bp genome, 2 samples x {c['reads_per_sample']} reads of {c['L']} bp"
            f"{' + reverse complements' if c['rc'] else ''}, {c['n_snps']} SNPs, {c['n_indels']} indels; "
            f"ebwt2clust -k 16 -m 2, clust2snp defaults, -x 4 -y 4 -z 4")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="C3", help="C3 = the configuration BASELINE.json's metric is quoted on (config 5 = C3 at 1/2/4/8 GPUs)")
    ap.add_argument("--scale", type=float, default=1.0, help="shrink the workload (debugging only)")
    ap.add_argument("--seed", type=int, default=1)
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--cpu-positions", type=float, default=None,
                    help="size of the CPU-baseline sample (default: 1.2e8 positions = about 11 s of reference time; the reference arm, "
                         "which builds its sample on the host, uses 3e7)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--scaling", default="strong", choices=["weak", "strong"],
                    help="N > 1: strong (default) = ONE workload cut into N contiguous eBWT ranges (BASELINE config 5 = C3 at 1/2/4/8 "
                         "GPUs); weak = one workload per GPU, glued end to end")
    ap.add_argument("--builder", default="auto", choices=["auto", "torch", "native"],
                    help="who builds the workload's index (data preparation): auto = torch for C1/C2 (and the library's builder is checked "
                         "against it), the library's own builder for C3-size workloads")
    ap.add_argument("--no-egsa-build", action="store_true", help="skip timing the library's EGSA builder on the workload's reads (N = 1 only)")
    ap.add_argument("--tiles", type=int, default=1,
                    help="resident-only study: tile the workload T times on the GPU (read ids shifted; every tile starts with "
                         "lcp = 0), e.g. --tiles 8 = 4.46e9 positions, C3/C4-sized shards; implies --no-e2e --no-cpu-baseline")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed (result counts, a seeded sample of the "
                         ".clusters records, the events) as DIR/<name>.npy, float32 / float64, under 63 MB: the same arguments "
                         "give the same inputs, so two builds can be compared output for output.  With N > 1 the counts are "
                         "global, the records and events rank 0's shard only.  The resident path only: not with --workload C4 "
                         "(streamed) or --impl reference")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl == "reference" or args.workload == "C4"):
        raise SystemExit("--dump-outputs covers the resident B200 path (--impl b200, workloads C1 - C3)")
    if args.impl == "reference":
        return reference_arm(args)

    import torch
    import torch.distributed as dist

    from ebwt2snp_b200 import api, sharding

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: there is no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    numa = bind_to_gpu_numa(local, torch)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    warmup = max(args.warmup, 3)
    if args.workload == "C4":
        return bench_c4_streamed(args, torch, dist, api, sharding, rank, world, local, dev)

    # ---- data: every rank owns one C2-size tile of a global eBWT of world * n positions (weak scaling) ----
    big = args.workload not in ("C1", "C2") and args.scale >= 0.5  # beyond what the torch builder fits on one GPU
    builder = args.builder if args.builder != "auto" else ("native" if big else "torch")
    # weak scaling (default): every rank owns its own workload-size tile of a global eBWT of world * n positions;
    # strong scaling (--scaling strong; BASELINE config C5): ONE workload, every rank builds the same index and keeps its
    # contiguous range of it
    strong = args.scaling == "strong" and world > 1
    rs, eg = make_dataset(args.workload, args.seed if strong else args.seed + rank, args.scale, dev, builder=builder)
    index_check = None
    if builder == "native":
        okc, nchk = check_egsa_sample(rs, eg)
        index_check = {"builder": "e2s_build_egsa_dev (the library's own radix sort)", "sampled_records": nchk, "order_lcp_bwt_consistent": okc,
                       "suffixes": int(eg["n"]), "build_seconds_incl_h2d_of_the_reads": eg["build_seconds"],
                       "suffixes_per_s": int(eg["n"]) / max(eg["build_seconds"], 1e-9)}
        log(f"[data] index property check on {nchk} sampled records: {okc}")
        if not okc:
            raise SystemExit("the index built by the library fails the order / LCP / BWT property check")
        args.no_egsa_build = True
    # ---- EGSA construction on the GPU (SURVEY.md 8(f) rank 1; data preparation, outside the timed step): the library's
    # builder on the same reads, timed, and compared element by element with the arrays the step below runs on ----
    egsa_build = None
    if not args.no_egsa_build and world == 1:
        from ebwt2snp_b200 import api as _api
        bctx = _api.Context(local)
        try:
            reads_t = torch.from_numpy(rs.reads).to(dev)
            bctx.build_egsa(reads_t[: max(1, min(1000, reads_t.shape[0]))])  # warm-up (allocator, module load)
            torch.cuda.synchronize()
            tb = time.perf_counter()
            mine = bctx.build_egsa(reads_t)
            tb = time.perf_counter() - tb
            same = all(bool(torch.equal(mine[k], eg[k])) for k in ("lcp", "text", "suff", "bwt"))
            egsa_build = {"suffixes": int(mine["n"]), "seconds": tb, "suffixes_per_s": mine["n"] / tb,
                          "equals_torch_builder": same, "api": "e2s_build_egsa_dev (2-bit keys, the library's own 8-bit radix passes per 64-bit key word)"}
            log(f"[egsa] native builder: {mine['n']} suffixes in {tb:.3f}s, equal to the torch builder: {same}")
            del mine, reads_t
        finally:
            bctx.close()
        torch.cuda.empty_cache()
    T = max(1, args.tiles)
    if T > 1:
        args.no_e2e = args.no_cpu_baseline = True
        if world > 1:
            raise SystemExit("--tiles is a single-GPU study")
    n_tile = int(eg["n"])
    n = n_tile * T
    n_all = [n]
    if strong:
        if T > 1:
            raise SystemExit("--tiles and --scaling strong do not combine")
        cuts = sharding.shard_cuts(n_tile, world)
        n_all = [cuts[g + 1] - cuts[g] for g in range(world)]
        n = n_all[rank]
    elif world > 1:
        t = torch.tensor([n], dtype=torch.int64, device=dev)
        g = [torch.zeros_like(t) for _ in range(world)]
        dist.all_gather(g, t)
        n_all = [int(x.item()) for x in g]
    global_off, n_global = sum(n_all[:rank]), sum(n_all)

    stream = torch.cuda.Stream(device=dev)
    ctx = api.Context(local, stream.cuda_stream)
    sh = ctx.shard(n, global_off, n_global)
    R0 = rs.reads.shape[0]
    if strong:  # my range of the one index, halos included (2 left, 151 right): every rank holds the whole index here
        a, b = max(0, global_off - sharding.HALO_L), min(n_global, global_off + n + sharding.HALO_R)
        sh.load_soa(eg["lcp"][a:b], eg["text"][a:b], eg["suff"][a:b], eg["bwt"][a:b], first=a, device=True)
        left = right = None
    else:
        for t in range(T):
            sh.load_soa(eg["lcp"], eg["text"] + t * R0 if t else eg["text"], eg["suff"], eg["bwt"], first=global_off + t * n_tile, device=True)
        # halo exchange over NCCL: my left neighbour's last 2 records, my right neighbour's first 151
        left, right = sharding.exchange_halo(eg["lcp"], eg["text"], eg["suff"], eg["bwt"], dev)
    if left is not None:
        sh.load_soa(left["lcp"], left["text"], left["suff"], left["bwt"], first=global_off - sharding.HALO_L, device=True)
    if right is not None:
        sh.load_soa(right["lcp"], right["text"], right["suff"], right["bwt"], first=global_off + n, device=True)
    torch.cuda.synchronize()
    t_seal = time.perf_counter()
    sh.seal()  # (the loads wrote the bit-sliced LCP and the base-code planes themselves: no kernel over the data here, see k_derive)
    seal_ms = 1e3 * (time.perf_counter() - t_seal)
    reads_dev = torch.from_numpy(rs.reads).to(dev)
    if T > 1:
        reads_dev = reads_dev.repeat(T, 1)
    reads_dev = reads_dev.contiguous().view(-1)
    R, L = rs.reads.shape[0] * T, rs.reads.shape[1]
    off_dev = (torch.arange(R + 1, dtype=torch.int64, device=dev) * L)
    ctx.stage_reads(reads_dev, off_dev, device=True, n_bases=R * L)
    params = api.default_params(rs.nreads1)

    host_rec = None
    rec_first = 0
    if not args.no_e2e:
        if strong:  # one eBWT from host buffers over the ranks: every rank stages ITS range + halos only
            rec_first, rec_end = max(0, global_off - 176), min(n_global, global_off + n + 152)
            host_rec = aos_records_pinned(eg, torch, rec_first, rec_end)
        else:
            host_rec = aos_records_pinned(eg, torch)
    # the same index as the BCR triple (ref:include.hpp:157-188) at BCR's usual widths: X.out.lcp 1 byte, X.out 1 byte (both pinned:
    # they cross PCIe), X.out.pairSA = suff(1) + text(4) in ordinary host memory (only the host reads it)
    host_soa = None
    if not args.no_e2e and world == 1 and lcp_fits_byte(eg, torch):
        host_soa = soa_triple_host(eg, torch)
    # generator arrays are no longer needed on the device
    for kk in ("lcp", "text", "suff", "bwt"):
        eg[kk] = None
    torch.cuda.empty_cache()

    # N > 1: the library's own NCCL communicator (one C call per step); E2S_PY_EXCHANGE=1 keeps the torch.distributed exchange
    comm = sharding.make_comm(ctx, dev) if (world > 1 and not os.environ.get("E2S_PY_EXCHANGE")) else None

    def step():
        """one pass of the hot path over the resident shard(s): K1, K2, summaries all-gather + merge, statistics
        all-gather, K3a/K3x/K3b/K4, event-count all-gather (ebwt2snp_b200/sharding.py)"""
        if world == 1:  # the same sequence inside the library: one C call, no Python between the kernels
            return sh.pipeline_resident(params, K_DEF, M_DEF)
        mg, st, cnt, ids = sharding.hot_path_step(sh, params, K_DEF, M_DEF, dev, comm=comm)
        step.ids = ids  # global .snp ids are assigned when the text is formatted: resolved after the timed loop
        return mg, st, cnt

    def sync_all():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    with torch.cuda.stream(stream):
        for _ in range(warmup):
            out = step()
        sync_all()
        ctx.timing(True)
        for kid in KERNELS:
            ctx.kernel_time(kid)
        launches0 = ctx.launches
        sampler = ClockSampler(local)
        sampler.start()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        sync_all()
        ev0.record(stream)
        for _ in range(args.steps):
            out = step()
        ev1.record(stream)
        sync_all()
        ms = ev0.elapsed_time(ev1)
        # the timed region lasts a few milliseconds, less than one nvidia-smi sampling period: the same steps continue
        # untimed (~0.6 s) so that the clock / throttle samples are taken under the load that was timed
        ktimes = {kid: ctx.kernel_time(kid) for kid in KERNELS}
        launches = ctx.launches - launches0
        ctx.timing(False)
        if args.dump_outputs and rank == 0:
            if world == 1:
                counts = {"n_written": out.n_written, "n_clust_out": out.n_clust_out, "max_clust_length": out.max_clust_length}
                snp = out.snp
            else:
                counts = {"n_written": out[0].total_written, "n_clust_out": out[0].n_clust_out, "max_clust_length": out[1].max_clust_length}
                snp = out[2]
            counts.update({f: getattr(snp, f) for f, _ in api.SnpCounts._fields_})
            dumped = (counts, *sh.cluster_fetch(), sh.events())  # fetched here, written once the clocks are sampled
        n_soak = 1000 if T == 1 else 150  # a fixed count: every rank must run the same number of (collective) steps
        for _ in range(n_soak):
            step()
        sync_all()
        clocks = sampler.stop()
        clocks["window"] = f"timed region + {n_soak} more of the same steps, untimed"
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, *dumped, api.Event, seed=args.seed)
        del dumped
        log(f"[dump] outputs of the last timed step written to {args.dump_outputs}")

    if world > 1:
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
        mg, st, cnt = out
        step.ids.resolve()
        # what the host-synchronised exchange between the phases costs by itself (same message size, no compute around it)
        torch.cuda.synchronize()
        probe_words = np.zeros(api.SUMMARY_WORDS + C.sizeof(api.Stats) // 8, dtype=np.uint64)
        for _ in range(3):
            sharding.all_gather_words(probe_words, dev)
        t_ex = time.perf_counter()
        for _ in range(20):
            sharding.all_gather_words(probe_words, dev)
        exchange_us = (time.perf_counter() - t_ex) / 20 * 1e6
    else:  # the one-call step returns the pipeline result; the histogram is still on the shard
        import types
        exchange_us = None
        mg = types.SimpleNamespace(total_written=out.n_written, n_clust_out=out.n_clust_out)
        cnt = out.snp
        st = sh.statistics(params.mcov_out, params.pval)
    value = n_global * args.steps / (ms * 1e-3)

    # ---- roofline of the two kernels that touch every position (this rank's shard) ----
    peak, peak_src = hbm_peak()
    m_own = sh.cluster_count()
    lcp_bytes = sh.lcp_bytes_resident()
    lo, hi = 2 * params.mcov_out, st.max_clust_length
    # positions inside analysed clusters: from the (global) histogram, scaled to this shard for world > 1
    pos_analysed = sum(int(st.hist[l]) * l for l in range(lo, hi + 1)) / world
    # algorithmic bytes per launch (DESIGN.md "Kernels"): what the kernel has to move for this shard
    fused = ktimes[api.KERNEL_SCAN][1] == 0             # K2 ran the BWT prefilter itself (e2s_cluster_prefilter): no K3a launch
    alg = {
        api.KERNEL_FLAGS: lcp_bytes * n + n / 4,        # resident LCP (1 B bit-sliced, else 4 B) read once + 2 bit masks written
        api.KERNEL_EMIT: n / 4 + 10 * m_own + (pos_analysed / 4 if fused else 0),  # masks read + records written (+ the 2-bit base codes inside analysed clusters)
        api.KERNEL_SCAN: pos_analysed / 4 + 10 * m_own,  # 2-bit base code (resident bit planes) of positions in analysed clusters + record list
        api.KERNEL_EXACT: 0,
        # K1 + K2 in one pass: the bit-sliced LCP (1 B/position) read once, the records written, the 2-bit base codes inside analysed clusters (fused prefilter)
        api.KERNEL_SCAN1: n + 10 * m_own + (pos_analysed / 4 if fused else 0),
        api.KERNEL_RESOLVE: 0, api.KERNEL_CAND: 0, api.KERNEL_EVENTS: 0, api.KERNEL_MERGE: 0,  # (latency-bound small kernels: times only)
    }
    streamed = {api.KERNEL_SCAN: n / 4 + 10 * m_own}    # the 16-byte plane loads also carry the positions outside clusters
    if fused:
        streamed[api.KERNEL_EMIT] = n / 2 + 10 * m_own + n / 4  # masks twice (count pass + write pass) + the bit planes
        streamed[api.KERNEL_SCAN1] = n + 10 * m_own + n / 4     # the whole plane array comes in with the tiles
    kern = {}
    ksum_ms = 0.0
    for kid, name in KERNELS.items():
        tot_ms, cnt_l = ktimes[kid]
        if not cnt_l:
            continue
        ksum_ms += tot_ms
        per = tot_ms / cnt_l
        kern[name] = {"ms": per, "alg_bytes": alg[kid], "GBps": alg[kid] / (per * 1e-3) / 1e9}
        if kid in streamed:
            kern[name]["streamed_bytes"] = streamed[kid]
            kern[name]["streamed_GBps"] = streamed[kid] / (per * 1e-3) / 1e9
    dom = max(kern, key=lambda kname: kern[kname]["ms"]) if kern else None
    traffic = None
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            traffic = json.load(f).get(dom)
        if isinstance(traffic, dict):  # per workload: one launch over the whole single-GPU shard of that workload
            traffic = traffic.get(args.workload) if (world == 1 and args.scale == 1.0 and T == 1) else None
    except Exception:
        pass
    roofline = None
    if dom:
        roofline = {"kernel": dom, "bound": "hbm", "achieved": kern[dom]["GBps"], "peak": peak, "unit": "GB/s",
                    "frac": kern[dom]["GBps"] / peak, "traffic": traffic, "peak_source": peak_src,
                    "ms_per_launch": kern[dom]["ms"], "alg_bytes_per_launch": kern[dom]["alg_bytes"],
                    "kernels": kern, "kernel_share_of_step": ksum_ms / ms if ms else None,
                    "fused_prefilter": bool(fused), "resident_lcp_bytes": lcp_bytes,
                    "note": "k_cluster_scan = LCP stencil (bit-sliced compare) + ranks + compaction + length histogram + BWT prefilter in one pass over the "
                            "bit-sliced LCP (1 B/position), one CTA per chunk of tiles; bound by instruction issue, not DRAM (DESIGN.md 3.1); "
                            "k_lcp_flags / k_cluster_emit only run for -m > 33 and for -k > 127 on shards with an LCP value > 127",
                    "pipeline": {"alg_bytes_per_step": sum(alg[k] for k in alg if ktimes[k][1]),
                                 "GBps": sum(alg[k] for k in alg if ktimes[k][1]) / (ms / args.steps * 1e-3) / 1e9,
                                 "frac_of_peak": sum(alg[k] for k in alg if ktimes[k][1]) / (ms / args.steps * 1e-3) / 1e9 / peak}}

    # ---- e2e: the C-ABI pipeline call from pinned host buffers, copies inside the timed region ----
    # N = 1: e2s_pipeline_host.  N > 1 (strong): ONE eBWT over the ranks, e2s_pipeline_host_sharded -- every rank streams its
    # range of the records through a chunked shard, one ncclAllGather of the summaries, phase 2 per rank.
    e2e = None
    if host_rec is not None:
        reads_pin = torch.from_numpy(rs.reads).view(-1).pin_memory()
        off_pin = (torch.arange(R + 1, dtype=torch.int64) * L).pin_memory()
        sh.close()  # free the resident shard: the pipeline call owns its own (chunked) one
        torch.cuda.empty_cache()
        rec10 = torch.empty((m_own + 64) * 10, dtype=torch.uint8, pin_memory=True)
        evbuf = (api.Event * (int(cnt.n_variants) + 16))()
        rec10_np = rec10.numpy()
        sharded_e2e = strong and comm is not None

        def e2e_call():
            if sharded_e2e:
                r3, _, _, _ = api.pipeline_host_sharded(ctx, comm, host_rec, rec_first, global_off, n, n_global, reads_pin, off_pin, params,
                                                        K_DEF, M_DEF, rec10=rec10_np, events=evbuf)
                return r3
            return ctx.pipeline_host(host_rec, n, reads_pin, off_pin, params, K_DEF, M_DEF, rec10=rec10_np, events=evbuf)

        res = e2e_call()
        sync_all()
        t0 = time.perf_counter()
        for _ in range(args.e2e_steps):
            res = e2e_call()
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        h2d_b, d2h_b = int(res.h2d_bytes), int(res.d2h_bytes)
        if world > 1:
            t = torch.tensor([dt, float(h2d_b), float(d2h_b)], dtype=torch.float64, device=dev)
            tmax = t.clone()
            dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
            dist.all_reduce(t, op=dist.ReduceOp.SUM)
            dt, h2d_b, d2h_b = float(tmax[0].item()), int(t[1].item()), int(t[2].item())
        # what the box delivers right now: pinned H2D copies on ALL ranks at the same time (what the e2e number is read against)
        sync_all()
        probe = h2d_probe(torch, dev)
        probe_sum = probe
        if world > 1:
            t = torch.tensor([probe], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.SUM)
            probe_sum = float(t.item())
        e2e = {"value": n_global * args.e2e_steps / dt, "unit": UNIT, "h2d_bytes_per_step": h2d_b,
               "h2d_probe_GBps": probe, "h2d_probe_concurrent_sum_GBps": probe_sum, "numa": numa,
               "d2h_bytes_per_step": d2h_b, "ms_per_step": 1e3 * dt / args.e2e_steps,
               "steps": args.e2e_steps,
               "api": ("e2s_pipeline_host_sharded (one eBWT over the ranks: each streams its range of the 13-byte records through a chunked shard)"
                       if sharded_e2e else "e2s_pipeline_host (13-byte .gesa records + reads in, .clusters records + events out; chunked shard)"),
               "chunk_positions": int(os.environ.get("E2S_CHUNK_POSITIONS", 1 << 28)),
               "h2d_GBps": h2d_b * args.e2e_steps / dt / 1e9,
               "fraction_of_concurrent_probe": (h2d_b * args.e2e_steps / dt / 1e9) / probe_sum if probe_sum else None,
               "n_events_rank0": int(res.snp.n_events), "n_written": int(res.n_written)}

    # ---- e2e_soa: the same job from the BCR triple, lean (e2s_pipeline_host_soa): lcp + bwt cross PCIe, text / suff of the
    # survivors only are fetched from the host's pairSA.  Same outputs as the e2e call above (compared).
    if host_soa is not None and e2e is not None:
        host_rec = None
        l8, b8, pair = host_soa
        want_rec = rec10[: int(res.n_written) * 10].clone()
        want_counts = (int(res.n_written), int(res.n_clust_out), int(res.max_clust_length), int(res.snp.n_candidates), int(res.snp.n_events))
        want_ev = api.events_format(list(evbuf)[: int(res.snp.n_variants)], params)

        def soa_call():
            return ctx.pipeline_host_soa(l8, b8, pair, n, reads_pin, off_pin, params, K_DEF, M_DEF, 1, 4, 1, rec10=rec10_np, events=evbuf)

        r2 = soa_call()
        same = (want_counts == (int(r2.n_written), int(r2.n_clust_out), int(r2.max_clust_length), int(r2.snp.n_candidates), int(r2.snp.n_events))
                and bool(torch.equal(want_rec, rec10[: int(r2.n_written) * 10]))
                and want_ev == api.events_format(list(evbuf)[: int(r2.snp.n_variants)], params))
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(args.e2e_steps):
            r2 = soa_call()
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        e2e["soa"] = {"value": n_global * args.e2e_steps / dt, "unit": UNIT, "ms_per_step": 1e3 * dt / args.e2e_steps,
                      "h2d_bytes_per_step": int(r2.h2d_bytes), "d2h_bytes_per_step": int(r2.d2h_bytes),
                      "h2d_GBps": int(r2.h2d_bytes) * args.e2e_steps / dt / 1e9,
                      "api": "e2s_pipeline_host_soa (BCR triple: X.out.lcp 1 byte + X.out cross PCIe in full; X.out.pairSA (suff 1 + text 4 bytes) stays "
                             "on the host, only the prefilter survivors' records are fetched from it)",
                      "outputs_equal_e2e": bool(same)}
        del want_rec, l8, b8, pair
        host_soa = None

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        # the CLI leg starts fresh processes on this GPU: release what this process still holds of the measured workload first
        host_rec = None
        if e2e is not None:
            rec10 = rec10_np = reads_pin = off_pin = None
        import gc
        gc.collect()
        torch.cuda.empty_cache()
        cpu = cpu_baseline_leg(args, dev, check_ctx=ctx)

    if rank == 0:
        c_ratio = m_own / n
        out = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": warmup,
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "strong" if strong else "weak", "vs_baseline": None,
            "dtype": "u32", "data": "synthetic",
            "config": {"workload": workload_name(args), "positions_per_gpu": n, "positions_total": n_global,
                       "parallelism": f"{world} contiguous eBWT shard(s), one per GPU; " + ("one ncclAllGather of the shard summaries per step, issued by the library on its stream (e2s_pipeline_sharded)" if comm is not None else ("no exchange (single shard: e2s_pipeline_resident)" if world == 1 else "torch.distributed all-gather of shard summaries")),
                       "l2": "the resident inputs a step streams (1.25 B/position, 4.25 on the 4-byte path: >= 0.7 GB per GPU at C2, 4.8 GB at C3) exceed the 126 MB L2; no flush needed",
                       "resident_layout": f"SoA: lcp u32 + text u32 + suff u32 + bwt u8; written by the loads: 2-bit base-code planes of the BWT + a bit-sliced LCP (7 bit planes + the descent plane, 1 B/position); the scan streams {'the bit-sliced copy (values above 127 saturated: exact for -k <= 127)' if lcp_bytes == 1 else 'the 4-byte LCP'}",
                       "scale": args.scale, "tiles": T, "exchange_us": exchange_us,
                       "seal": {"ms": seal_ms, "kernels_over_the_data": 0,
                                "note": "the bit-sliced LCP and the base-code planes are written by the loads (k_derive): sealing is a 4-byte read-back"}},
            "value_one_pass": n_global * args.steps / (ms * 1e-3 + args.steps * seal_ms * 1e-3),
            "clocks": clocks, "e2e": e2e, "egsa_build": egsa_build, "index_check": index_check, "gpu_launches": int(launches), "roofline": roofline, "cpu_baseline": cpu,
            "results": {"n_written": int(mg.total_written), "n_clust_out": int(mg.n_clust_out),
                        "max_clust_length": int(st.max_clust_length), "n_analysed_rank0": int(cnt.n_analysed),
                        "n_candidates_rank0": int(cnt.n_candidates), "n_events_rank0": int(cnt.n_events),
                        "clusters_per_position": c_ratio, "fraction_in_analysed_clusters": pos_analysed / n},
        }
        print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
