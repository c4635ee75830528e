"""Timing tool (not part of the library): the ragged index builder whole (e2s_build_egsa_ragged_dev) next to the same index built in
P = 2, 4 and 8 key ranges (e2s_build_egsa_ragged_range_dev, quantile cuts of sharding.key_range_cuts, each range written straight to its
place in one set of device arrays).  C2-size read set (synth config C2) trimmed to 70..100 bases with a seeded length draw.

    python scripts/bench_build_ranges.py [--scale 1.0] [--reps 3] [--seed 1] [--out FILE]

Prints one JSON line: ms per build (host clock around synchronised calls, best and median of --reps after a warm-up of every shape),
suffixes/s, the share of the selection sweeps (k_range_select, from a torch.profiler trace of one extra build per P), whether every P
gives the whole build's arrays, and the GPU's name and power limit read in the same run.  Needs a GPU; writes only --out."""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from ebwt2snp_b200 import api, sharding, synth  # noqa: E402
from ebwt2snp_b200.api import _ptr  # noqa: E402


def gpu_info():
    import torch
    info = {"gpu": torch.cuda.get_device_name(0)}
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=60)
        info["power_limit_and_max_sm_clock"] = r.stdout.strip() or r.stderr.strip()
    except OSError as e:
        info["power_limit_and_max_sm_clock"] = "not read: %s" % e
    return info


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--scale", type=float, default=1.0)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--seed", type=int, default=1)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_build_ranges: no CUDA device")
    rs = synth.make_config("C2", seed=a.seed, scale=a.scale)
    R, L = rs.reads.shape
    lens = np.random.default_rng(a.seed).integers(70, L + 1, size=R)
    bases = rs.reads[np.arange(L)[None, :] < lens[:, None]]  # row-major: every read's kept bases, back to back
    off = np.zeros(R + 1, dtype=np.uint64)
    off[1:] = np.cumsum(lens)
    n = int(off[R]) + R
    dev = torch.device("cuda", 0)
    ctx = api.Context(0)
    lib = ctx.lib
    bases_t = torch.from_numpy(bases).to(dev)
    whole = {k: torch.empty(n, dtype=torch.int32, device=dev) for k in ("lcp", "text", "suff")}
    whole["bwt"] = torch.empty(n, dtype=torch.uint8, device=dev)
    part = {k: torch.empty_like(v) for k, v in whole.items()}
    cuts = {P: sharding.key_range_cuts(P, (bases, off), sample=1 << 18, seed=P) for P in (2, 4, 8)}

    def build_whole():
        ctx._ck(lib.e2s_build_egsa_ragged_dev(ctx.h, _ptr(bases_t), off.ctypes.data, R, _ptr(whole["lcp"]), _ptr(whole["text"]),
                                              _ptr(whole["suff"]), _ptr(whole["bwt"])))

    def build_ranges(P):
        at, bt, bs = 0, 0xFFFFFFFF, 0
        for lo, hi in cuts[P]:
            m, first = C.c_uint64(0), C.c_uint64(0)
            ptrs = [part[k].data_ptr() + at * part[k].element_size() for k in ("lcp", "text", "suff", "bwt")]
            ctx._ck(lib.e2s_build_egsa_ragged_range_dev(ctx.h, _ptr(bases_t), off.ctypes.data, R, lo, hi, bt, bs, n - at,
                                                        *[C.c_void_p(p) for p in ptrs], C.byref(m), C.byref(first)))
            assert first.value == at
            at += m.value
            if m.value:
                bt, bs = int(part["text"][at - 1]), int(part["suff"][at - 1])
        assert at == n

    def timed(fn):
        torch.cuda.synchronize(dev)
        t = time.perf_counter()
        fn()
        torch.cuda.synchronize(dev)
        return (time.perf_counter() - t) * 1e3

    runs = {"whole": build_whole}
    runs.update({"P%d" % P: (lambda P=P: build_ranges(P)) for P in (2, 4, 8)})
    for fn in runs.values():  # warm-up of every shape
        fn()
    ms = {k: [] for k in runs}
    equal = {}
    for _ in range(a.reps):  # alternate the variants
        for k, fn in runs.items():
            ms[k].append(timed(fn))
            if k != "whole":
                equal[k] = equal.get(k, True) and all(torch.equal(part[x], whole[x]) for x in whole)

    share = {}
    from torch.profiler import ProfilerActivity, profile
    for k, fn in runs.items():
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            fn()
            torch.cuda.synchronize(dev)
        tot = sel = 0.0
        cnt = 0
        for ev in prof.key_averages():
            t = getattr(ev, "device_time_total", None)
            if t is None:
                t = getattr(ev, "cuda_time_total", 0.0)
            if "k_" not in ev.key:
                continue
            tot += t
            if "k_range_select" in ev.key:
                sel += t
                cnt += ev.count
        share[k] = {"kernel_ms": round(tot / 1e3, 3), "select_ms": round(sel / 1e3, 3), "select_launches": cnt,
                    "select_share": round(sel / tot, 4) if tot else None}

    res = {"tool": "bench_build_ranges", "config": "C2 trimmed to 70..%d bases" % L, "scale": a.scale, "reads": R, "suffixes": n,
           "ids": "64-bit" if R > (1 << (32 - int(L).bit_length())) else "32-bit",
           "ms_best": {k: round(min(v), 2) for k, v in ms.items()}, "ms_median": {k: round(statistics.median(v), 2) for k, v in ms.items()},
           "suffixes_per_s": {k: float("%.4g" % (n / (min(v) / 1e3))) for k, v in ms.items()},
           "ratio_to_whole": {k: round(min(v) / min(ms["whole"]), 3) for k, v in ms.items()},
           "kernels": share, "outputs_equal_whole": equal,
           "timing": "host clock around synchronised calls, best / median of %d after a warm-up; kernel times from torch.profiler, "
                     "one extra build each" % a.reps}
    res.update(gpu_info())
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")
    ctx.close()


if __name__ == "__main__":
    main()
