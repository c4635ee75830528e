"""-m gpu: byte parity on the NAMED configs of BASELINE.json (SURVEY.md 8(d)), against the unmodified reference run on
the same files (oracle/_ref where it is built, else the oracle's restatement of it: tests/helpers.py:reference_outputs).

  C1  exactly as stated (1 Mbp genome, 2 x 50 k reads of 100 bp, 1 000 SNPs, no reverse complements): file against file.
  C2  the whole E. coli-size set (5.6e8 positions, ~2 min of the single-threaded reference): file against file.
      E2S_SKIP_SLOW=1 skips it (development runs); the driver's round-end run keeps it.
  C3  the chr20-size set cannot go through the reference in one piece in a test (14 min, 50 GB of records), but the
      stencil is local: windows of the C3 index cut where lcp < k (no cluster can span such a position) are complete
      inputs of their own.  >= 24 windows (the first, the last with the real phantom tail, one across every N = 8
      shard cut, the rest at seeded random places): reference and CUDA path on each window's files byte for byte,
      then the records and events of the ONE full-size run must equal the windows' in every window interior, and the
      full-size run cut into 8 shards (run in sequence + host merge) must reproduce the single-shard records.
"""
import os
import shutil
import subprocess
import tempfile

import numpy as np
import pytest

from ebwt2snp_b200 import api, sharding, synth
from oracle import oracle as O
from tests import helpers as H

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "ebwt2snp_b200", "bin")
K, M = 16, 2


def scratch_dir(need_bytes):
    base = "/dev/shm" if os.path.isdir("/dev/shm") and shutil.disk_usage("/dev/shm").free > need_bytes * 1.2 else None
    return tempfile.mkdtemp(prefix="e2s_named_", dir=base)


def run_cli(tool, *args, env=None):
    e = dict(os.environ)
    e.update(env or {})
    return subprocess.run([os.path.join(BIN, tool), *[str(a) for a in args]], capture_output=True, text=True, env=e, timeout=3600)


def both_tool_chains(fa, eg, reads, nreads1, out_dir):
    """reference, then this repository's CLIs, on the same input files -> ((clusters, snp) of each, stdout counts)"""
    snp = os.path.join(out_dir, "ALL.snp")
    ref_cl, ref_snp, ncl, info = H.reference_outputs(fa, eg, reads, nreads1)
    assert info["returncode"] == 0
    o1 = run_cli("ebwt2clust", "-i", fa, "-x", 4, "-y", 4, "-z", 4)
    assert o1.returncode == 0, o1.stderr
    o2 = run_cli("clust2snp", "-i", fa, "-n", nreads1, "-x", 4, "-y", 4, "-z", 4)
    assert o2.returncode == 0, o2.stderr
    our_cl, our_snp = open(fa + ".clusters", "rb").read(), open(snp, "rb").read()

    def first_int(out, prefix):
        for line in out.splitlines():
            if line.startswith(prefix):
                return int(line.split()[1])
    return (ref_cl, ref_snp, ncl, info["n_candidates"], info["allowed"]), (
        our_cl, our_snp, first_int(o1.stdout, "Done. "), first_int(o2.stdout, "Done. "), o2.stdout)


@pytest.mark.parametrize("name", ["C1", "C2"])
def test_named_config_file_vs_file(built, name):
    if name == "C2" and os.environ.get("E2S_SKIP_SLOW"):
        pytest.skip("E2S_SKIP_SLOW set")
    import torch
    rs = synth.make_config(name, seed=1)
    e = synth.build_egsa(rs.reads, device="cuda")
    n = int(e["n"])
    if name == "C1":
        assert n == 10_100_000 and rs.nreads1 == 50_000 and len(rs.snp_pos) == 1000  # BASELINE config 1 as stated
    eg = {k: (v.cpu().numpy() if hasattr(v, "cpu") else v) for k, v in e.items()}
    del e
    torch.cuda.empty_cache()
    d = scratch_dir(n * 15)
    try:
        fa = synth.write_dataset(d, rs, eg, fixed_headers=True)
        ref, our = both_tool_chains(fa, eg, rs.reads, rs.nreads1, d)
        assert our[0] == ref[0], f"{name}: .clusters differ"
        assert our[1] == ref[1], f"{name}: .snp differ"
        assert our[2] == ref[2] and our[3] == ref[3]
        assert f"Cluster sizes allowed: [{ref[4][0]},{ref[4][1]}]" in our[4]
        assert len(ref[1]) > 0
        # the same through the C ABI in one call (fused scan + prefilter): e2s_pipeline_host from the file's records
        ctx = api.Context(0)
        rec = np.fromfile(fa + ".gesa", dtype=np.uint8)
        p = api.default_params(rs.nreads1)
        m = len(ref[0]) // 10
        rec10 = np.empty((m + 16) * 10, dtype=np.uint8)
        evbuf = (api.Event * (ref[3] + 16))()
        res = ctx.pipeline_host(rec, n, rs.reads.reshape(-1), O.uniform_read_offsets(*rs.reads.shape), p, K, M, rec10=rec10, events=evbuf)
        assert res.n_written == m and rec10[: m * 10].tobytes() == ref[0]
        assert res.snp.n_candidates == ref[3]
        assert api.events_format(list(evbuf)[: res.snp.n_variants], p) == ref[1]
        ctx.close()
    finally:
        shutil.rmtree(d, ignore_errors=True)


# ---------------------------------------------------------------------------------------------------------------------
# C3
# ---------------------------------------------------------------------------------------------------------------------
WINDOW = 6_000_000
MARGIN = 400  # positions before a window's end whose records are left out of the interior comparisons (tail rule)


@pytest.fixture(scope="module")
def c3(built):
    import torch
    if torch.cuda.get_device_properties(0).total_memory < 150 << 30:
        pytest.skip("needs a 180 GB B200")
    scale = float(os.environ.get("E2S_C3_SCALE", "1.0"))  # development knob; the driver runs the real size
    rs = synth.make_config("C3", seed=1, scale=scale)
    ctx = api.Context(0)
    eg = ctx.build_egsa(rs.reads)
    ctx.stage_reads(torch.from_numpy(rs.reads).cuda().view(-1),
                    torch.arange(rs.reads.shape[0] + 1, dtype=torch.int64, device="cuda") * rs.reads.shape[1],
                    device=True, n_bases=rs.reads.size)
    yield rs, eg, ctx
    ctx.close()


def window_starts(eg, n_windows=24, seed=5):
    """[(a, b, why)]: a = a position with lcp < K (nothing can span it), b - a = WINDOW (b = n for the last window)"""
    import torch
    n = int(eg["n"])
    lcp = eg["lcp"]
    W = min(WINDOW, n // 4)

    def snap(pos):  # the last position <= pos with lcp < K
        pos = max(0, min(int(pos), n - W))
        lo = max(0, pos - 100_000)
        idx = torch.nonzero(lcp[lo:pos + 1] < K)
        return lo + int(idx[-1]) if len(idx) else 0

    R = int(eg["R"])  # the first R records are the terminator suffixes (lcp 0): the first window with clusters starts there
    wins = [(0, W, "first"), (snap(n - W), n, "last (phantom tail)"), (snap(R - 1000), None, "where the terminator suffixes end")]
    for c in sharding.shard_cuts(n, 8)[1:-1]:
        wins.append((snap(c - W // 2), None, f"across the N=8 shard cut at {c}"))
    rng = np.random.default_rng(seed)
    while len(wins) < n_windows:
        wins.append((snap(int(rng.integers(W, n - 2 * W))), None, "random"))
    return [(a, b if b is not None else a + W, why) for a, b, why in wins]


def window_dataset(rs, eg, a, b):
    """the records [a, b) as an index of their own: read ids renumbered densely (order kept, so `text < -n` still splits
    the samples), the FASTA holds just those reads"""
    sl = {k: eg[k][a:b].cpu().numpy() for k in ("lcp", "text", "suff", "bwt")}
    uniq, inv = np.unique(sl["text"].view(np.uint32), return_inverse=True)
    sub = dict(lcp=sl["lcp"].view(np.uint32), text=inv.astype(np.uint32), suff=sl["suff"].view(np.uint32), bwt=sl["bwt"], n=b - a)
    reads = np.ascontiguousarray(rs.reads[uniq])
    n1 = int(np.searchsorted(uniq, rs.nreads1))
    return sub, reads, n1


def event_key(ev, shift=0):
    return (ev.cluster_start - shift, ev.D, ev.gap, ev.supp0, ev.supp1, ev.keep, ev.right_len, bytes(ev.left0), bytes(ev.left1), bytes(ev.right))


def test_c3_windows_vs_reference_and_full_run(c3):
    import torch
    rs, eg, ctx = c3
    n = int(eg["n"])
    p = api.default_params(rs.nreads1)
    # ---- the ONE full-size run (BASELINE config 3 / 5 on one GPU) ----
    sh = ctx.shard(n)
    sh.load_soa(eg["lcp"], eg["text"], eg["suff"], eg["bwt"], device=True)
    sh.seal()
    res = sh.pipeline_resident(p, K, M)
    g_start, g_len = sh.cluster_fetch()
    g_events = [event_key(ev) for ev in sh.events()]
    mcl = res.max_clust_length
    sh.close()
    assert len(g_start) == res.n_written and res.snp.n_candidates > 0
    g_ev_start = np.array([e[0] for e in g_events], dtype=np.uint64)

    wins = window_starts(eg)
    assert len(wins) >= 24
    d = scratch_dir(WINDOW * 140)
    wctx = api.Context(0)
    try:
        for wi, (a, b, why) in enumerate(wins):
            sub, reads, n1 = window_dataset(rs, eg, a, b)
            assert n1 >= 1
            wdir = os.path.join(d, f"w{wi}")
            wrs = synth.ReadSet(reads=reads, nreads1=n1, genome1=None, genome2=None, snp_pos=None, indels=[])
            fa = synth.write_dataset(wdir, wrs, sub, fixed_headers=True)
            ref_cl, ref_snp, ncl, info = H.reference_outputs(fa, sub, reads, n1)
            # ---- the CUDA path on the window's own files (C ABI, from the .gesa records) ----
            rec = np.fromfile(fa + ".gesa", dtype=np.uint8)
            wsh = wctx.shard(b - a)
            wsh.load_gesa(rec, 0, b - a)
            wsh.seal()
            wp = api.default_params(n1)
            wctx.stage_reads(reads, O.uniform_read_offsets(*reads.shape))
            hi = b - MARGIN if b < n else n + 1
            lo_i, hi_i = np.searchsorted(g_start, a), np.searchsorted(g_start, hi)
            if len(ref_cl) == 0:  # e.g. the first window: nothing but terminator suffixes (the reference then divides by zero)
                nw, nc = wsh.cluster_lm(K, M)
                assert nw == 0 and (nc & 0xFFFFFFFF) == ncl and lo_i == hi_i
                wsh.close()
                shutil.rmtree(wdir, ignore_errors=True)
                continue
            wres = wsh.pipeline_resident(wp, K, M)
            assert wsh.cluster_fetch_packed() == ref_cl, f"window {wi} ({why}): .clusters differ"
            assert (wres.n_clust_out & 0xFFFFFFFF) == ncl
            assert (2 * wp.mcov_out, wres.max_clust_length) == info["allowed"]
            if ref_snp is not None:
                assert wres.snp.n_candidates == info["n_candidates"]
                assert api.events_format(wsh.events(), wp) == ref_snp, f"window {wi} ({why}): .snp differ"
            else:
                assert wres.snp.n_candidates == 0
            if wi in (0, 1, 2):  # and file against file through the CLIs
                assert run_cli("ebwt2clust", "-i", fa, "-x", 4, "-y", 4, "-z", 4).returncode == 0
                assert open(fa + ".clusters", "rb").read() == ref_cl
                if ref_snp is not None:
                    assert run_cli("clust2snp", "-i", fa, "-n", n1, "-x", 4, "-y", 4, "-z", 4).returncode == 0
                    assert open(os.path.join(wdir, "ALL.snp"), "rb").read() == ref_snp
            # ---- the full-size run agrees with the window in the window's interior ----
            ws, wl = wsh.cluster_fetch()
            keep = ws + np.uint64(a) < np.uint64(hi)
            assert np.array_equal(g_start[lo_i:hi_i], ws[keep] + np.uint64(a)), f"window {wi} ({why}): records of the full run differ"
            assert np.array_equal(g_len[lo_i:hi_i], wl[keep])
            # events with the FULL run's max_clust_length (the window's own statistics may choose another one)
            wsh.find_events(wp, mcl)
            w_events = [event_key(ev, 0) for ev in wsh.events()]
            w_events = [(e[0] + a,) + e[1:] for e in w_events if e[0] + a < hi]
            sel = (g_ev_start >= a) & (g_ev_start < hi)
            assert [g_events[i] for i in np.flatnonzero(sel)] == w_events, f"window {wi} ({why}): events of the full run differ"
            wsh.close()
            shutil.rmtree(wdir, ignore_errors=True)
    finally:
        wctx.close()
        shutil.rmtree(d, ignore_errors=True)

    # ---- the same index cut into 8 shards (BASELINE config 5's cuts), run one after the other + host merge ----
    cuts = sharding.shard_cuts(n, 8)
    sums, parts = [], []
    for lo, hi in zip(cuts[:-1], cuts[1:]):
        s8 = ctx.shard(hi - lo, lo, n)
        x, y = max(0, lo - 2), min(n, hi + 151)
        s8.load_soa(eg["lcp"][x:y], eg["text"][x:y], eg["suff"][x:y], eg["bwt"][x:y], first=x, device=True)
        s8.seal()
        sums.append(s8.cluster_run(K, M))
        s8.cluster_finalize(api.ClusterMerged())
        parts.append(s8.cluster_fetch())
        s8.close()
    S, L = [], []
    for g, (ps, pl) in enumerate(parts):
        mg = api.cluster_merge(sums, g)
        if mg.n_prepend and mg.prepend_written:
            S.append(np.array([mg.prepend_start], dtype=np.uint64))
            L.append(np.array([mg.prepend_len], dtype=np.uint16))
        S.append(ps)
        L.append(pl)
        for i in range(mg.n_append):
            S.append(np.array([mg.append_start[i]], dtype=np.uint64))
            L.append(np.array([mg.append_len[i]], dtype=np.uint16))
    assert mg.n_clust_out == res.n_clust_out and mg.total_written == res.n_written
    assert np.array_equal(np.concatenate(S), g_start) and np.array_equal(np.concatenate(L), g_len)
