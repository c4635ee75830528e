"""-m gpu: the index of reads of any lengths built key range by key range (e2s_build_egsa_ragged_range_dev, and the host path
e2s_build_egsa_ragged / build_gesa that switches to ranges when the whole index does not fit) against the oracle's comparison sort."""
import ctypes as C
import os

import numpy as np
import pytest

from ebwt2snp_b200 import api, sharding, synth
from ebwt2snp_b200.api import _ptr
from oracle import oracle as O
from tests.test_builder_gpu import key_of, make_case, ragged_from_genome, run

pytestmark = pytest.mark.gpu

KEYS = ("text", "suff", "lcp", "bwt")


@pytest.fixture(scope="module")
def ctx(built):
    c = api.Context(0)
    yield c
    c.close()


@pytest.fixture
def ids(monkeypatch, request):
    """E2S_BUILD_IDS64 on / off for the test"""
    if request.param:
        monkeypatch.setenv("E2S_BUILD_IDS64", "1")
    else:
        monkeypatch.delenv("E2S_BUILD_IDS64", raising=False)
    monkeypatch.delenv("E2S_BUILD_RANGE_RECORDS", raising=False)
    return request.param


def host(a, key):
    a = a.cpu().numpy() if hasattr(a, "cpu") else np.asarray(a)
    return a.view(np.uint32) if key != "bwt" else a


def index_keys(bases, off, want):
    return sharding.first_key_words((bases, off), want["text"].astype(np.int64), want["suff"].astype(np.int64))


def hand_cuts(keys):
    """cuts at and just past the key-0 run and the heaviest other key (a run of equal keys is never split: the cut lands at its edge),
    fixed prefixes, and an empty range [x, x + 1) at a key no suffix has"""
    vals, cnt = np.unique(keys, return_counts=True)
    nz = vals[1:], cnt[1:]
    heavy = int(nz[0][np.argmax(nz[1])]) if len(nz[0]) else key_of(b"C")
    present = set(int(v) for v in vals)
    x = key_of(b"CGTC") + 1
    while x in present or x + 1 in present:
        x += 7
    cuts = {1, key_of(b"AC"), heavy, heavy + 1, key_of(b"CGT"), x, x + 1, key_of(b"G"), key_of(b"T" * 32)}
    cuts = [0] + sorted(c for c in cuts if 0 < c < 1 << 64) + [0]
    return list(zip(cuts[:-1], cuts[1:])), (x, x + 1)


def range_call(ctx, bases_t, off, lo, hi, cap, before=None):
    """e2s_build_egsa_ragged_range_dev through ctypes: (rc, n_records, first_position) -- for the refusals the wrapper raises on"""
    import torch
    dev = torch.device("cuda", ctx.device)
    out = [torch.empty(max(cap, 1), dtype=torch.int32, device=dev) for _ in range(3)] + [torch.empty(max(cap, 1), dtype=torch.uint8, device=dev)]
    n_rec, first = C.c_uint64(12345), C.c_uint64(12345)
    bt, bs = (0xFFFFFFFF, 0) if before is None else before
    torch.cuda.synchronize(dev)
    rc = ctx.lib.e2s_build_egsa_ragged_range_dev(ctx.h, _ptr(bases_t), off.ctypes.data, len(off) - 1, lo, hi, bt, bs, cap,
                                                 *[_ptr(t) for t in out], C.byref(n_rec), C.byref(first))
    return rc, int(n_rec.value), int(first.value)


def check_chain(ctx, bases, off, want, ranges, what, empty=None):
    """ranges in key order, each told the last record of the one before: the concatenation is the oracle's index array for array"""
    import torch
    bases_t = torch.from_numpy(np.ascontiguousarray(bases).reshape(-1) if len(bases) else np.zeros(1, np.uint8)).cuda(ctx.device)
    n = want["n"]
    at, before = 0, None
    for lo, hi in ranges:
        part = ctx.build_egsa_ragged_range(bases_t, off, lo, hi, before=before)
        alone = ctx.build_egsa_ragged_range(bases_t, off, lo, hi)
        m = part["n"]
        tag = (what, hex(lo), hex(hi))
        assert part["first"] == at and alone["first"] == at and alone["n"] == m, tag
        for key in KEYS:
            got, solo = host(part[key], key), host(alone[key], key)
            assert np.array_equal(got, want[key][at:at + m]), (key,) + tag
            if key == "lcp" and m:
                assert solo[0] == 0 and np.array_equal(solo[1:], want[key][at + 1:at + m]), tag
            else:
                assert np.array_equal(solo, want[key][at:at + m]), (key,) + tag
        if (lo, hi) == empty:
            assert m == 0, tag
        if m:
            rc, m2, _ = range_call(ctx, bases_t, off, lo, hi, m - 1, before)
            assert rc == api.ERR_ARG and m2 == m, tag
            before = (int(want["text"][at + m - 1]), int(want["suff"][at + m - 1]))
        at += m
    assert at == n, what


@pytest.mark.parametrize("ids", [False, True], indirect=True)
@pytest.mark.parametrize("name", ["tiny", "genome", "two_length_places", "skewed", "many_tiles"])
def test_ragged_ranges_tile_the_index(ctx, ids, name):
    """hand-made cuts (key-0 run, the heaviest key, an empty range) and key_range_cuts quantiles with 2, 3 and 7 parts"""
    bases, off = make_case(name)
    want = O.build_egsa_ragged(bases, off)
    hand, empty = hand_cuts(index_keys(bases, off, want))
    check_chain(ctx, bases, off, want, hand, (name, "hand"), empty)
    for parts in (2, 3, 7):
        cuts = sharding.key_range_cuts(parts, (bases, off), sample=1 << 14, seed=parts)
        check_chain(ctx, bases, off, want, cuts, (name, parts))


@pytest.mark.parametrize("ids", [False, True], indirect=True)
def test_equal_length_reads_agree_across_range_entry_points(ctx, ids):
    """equal-length reads through the ragged range entry point give the records of e2s_build_egsa_range_dev on the same cuts"""
    rs = synth.make_read_set(G=20_000, reads_per_sample=2_000, L=100, n_snps=30, n_indels=2, rc=True, seed=78)
    R, L = rs.reads.shape
    off = np.arange(R + 1, dtype=np.uint64) * np.uint64(L)
    cuts = [(0, key_of(b"AC")), (key_of(b"AC"), key_of(b"CGTC")), (key_of(b"CGTC"), key_of(b"G")), (key_of(b"G"), 0)]
    cuts += sharding.key_range_cuts(3, rs.reads, sample=1 << 14)
    for lo, hi in cuts:
        a = ctx.build_egsa_range(rs.reads, lo, hi)
        b = ctx.build_egsa_ragged_range(rs.reads.reshape(-1), off, lo, hi)
        assert a["n"] == b["n"] and a["first"] == b["first"], (hex(lo), hex(hi))
        for key in KEYS:
            assert np.array_equal(host(a[key], key), host(b[key], key)), (key, hex(lo), hex(hi))


def host_build(ctx, bases, off):
    """e2s_build_egsa_ragged (host in / out) through ctypes: (rc, message, dict of arrays)"""
    off = np.ascontiguousarray(off, dtype=np.uint64)
    R = len(off) - 1
    n = int(off[R]) + R
    out = {k: np.zeros(n, dtype=np.uint32) for k in ("lcp", "text", "suff")}
    out["bwt"] = np.zeros(n, dtype=np.uint8)
    b = np.ascontiguousarray(bases, dtype=np.uint8).reshape(-1)
    rc = ctx.lib.e2s_build_egsa_ragged(ctx.h, _ptr(b), off.ctypes.data, R, _ptr(out["lcp"]), _ptr(out["text"]), _ptr(out["suff"]),
                                       _ptr(out["bwt"]))
    msg = ctx.lib.e2s_last_error(ctx.h).decode() if rc else ""
    return rc, msg, out


def host_slices(n, cap):
    """the key-space slices the host path starts from (build_egsa_host_ranges)"""
    parts = (n + cap - 1) // cap
    parts += parts // 4 + 1
    return [((i << 64) // parts, ((i + 1) << 64) // parts if i + 1 < parts else 1 << 64) for i in range(parts)]


def test_host_path_forced_ranges(ctx, monkeypatch):
    """E2S_BUILD_RANGE_RECORDS at several caps, one of which makes a starting slice hold more than the cap (cut in two on the way),
    and with 64-bit ids: the arrays equal the unforced call and the oracle"""
    rng = np.random.default_rng(41)
    bases, off = ragged_from_genome(rng, 40_000, 3_000, 0, 150)
    want = O.build_egsa_ragged(bases, off)
    n = want["n"]
    keys = index_keys(bases, off, want)
    monkeypatch.delenv("E2S_BUILD_RANGE_RECORDS", raising=False)
    monkeypatch.delenv("E2S_BUILD_IDS64", raising=False)
    l0 = ctx.launches
    rc, msg, whole = host_build(ctx, bases, off)
    assert rc == 0, msg
    whole_launches = ctx.launches - l0
    k0 = int(np.count_nonzero(keys == 0))
    caps = [n // 2 + 1, n // 5, max(k0 + 1, n // 16)]
    split = False
    for cap in caps:
        assert cap > k0
        split |= any(int(np.count_nonzero((keys >= lo) & (keys < hi))) > cap for lo, hi in host_slices(n, cap))
    assert split
    for env in [{"E2S_BUILD_RANGE_RECORDS": str(c)} for c in caps] + [{"E2S_BUILD_RANGE_RECORDS": str(caps[1]), "E2S_BUILD_IDS64": "1"}]:
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        l0 = ctx.launches
        rc, msg, got = host_build(ctx, bases, off)
        launches = ctx.launches - l0
        monkeypatch.delenv("E2S_BUILD_RANGE_RECORDS", raising=False)
        monkeypatch.delenv("E2S_BUILD_IDS64", raising=False)
        assert rc == 0, (env, msg)
        assert launches > whole_launches, (env, launches, whole_launches)  # the ranges were taken
        for key in KEYS:
            assert np.array_equal(got[key], whole[key]) and np.array_equal(got[key], want[key]), (env, key)


def test_host_path_refuses_a_heavy_key(ctx, monkeypatch):
    """poly-A reads put more suffixes under key 0 than the forced cap: a clean refusal, not a wrong index"""
    rng = np.random.default_rng(43)
    b, o = ragged_from_genome(rng, 20_000, 500, 40, 120)
    parts = [b] + [np.full(int(l), ord("A"), dtype=np.uint8) for l in rng.integers(32, 100, size=400)]
    lens = np.concatenate([np.diff(o.astype(np.int64)), [len(p) for p in parts[1:]]])
    off = np.zeros(len(lens) + 1, dtype=np.uint64)
    off[1:] = np.cumsum(lens)
    bases = np.concatenate(parts)
    keys = sharding.first_key_words((bases, off), np.repeat(np.arange(len(lens)), lens + 1), np.concatenate([np.arange(l + 1) for l in lens]))
    k0 = int(np.count_nonzero(keys == 0))
    cap = k0 - 1000
    assert cap > 4096
    monkeypatch.setenv("E2S_BUILD_RANGE_RECORDS", str(cap))
    rc, msg, _ = host_build(ctx, bases, off)
    assert rc == api.ERR_UNSUPPORTED and "32-symbol prefix" in msg, (rc, msg)


def test_build_gesa_forced_ranges_on_a_ragged_fasta(built, tmp_path, monkeypatch):
    """build_gesa on trimmed reads: .gesa and the BCR triple (-b) byte-identical with and without forced ranges; a forced cap below
    the key-0 run is refused (the forced ranges are really taken)"""
    rs = synth.make_read_set(G=20_000, reads_per_sample=2_500, L=100, n_snps=30, n_indels=0, rc=True, seed=33)
    rng = np.random.default_rng(6)
    lens = rng.integers(70, 101, size=rs.reads.shape[0])
    n = int(lens.sum()) + len(lens)
    monkeypatch.delenv("E2S_BUILD_RANGE_RECORDS", raising=False)
    monkeypatch.delenv("E2S_BUILD_IDS64", raising=False)
    outs = {}
    for j, env in enumerate([None, {"E2S_BUILD_RANGE_RECORDS": str(n // 3)}, {"E2S_BUILD_RANGE_RECORDS": str(n // 7), "E2S_BUILD_IDS64": "1"}]):
        for bcr in (False, True):
            d = tmp_path / f"v{j}{int(bcr)}"
            os.makedirs(d)
            fa = str(d / "ALL.fasta")
            with open(fa, "wb") as f:
                for r in range(len(lens)):
                    f.write(b">r%d\n" % r + rs.reads[r, :lens[r]].tobytes() + b"\n")
            r = run("build_gesa", "-i", fa, "-x", 1, "-y", 4, "-z", 1, *(["-b"] if bcr else []), env=env)
            assert r.returncode == 0, r.stdout + r.stderr
            exts = (".out", ".out.lcp", ".out.pairSA") if bcr else (".gesa",)
            outs[(j, bcr)] = [open(fa + x, "rb").read() for x in exts]
    r = run("build_gesa", "-i", str(tmp_path / "v00" / "ALL.fasta"), env={"E2S_BUILD_RANGE_RECORDS": str(len(lens))})
    assert r.returncode == 3 and "32-symbol prefix" in r.stdout, r.stdout + r.stderr
    for bcr in (False, True):
        assert len(outs[(0, bcr)][0]) > 0
        assert outs[(1, bcr)] == outs[(0, bcr)] and outs[(2, bcr)] == outs[(0, bcr)], bcr


def test_host_path_chooses_ranges_when_the_device_is_nearly_full(ctx, monkeypatch):
    """with all but a few hundred MB of free device memory held by a tensor, e2s_build_egsa_ragged sees that the whole index would
    not fit, takes key ranges on its own (more launches than the whole build) and still writes the oracle's index"""
    import torch
    monkeypatch.delenv("E2S_BUILD_RANGE_RECORDS", raising=False)
    monkeypatch.delenv("E2S_BUILD_IDS64", raising=False)
    rng = np.random.default_rng(45)
    bases, off = ragged_from_genome(rng, 2_000_000, 150_000, 60, 140)
    R = len(off) - 1
    n = int(off[R]) + R
    want = O.build_egsa_ragged(bases, off)
    rc, msg, _ = host_build(ctx, bases[: int(off[100])], off[:101])  # modules loaded, nothing left to allocate lazily
    assert rc == 0, msg
    l0 = ctx.launches
    rc, msg, whole = host_build(ctx, bases, off)
    assert rc == 0, msg
    whole_launches = ctx.launches - l0
    need = n * 38  # outputs + 32-bit-id scratch per suffix
    leave = 400 << 20
    assert need > leave / 0.92 + (64 << 20)
    dev = torch.device("cuda", ctx.device)
    torch.cuda.synchronize(dev)
    torch.cuda.empty_cache()
    hold = None
    try:
        free, _ = torch.cuda.mem_get_info(dev)
        assert free > leave + (1 << 30), free
        hold = torch.empty(free - leave, dtype=torch.uint8, device=dev)
        torch.cuda.synchronize(dev)
        free_after, _ = torch.cuda.mem_get_info(dev)
        assert free_after < need, free_after
        l0 = ctx.launches
        rc, msg, got = host_build(ctx, bases, off)
        launches = ctx.launches - l0
    finally:
        del hold
        torch.cuda.empty_cache()
    assert rc == 0, msg
    assert launches > whole_launches, (launches, whole_launches)
    for key in KEYS:
        assert np.array_equal(got[key], want[key]) and np.array_equal(whole[key], want[key]), key
