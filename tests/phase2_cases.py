"""Designed phase-2 (clust2snp) inputs: lcp / text / suff / bwt arrays and a read collection written directly, with no suffix
sort, each planting a few clusters that reach one branch of find_variants, the candidate selection, consensus / support,
distance() or the context and read handling.

clust2snp accepts any index file, so the CUDA path must match the oracle on any index, not only on sorted ones.  Every case
also carries what it was designed to produce (`expect`): the counts and, per kept event in output order, its kind
(SNP / INDEL), type string and the two supports.  tests/test_phase2_cases_nogpu.py checks the oracle against that, so a
case that silently stops reaching its branch fails there; tests/test_phase2_paths_gpu.py compares the CUDA paths with the
oracle on the same cases.

Layout: records with LCP 0 separate the clusters, so with -k 16 every planted cluster is one run of LCP >= 16 whose values
never fall to a strict local minimum (no split).  A planted record's left context is written into its read at
[suff - k_left, suff) and its right context from suff on.  Sample 0 reads get the ids below nreads1.
"""
from __future__ import annotations

import re
from dataclasses import dataclass

import numpy as np

from oracle import oracle as O

K = 16          # ebwt2clust -k for every case
MIN_LEN = 2     # ebwt2clust -m
ACGT = b"ACGT"
DEFAULTS = dict(k_left=31, k_right=30, mcov_out=5, max_gap=10, consensus_reads=20, max_err=2, max_snvs=3)


# ---- distance() as specified (ref:clust2snp.cpp:254-302): used only to choose contexts with a wanted outcome ------------
def _dh(a: bytes, b: bytes) -> int:
    n = min(len(a), len(b))
    return sum(a[len(a) - 1 - i] != b[len(b) - 1 - i] for i in range(n))


def dist_table(a: bytes, b: bytes, max_gap: int):
    """(d0, ab[g], ba[g]) for g = 1..max_gap (index g - 1), ab = dH(a without g chars on the right, b) + g"""
    n = len(a)
    return _dh(a, b), [_dh(a[:n - g], b) + g for g in range(1, max_gap + 1)], [_dh(a, b[:n - g]) + g for g in range(1, max_gap + 1)]


def distance(a: bytes, b: bytes, max_gap: int):
    d0, ab, ba = dist_table(a, b, max_gap)
    if not ab:
        return d0, 0
    mab, mba = min(ab), min(ba)
    gab, gba = ab.index(mab) + 1, ba.index(mba) + 1
    if d0 < mab and d0 < mba:
        return d0, 0
    if mab < mba:
        return mab - gab, gab
    return mba - gba, -gba


def type_string(l0: bytes, l1: bytes, gap: int) -> bytes:
    kl = len(l0)
    if gap == 0:
        return l0[-1:] + b"/" + l1[-1:]
    if gap > 0:
        return l0[kl - gap:] + b"/"
    return b"/" + l1[kl + gap:]


# ---- the case -----------------------------------------------------------------------------------------------------------
@dataclass
class Case:
    name: str
    lcp: np.ndarray
    text: np.ndarray
    suff: np.ndarray
    bwt: np.ndarray
    bases: np.ndarray
    off: np.ndarray
    nreads1: int
    params: dict
    pval: float
    max_clust_length: int
    clusters: list                      # planted (start, len)
    expect: dict                        # n_analysed / n_candidates / n_variants / n_events / saw_n (when given) + events
    refuse: bool = False                # the right context starts past its read's end: both must refuse
    groups: tuple = ()                  # the subsets of the GPU test this case belongs to
    note: str = ""

    @property
    def n(self):
        return len(self.lcp)

    def oparams(self):
        return O.default_params(self.nreads1, **self.params)


class Builder:
    def __init__(self, seed, **params):
        self.rng = np.random.default_rng(seed)
        self.params = dict(DEFAULTS, **params)
        self.reads = ([], [])           # per sample: bytes
        self.rows = []                  # (read handle or None, suff, lcp, bwt byte)
        self.clusters = []
        self.gap(3)

    @property
    def kl(self):
        return self.params["k_left"]

    @property
    def kr(self):
        return self.params["k_right"]

    def rand(self, n, alphabet=ACGT) -> bytes:
        a = np.frombuffer(alphabet, dtype=np.uint8)
        return a[self.rng.integers(0, len(a), size=n)].tobytes()

    def read(self, sample, data: bytes):
        self.reads[sample].append(bytes(data))
        return (sample, len(self.reads[sample]) - 1)

    def gap(self, n=2):
        self.rows.extend([(None, 0, 0, ord("T"))] * n)

    def member(self, sample, left: bytes, right: bytes, bwt=None, lcp=None, pre=b""):
        """a record whose own read is pre + left + right, suff = len(pre + left)"""
        h = self.read(sample, pre + left + right)
        return (h, len(pre) + len(left), max(K, self.kr) if lcp is None else lcp, left[-1] if bwt is None else
                (ord(bwt) if isinstance(bwt, str) else bwt))

    def cluster(self, rows):
        start = len(self.rows)
        lc = [r[2] for r in rows]
        assert min(lc) >= K
        self.rows.extend(rows)
        self.clusters.append((start, len(rows)))
        self.gap(2)
        return start

    def snp_contexts(self, a0=b"A", a1=b"C", kl=None, max_gap=None):
        """two left contexts that differ in their last character only, with distance() = (1, 0)"""
        kl = self.kl if kl is None else kl
        g = self.params["max_gap"] if max_gap is None else max_gap
        while True:
            c = self.rand(kl - 1)
            l0, l1 = c + a0, c + a1
            if kl == 1 or distance(l0, l1, g) == (1, 0):
                return l0, l1

    def snp_cluster(self, n0, n1, a0="A", a1="C", extra0=(), extra1=(), lcp=None, right=None):
        """n0 sample-0 records with allele a0 and n1 sample-1 records with a1 whose contexts differ in the last character;
        extra0 / extra1: more rows appended after each sample's records"""
        l0, l1 = self.snp_contexts(a0.encode(), a1.encode())
        right = self.rand(self.kr) if right is None else right
        rows = [self.member(0, l0, right, lcp=lcp) for _ in range(n0)] + list(extra0)
        rows += [self.member(1, l1, right, lcp=lcp) for _ in range(n1)] + list(extra1)
        self.cluster(rows)
        return l0, l1, right

    def build(self, name, expect, pval=1.0, mcl=None, uniform=False, refuse=False, groups=(), note="", extra_reads=()):
        for s, data in extra_reads:
            self.read(s, data)
        reads = list(self.reads[0]) + list(self.reads[1])
        if uniform:
            L = max(len(r) for r in reads)
            reads = [r + self.rand(L - len(r)) for r in reads]
        nreads1 = len(self.reads[0])
        lcp = np.zeros(len(self.rows) + 3, dtype=np.uint32)
        text = np.zeros_like(lcp)
        suff = np.zeros_like(lcp)
        bwt = np.full(len(lcp), ord("T"), dtype=np.uint8)
        for i, (h, sf, lc, b) in enumerate(self.rows):
            if h is not None:
                text[i] = h[1] + (nreads1 if h[0] else 0)
            suff[i], lcp[i], bwt[i] = sf, lc, b
        bases = np.frombuffer(b"".join(reads), dtype=np.uint8).copy()
        off = np.zeros(len(reads) + 1, dtype=np.uint64)
        off[1:] = np.cumsum([len(r) for r in reads])
        es, el, _, _ = O.cluster_lm(lcp, bwt, K, MIN_LEN)
        assert list(zip(es.tolist(), el.tolist())) == self.clusters, name
        mcov = self.params["mcov_out"]
        st = O.statistics(es, el, mcov, pval)
        if mcl is None:  # pval 1: the longest cluster, unless a shorter one than 2 mcov keeps the sum below n_bases
            lens = [l for _, l in self.clusters]
            mcl = max(lens) if min(lens) >= 2 * mcov else O.MAX_C_LEN
        assert st.max_clust_length == mcl, (name, st.max_clust_length, mcl)
        return Case(name, lcp, text, suff, bwt, bases, off, nreads1, dict(self.params), pval, st.max_clust_length,
                    list(self.clusters), expect, refuse, tuple(groups), note)


def ev(kind, typ, s0, s1):
    return (kind, typ if isinstance(typ, bytes) else typ.encode(), s0, s1)


def snp_ev(l0, l1, s0, s1):
    return ev("SNP", type_string(l0, l1, 0), s0, s1)


def counts(cand, var, evs, **kw):
    d = dict(n_candidates=cand, n_variants=var, n_events=len(evs), events=list(evs))
    d.update(kw)
    return d


# ---- find_variants -------------------------------------------------------------------------------------------------------
def find_variants_cases():
    out = []
    # count = mcov (flagged) and mcov - 1 (not), in either sample
    b = Builder(101)
    l0, l1, _ = b.snp_cluster(5, 5)
    b.snp_cluster(4, 5)
    b.snp_cluster(5, 4)
    out.append(b.build("fv_count_mcov", counts(1, 1, [snp_ev(l0, l1, 5, 5)], n_analysed=1)))  # (the 9-record ones are too short)
    b = Builder(102, mcov_out=3)
    l0, l1, _ = b.snp_cluster(3, 3)
    b.snp_cluster(2, 4)
    b.snp_cluster(4, 2)
    out.append(b.build("fv_count_mcov3", counts(1, 1, [snp_ev(l0, l1, 3, 3)], n_analysed=3)))

    # union of 3 letters (two candidates) vs 4 letters (none); equal frequent sets; 3 frequent codes in one sample
    b = Builder(103)
    c = b.rand(b.kl - 1)
    right = b.rand(b.kr)
    ctx = {a: c + a.encode() for a in "ACGT"}
    rows = [b.member(0, ctx["A"], right) for _ in range(5)] + [b.member(0, ctx["C"], right) for _ in range(5)]
    rows += [b.member(1, ctx["G"], right) for _ in range(6)]
    b.cluster(rows)
    rows = [b.member(0, ctx["A"], right) for _ in range(5)] + [b.member(0, ctx["C"], right) for _ in range(5)]
    rows += [b.member(1, ctx["G"], right) for _ in range(5)] + [b.member(1, ctx["T"], right) for _ in range(5)]
    b.cluster(rows)  # 4 letters
    rows = [b.member(0, ctx["A"], right) for _ in range(5)] + [b.member(0, ctx["C"], right) for _ in range(5)]
    rows += [b.member(1, ctx["A"], right) for _ in range(5)] + [b.member(1, ctx["C"], right) for _ in range(5)]
    b.cluster(rows)  # equal sets
    rows = [b.member(0, ctx[a], right) for a in "ACG" for _ in range(5)] + [b.member(1, ctx["A"], right) for _ in range(5)]
    b.cluster(rows)  # three frequent codes in sample 0
    out.append(b.build("fv_union_and_sets", counts(2, 2, [snp_ev(ctx["A"], ctx["G"], 5, 6), snp_ev(ctx["C"], ctx["G"], 5, 6)],
                                                     n_analysed=4)))

    # two allele pairs in one cluster: f0 = {A, C}, f1 = {C, G}: (A,C), (A,G), (C,G) in that order, (C,C) skipped
    b = Builder(104)
    rows = [b.member(0, ctx["A"], right) for _ in range(5)] + [b.member(1, ctx["G"], right) for _ in range(6)]
    rows += [b.member(0, ctx["C"], right) for _ in range(7)] + [b.member(1, ctx["C"], right) for _ in range(8)]
    b.cluster(rows)
    out.append(b.build("fv_two_pairs_nested", counts(3, 3, [snp_ev(ctx["A"], ctx["C"], 5, 8), snp_ev(ctx["A"], ctx["G"], 5, 6),
                                                            snp_ev(ctx["C"], ctx["G"], 7, 6)])))

    # max LCP = k_right (flagged) vs k_right - 1 (not); LCP rises to a plateau shared by several records: the first gives the
    # right context
    b = Builder(105)
    l0, l1, _ = b.snp_cluster(5, 5, lcp=30)
    b.snp_cluster(5, 5, lcp=29)
    out.append(b.build("fv_max_lcp_k_right", counts(1, 1, [snp_ev(l0, l1, 5, 5)])))
    b = Builder(106)
    l0, l1 = b.snp_contexts()
    rows = [b.member(0, l0, b.rand(b.kr), lcp=v) for v in (30, 31, 35, 35)] + [b.member(1, l1, b.rand(b.kr), lcp=v) for v in (35, 34, 33, 32, 31)]
    rows.insert(1, b.member(0, l0, b.rand(b.kr), lcp=30))
    b.cluster(rows)
    first_max = b.reads[0][2]
    out.append(b.build("fv_lcp_argmax_first", counts(1, 1, [snp_ev(l0, l1, 5, 5)], right=first_max[b.kl:b.kl + b.kr])))
    b = Builder(107)
    l0, l1 = b.snp_contexts()
    rows = [b.member(1, l1, b.rand(b.kr), lcp=v) for v in (30, 40, 40)] + [b.member(0, l0, b.rand(b.kr), lcp=v) for v in (40, 40, 40, 40, 40)]
    rows += [b.member(1, l1, b.rand(b.kr), lcp=v) for v in (39, 38)]
    b.cluster(rows)
    out.append(b.build("fv_lcp_argmax_sample1", counts(1, 1, [snp_ev(l0, l1, 5, 5)], right=b.reads[1][1][b.kl:b.kl + b.kr])))

    # suff = k_left (a candidate: context = the read's first k_left bytes) vs k_left - 1 (counted, never a candidate)
    b = Builder(108)
    l0, l1 = b.snp_contexts()
    right = b.rand(b.kr)
    rows = [b.member(0, l0, right), b.member(0, l0[1:], right, bwt="A"), b.member(0, l0, right, pre=b.rand(3)),
            b.member(0, l0[1:], right, bwt="A"), b.member(0, l0, right)]
    rows += [b.member(1, l1[1:], right, bwt="C")] + [b.member(1, l1, right) for _ in range(4)]
    b.cluster(rows)
    out.append(b.build("fv_suff_k_left", counts(1, 1, [snp_ev(l0, l1, 3, 4)])))

    # lower-case BWT bytes count in the histogram but are never candidates (raw byte compare)
    b = Builder(109)
    l0, l1 = b.snp_contexts()
    right = b.rand(b.kr)
    rows = [b.member(0, l0, right) for _ in range(5)] + [b.member(1, l1, right, bwt="c") for _ in range(2)]
    rows += [b.member(1, l1, right) for _ in range(3)]
    b.cluster(rows)
    rows = [b.member(0, l0, right) for _ in range(5)] + [b.member(1, l1, right, bwt="c") for _ in range(5)]
    b.cluster(rows)  # frequent {C} in sample 1, no candidate read: not a candidate
    out.append(b.build("fv_lowercase_bwt", counts(1, 1, [snp_ev(l0, l1, 5, 3)])))

    # analysed lengths: 2 mcov - 1 (not), 2 mcov, max_clust_length, max_clust_length + 1 (not)
    b = Builder(110)
    b.snp_cluster(5, 4)
    l0, l1, _ = b.snp_cluster(5, 5)
    evs = [snp_ev(l0, l1, 5, 5)]
    b.snp_cluster(7, 6)  # 13: one too long
    for _ in range(10):
        l0, l1, _ = b.snp_cluster(6, 6)
        evs.append(snp_ev(l0, l1, 6, 6))
    out.append(b.build("fv_cluster_lengths", counts(11, 11, evs, n_analysed=11), pval=0.85, mcl=12))

    # text = nreads1 - 1 (sample 0) and nreads1 (sample 1)
    b = Builder(111)
    l0, l1 = b.snp_contexts()
    right = b.rand(b.kr)
    for _ in range(3):
        b.read(0, b.rand(80))
    h1 = b.read(1, l1 + right)
    for _ in range(3):
        b.read(1, b.rand(80))
    h0 = b.read(0, l0 + right)
    rows = [(h0, b.kl, 30, ord("A"))] * 5 + [(h1, b.kl, 30, ord("C"))] * 5
    b.cluster(rows)
    case = b.build("fv_text_at_nreads1", counts(1, 1, [snp_ev(l0, l1, 5, 5)]))
    assert set(case.text[case.clusters[0][0]:sum(case.clusters[0])].tolist()) == {case.nreads1 - 1, case.nreads1}
    out.append(case)
    return out


# ---- candidates: supporting reads per sample vs -c ------------------------------------------------------------------------
C_VALUES = (1, 20, 32, 33, 64, 65, 100, 150, 1000)


def candidate_cases():
    out = []
    for c in C_VALUES:
        cap = min(c, 150)
        b = Builder(200 + c, consensus_reads=c)
        evs, ncand = [], 0
        # (a cluster holds at most 150 records and the other sample needs mcov_out = 5 of them: 145 is the largest support)
        ns = sorted({n for n in (1, 31, 32, 33, 64, 65, 127, 128, 145, cap - 1, cap, cap + 1) if 1 <= n <= 145})
        for n in ns:
            for side in (0, 1):
                n0, n1 = (n, 5) if side == 0 else (5, n)
                # n supporting records; the frequency threshold is met with records whose suff < k_left when n < 5
                l0, l1 = b.snp_contexts()
                right = b.rand(b.kr)
                rows = [b.member(0, l0, right) for _ in range(n0)] + [b.member(0, l0[1:], right, bwt="A") for _ in range(5 - n0)]
                rows += [b.member(1, l1, right) for _ in range(n1)] + [b.member(1, l1[1:], right, bwt="C") for _ in range(5 - n1)]
                b.cluster(rows)
                evs.append(snp_ev(l0, l1, min(n0, cap), min(n1, cap)))
                ncand += 1
        # one sample whose reads share no consensus: a candidate, not a variant
        l0, _ = b.snp_contexts()
        rows = [b.member(0, l0, b.rand(b.kr)) for _ in range(5)] + [b.member(1, b.rand(b.kl - 1) + b"C", b.rand(b.kr)) for _ in range(5)]
        b.cluster(rows)
        groups = ("subset",) if c in (33, 100) else ()
        # (with -c 1 the one read of sample 1 is its own consensus: a variant, too far from sample 0 to be kept)
        out.append(b.build(f"cand_c{c}", counts(ncand + 1, ncand + (cap == 1), evs), groups=groups,
                           note=f"supporting reads {ns} in either sample"))
    # with -m 1 one record makes an allele frequent: supports up to 149, next to the 150-record cap
    for c in (100, 150, 1000):
        cap = min(c, 150)
        b = Builder(250 + c, consensus_reads=c, mcov_out=1)
        evs = []
        for n0, n1 in ((149, 1), (1, 149), (148, 2), (2, 148)):
            l0, l1, _ = b.snp_cluster(n0, n1)
            evs.append(snp_ev(l0, l1, min(n0, cap), min(n1, cap)))
        out.append(b.build(f"cand_c{c}_m1", counts(len(evs), len(evs), evs), groups=("subset",) if c == 150 else ()))
    return out


# ---- consensus / support --------------------------------------------------------------------------------------------------
def _column_cluster(columns, n_reads, base):
    """n_reads contexts = base with the given columns {position: chars per read} overwritten"""
    ctxs = []
    for j in range(n_reads):
        c = bytearray(base)
        for pos, chars in columns.items():
            c[pos] = ord(chars[j])
        ctxs.append(bytes(c))
    return ctxs


def consensus(ctxs):
    """cons::increment (ref:include.hpp:334-371): counts by base_to_int, the stored char is the read's that took the lead"""
    code = {ord(x): i for i, x in enumerate("ACGT")}
    code.update({ord(x): i for i, x in enumerate("acgt")})
    kl = len(ctxs[0])
    out = bytearray(b"A" * kl)
    for i in range(kl):
        cnt = [0, 0, 0, 0]
        for c in ctxs:
            v = code.get(c[i], 0)
            cnt[v] += 1
            if cnt[v] > cnt[code.get(out[i], 0)]:
                out[i] = c[i]
    return bytes(out)


def consensus_cases():
    out = []
    # per-column ties: the first base to reach the final maximum wins (order-dependent), an all-'a' column keeps 'A',
    # a column of 'c' then 'C' keeps the 'c'
    b = Builder(301, max_err=31, max_snvs=31)  # every read supports, every pair is kept: the .snp shows both consensus strings
    base0 = bytearray(b.rand(b.kl - 1) + b"A")
    base1 = bytearray(bytes(base0[:-1]) + b"C")
    cols0 = {3: "CGGCTA", 7: "GCCGAT", 11: "aaaaaa", 15: "cCCCCC", 19: "TTAACC", 22: "ACGTAC"}
    cols1 = {3: "GCCGTT", 9: "aAaAaA", 13: "tTtGGG", 20: "CAAC" + "TT", 25: "GGTTAA"}
    c0 = _column_cluster(cols0, 6, base0)
    c1 = _column_cluster(cols1, 6, base1)
    right = b.rand(b.kr)
    rows = [b.member(0, x, right, bwt="A") for x in c0] + [b.member(1, x, right, bwt="C") for x in c1]
    b.cluster(rows)
    k0, k1 = consensus(c0), consensus(c1)
    assert [k0[i:i + 1] for i in (3, 7, 11, 15, 19, 22)] == [b"G", b"C", b"A", b"c", b"T", b"A"]
    assert [k1[i:i + 1] for i in (3, 9, 13, 20, 25)] == [b"C", b"A", b"t", b"A", b"G"]
    assert distance(k0, k1, b.params["max_gap"])[1] == 0
    out.append(b.build("cons_column_ties", counts(1, 1, [snp_ev(k0, k1, 6, 6)], consensus=(k0, k1)), groups=("subset", "reads")))

    # reads at exactly max_err and max_err + 1 mismatches of the consensus; the same with max_err = 0 and with k_left > 32
    for name, kw, e in (("cons_max_err2", {}, 2), ("cons_max_err0", {"max_err": 0}, 0), ("cons_max_err1_kl40", {"k_left": 40, "k_right": 35, "max_err": 1}, 1)):
        b = Builder(302 + e, **kw)
        l0, l1 = b.snp_contexts()
        right = b.rand(b.kr)

        def mut(ctx, k, at=1):
            c = bytearray(ctx)
            for p in range(at, at + 2 * k, 2):
                c[p] = ord("T") if c[p] != ord("T") else ord("G")
            return bytes(c)
        rows = [b.member(0, l0, right) for _ in range(4)] + [b.member(0, mut(l0, e), right), b.member(0, mut(l0, e + 1), right)]
        rows += [b.member(1, l1, right) for _ in range(4)] + [b.member(1, mut(l1, e + 1, 5), right), b.member(1, mut(l1, e, 7), right)]
        b.cluster(rows)
        out.append(b.build(name, counts(1, 1, [snp_ev(l0, l1, 5, 5)])))
    return out


# ---- distance ------------------------------------------------------------------------------------------------------------
def _indel_pair(b, g, kl, max_gap):
    """(l0, l1) with a planted indel of |g| at the right end: gap > 0 = l1 is X + l0[:kl-g] (higher path), gap < 0 the reverse"""
    for _ in range(1000):
        a = b.rand(kl)
        x = b.rand(abs(g))
        bb = x + a[:kl - abs(g)]
        l0, l1 = (a, bb) if g > 0 else (bb, a)
        if distance(l0, l1, max_gap) == (0, g):
            return l0, l1
    raise AssertionError(f"no context pair with a winning indel of {g} (k_left {kl}, max_gap {max_gap})")


def _search_pair(b, kl, max_gap, pred, alphabet=b"AC"):
    for _ in range(200000):
        l0, l1 = b.rand(kl, alphabet), b.rand(kl, alphabet)
        d0, ab, ba = dist_table(l0, l1, max_gap)
        if pred(d0, ab, ba):
            return l0, l1
    raise AssertionError("no context pair found")


def _pair_cluster(b, l0, l1, n0=5, n1=5):
    right = b.rand(b.kr)
    b.cluster([b.member(0, l0, right, bwt="A") for _ in range(n0)] + [b.member(1, l1, right, bwt="C") for _ in range(n1)])
    D, g = distance(l0, l1, b.params["max_gap"])
    return D, g, ev("SNP" if g == 0 else "INDEL", type_string(l0, l1, g), n0, n1)


def distance_cases():
    out = []
    for kl, mg in ((31, 10), (32, 32), (40, 12), (64, 64), (128, 128)):
        b = Builder(400 + kl, k_left=kl, k_right=30, max_gap=mg)
        evs = []
        # a planted indel of g wins while g stays below the Hamming distance of the unshifted contexts (about 3/4 k_left for
        # random ones): every g up to 12, then g around the 32-lane strides of K4's distance loop, up to 0.6 k_left
        lim = min(mg, int(0.6 * kl))
        gs = sorted({g for g in list(range(1, 13)) + [16, 20, 31, 32, 33, 38, 40, 63, 64, 65, 70, lim] if g <= lim})
        for g in gs:
            for sg in (1, -1):
                l0, l1 = _indel_pair(b, sg * g, kl, mg)
                D, gg, e = _pair_cluster(b, l0, l1)
                assert (D, gg) == (0, sg * g)
                evs.append(e)
        out.append(b.build(f"dist_indels_kl{kl}_g{mg}", counts(len(evs), len(evs), evs),
                           groups=("subset",) if kl in (32, 128) else ()))

    def mins(ab):
        m = min(ab)
        return m, [i for i, v in enumerate(ab) if v == m]
    preds = {
        "d0_eq_min_ab": lambda d0, ab, ba: d0 == min(ab) < min(ba),
        "min_ab_eq_min_ba": lambda d0, ab, ba: min(ab) == min(ba) < d0,
        "all_three_equal": lambda d0, ab, ba: d0 == min(ab) == min(ba),
        "ab_minima_several_g": lambda d0, ab, ba: len(mins(ab)[1]) >= 2 and min(ab) < min(ba) and min(ab) <= d0,
        "ba_minima_several_g": lambda d0, ab, ba: len(mins(ba)[1]) >= 2 and min(ba) <= min(ab) and min(ba) <= d0,
    }
    for kl, mg in ((12, 5), (31, 10), (36, 8)):
        b = Builder(450 + kl, k_left=kl, k_right=20, max_gap=mg, max_snvs=kl)
        evs = []
        for nm, pr in preds.items():
            l0, l1 = _search_pair(b, kl, mg, pr)
            evs.append(_pair_cluster(b, l0, l1)[2])
        out.append(b.build(f"dist_ties_kl{kl}", counts(len(evs), len(evs), evs), note=" ".join(preds)))

    # D = max_snvs (kept) and max_snvs + 1 (a variant, not kept)
    b = Builder(480)
    evs = []
    for D in (3, 4, 0):
        while True:
            l0 = b.rand(b.kl)
            l1 = bytearray(l0)
            for p in b.rng.choice(b.kl, size=D, replace=False):
                l1[p] = ord("ACGT"[("ACGT".index(chr(l1[p])) + 1) % 4])
            l1 = bytes(l1)
            if distance(l0, l1, 10) == (D, 0):
                break
        _, _, e = _pair_cluster(b, l0, l1)
        if D <= 3:
            evs.append(e)
    out.append(b.build("dist_max_snvs", counts(3, 3, evs)))
    return out


# ---- context lengths -----------------------------------------------------------------------------------------------------
KL_VALUES = (1, 2, 31, 32, 33, 64, 127, 128)
KR_VALUES = (1, 30, 32, 33, 128)


def context_cases():
    out = []
    for kl in KL_VALUES:
        for kr in KR_VALUES:
            for mg in sorted({1, kl}):
                b = Builder(1000 + kl * 7 + kr * 3 + mg, k_left=kl, k_right=kr, max_gap=mg)
                evs = []
                l0, l1 = b.snp_contexts(max_gap=mg)
                D, g = distance(l0, l1, mg)
                assert (D, g) == ((0, -1) if kl == 1 else (1, 0))
                kind = "SNP" if g == 0 else "INDEL"
                # a full right context; one cut by the read end; an empty one (right_pos = read length)
                for rlen in (kr, max(kr // 2, 1) if kr > 1 else 0, 0):
                    right = b.rand(kr)[:rlen]
                    b.cluster([b.member(0, l0, right) for _ in range(5)] + [b.member(1, l1, b.rand(kr)) for _ in range(6)])
                    evs.append(ev(kind, type_string(l0, l1, g), 5, 6) + (len(right),))
                grp = ("subset",) if kl in (32, 33, 128) and mg == kl else ()
                out.append(b.build(f"ctx_L{kl}_R{kr}_g{mg}", counts(3, 3, [e[:4] for e in evs], right_lens=[e[4] for e in evs]),
                                   groups=grp))
    # right_pos past the read's end: the reference's substr throws
    b = Builder(1999)
    l0, l1 = b.snp_contexts()
    h = b.read(1, b.rand(40))
    rows = [b.member(0, l0, b.rand(b.kr), lcp=30) for _ in range(5)] + [b.member(1, l1, b.rand(b.kr), lcp=30) for _ in range(5)]
    rows.append((h, 41, 31, ord("G")))  # the LCP maximum: its suffix starts one past the end of its 40-base read
    b.cluster(rows)
    out.append(b.build("ctx_right_pos_past_end", counts(1, 1, []), refuse=True))
    return out


# ---- reads ---------------------------------------------------------------------------------------------------------------
def reads_cases():
    out = []

    def base_case(seed, ragged=False, **kw):
        """six SNP clusters of 5 + 6 records; ragged: random read starts, empty reads, one right context cut per cluster"""
        b = Builder(seed, **kw)
        evs = []
        for _ in range(6):
            l0, l1 = b.snp_contexts()
            right = b.rand(b.kr)
            pre = (lambda: b.rand(int(b.rng.integers(0, 25)))) if ragged else (lambda: b"")
            rows = [b.member(0, l0, right, pre=pre(), bwt="A") for _ in range(5)]
            rows += [b.member(1, l1, (right[:int(b.rng.integers(0, b.kr))] if ragged and k == 0 else right), pre=pre(), bwt="C")
                     for k in range(6)]
            if ragged:
                b.read(0, b"")
                b.read(1, b"")
            b.cluster(rows)
            evs.append(snp_ev(l0, l1, 5, 6))
        return b, evs
    b, evs = base_case(501)
    out.append(b.build("reads_upper_uniform", counts(6, 6, evs, saw_n=0), uniform=True, groups=("subset", "reads")))
    b, evs = base_case(502)
    lower = bytearray(b.rand(60))
    lower[17] = ord("g")
    out.append(b.build("reads_one_lowercase_outside", counts(6, 6, evs, saw_n=0), uniform=True, groups=("subset", "reads"),
                       extra_reads=[(0, bytes(lower))]))

    b, evs = base_case(503)
    # one sample-0 read of one cluster with a lower-case base inside its context (1 mismatch: still supported)
    r = bytearray(b.reads[0][6])
    r[4] = r[4] | 0x20
    b.reads[0][6] = bytes(r)
    out.append(b.build("reads_lowercase_in_context", counts(6, 6, evs, saw_n=0), uniform=True, groups=("subset", "reads")))

    b, evs = base_case(504)
    r = bytearray(b.reads[1][13])
    r[3], r[9] = ord("R"), ord("-")
    b.reads[1][13] = bytes(r)
    out.append(b.build("reads_iupac_in_context", counts(6, 6, evs, saw_n=0), uniform=True, groups=("subset", "reads"),
                       extra_reads=[(1, b"ACGTRYACGT-ACGT")]))
    b, evs = base_case(505)
    out.append(b.build("reads_iupac_outside_context", counts(6, 6, evs, saw_n=0), uniform=True, groups=("subset", "reads"),
                       extra_reads=[(0, b"ACGTRACGT"), (1, b"AC-GT")]))
    b, evs = base_case(506, ragged=True)
    out.append(b.build("reads_ragged_with_empty", counts(6, 6, evs, saw_n=0), groups=("subset", "reads"),
                       extra_reads=[(0, b""), (1, b"")]))
    b, evs = base_case(507, ragged=True, k_left=40, k_right=35, max_gap=12)
    out.append(b.build("reads_ragged_kl40", counts(6, 6, evs, saw_n=0), groups=("subset", "reads")))
    # an N inside one context: the reference draws rand() % 4 there, so only the text (N counted as 'A' on both sides) and
    # the saw_n flag are compared
    b, evs = base_case(508)
    r = bytearray(b.reads[0][8])
    r[10] = ord("N")
    b.reads[0][8] = bytes(r)
    out.append(b.build("reads_n_in_context", counts(6, 6, evs, saw_n=1), uniform=True, groups=("subset", "reads")))
    return out


# ---- volume --------------------------------------------------------------------------------------------------------------
def volume_case(n_clusters=100_000, n_pos=3_000_000, seed=900):
    """n_clusters designed SNP clusters of 10-14 records in n_pos positions with default options: several K3x / K3b / K4
    rounds and an overflow of the first flagged-list capacity guess (n_clusters >> m / 256 + 2048).  Every 7th cluster
    carries 4 substitutions (a variant, not kept), every 11th an indel of 1-3 (an INDEL event)."""
    rng = np.random.default_rng(seed)
    kl, kr = 31, 30
    P = 4096  # read pairs, reused by many clusters
    L = 100
    r0 = np.frombuffer(ACGT, dtype=np.uint8)[rng.integers(0, 4, size=(P, L))]
    r1 = r0.copy()
    at = 40  # suff of every planted record: left context [9, 40), right context [40, 70)
    kind = np.arange(P) % 77
    lut = np.zeros(256, dtype=np.uint8)
    lut[np.frombuffer(ACGT, dtype=np.uint8)] = np.frombuffer(b"CGTA", dtype=np.uint8)
    r1[:, at - 1] = lut[r0[:, at - 1]]                       # the SNP
    sub = kind % 7 == 0
    for q in (at - 5, at - 12, at - 20):                    # + 3 substitutions: D = 4
        r1[sub, q] = lut[r0[sub, q]]
    for p in np.nonzero(~sub & (kind % 11 == 0))[0]:         # an insertion of 1-3 bases on the lower path: INDEL, D = 0
        g = 1 + p % 3
        r1[p, at - kl:at] = np.concatenate([np.frombuffer(ACGT, dtype=np.uint8)[rng.integers(0, 4, size=g)], r0[p, at - kl:at - g]])
    reads = np.concatenate([r0, r1])
    sizes = rng.integers(5, 8, size=(n_clusters, 2))   # records per sample
    lens = sizes.sum(1)
    gap = n_pos // n_clusters - int(lens.mean()) - 1
    assert gap >= 2
    lcp = np.zeros(n_pos, dtype=np.uint32)
    text = np.zeros(n_pos, dtype=np.uint32)
    suff = np.full(n_pos, 0, dtype=np.uint32)
    bwt = np.full(n_pos, ord("T"), dtype=np.uint8)
    starts = 3 + np.concatenate([[0], np.cumsum(lens + gap)[:-1]])
    assert starts[-1] + lens[-1] + 3 < n_pos
    pair = rng.integers(0, P, size=n_clusters)
    idx = np.repeat(starts, lens) + (np.arange(lens.sum()) - np.repeat(np.cumsum(lens) - lens, lens))
    in_cl = np.repeat(np.arange(n_clusters), lens)
    pos_in = idx - starts[in_cl]
    s1 = pos_in >= sizes[in_cl, 0]
    lcp[idx] = 30                                      # the first record gives the right context
    text[idx] = pair[in_cl] + np.where(s1, P, 0)
    suff[idx] = at
    bwt[idx] = np.where(s1, lut[r0[pair[in_cl], at - 1]], r0[pair[in_cl], at - 1])  # (an indel pair's context keeps no SNP)
    off = O.uniform_read_offsets(2 * P, L)
    kept = n_clusters - int(np.sum(sub[pair]))
    return Case("volume", lcp, text, suff, bwt, reads.reshape(-1).copy(), off, P, dict(DEFAULTS), 0.99, int(lens.max()),
                list(zip(starts.tolist(), lens.tolist())),
                dict(n_analysed=n_clusters, n_candidates=n_clusters, n_variants=n_clusters, n_events=kept),
                groups=("subset",), note="volume")


def cli_case():
    """ragged reads for `clust2snp -c 100 -L 40 -R 33 -g 12 -e 1 -p 1`: supports above 32 and 64 (K4's general path), indels
    of both signs, SNPs with a read at max_err + 1 mismatches, right contexts cut by the read end"""
    b = Builder(700, k_left=40, k_right=33, max_gap=12, max_err=1, consensus_reads=100)
    evs = []

    def pre():
        return b.rand(int(b.rng.integers(0, 30)))
    for n0, n1 in ((70, 45), (33, 5), (5, 32), (6, 7)):
        l0, l1 = b.snp_contexts()
        right = b.rand(int(b.rng.integers(10, b.kr + 5)))
        rows = [b.member(0, l0, right, pre=pre()) for _ in range(n0)] + [b.member(1, l1, right, pre=pre()) for _ in range(n1)]
        rows.append(b.member(1, l1[:3] + l1[3:5].translate(bytes.maketrans(b"ACGT", b"CGTA")) + l1[5:], right, pre=pre()))
        b.cluster(rows)
        evs.append(snp_ev(l0, l1, min(n0, 100), min(n1, 100)))
    for g in (3, -5, 12):
        l0, l1 = _indel_pair(b, g, b.kl, b.params["max_gap"])
        right = b.rand(b.kr)
        b.cluster([b.member(0, l0, right, pre=pre(), bwt="G") for _ in range(6)] + [b.member(1, l1, right, pre=pre(), bwt="T") for _ in range(8)])
        evs.append(ev("INDEL", type_string(l0, l1, g), 6, 8))
    return b.build("cli_ragged", counts(len(evs), len(evs), evs))


def all_cases():
    return find_variants_cases() + candidate_cases() + consensus_cases() + distance_cases() + context_cases() + reads_cases()


# ---- .snp parsing --------------------------------------------------------------------------------------------------------
HDR = re.compile(rb">(SNP|INDEL)_(higher|lower)_path_(\d+)\|P_1:(\d+)_([^|]*)\|(\d+)\|nb_pol_1")


def parse_snp(text: bytes):
    """-> [(kind, type, supp0, supp1, right_len, left0, left1, right)] from the .snp bytes"""
    lines = text.split(b"\n")
    assert lines[-1] == b""
    out = []
    for i in range(0, len(lines) - 1, 4):
        h0, s0, h1, s1 = lines[i:i + 4]
        m0, m1 = HDR.fullmatch(h0), HDR.fullmatch(h1)
        assert m0 and m1 and m0.group(2) == b"higher" and m1.group(2) == b"lower", (h0, h1)
        assert m0.group(3) == m1.group(3) and m0.group(5) == m1.group(5)
        rl = int(m0.group(4))
        out.append((m0.group(1).decode(), m0.group(5), int(m0.group(6)), int(m1.group(6)), rl, s0[:len(s0) - rl], s1[:len(s1) - rl],
                    s0[len(s0) - rl:]))
    return out
