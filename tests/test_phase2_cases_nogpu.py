"""The designed phase-2 cases (tests/phase2_cases.py) through the oracle: each must produce what it was designed to produce, so
every case is known to reach its branch before the CUDA path is compared with the oracle on it (test_phase2_paths_gpu.py)."""
import numpy as np
import pytest

from oracle import oracle as O
from tests import phase2_cases as P

CASES = P.all_cases() + [P.cli_case()]


def run_oracle(case):
    es, el, _, _ = O.cluster_lm(case.lcp, case.bwt, P.K, P.MIN_LEN)
    return O.find_events(case.lcp, case.text, case.suff, case.bwt, es, el, case.oparams(), case.max_clust_length, case.bases,
                         case.off)


@pytest.mark.parametrize("case", CASES, ids=[c.name for c in CASES])
def test_oracle_shows_planted_expectation(case):
    x = case.expect
    if case.refuse:
        with pytest.raises(ValueError, match="crash"):
            run_oracle(case)
        return
    text, res = run_oracle(case)
    got = P.parse_snp(text)
    assert [g[:4] for g in got] == x["events"]
    assert (res.n_candidates, res.n_variants, res.n_events) == (x["n_candidates"], x["n_variants"], x["n_events"])
    if "n_analysed" in x:
        assert res.n_analysed == x["n_analysed"]
    if "saw_n" in x:
        assert bool(res.flags & O.FLAG_SAW_N) == bool(x["saw_n"])
    if "right" in x:
        assert got[0][7] == x["right"]
    if "right_lens" in x:
        assert [g[4] for g in got] == x["right_lens"]
    if "consensus" in x:
        assert (got[0][5], got[0][6]) == x["consensus"]


def test_cases_cover_the_grid():
    names = {c.name for c in CASES}
    for kl in P.KL_VALUES:
        for kr in P.KR_VALUES:
            assert f"ctx_L{kl}_R{kr}_g1" in names and f"ctx_L{kl}_R{kr}_g{kl}" in names
    for c in P.C_VALUES:
        assert f"cand_c{c}" in names


def test_support_above_64_with_c100():
    """-c 100: supports above 64 (the restatement used to stop at 64 reads per sample) and above the uint8-friendly 32"""
    case = next(c for c in CASES if c.name == "cand_c100")
    text, _ = run_oracle(case)
    supports = [s for g in P.parse_snp(text) for s in g[2:4]]
    assert max(supports) == 100 and 99 in supports and 65 < sorted(supports)[-3]


def test_supports_up_to_the_cluster_size():
    """supports past 127 (a signed 8-bit field) up to 145 (-m 5) and 149 (-m 1) next to the 150-record cluster limit"""
    def supports(name):
        text, _ = run_oracle(next(c for c in CASES if c.name == name))
        return {s for g in P.parse_snp(text) for s in g[2:4]}
    for c in (150, 1000):
        assert {1, 31, 32, 33, 64, 65, 127, 128, 145} <= supports(f"cand_c{c}")
        assert {148, 149} <= supports(f"cand_c{c}_m1")
    assert max(supports("cand_c100")) == 100 and max(supports("cand_c100_m1")) == 100


def test_indels_past_the_32_lane_strides():
    """planted indels whose winning gap is served by the second and third iteration of K4's strided distance loop"""
    for name, want in (("dist_indels_kl128_g128", {32, 33, 63, 64, 65, 70, 76}), ("dist_indels_kl64_g64", {31, 32, 33, 38})):
        text, _ = run_oracle(next(c for c in CASES if c.name == name))
        types = [g[1] for g in P.parse_snp(text) if g[0] == "INDEL"]
        gaps = {len(t) - 1 if t.endswith(b"/") else 1 - len(t) for t in types}  # "XX/": higher path, "/XX": lower path
        assert want <= gaps and {-g for g in want} <= gaps, name


def test_oracle_accepts_any_consensus_reads():
    case = next(c for c in CASES if c.name == "cand_c1000")
    assert case.params["consensus_reads"] == 1000
    _, res = run_oracle(case)
    assert res.n_events > 0
    p = case.oparams()
    p.consensus_reads = 0
    es, el, _, _ = O.cluster_lm(case.lcp, case.bwt, P.K, P.MIN_LEN)
    with pytest.raises(ValueError, match="supports"):
        O.find_events(case.lcp, case.text, case.suff, case.bwt, es, el, p, case.max_clust_length, case.bases, case.off)


def test_volume_case():
    case = P.volume_case()
    text, res = run_oracle(case)
    x = case.expect
    assert (res.n_analysed, res.n_candidates, res.n_variants, res.n_events) == (
        x["n_analysed"], x["n_candidates"], x["n_variants"], x["n_events"])
    kinds = [g[0] for g in P.parse_snp(text)]
    assert kinds.count("INDEL") > 1000 and kinds.count("SNP") > 50_000
    st = O.statistics(*O.cluster_lm(case.lcp, case.bwt, P.K, P.MIN_LEN)[:2], 5, case.pval)
    assert st.max_clust_length == case.max_clust_length
    # far more flagged clusters than one K3x round of a 148-SM device (148 * 16 * 32) and the first capacity guess
    assert x["n_candidates"] > 148 * 16 * 32 and x["n_candidates"] > len(case.clusters) // 256 + 2048
    assert np.all(np.diff([s for s, _ in case.clusters]) > 0)
