"""The key-range helpers of sharding.py on ragged collections (bases, off), checked against the oracle's index (no GPU): the first key
words that e2s_build_egsa_ragged_range_dev compares with its range are ordered along the index, and key_range_cuts splits it evenly."""
import numpy as np

from ebwt2snp_b200 import sharding
from oracle import oracle as O
from tests.test_builder_gpu import BASES, make_case, ragged_from_genome


def with_empty_and_long(rng):
    """empty reads, reads shorter and longer than 32 bases (up to five key words)"""
    return ragged_from_genome(rng, 8_000, 1_500, 0, 150)


def index_keys(bases, off, e):
    return sharding.first_key_words((bases, off), e["text"].astype(np.int64), e["suff"].astype(np.int64))


def test_first_key_words_are_ordered_along_the_ragged_index():
    rng = np.random.default_rng(3)
    for bases, off in (with_empty_and_long(rng), make_case("tiny"), make_case("two_length_places"), make_case("skewed")):
        e = O.build_egsa_ragged(bases, off)
        keys = index_keys(bases, off, e)
        assert len(keys) == e["n"]
        assert np.all(keys[1:] >= keys[:-1])
        assert np.count_nonzero(keys == 0) >= len(off) - 1  # every terminator suffix has key 0


def test_first_key_words_agree_between_matrix_and_ragged_forms():
    rng = np.random.default_rng(4)
    R, L = 300, 45
    reads = BASES[rng.integers(0, 4, size=(R, L))]
    off = np.arange(R + 1, dtype=np.uint64) * np.uint64(L)
    rows, cols = rng.integers(0, R, size=5000), rng.integers(0, L + 1, size=5000)
    assert np.array_equal(sharding.first_key_words(reads, rows, cols), sharding.first_key_words((reads.reshape(-1), off), rows, cols))


def test_ragged_cuts_tile_the_key_space_and_balance_the_records():
    rng = np.random.default_rng(5)
    bases, off = ragged_from_genome(rng, 60_000, 6_000, 50, 150)  # no heavy key: a random genome, the key-0 run is R of ~600 k
    e = O.build_egsa_ragged(bases, off)
    keys = index_keys(bases, off, e)
    n = e["n"]
    k0 = int(np.count_nonzero(keys == 0))
    for parts in (2, 3, 5, 7, 8):
        cuts = sharding.key_range_cuts(parts, (bases, off), sample=1 << 15, seed=parts)
        assert len(cuts) == parts and cuts[0][0] == 0 and cuts[-1][1] == 0
        for (lo, hi), (lo2, _) in zip(cuts[:-1], cuts[1:]):
            assert lo < hi == lo2
        counts = [int(np.count_nonzero((keys >= lo) & ((keys < hi) | (hi == 0)))) for lo, hi in cuts]
        assert sum(counts) == n
        assert all(abs(c - n / parts) <= 0.25 * n / parts for c in counts), (parts, counts)
        assert counts[0] >= k0  # the key-0 run stays in the first range


def test_key_zero_run_stays_in_the_first_range_when_it_is_heavy():
    """poly-A reads: key 0 holds far more than n / parts suffixes; it is never split, the later cuts are strictly increasing"""
    bases, off = make_case("skewed")
    e = O.build_egsa_ragged(bases, off)
    keys = index_keys(bases, off, e)
    k0 = int(np.count_nonzero(keys == 0))
    assert k0 > e["n"] // 4
    for parts in (2, 4, 7):
        cuts = sharding.key_range_cuts(parts, (bases, off), sample=1 << 14, seed=1)
        assert cuts[0] == (0, cuts[1][0]) and cuts[1][0] >= 1
        assert all(lo < hi for lo, hi in cuts[:-1])
        first = int(np.count_nonzero(keys < cuts[0][1]))
        assert first >= k0
