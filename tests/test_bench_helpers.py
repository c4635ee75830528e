"""not gpu: bench.py's sampled property check of an index (what vouches for the C3-size index nobody else can build):
passes on a correct index, fails on a wrong LCP value, on two swapped records and on a wrong BWT byte."""
import importlib.util
import os

import numpy as np

from ebwt2snp_b200 import synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench():
    spec = importlib.util.spec_from_file_location("bench_module", os.path.join(ROOT, "bench.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


def test_index_property_check_detects_damage():
    b = _bench()
    rs = synth.make_config("tiny", seed=9)
    eg = synth.build_egsa(rs.reads)
    ok, n_checked = b.check_egsa_sample(rs, eg, samples=30000)
    assert ok and n_checked > 30000
    n = int(eg["n"])
    every = dict(samples=4 * n)  # (nearly) every record gets sampled

    bad = dict(eg)
    lcp = eg["lcp"].clone()
    lcp[n // 2] += 1
    bad["lcp"] = lcp
    assert not b.check_egsa_sample(rs, bad, **every)[0]

    bad = dict(eg)
    t, s = eg["text"].clone(), eg["suff"].clone()
    i = n // 3
    t[[i, i + 1]] = t[[i + 1, i]]
    s[[i, i + 1]] = s[[i + 1, i]]
    bad["text"], bad["suff"] = t, s
    assert not b.check_egsa_sample(rs, bad, **every)[0]

    bad = dict(eg)
    bw = eg["bwt"].clone()
    j = int(np.flatnonzero(eg["suff"].numpy() > 0)[1234])
    bw[j] = ord("A") if bw[j] != ord("A") else ord("C")
    bad["bwt"] = bw
    assert not b.check_egsa_sample(rs, bad, **every)[0]


def test_dump_outputs_files_sample_and_budget(tmp_path, monkeypatch):
    """--dump-outputs: float32 / float64 .npy files only, the same files for the same outputs, a seeded sample of records and
    events once they exceed the budget, contexts cut to the bytes the events use"""
    from ebwt2snp_b200 import api
    b = _bench()
    monkeypatch.setattr(b, "DUMP_CLUSTER_SAMPLE", 1000)
    monkeypatch.setattr(b, "DUMP_EVENT_BYTES", 300 * (2 * 8 + 6 * 4 + 3 * 4 * 31))
    rng = np.random.default_rng(2)
    start = np.sort(rng.choice(1 << 40, size=5000, replace=False)).astype(np.uint64)
    ln = rng.integers(2, 70, size=5000).astype(np.uint16)
    events = []
    for i in range(500):
        e = api.Event(D=int(rng.integers(0, 3)), gap=int(rng.integers(-5, 5)), supp0=i, supp1=i + 1, right_len=30, keep=i % 2,
                      cluster_start=int(start[i * 10]))
        e.left0 = e.left1 = bytes(rng.choice(list(b"ACGT"), size=31).astype(np.uint8))
        e.right = bytes(rng.choice(list(b"ACGT"), size=30).astype(np.uint8))
        events.append(e)
    counts = {"n_written": 5000, "n_events": 500, "max_clust_length": 69}
    a = b.dump_outputs(str(tmp_path / "a"), counts, start, ln, events, api.Event, seed=1)
    b.dump_outputs(str(tmp_path / "b"), counts, start, ln, events, api.Event, seed=1)
    names = sorted(os.listdir(tmp_path / "a"))
    assert names == sorted(f"{k}.npy" for k in a) and names == sorted(os.listdir(tmp_path / "b"))
    for f in names:
        x, y = np.load(tmp_path / "a" / f), np.load(tmp_path / "b" / f)
        assert x.dtype in (np.float32, np.float64) and np.array_equal(x, y), f
    assert a["counts"].tolist() == [69, 500, 5000]  # max_clust_length, n_events, n_written: sorted by name
    idx = a["cluster_index"].astype(np.int64)
    assert len(idx) == 1000 and np.all(np.diff(idx) > 0)
    assert np.array_equal(a["cluster_start"], start[idx].astype(np.float64)) and np.array_equal(a["cluster_len"], ln[idx])
    keep = a["event_index"].astype(np.int64)
    assert len(keep) == 300 and a["event_left0"].shape == (300, 31)
    assert a["event_fields"][:, 2].tolist() == keep.tolist()  # supp0 = the event's index
    assert bytes(a["event_right"][0].astype(np.uint8)) == bytes(events[keep[0]].right) + b"\0"
    assert sum(v.nbytes for v in a.values()) < 64 << 20
    small = b.dump_outputs(str(tmp_path / "c"), counts, start[:10], ln[:10], [], api.Event)
    assert len(small["cluster_index"]) == 10 and small["event_left0"].shape == (0, 0)
