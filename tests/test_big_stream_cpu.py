"""CPU: the library construction of the exact reference (exact_ref.library_hits / stream_hits / library_counts / stream_counts,
big_stream.layout) against the direct reference (exact_ref.scan, test_sdk_selection_cpu.exact_counts) on the stream itself. The layout
is big_stream's with X = 2^24 instead of 2^32: about 25 Mbases, with the same placement rules, periodic read and exception bytes as the
stream of more than 2^32 bases the GPU tests (test_gpu_past_2_32.py) build."""
import numpy as np
import pytest

import big_stream
import exact_ref
from test_sdk_selection_cpu import exact_counts

X = 1 << 24
LONG = (1 << 22) - 1


@pytest.fixture(scope="module")
def small():
    L = big_stream.layout(X, filler_len=1 << 16, n_filler=16, long_len=LONG, genome=500_000, hit_reads=800, seed=8200)
    bases, off = big_stream.materialise(L)
    return L, bases, off


def test_layout_places_its_reads(small):
    L, bases, off = small
    r, D = L["rows"], L["D"]
    assert off[r["S"]] < X < off[r["S"] + 1], "S straddles X"
    assert off[r["E"]] == off[r["T"]] == off[r["E"] + 1] == X + D, "E is empty and it and T start at X + D"
    assert D == off[r["suffix"]] and D % 4 != 0
    assert off[r["P"] + 1] - off[r["P"]] == LONG and off[r["P"]] > X
    assert off[-1] > X + D + LONG
    other = ~np.isin(bases, np.frombuffer(b"ACGT", dtype=np.uint8))
    assert other[:X].any() and other[X:].any(), "bytes other than ACGT on both sides of X"
    n_hit = 2 * 800
    assert sorted(L["order"][(L["order"] >= 16) & (L["order"] < 16 + n_hit)].tolist()) == list(range(16, 16 + n_hit)), "hit reads once each"


def test_library_hits_equal_the_direct_scan(small):
    L, bases, off = small
    k, kmers, r = L["k"], L["kmers"], L["rows"]
    lib_hits = exact_ref.library_hits(L["lib"], k, kmers)
    want = exact_ref.scan(bases, off, k, kmers)
    got = exact_ref.stream_hits(lib_hits, L["order"])
    for w, g in zip(want, got):
        assert np.array_equal(w, g)
    for i, lr in enumerate(L["lib"]):
        if i < 16 or i >= 16 + 1600 + 4:
            assert lib_hits[i][0].shape[0] == 0, "fillers and pads have no hit"
    ro = want[0].astype(np.int64)
    for row in ("S", "T", "P"):
        assert ro[r[row] + 1] > ro[r[row]], f"{row} has hits"
    p_pos = want[2][ro[r["P"]]:ro[r["P"] + 1]].astype(np.int64)
    assert p_pos.min() > LONG - 512 and p_pos.max() == LONG, "P's hits lie in its last 512 bases, one ends at its last base"
    # the suffix: the stream from read `suffix` on, in its own coordinates
    s0 = r["suffix"]
    sub = off[s0:] - off[s0]
    want_s = exact_ref.scan(bases[int(off[s0]):], sub, k, kmers)
    got_s = exact_ref.stream_hits(lib_hits, L["order"][s0:])
    for w, g in zip(want_s, got_s):
        assert np.array_equal(w, g)
    assert sub[r["T"] - s0] == X


def test_library_counts_equal_the_direct_count(small):
    L, bases, off = small
    k = L["k"]
    lib_counts = exact_ref.library_counts(L["lib"], k)
    raw = bases.tobytes()
    for mc in (1, 2):
        wk, wc = exact_counts(raw, off, k, min_count=mc)
        gk, gc = exact_ref.stream_counts(lib_counts, L["order"], min_count=mc)
        assert np.array_equal(wk, gk) and np.array_equal(wc.astype(np.int64), gc)
        if mc == 1:
            c = gc
    assert c.min() == 1 and (c == 2).any() and c.max() > 50                  # the GPU layout reaches counts in the hundreds
    hist, n_windows, n_distinct, max_count = exact_ref.spectrum(c, 1000)
    assert n_distinct == c.shape[0] and n_windows == int(c.sum()) and max_count == int(c.max())
    assert np.array_equal(hist[:999], np.bincount(c[c < 1000] - 1, minlength=999)) and hist[999] == int((c >= 1000).sum())
    # a slice in place (as jf_occurrences counts a file): the reads from T on
    t = L["rows"]["T"]
    sk, sc = exact_counts(raw[int(off[t]):], off[t:] - off[t], k, min_count=2)
    gk, gc = exact_ref.stream_counts(lib_counts, L["order"][t:], min_count=2)
    assert np.array_equal(sk, gk) and np.array_equal(sc.astype(np.int64), gc)
