"""CPU: the numpy / scipy reference (exact_ref.py) against the C oracle and the stored golden vectors, stage by stage. The GPU tests
of test_gpu_exact_reference.py take the reference as their judge at sizes the oracle cannot reach; these tests are why it may."""
import numpy as np
import pytest

import compare
import datagen
import exact_ref
import golden_util


def _pack(reads):
    seqs = [r.encode() if isinstance(r, str) else datagen.to_ascii(r).encode() for r in reads]
    off = np.zeros(len(seqs) + 1, dtype=np.uint64)
    np.cumsum([len(s) for s in seqs], out=off[1:])
    return b"".join(seqs), off


def _check_against_oracle(oracle, bases, off, k, kmers, fraction, min_size, pivot_min_scores=()):
    kmers = np.unique(np.asarray(kmers, dtype=np.uint64))
    ro, kid, pos = exact_ref.scan(bases, off, k, kmers, chunk_bases=1 << 16)   # small chunks: reads cross no chunk, several chunks run
    o_ro, o_kid, o_pos = oracle.scan(bases, off, k, kmers)
    assert np.array_equal(ro, o_ro) and np.array_equal(kid, o_kid) and np.array_equal(pos, o_pos), "hits differ"
    io, ir = exact_ref.index(ro, kid, len(kmers))
    o_io, o_ir = oracle.index(o_ro, o_kid, len(kmers))
    assert np.array_equal(io, o_io) and np.array_equal(ir, o_ir), "index differs"
    x, y, s = exact_ref.pairs(ro, kid, len(kmers))
    cx, cy, cs = oracle.canonical_sort(*oracle.connections(o_ro, o_kid, o_io, o_ir, min_score=1))
    ux, uy, us = compare.undirected(cx, cy, cs)
    assert np.array_equal(x, ux) and np.array_equal(y, uy) and np.array_equal(s.astype(np.uint64), us), "pair scores differ"
    # selection: the oracle's first n entries of its canonical directed list
    sel = exact_ref.select(x, y, s, fraction=fraction)
    n = int(len(cx) * fraction)
    assert sel["n_directed"] == n and sel["cut_score"] == (int(cs[n - 1]) if n else 0), "cut differs"
    want = {(min(a, b), max(a, b), int(c)) for a, b, c in zip(cx[:n].tolist(), cy[:n].tolist(), cs[:n].tolist())}
    assert set(zip(sel["x"].tolist(), sel["y"].tolist(), sel["score"].tolist())) == want, "selected set differs"
    comp = exact_ref.components(len(off) - 1, sel["x"], sel["y"], min_size)
    co, cm, _, _, _ = oracle.union_find(cx[:n], cy[:n], min_size=min_size)
    want_c = compare.components_partition(co, cm)
    got_c = sorted(tuple(int(v) for v in np.nonzero(comp["label"] == c)[0] + 1) for c in comp["comp_label"])
    assert got_c == want_c, "components differ"
    assert comp["comp_size"].tolist() == [len(c) for c in sorted(want_c, key=lambda c: c[0])]
    # threshold mode: score > S
    if len(s):
        S = int(np.median(s))
        t = exact_ref.select(x, y, s, score_threshold=S)
        m = s > S
        assert t["n_directed"] == 2 * int(m.sum()) and np.array_equal(t["x"], x[m]) and np.array_equal(t["score"], s[m])
    for ms in pivot_min_scores:
        n_reads = len(off) - 1
        pv = np.unique(np.random.default_rng(ms).integers(1, n_reads + 1, max(4, n_reads // 20))).astype(np.uint32)
        px, py, ps = exact_ref.pairs(ro, kid, len(kmers), min_score=ms, pivots=pv)
        ox, oy, os_ = oracle.connections(o_ro, o_kid, o_io, o_ir, min_score=ms, pivots=pv)
        want_p = {(min(a, b), max(a, b)): int(c) for a, b, c in zip(ox.tolist(), oy.tolist(), os_.tolist())}
        assert {(a, b): int(c) for a, b, c in zip(px.tolist(), py.tolist(), ps.tolist())} == want_p, f"subset pairs differ (min_score {ms})"
        assert len(want_p) > 0
    return s


@pytest.mark.parametrize("seed", range(10))
def test_reference_matches_oracle_fuzz(oracle, seed):
    _, reads, k, fraction, min_size, _ = datagen.fuzz_case(seed)
    bases, off = _pack(reads)
    hap = datagen.fuzz_case(seed)[0]
    _check_against_oracle(oracle, bases, off, k, datagen.discriminative_kmers(hap, k), fraction, min_size)


def test_reference_matches_oracle_config1_like(oracle):
    a = datagen.random_genome(20000, 1000)
    b = datagen.mutate(a, 0.03, 1001)
    reads = datagen.sample_reads(a, 4000, 150, 1, error_rate=0.005) + datagen.sample_reads(b, 4000, 150, 2, error_rate=0.005)
    bases, off = _pack(reads)
    s = _check_against_oracle(oracle, bases, off, 19, datagen.discriminative_kmers([a, b], 19), 0.15, 30)
    assert len(s) > 10000


def test_reference_matches_oracle_long_reads(oracle):
    a = datagen.random_genome(120000, 2019)
    b = datagen.mutate(a, 0.02, 2020)
    reads = datagen.sample_reads(a, 300, 7800, 3, error_rate=0.08, length_sigma=0.6, max_len=60000) + \
        datagen.sample_reads(b, 300, 7800, 4, error_rate=0.08, length_sigma=0.6, max_len=60000)
    bases, off = _pack(reads)
    _check_against_oracle(oracle, bases, off, 19, datagen.discriminative_kmers([a, b], 19), 0.15, 5)


def test_reference_matches_oracle_pivot_subsets(oracle):
    a = datagen.random_genome(30000, 31)
    b = datagen.mutate(a, 0.03, 32)
    reads = datagen.sample_reads(a, 250, 1200, 5) + datagen.sample_reads(b, 250, 1200, 6)
    bases, off = _pack(reads)
    _check_against_oracle(oracle, bases, off, 19, datagen.discriminative_kmers([a, b], 19), 0.3, 10, pivot_min_scores=(1, 20))


def test_reference_duplicate_hits_multiply():
    """a k-mer present m times in x and n times in y contributes m * n"""
    rng = np.random.default_rng(7)
    X = datagen.to_ascii(rng.integers(0, 4, 40, dtype=np.uint8)); Y = datagen.to_ascii(rng.integers(0, 4, 40, dtype=np.uint8))
    bases, off = _pack([X + Y + X, X, Y + X + X + X, Y, "ACGT"])
    codes = np.frombuffer(X.encode(), dtype=np.uint8)
    kmers = np.unique(datagen.canonical_kmers(np.array([b"ACGT".index(c) for c in codes[:19]], dtype=np.uint8), 15))
    ro, kid, pos = exact_ref.scan(bases, off, 15, kmers)
    x, y, s = exact_ref.pairs(ro, kid, len(kmers))
    assert list(zip(x.tolist(), y.tolist(), s.tolist())) == [(1, 2, 10), (1, 3, 30), (2, 3, 15)]


def _all_acgt(bases):
    return set(np.unique(np.frombuffer(bases, dtype=np.uint8)).tolist()) <= set(b"ACGT")


@pytest.mark.parametrize("name", golden_util.CASES)
def test_reference_matches_golden(name):
    c = golden_util.load_case(name)
    ref = c["ref"]
    kmers = np.asarray(c["kmers"], dtype=np.uint64)
    ro, kid, pos = exact_ref.scan(c["bases"], c["seq_off"], c["k"], kmers)
    compare.check_hits(ref, ro, kid, pos, kmers)
    io, ir = exact_ref.index(ro, kid, len(kmers))
    compare.check_index(ref, io, ir, kmers)
    x, y, s = exact_ref.pairs(ro, kid, len(kmers))
    ux, uy, us = compare.undirected(ref["conn_x"], ref["conn_y"], ref["conn_score"])
    assert np.array_equal(x, ux) and np.array_equal(y, uy) and np.array_equal(s.astype(np.uint64), us)
    sel = exact_ref.select(x, y, s, fraction=c["fraction"])
    assert sel["n_directed"] == ref["cut_n"] and sel["cut_score"] == ref["cut_score"]
    comp = exact_ref.components(len(c["seq_off"]) - 1, sel["x"], sel["y"], c["min_size"])
    got = sorted(tuple(int(v) for v in np.nonzero(comp["label"] == l)[0] + 1) for l in comp["comp_label"])
    assert got == compare.components_partition(ref["comp_off"], ref["comp_read"])


def test_golden_cases_cover_the_reference():
    """at least four of the golden cases are plain ACGT, and at least one holds other bytes, so the comparison above also judges the
    reference's rule for bytes other than ACGT"""
    plain = [_all_acgt(golden_util.load_case(n)["bases"]) for n in golden_util.CASES]
    assert sum(plain) >= 4 and not all(plain)
