"""GPU: the CUDA path against the numpy / scipy reference (exact_ref.py) in the regimes only large or extreme inputs reach, where
the C oracle is too slow to judge. Every stage a test runs is compared value for value, and every test asserts the metric or input
property that proves it reached its regime, so that a later change to a threshold cannot move it back onto an easier path:

  - scan: hit-buffer capacity from a count-only sample (first scan of more than 32 MiB), from the previous scan's density followed
    by an overflow and an exact rerun, a device input at an unaligned address, lookups in the table's sorted overflow region
  - pair count: min-hash pivot order with the first pass, its redo, tier 2 and the heavy tier in one run, rows with more long lists
    than the first pass defers, pivot subsets, min_score inside the score distribution, scores at the 32-bit limit
  - selection: cuts in a non-zero high bin of the 16 + 16 bit radix select, tie runs over many selection chunks
"""
import numpy as np
import pytest

import datagen
import exact_ref

pytestmark = pytest.mark.gpu

HGA_E_OVERFLOW = 5
SEL_CHUNK = 2048          # pairs per block of the selection kernels (hga_select.cu)


def _pack(reads):
    seqs = [r.encode() if isinstance(r, str) else datagen.to_ascii(r).encode() for r in reads]
    off = np.zeros(len(seqs) + 1, dtype=np.uint64)
    np.cumsum([len(s) for s in seqs], out=off[1:])
    return b"".join(seqs), off


def _rand(rng, n):
    return datagen.to_ascii(rng.integers(0, 4, n, dtype=np.uint8))


def _check_hits(h, want):
    row_off, kid, pos = h.get_hits()
    assert np.array_equal(row_off, want[0]), "row offsets differ"
    assert np.array_equal(kid, want[1]), "hit k-mer ids differ"
    assert np.array_equal(pos, want[2]), "hit positions differ"


def _check_index(h, hits, n_kmers):
    inv_off, inv_read = h.get_index()
    w_off, w_read = exact_ref.index(hits[0], hits[1], n_kmers)
    assert np.array_equal(inv_off, w_off) and np.array_equal(inv_read, w_read), "inverted index differs"


def _check_pairs(h, want):
    x, y, s, _ = h.get_pairs()
    assert x.shape[0] == want[0].shape[0], f"{x.shape[0]} pairs, want {want[0].shape[0]}"
    assert np.array_equal(x, want[0]) and np.array_equal(y, want[1]), "pair sets differ"
    assert np.array_equal(s.astype(np.int64), want[2]), "pair scores differ"


def _check_selection(h, want, fraction=0.15, score_threshold=0):
    h.select_edges(fraction=fraction, score_threshold=score_threshold)
    sel = h.get_selection()
    ref = exact_ref.select(*want, fraction=fraction, score_threshold=score_threshold)
    assert sel["n_directed"] == ref["n_directed"] and sel["cut_score"] == ref["cut_score"], "cut differs"
    o = np.lexsort((sel["y"], sel["x"]))
    assert np.array_equal(sel["x"][o], ref["x"]) and np.array_equal(sel["y"][o], ref["y"]), "selected set differs"
    assert np.array_equal(sel["score"][o].astype(np.int64), ref["score"]), "selected scores differ"
    return ref


def _check_components(h, n_reads, sel, min_size):
    h.components(min_size=min_size)
    comp = h.get_components()
    ref = exact_ref.components(n_reads, sel["x"], sel["y"], min_size)
    assert comp["read_id_first"] == 1
    assert np.array_equal(comp["label"], ref["label"]), "component labels differ"
    assert np.array_equal(comp["comp_label"], ref["comp_label"]) and np.array_equal(comp["comp_size"], ref["comp_size"]), "components differ"


def test_long_reads_above_both_size_thresholds():
    """~40 Mbases of long diploid reads on a fresh handle: the hit buffers are sized from a 1/64 count-only sample (> 32 MiB of
    bases), the pivots take the min-hash order (> 4096 rows), and the normal pair tiers run"""
    import hga_b200
    k = 19
    a = datagen.random_genome(2_000_000, 7101)
    b = datagen.mutate(a, 0.01, 7102)
    reads = datagen.sample_reads(a, 4000, 5000, 7103, error_rate=0.02, length_sigma=0.5, min_len=500, max_len=40000) + \
        datagen.sample_reads(b, 4000, 5000, 7104, error_rate=0.02, length_sigma=0.5, min_len=500, max_len=40000)
    reads = [reads[i] for i in np.random.default_rng(7105).permutation(len(reads))]
    bases, off = _pack(reads)
    kmers = datagen.discriminative_kmers([a, b], k)
    hits = exact_ref.scan(bases, off, k, kmers)
    pairs = exact_ref.pairs(hits[0], hits[1], len(kmers))
    with hga_b200.Handle(kmers, k) as h:
        h.scan(bases, off)
        m = h.metrics()
        assert m["n_bases"] == len(bases) > 32 << 20 and m["n_reads"] == len(reads) > 4096
        _check_hits(h, hits)
        h.build_index()
        _check_index(h, hits, len(kmers))
        h.pair_count(min_score=1)
        _check_pairs(h, pairs)
        sel = _check_selection(h, pairs, fraction=0.15)
        _check_components(h, len(reads), sel, 10)
    assert pairs[0].shape[0] > 50_000


def test_denser_second_scan_overflows_and_reruns():
    """a second scan on the same handle is sized from the first one's hit density; a denser input overflows that estimate and
    reruns with the exact count. Then the same input through hga_scan_device with a base pointer that is not 16 B aligned."""
    import torch
    import hga_b200
    k = 21
    dense = datagen.random_genome(1_500_000, 7201)
    other = datagen.random_genome(1_500_000, 7202)
    kmers = np.unique(datagen.canonical_kmers(dense, k))          # every window of a read of `dense` is a hit
    first = datagen.sample_reads(dense, 2600, 5000, 7203, length_sigma=0.3, min_len=1000) + \
        datagen.sample_reads(other, 5000, 5000, 7204, length_sigma=0.3, min_len=1000)
    first = [first[i] for i in np.random.default_rng(7205).permutation(len(first))]
    second = datagen.sample_reads(dense, 7600, 5000, 7206, length_sigma=0.3, min_len=1000)
    b1, o1 = _pack(first)
    b2, o2 = _pack(second)
    h1 = exact_ref.scan(b1, o1, k, kmers)
    h2 = exact_ref.scan(b2, o2, k, kmers)
    d1, d2 = h1[1].shape[0] / len(b1), h2[1].shape[0] / len(b2)
    assert len(b1) > 32 << 20 and len(b2) > 32 << 20 and d2 > 1.3 * d1, (d1, d2)
    with hga_b200.Handle(kmers, k) as h:
        h.scan(b1, o1)
        _check_hits(h, h1)
        h.build_index()
        _check_index(h, h1, len(kmers))
        h.scan(b2, o2)
        assert h.metrics()["scan_retries"] == 1, "the denser scan was meant to overflow its estimated hit buffer"
        _check_hits(h, h2)
        h.build_index()
        _check_index(h, h2, len(kmers))
        lead = 5
        buf = torch.zeros(len(b2) + 64, dtype=torch.uint8, device="cuda")
        assert (buf.data_ptr() + lead) % 16 != 0
        buf[lead:lead + len(b2)].copy_(torch.from_numpy(np.frombuffer(b2, dtype=np.uint8).copy()))
        d_off = torch.from_numpy(o2.astype(np.int64)).cuda()
        torch.cuda.synchronize()
        h.scan_device(buf.data_ptr() + lead, d_off.data_ptr(), len(second), len(b2))
        _check_hits(h, h2)
        del buf, d_off


def _tier_case():
    """4 500 reads sharing pieces of one 100 bp segment (every ninth holds its piece twice), 150 reads sharing another 100 bp
    segment whole, 500 background long reads of a diploid genome and 30 reads without any hit, ids shuffled"""
    rng = np.random.default_rng(7301)
    k = 21
    seg1, seg2 = _rand(rng, 100), _rand(rng, 100)
    reads, group1, group2, nohit = [], [], [], []
    for i in range(4500):
        a0 = int(rng.integers(0, 21)); L = int(rng.integers(60, 100 - a0 + 1))
        piece = seg1[a0:a0 + L]
        body = piece + _rand(rng, 10) + piece if i % 9 == 0 else piece
        reads.append(_rand(rng, 60) + body + _rand(rng, 40)); group1.append(len(reads))
    for _ in range(150):
        reads.append(_rand(rng, 50) + seg2 + _rand(rng, 50)); group2.append(len(reads))
    ga = datagen.random_genome(1_000_000, 7302)
    gb = datagen.mutate(ga, 0.01, 7303)
    bg = datagen.sample_reads(ga, 250, 3000, 7304, error_rate=0.01) + datagen.sample_reads(gb, 250, 3000, 7305, error_rate=0.01)
    background = list(range(len(reads) + 1, len(reads) + 1 + len(bg)))
    reads += [datagen.to_ascii(r) for r in bg]
    for _ in range(30):
        reads.append(_rand(rng, 200)); nohit.append(len(reads))
    kmers = np.unique(np.concatenate([datagen.canonical_kmers(_to_codes(seg1), k), datagen.canonical_kmers(_to_codes(seg2), k),
                                      datagen.discriminative_kmers([ga, gb], k)]))
    perm = rng.permutation(len(reads))              # new id of old id i + 1 = inv[i] + 1
    inv = np.empty_like(perm); inv[perm] = np.arange(len(perm))
    ids = lambda old: (inv[np.asarray(old, dtype=np.int64) - 1] + 1).astype(np.int64)
    return k, [reads[i] for i in perm], kmers, ids(group1), ids(group2), ids(background), ids(nohit)


def _to_codes(s):
    return np.array([b"ACGT".index(c) for c in s.encode()], dtype=np.uint8)


def _assert_all_tiers(m):
    assert m["redo_pivots"] > 0 and m["mid_pivots"] > 0 and m["heavy_pivots"] > 0, \
        f"tiers: redo {m['redo_pivots']}, tier 2 {m['mid_pivots']}, heavy {m['heavy_pivots']}"


def test_all_pair_tiers_in_one_run():
    """first pass, its redo, tier 2 and the heavy tier in one run with min-hash order, for min_score 1 and a min_score inside the
    score distribution, and again for a pivot subset drawn from every tier plus pivots without hits"""
    import hga_b200
    k, reads, kmers, g1, g2, bg, nohit = _tier_case()
    n = len(reads)
    bases, off = _pack(reads)
    hits = exact_ref.scan(bases, off, k, kmers)
    full = exact_ref.pairs(hits[0], hits[1], len(kmers))
    # regime of the 150-read group: more than PW_DEFER (32) lists longer than PW_LONG (96) in a row whose partners fit the first pass
    lens = np.diff(exact_ref.index(hits[0], hits[1], len(kmers))[0].astype(np.int64))
    ro = hits[0].astype(np.int64)
    partners = np.bincount(full[0].astype(np.int64), minlength=n + 1) + np.bincount(full[1].astype(np.int64), minlength=n + 1)
    for r in g2[:10]:
        assert int((lens[hits[1][ro[r - 1]:ro[r]]] > 96).sum()) > 32 and partners[r] < 384
    assert np.all(np.diff(ro)[nohit - 1] == 0)
    mid_score = int(np.median(full[2]))
    assert full[2].min() < mid_score < full[2].max()
    with hga_b200.Handle(kmers, k) as h:
        h.scan(bases, off)
        assert h.metrics()["n_reads"] == n > 4096
        _check_hits(h, hits)
        h.build_index()
        _check_index(h, hits, len(kmers))
        for ms in (1, mid_score):
            want = exact_ref.restrict(*full, min_score=ms)
            h.pair_count(min_score=ms)
            _assert_all_tiers(h.metrics())
            _check_pairs(h, want)
            sel = _check_selection(h, want, fraction=0.15)
            _check_components(h, n, sel, 2)
        # subset: 300 of the big group are no pivots, so a pivot of that group has 300 + (pivots of the group above it) partners,
        # 300 .. 4 500: every tier
        rng = np.random.default_rng(7306)
        pv = np.sort(np.concatenate([np.setdiff1d(g1, rng.choice(g1, 300, replace=False)), rng.choice(g2, 20, replace=False),
                                     rng.choice(bg, 20, replace=False), nohit[:10]])).astype(np.uint32)
        for ms in (1, mid_score):
            want = exact_ref.restrict(*full, min_score=ms, pivots=pv)
            h.pair_count(min_score=ms, pivots=pv)
            _assert_all_tiers(h.metrics())
            _check_pairs(h, want)
            sel = _check_selection(h, want, score_threshold=mid_score)
            _check_components(h, n, sel, 2)


@pytest.mark.parametrize("k", [15, 19, 31])
def test_scan_lookups_in_table_overflow_region(monkeypatch, k):
    """the k-mer set is every canonical k-mer of a 3 Mbp genome and the reads tile that genome, so every key is looked up; keys
    whose bucket is full sit in the sorted overflow region (bisection). At the default load that happens for k = 15 and 19 with
    these genomes; for k = 31 the table is built at load 0.9."""
    import hga_b200
    g = datagen.random_genome(3_000_000, 4000 + k)
    kmers = np.unique(datagen.canonical_kmers(g, k))
    reads = []
    for i, s in enumerate(range(0, g.shape[0], 1500)):
        r = g[s:s + 2000]
        reads.append(datagen.COMP[r[::-1]] if i % 2 else r)
    bases, off = _pack(reads)
    hits = exact_ref.scan(bases, off, k, kmers)
    assert np.all(np.bincount(hits[1], minlength=len(kmers)) > 0), "every key is meant to be hit"
    if k == 31:
        monkeypatch.setenv("HGA_TABLE_LOAD", "0.9")
    with hga_b200.Handle(kmers, k) as h:
        h.scan(bases, off)
        assert h.metrics()["table_overflow_keys"] > 0
        _check_hits(h, hits)


def test_selection_cut_in_high_bin():
    """scores of 2^16 and more (poly-A and tandem-repeat reads of graded lengths): the cut falls into a non-zero high bin of the
    radix select that holds several distinct scores"""
    import hga_b200
    k = 15
    unit = "ACGTC"
    reads = ["A" * (k - 1 + 300 + 3 * i) for i in range(30)]
    reads += [unit * (300 + 7 * i) for i in range(30)]
    reads += ["A" * (k - 1 + 250 + 5 * i) + "G" + unit * (200 + 9 * i) for i in range(10)]
    rng = np.random.default_rng(7401)
    reads = [reads[i] for i in rng.permutation(len(reads))]
    kmers = np.unique(np.concatenate([np.zeros(1, dtype=np.uint64), datagen.canonical_kmers(_to_codes(unit * 8), k)]))
    bases, off = _pack(reads)
    hits = exact_ref.scan(bases, off, k, kmers)
    full = exact_ref.pairs(hits[0], hits[1], len(kmers))
    assert full[2].min() >= 1 << 16
    with hga_b200.Handle(kmers, k) as h:
        h.scan(bases, off)
        _check_hits(h, hits)
        h.build_index()
        h.pair_count(min_score=1)
        _check_pairs(h, full)
        for f in (0.05, 0.2, 0.5, 0.9):
            ref = _check_selection(h, full, fraction=f)
            cut = ref["cut_score"]
            assert cut >> 16 > 0 and np.unique(full[2][(full[2] >> 16) == (cut >> 16)]).shape[0] > 1
        sel = _check_selection(h, full, score_threshold=int(np.median(full[2])))
        _check_components(h, len(reads), sel, 2)


def test_selection_tie_run_over_many_chunks():
    """a run of more than 5 x 2048 pairs with the same score (identical reads) between a group above and a group below it; the cut
    at the run's first, middle and last pair, each with an odd number r of directed slots left for the ties"""
    import hga_b200
    k = 21
    rng = np.random.default_rng(7501)
    s_above, s_tie, s_below = _rand(rng, 250), _rand(rng, 200), _rand(rng, 150)
    reads = [s_above] * 30 + [s_tie] * 160 + [s_below] * 100
    reads = [reads[i] for i in rng.permutation(len(reads))]
    kmers = np.unique(np.concatenate([datagen.canonical_kmers(_to_codes(s), k) for s in (s_above, s_tie, s_below)]))
    bases, off = _pack(reads)
    hits = exact_ref.scan(bases, off, k, kmers)
    full = exact_ref.pairs(hits[0], hits[1], len(kmers))
    P = full[0].shape[0]
    tie = int(np.unique(full[2])[1])
    above, T = int((full[2] > tie).sum()), int((full[2] == tie).sum())
    assert T == 160 * 159 // 2 > 5 * SEL_CHUNK and above == 30 * 29 // 2
    with hga_b200.Handle(kmers, k) as h:
        h.scan(bases, off)
        h.build_index()
        h.pair_count(min_score=1)
        _check_pairs(h, full)
        for n, quota in ((2 * above + 1, 1), (2 * (above + T // 2) + 1, T // 2 + 1), (2 * (above + T) - 1, T)):
            f = (n + 0.5) / (2 * P)
            assert int(2 * P * f) == n and (n - 2 * above) % 2 == 1
            ref = _check_selection(h, full, fraction=f)
            assert ref["cut_score"] == tie and int((ref["score"] == tie).sum()) == quota
        sel = _check_selection(h, full, fraction=(2 * (above + T // 2) + 1.5) / (2 * P))
        _check_components(h, len(reads), sel, 2)
        _check_selection(h, full, score_threshold=tie)
        _check_selection(h, full, score_threshold=tie - 1)


def _poly_a_case(hits_each, heavy):
    """two poly-A reads with hits_each hits of k-mer 0 each (k = 15); heavy: and 3 200 short reads with one hit each, so that both
    long reads have more than 3 072 partners (heavy tier)"""
    k = 15
    reads = ["A" * (hits_each + k - 1)] * 2
    if heavy:
        reads += ["C" + "A" * k + "C"] * 3200
    bases, off = _pack(reads)
    kmers = np.zeros(1, dtype=np.uint64)
    return k, bases, off, kmers


@pytest.mark.parametrize("layout", ["plain", "heavy", "subset"])
def test_pair_scores_at_the_32_bit_limit(layout):
    """65 535 hits each: the score 65 535^2 = 4 294 836 225 fits 32 bits and comes back exactly; 65 536 hits each: the score 2^32
    does not fit, and pair_count fails with HGA_E_OVERFLOW instead of returning a wrapped score"""
    import hga_b200
    heavy = layout != "plain"
    pivots = np.array([1], dtype=np.uint32) if layout == "subset" else None
    k, bases, off, kmers = _poly_a_case(65535, heavy)
    hits = exact_ref.scan(bases, off, k, kmers)
    want = exact_ref.pairs(hits[0], hits[1], 1, pivots=pivots)
    assert want[0][0] == 1 and want[1][0] == 2 and want[2][0] == 65535 * 65535 == 4_294_836_225
    with hga_b200.Handle(kmers, k) as h:
        h.scan(bases, off)
        _check_hits(h, hits)
        h.build_index()
        h.pair_count(min_score=1, pivots=pivots)
        if heavy:
            assert h.metrics()["heavy_pivots"] > 0
        _check_pairs(h, want)
    k, bases, off, kmers = _poly_a_case(65536, heavy)
    with hga_b200.Handle(kmers, k) as h:
        h.scan(bases, off)
        h.build_index()
        with pytest.raises(hga_b200.HgaError) as e:
            h.pair_count(min_score=1, pivots=pivots)
        assert e.value.code == HGA_E_OVERFLOW and "2^32" in str(e.value)
        if heavy:
            assert h.metrics()["heavy_pivots"] > 0
        with pytest.raises(hga_b200.HgaError):
            h.get_pairs()                                   # no pairs after the failed count
