"""GPU: merge and enrichment (hga_enrich, hga_enrich_ex, hga_enrich_full) against the numpy / scipy reference (exact_ref.enrich) at
a selection of more than 2^18 edges, where the small inputs of the other tests leave parts of hga_enrich_run idle: the root-replay
pre-filter walks several doubling batches and reruns its survivors in small batches, the concurrent hook unites edges, the
connection list needs the GPU canonical sort. The tail block runs on long reads of one genome, where about a hundred scaffold cores
fall into multi-member spectral clusters, so the GPU tail amplification and the second merge both work on many cores.
Every output is compared value for value, and every test asserts what shows it reached its regime. The replay line that
HGA_ENRICH_TIMING=1 prints ("N of M selected edges replayed") gives the pre-filter's counts."""
import numpy as np
import pytest

import compare
import datagen
import exact_ref
from test_exact_ref_enrich_cpu import ENRICH_MIN, FRACTION, MIN_SIZE, SC_SCORE, _replayed, loci  # noqa: F401  (loci is a fixture)

pytestmark = pytest.mark.gpu

TAIL_K = 21


@pytest.fixture(scope="module")
def plain(loci):
    """exact_ref's scaffold list (fraction mode) and its enrichment"""
    x, y, s = loci["pairs"]
    sel = exact_ref.select(x, y, s, fraction=FRACTION)
    ex, ey, _ = exact_ref.directed_fraction(x, y, s, sel["n_directed"])
    return dict(M=len(sel["x"]), ex=ex, ey=ey, want=exact_ref.enrich(loci["ro"], loci["kid"], len(loci["kmers"]), ex, ey, MIN_SIZE, ENRICH_MIN))


@pytest.fixture(scope="module")
def tails():
    """the tail block's input: long reads of one 400 kb diploid genome, so that scaffold cores overlap at their tails and the spectral
    clustering groups them (with the short reads of `loci` the cores are independent and no tail connection is strong)"""
    a = datagen.random_genome(400_000, 7401); b = datagen.mutate(a, 0.03, 7402)
    n = int(12 * 400_000 / 1800)
    reads = datagen.sample_reads(a, n, 1800, 7403, error_rate=0.02, length_sigma=0.4) + datagen.sample_reads(b, n, 1800, 7404, error_rate=0.02, length_sigma=0.4)
    seqs = [datagen.to_ascii(reads[i]).encode() for i in np.random.default_rng(7405).permutation(len(reads))]
    off = np.zeros(len(seqs) + 1, dtype=np.uint64)
    np.cumsum([len(s) for s in seqs], out=off[1:])
    L = dict(bases=b"".join(seqs), off=off, kmers=datagen.discriminative_kmers([a, b], TAIL_K))
    L["ro"], L["kid"], L["pos"] = exact_ref.scan(L["bases"], off, TAIL_K, L["kmers"])
    x, y, s = exact_ref.pairs(L["ro"], L["kid"], len(L["kmers"]))
    L["ex"], L["ey"], _ = exact_ref.directed_fraction(x, y, s, exact_ref.select(x, y, s, fraction=0.15)["n_directed"])
    L["want"] = exact_ref.enrich(L["ro"], L["kid"], len(L["kmers"]), L["ex"], L["ey"], MIN_SIZE, ENRICH_MIN)
    return L


def _handle(L, fraction=FRACTION, k=19):
    import hga_b200
    h = hga_b200.Handle(L["kmers"], k)
    h.scan(L["bases"], L["off"])
    h.build_index()
    if fraction:
        h.pair_count(min_score=1)
        h.select_edges(fraction=fraction)
    return h


def _result(h):
    e = h.get_enrichment()
    ko, kk = h.get_core_kmers()
    po, pr = h.get_purged_index()
    co = e["core_off"].astype(np.int64); fo = e["final_off"].astype(np.int64); ko = ko.astype(np.int64)
    assert e["read_id_first"] == 1
    return dict(core_id=e["core_id"], core_kmers=[kk[ko[i]:ko[i + 1]] for i in range(len(ko) - 1)],
                core_reads=[e["core_read"][co[i]:co[i + 1]] for i in range(len(co) - 1)], purged_off=po, purged_read=pr,
                econn=(e["conn_x"], e["conn_y"], e["conn_score"].astype(np.uint64)), final_id=e["final_id"],
                final_reads=[e["final_read"][fo[i]:fo[i + 1]] for i in range(len(fo) - 1)], assignment=e["assignment"])


def _check(h, want, kmers):
    got = _result(h)
    compare.check_enrichment(compare.enrichment_as_dump(want, kmers), got, kmers)
    assert np.array_equal(got["assignment"], want["assignment"]), "assignment differs"
    m = h.metrics()
    assert m["n_cores"] == len(want["core_id"]) and m["n_enrich_connections"] == len(want["econn"][0])
    assert m["n_final_components"] == len(want["final_id"])
    return got


def _same(a, b):
    for key in ("core_id", "purged_off", "purged_read", "final_id", "assignment"):
        assert np.array_equal(a[key], b[key]), key
    for key in ("core_kmers", "core_reads", "econn", "final_reads"):
        assert len(a[key]) == len(b[key]) and all(np.array_equal(p, q) for p, q in zip(a[key], b[key])), key


def test_enrich_many_loci(loci, plain, monkeypatch, capfd):
    """hga_enrich: more than 2^18 selected edges (three or more doubling batches), more than 2^16 of them replayed (so more than 2^16
    survived the batches and the second level ran) but fewer than all, >= 64 cores, more than 2^16 enrichment connections. A second
    run on the same handle may keep another superset of edges in the concurrent hook; its result must not change."""
    want = plain["want"]
    assert len(want["core_id"]) >= 64 and len(want["econn"][0]) > 1 << 16
    monkeypatch.setenv("HGA_ENRICH_TIMING", "1")
    with _handle(loci) as h:
        h.enrich(min_size=MIN_SIZE, enrichment_min_score=ENRICH_MIN)
        N, M = _replayed(capfd)
        assert M == plain["M"] > 1 << 18 and (1 << 16) < N < M, (N, M)
        first = _check(h, want, loci["kmers"])
        h.enrich(min_size=MIN_SIZE, enrichment_min_score=ENRICH_MIN)
        N2, _ = _replayed(capfd)
        assert (1 << 16) < N2 < M, N2
        _same(_result(h), first)


def test_enrich_ex_many_loci_with_a_size_limit(loci, plain, monkeypatch, capfd):
    """hga_enrich_ex with max_size below the largest unlimited scaffold component: the limit skips unions, the host replays every
    selected edge (the d_key / d_kept swap path)"""
    free, _ = exact_ref.union_find(plain["ex"], plain["ey"], MIN_SIZE)
    limit = max(len(c) for c in free) // 2
    want = exact_ref.enrich(loci["ro"], loci["kid"], len(loci["kmers"]), plain["ex"], plain["ey"], MIN_SIZE, ENRICH_MIN, max_size=limit)
    assert max(len(c) for c in want["scaffold"]) <= limit and len(want["core_id"]) >= 64
    monkeypatch.setenv("HGA_ENRICH_TIMING", "1")
    with _handle(loci) as h:
        h.enrich(min_size=MIN_SIZE, enrichment_min_score=ENRICH_MIN, max_size=limit)
        N, M = _replayed(capfd)
        assert N == M == plain["M"], (N, M)
        _check(h, want, loci["kmers"])


def test_enrich_many_loci_sc_score(loci, monkeypatch, capfd):
    """pivot subset (reads with >= S hits), pair_count(min_score = S), select_edges(score > S), enrich: more than 2^16 selected
    edges, the filter drops some, and selected one-pivot pairs hold their pivot as the larger id, so the host's swap into
    (pivot, other) decides the replay order. Judged with the literal directed list get_connections emits."""
    ro, kid = loci["ro"], loci["kid"]
    pivots = np.nonzero(np.diff(ro.astype(np.int64)) >= SC_SCORE)[0] + 1
    x, y, s = exact_ref.pairs(ro, kid, len(loci["kmers"]), min_score=SC_SCORE, pivots=pivots)
    ex, ey, _ = exact_ref.directed_pivots(x, y, s, pivots, SC_SCORE)
    want = exact_ref.enrich(ro, kid, len(loci["kmers"]), ex, ey, MIN_SIZE, ENRICH_MIN)
    is_pivot = np.zeros(len(loci["off"]) + 1, dtype=bool)
    is_pivot[pivots] = True
    monkeypatch.setenv("HGA_ENRICH_TIMING", "1")
    with _handle(loci, fraction=0) as h:
        h.pair_count(min_score=SC_SCORE, pivots=pivots.astype(np.uint32))
        h.select_edges(score_threshold=SC_SCORE)
        sel = h.get_selection()
        sx, sy = sel["x"].astype(np.int64), sel["y"].astype(np.int64)
        lo, hi = np.minimum(sx, sy), np.maximum(sx, sy)
        assert (~is_pivot[lo] & is_pivot[hi]).sum() > 100, "no selected one-pivot pair has its pivot as the larger id"
        h.enrich(min_size=MIN_SIZE, enrichment_min_score=ENRICH_MIN)
        N, M = _replayed(capfd)
        assert M == len(sx) == (s > SC_SCORE).sum() > 1 << 16 and N < M, (N, M)
        _check(h, want, loci["kmers"])


def _tail_inputs(L, want):
    """what hga_enrich_run hands the tail stage, rebuilt from exact_ref: hits by read sorted by (k-mer id, position), read lengths,
    the scaffold components in survivor order (survivor first, then ascending) with their spanning trees in replay order, and the
    purged index after the first merge"""
    n = len(L["off"]) - 1
    rows = np.repeat(np.arange(n), np.diff(L["ro"].astype(np.int64)))
    o = np.lexsort((L["pos"], L["kid"], rows))
    order = np.argsort([int(c[0]) for c in want["scaffold"]])
    comps = [want["scaffold"][i] for i in order]
    trees = [want["trees"][i] for i in order]
    off = L["off"].astype(np.int64)
    cat = lambda parts: np.concatenate(parts) if parts else np.zeros(0, np.int64)
    st = want["first_merge"]
    return dict(row_off=L["ro"], kmer_id=L["kid"][o], pos=L["pos"][o], read_len=np.diff(off), avg_read_length=int((off[-1] - off[0]) // n),
                comp_off=np.cumsum([0] + [len(c) for c in comps]), comp_member=cat(comps), tree_off=np.cumsum([0] + [len(t[0]) for t in trees]),
                tree_x=cat([t[0] for t in trees]), tree_y=cat([t[1] for t in trees]), purged_off=st.inv_off, purged_read=st.inv_id)


def _run_full(h, L):
    h.enrich_full(L["off"], min_size=MIN_SIZE, enrichment_min_score=ENRICH_MIN, tail_amplification_min_score=40, spectral_dims=16)
    return h.get_tail_block(), _result(h)


def _check_full(L, t, got):
    import hga_b200
    want = L["want"]
    assert t["ran"] and t["n_scaffold_cores"] == len(want["scaffold"]) > 2
    tx, ty, ts = hga_b200.capi.host_tail_connections(amplification_min_score=40, **_tail_inputs(L, want))
    assert np.array_equal(t["conn_x"], tx) and np.array_equal(t["conn_y"], ty) and np.array_equal(t["conn_score"], ts), "tail connections differ"
    strong = ts > 5
    clusters = [c for c in hga_b200.capi.spectral_clustering(tx[strong], ty[strong], ts[strong], dims=16) if len(c)]
    assert len(t["clusters"]) == len(clusters) and all(np.array_equal(a, b) for a, b in zip(t["clusters"], clusters)), "spectral clusters differ"
    assert max(len(c) for c in clusters) > 1, "no multi-member cluster: the second merge did not run"
    full = exact_ref.enrich(L["ro"], L["kid"], len(L["kmers"]), L["ex"], L["ey"], MIN_SIZE, ENRICH_MIN, clusters=clusters)
    compare.check_enrichment(compare.enrichment_as_dump(full, L["kmers"]), got, L["kmers"])
    assert np.array_equal(got["assignment"], full["assignment"]), "assignment differs"


def test_enrich_full_at_scale(tails):
    """hga_enrich_full: the tail block runs on many cores (gpu_tail_amplify judged by the host amplification of the same state), at
    least one spectral cluster has several members (the second-merge kernels run), everything after the block against exact_ref
    with those clusters as the second merge"""
    with _handle(tails, fraction=0.15, k=TAIL_K) as h:
        t, got = _run_full(h, tails)
    _check_full(tails, t, got)


def test_enrich_buffers_reused_on_one_handle(tails):
    """enrich_full, enrich, enrich_full on one handle: the purged / purged2 buffers change places and d_enr_parent serves as the
    cluster map between these calls; every result equals its first-run counterpart"""
    with _handle(tails, fraction=0.15, k=TAIL_K) as h:
        t1, a = _run_full(h, tails)
        h.enrich(min_size=MIN_SIZE, enrichment_min_score=ENRICH_MIN)
        _check(h, tails["want"], tails["kmers"])
        assert not h.get_tail_block()["ran"]
        t3, c = _run_full(h, tails)
    _same(a, c)
    assert all(np.array_equal(p, q) for p, q in zip(t1["clusters"], t3["clusters"])) and len(t1["clusters"]) == len(t3["clusters"])
    _check_full(tails, t1, a)
