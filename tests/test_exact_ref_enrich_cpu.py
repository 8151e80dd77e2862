"""CPU: the scaffold union_find, merge and enrichment stages of exact_ref.py against the C oracle (stage by stage), the stored
golden vectors and a literal restatement of the purge; then the reference as the judge of hga_enrich_run's own source compiled for
the host (test_kernel_bodies_on_host.py) at a selection of more than 2^18 edges, where the doubling batches of the root-replay
pre-filter and its second level run. The host build runs the kernels one thread at a time, so it can show a logic error in the
batching but no race; tests/test_gpu_exact_enrichment.py runs the same inputs on the GPU."""
import ctypes as C
import re

import numpy as np
import pytest

import compare
import datagen
import exact_ref
import golden_util
import oracle_lib
from test_kernel_bodies_on_host import _emu_collect, _p, host_enrich  # noqa: F401  (host_enrich is a fixture)

REPLAYED = re.compile(r"hga_enrich: (\d+) of (\d+) selected edges replayed")


def _pack(reads):
    seqs = [r.encode() if isinstance(r, str) else datagen.to_ascii(r).encode() for r in reads]
    off = np.zeros(len(seqs) + 1, dtype=np.uint64)
    np.cumsum([len(s) for s in seqs], out=off[1:])
    return b"".join(seqs), off


def _scaffold_list(ro, kid, n_kmers, fraction=0.15, sc_score=0):
    """the directed list run_clustering hands to union_find, built from exact_ref's pair scores"""
    if sc_score:
        pivots = np.nonzero(np.diff(np.asarray(ro, dtype=np.int64)) >= sc_score)[0] + 1
        x, y, s = exact_ref.pairs(ro, kid, n_kmers, min_score=sc_score, pivots=pivots)
        return exact_ref.directed_pivots(x, y, s, pivots, sc_score)
    x, y, s = exact_ref.pairs(ro, kid, n_kmers)
    return exact_ref.directed_fraction(x, y, s, exact_ref.select(x, y, s, fraction=fraction)["n_directed"])


def _check_union_find(got, want):
    comps, trees = got
    co, cm, to, tx, ty = want
    co = co.astype(np.int64)
    assert compare.components_partition(co, cm) == sorted(tuple(int(v) for v in np.sort(c)) for c in comps), "components differ"
    assert sorted(int(cm[co[i]]) for i in range(len(co) - 1)) == sorted(int(c[0]) for c in comps), "roots differ"
    assert all(np.array_equal(c[1:], np.sort(c[1:])) for c in comps)
    got_t = np.cumsum([0] + [len(t[0]) for t in trees])
    assert compare.tree_edges(got_t, np.concatenate([t[0] for t in trees] + [np.zeros(0, np.int64)]),
                              np.concatenate([t[1] for t in trees] + [np.zeros(0, np.int64)])) == compare.tree_edges(to, tx, ty), "spanning trees differ"


def _check_against_oracle(oracle, bases, off, k, kmers, min_size, enrich_min, fraction=0.15, sc_score=0, max_size=-1):
    kmers = np.unique(np.asarray(kmers, dtype=np.uint64))
    ro, kid, _ = exact_ref.scan(bases, off, k, kmers)
    ex, ey, es = _scaffold_list(ro, kid, len(kmers), fraction, sc_score)
    res = oracle.run(bases, off, k, kmers, fraction=fraction, min_size=min_size, sc_score=sc_score, max_size=max_size)
    n = res["cut_n"]
    sx, sy, ss = res["conn"]
    assert np.array_equal(ex, sx[:n]) and np.array_equal(ey, sy[:n]) and np.array_equal(es, ss[:n].astype(np.int64)), "directed scaffold list differs"
    _check_union_find(exact_ref.union_find(ex, ey, min_size, max_size), oracle.union_find(sx[:n], sy[:n], min_size=min_size, max_size=max_size))
    got = exact_ref.enrich(ro, kid, len(kmers), ex, ey, min_size, enrich_min, max_size=max_size)
    want = oracle_lib.enrich(oracle, res, len(kmers), min_size=min_size, enrich_min=enrich_min)
    compare.check_enrichment(compare.enrichment_as_dump(want, kmers), got, kmers)
    # the restricted union_find of the enrichment on its own
    cx, cy, _ = got["econn"]
    _check_union_find(exact_ref.union_find(cx, cy, 2, restricted=got["core_id"]),
                      oracle.union_find(cx, cy, min_size=2, restricted=got["core_id"]))
    return got


@pytest.mark.parametrize("seed", range(10))
def test_enrich_reference_matches_oracle_fuzz(oracle, seed):
    haps, reads, k, fraction, min_size, enrich_min = datagen.fuzz_case(seed)
    bases, off = _pack(reads)
    _check_against_oracle(oracle, bases, off, k, datagen.discriminative_kmers(haps, k), min_size, enrich_min, fraction=fraction)


def _parity_input(seed):
    """the 12 000 short reads of test_gpu_parity.py's sc_max_size (seed 71) and sc_score (seed 61) cases"""
    a = datagen.random_genome(30000, seed); b = datagen.mutate(a, 0.03, seed + 1)
    reads = datagen.sample_reads(a, 6000, 150, seed + 2, error_rate=0.005) + datagen.sample_reads(b, 6000, 150, seed + 3, error_rate=0.005)
    bases, off = _pack(reads)
    return bases, off, datagen.discriminative_kmers([a, b], 19)


@pytest.mark.parametrize("max_size", [40, 120])
def test_enrich_reference_matches_oracle_sc_max_size(oracle, max_size):
    bases, off, kmers = _parity_input(71)
    got = _check_against_oracle(oracle, bases, off, 19, kmers, 10, 20, max_size=max_size)
    assert len(got["core_id"]) >= 2 and max(len(r) for r in got["core_reads"]) <= max_size


def test_enrich_reference_matches_oracle_sc_score(oracle):
    bases, off, kmers = _parity_input(61)
    got = _check_against_oracle(oracle, bases, off, 19, kmers, 10, 20, sc_score=60)
    assert len(got["core_id"]) >= 2


def _golden_reference(c, clusters=None):
    kmers = np.asarray(c["kmers"], dtype=np.uint64)
    ro, kid, _ = exact_ref.scan(c["bases"], c["seq_off"], c["k"], kmers)
    ex, ey, _ = _scaffold_list(ro, kid, len(kmers), c["fraction"])
    return exact_ref.enrich(ro, kid, len(kmers), ex, ey, c["min_size"], c["enrich"], clusters=clusters)


@pytest.mark.parametrize("name", golden_util.ENRICH_CASES)
def test_enrich_reference_matches_golden(name):
    c = golden_util.load_case(name)
    got = _golden_reference(c)
    compare.check_enrichment(c["ref"], got, c["kmers"])
    assert len(got["core_id"]) == c["ref"]["cores"] and len(got["final_id"]) == c["ref"]["final_components"]


@pytest.mark.parametrize("name", golden_util.FULL_CASES)
def test_enrich_reference_with_second_merge_matches_golden(name):
    """the full_* dumps: the reference's spectral clusters given as the second merge"""
    c = golden_util.load_case(name)
    ref = c["ref"]
    so = ref["spectral_off"].astype(np.int64)
    clusters = []
    for i in range(len(so) - 1):
        m = ref["spectral_member"][so[i]:so[i + 1]].astype(np.int64)
        first = int(ref["spectral_first"][i])
        clusters.append(np.concatenate([[first], m[m != first]]))
    assert any(len(cl) > 1 for cl in clusters), "no cluster with several members: the second merge would not run"
    got = _golden_reference(c, clusters)
    assert len(got["scaffold"]) == ref["merged_scaffolds"]
    compare.check_enrichment(ref, got, c["kmers"])


def test_vectorized_purge_matches_the_walk():
    """exact_ref.purge against the reference's two-pointer walk, list by list: lists with repeated ids (a survivor holding a k-mer
    several times), removal lists that name ids the list does not hold, entries above the largest removed id, untouched lists"""
    rng = np.random.default_rng(11)
    n_kmers, n_ids = 400, 60
    lists = [np.sort(rng.integers(1, n_ids, rng.integers(0, 25))) for _ in range(n_kmers)]
    removal = [np.sort(rng.integers(1, n_ids, rng.integers(0, 12))) if rng.random() < 0.8 else np.zeros(0, np.int64) for _ in range(n_kmers)]
    for i in range(0, n_kmers, 7):               # removal ids that all lie in the list: the walk ends inside it
        if len(lists[i]):
            removal[i] = np.sort(rng.choice(lists[i], max(1, len(lists[i]) // 3)))
    off = np.cumsum([0] + [len(l) for l in lists])
    rk = np.concatenate([np.full(len(r), k) for k, r in enumerate(removal)]); ri = np.concatenate(removal)
    p_off, p_id = exact_ref.purge(off, np.concatenate(lists), rk, ri)
    for k in range(n_kmers):
        want = purge_or_keep(lists[k], removal[k])
        assert p_id[p_off[k]:p_off[k + 1]].tolist() == want, k
    dropped_above = sum(1 for l, r in zip(lists, removal) if len(r) and (l > r.max()).any())
    stale = sum(1 for l, r in zip(lists, removal) if len(r) and any((l == v).sum() > (r == v).sum() > 0 and v < r.max() for v in np.unique(l)))
    assert dropped_above > 50 and stale > 20


def purge_or_keep(lst, removal):
    """a k-mer that is not in the removal map keeps its list (merge_components only rewrites the lists of the map's keys)"""
    return [int(v) for v in lst] if len(removal) == 0 else [int(v) for v in exact_ref.purge_walk(list(lst), list(removal))]


# ---- hga_enrich_run compiled for the host, judged by exact_ref at a selection of more than 2^18 edges ------------------------------

LOCI = dict(n_loci=80, locus_len=3000, reads_per_haplotype=800, read_len=150, seed=7300, repeat_every=4)
MIN_SIZE, ENRICH_MIN, FRACTION = 5, 2, 0.1


@pytest.fixture(scope="module")
def loci():
    bases, off, kmers = datagen.many_loci_case(**LOCI)
    ro, kid, pos = exact_ref.scan(bases, off, 19, kmers)
    return dict(bases=bases, off=off, kmers=kmers, ro=ro, kid=kid, pos=pos, pairs=exact_ref.pairs(ro, kid, len(kmers)))


def _emu(lib, L, sel, max_size=-1, pivots=None):
    n = len(L["off"]) - 1
    rows = np.repeat(np.arange(n), np.diff(L["ro"].astype(np.int64)))
    o = np.lexsort((L["pos"], L["kid"], rows))
    kid, pos = np.ascontiguousarray(L["kid"][o]), np.ascontiguousarray(L["pos"][o])
    inv_off, inv_read = exact_ref.index(L["ro"], L["kid"], len(L["kmers"]))
    flag = None
    if pivots is not None:
        flag = np.zeros(n + 1, dtype=np.uint8)
        flag[np.asarray(pivots, dtype=np.int64) - 1] = 1
    arr = lambda a, dt: np.ascontiguousarray(a, dtype=dt)
    sx, sy, ss = arr(sel["x"], np.uint32), arr(sel["y"], np.uint32), arr(sel["score"], np.uint32)
    ro, inv_off, inv_read, read_off = arr(L["ro"], np.uint64), arr(inv_off, np.uint64), arr(inv_read, np.uint32), arr(L["off"], np.uint64)
    rc = lib.emu_enrich(C.c_uint64(n), C.c_uint64(len(L["kmers"])), _p(ro), _p(kid), _p(pos), _p(inv_off), _p(inv_read), C.c_uint64(len(sx)), _p(sx), _p(sy), _p(ss),
                        _p(read_off), MIN_SIZE, C.c_uint32(ENRICH_MIN), C.c_uint32(40), 16, 0, int(max_size), _p(flag) if flag is not None else None)
    assert rc == 0, lib.emu_last_error()
    return _emu_collect(lib)[0]


def _replayed(capfd):
    m = REPLAYED.findall(capfd.readouterr().err)
    assert len(m) == 1, "the replay line of HGA_ENRICH_TIMING is missing"
    return int(m[0][0]), int(m[0][1])


def test_enrich_run_on_host_at_scale(host_enrich, loci, monkeypatch, capfd):
    """M > 2^18 selected edges: at least three doubling batches; more than 2^16 edges replayed, so at least as many survived the
    doubling batches and the second level ran; fewer than M, so the filter dropped edges"""
    x, y, s = loci["pairs"]
    sel = exact_ref.select(x, y, s, fraction=FRACTION)
    ex, ey, _ = exact_ref.directed_fraction(x, y, s, sel["n_directed"])
    want = exact_ref.enrich(loci["ro"], loci["kid"], len(loci["kmers"]), ex, ey, MIN_SIZE, ENRICH_MIN)
    monkeypatch.setenv("HGA_ENRICH_TIMING", "1")
    got = _emu(host_enrich, loci, sel)
    N, M = _replayed(capfd)
    assert M == len(sel["x"]) > 1 << 18 and (1 << 16) < N < M, (N, M)
    assert len(want["core_id"]) >= 64 and len(want["econn"][0]) > 1 << 16
    compare.check_enrichment(compare.enrichment_as_dump(want, loci["kmers"]), got, loci["kmers"])


def test_enrich_run_on_host_at_scale_with_a_size_limit(host_enrich, loci):
    """max_size below the largest unlimited scaffold component: the host replays every edge under the limit"""
    x, y, s = loci["pairs"]
    sel = exact_ref.select(x, y, s, fraction=FRACTION)
    ex, ey, _ = exact_ref.directed_fraction(x, y, s, sel["n_directed"])
    free, _ = exact_ref.union_find(ex, ey, MIN_SIZE)
    limit = max(len(c) for c in free) // 2
    want = exact_ref.enrich(loci["ro"], loci["kid"], len(loci["kmers"]), ex, ey, MIN_SIZE, ENRICH_MIN, max_size=limit)
    assert max(len(c) for c in want["scaffold"]) <= limit and len(want["core_id"]) >= 64
    got = _emu(host_enrich, loci, sel, max_size=limit)
    compare.check_enrichment(compare.enrichment_as_dump(want, loci["kmers"]), got, loci["kmers"])


SC_SCORE = 55


def test_enrich_run_on_host_at_scale_with_sc_score(host_enrich, loci, monkeypatch, capfd):
    """pivot subset (reads with >= S hits), score > S: the host swaps one-pivot pairs into (pivot, other) before the replay"""
    ro, kid = loci["ro"], loci["kid"]
    pivots = np.nonzero(np.diff(ro.astype(np.int64)) >= SC_SCORE)[0] + 1
    x, y, s = exact_ref.pairs(ro, kid, len(loci["kmers"]), min_score=SC_SCORE, pivots=pivots)
    sel = exact_ref.select(x, y, s, score_threshold=SC_SCORE)
    ex, ey, _ = exact_ref.directed_pivots(x, y, s, pivots, SC_SCORE)
    is_pivot = np.zeros(len(loci["off"]) + 1, dtype=bool)
    is_pivot[pivots] = True
    sx, sy = sel["x"].astype(np.int64), sel["y"].astype(np.int64)
    assert (~is_pivot[sx] & is_pivot[sy]).sum() > 100, "no selected one-pivot pair has its pivot as the larger id"
    want = exact_ref.enrich(ro, kid, len(loci["kmers"]), ex, ey, MIN_SIZE, ENRICH_MIN)
    monkeypatch.setenv("HGA_ENRICH_TIMING", "1")
    got = _emu(host_enrich, loci, sel, pivots=pivots)
    N, M = _replayed(capfd)
    assert M == len(sx) > 1 << 16 and N < M, (N, M)
    assert len(want["core_id"]) >= 64
    compare.check_enrichment(compare.enrichment_as_dump(want, loci["kmers"]), got, loci["kmers"])
