"""Order-independent comparisons between a hot-path result expressed on (row_off, hit_kid, hit_pos, ...) with
k-mer ids indexing a SORTED k-mer array, and a ref_driver dump (tests/refdump.py) or a golden npz."""
import numpy as np


def hits_as_ref(row_off, hit_kid, hit_pos, kmers_sorted):
    """-> (hit_read, hit_kmer) sorted by (read, kmer value) and first-occurrence triples (read, kmer, pos)."""
    row_off = np.asarray(row_off).astype(np.int64)
    n_reads = row_off.shape[0] - 1
    read = np.repeat(np.arange(1, n_reads + 1, dtype=np.uint32), np.diff(row_off))
    kmer = np.asarray(kmers_sorted, dtype=np.uint64)[np.asarray(hit_kid, dtype=np.int64)]
    pos = np.asarray(hit_pos, dtype=np.uint32)
    order = np.lexsort((pos, kmer, read))
    read, kmer, pos = read[order], kmer[order], pos[order]
    first = np.ones(read.shape[0], dtype=bool)
    first[1:] = (read[1:] != read[:-1]) | (kmer[1:] != kmer[:-1])
    return read, kmer, (read[first], kmer[first], pos[first])


def check_hits(ref, row_off, hit_kid, hit_pos, kmers_sorted):
    read, kmer, (fr, fk, fp) = hits_as_ref(row_off, hit_kid, hit_pos, kmers_sorted)
    assert np.array_equal(read, ref["hit_read"]), "per-read hit lists differ (read ids)"
    assert np.array_equal(kmer, ref["hit_kmer"]), "per-read hit lists differ (k-mer values)"
    assert np.array_equal(fr, ref["firstpos_read"]) and np.array_equal(fk, ref["firstpos_kmer"])
    assert np.array_equal(fp, ref["firstpos_pos"]), "first-occurrence positions differ"


def check_index(ref, inv_off, inv_read, kmers_sorted):
    assert np.array_equal(np.asarray(kmers_sorted, dtype=np.uint64), ref["inv_kmer"])
    assert np.array_equal(np.asarray(inv_off, dtype=np.uint64), ref["inv_off"])
    assert np.array_equal(np.asarray(inv_read, dtype=np.uint32), ref["inv_read"])


def undirected(cx, cy, cs):
    """directed canonical list -> unique (x<y, score) sorted by (x, y)"""
    cx = np.asarray(cx, dtype=np.int64); cy = np.asarray(cy, dtype=np.int64); cs = np.asarray(cs, dtype=np.uint64)
    m = cx < cy
    x, y, s = cx[m], cy[m], cs[m]
    o = np.lexsort((y, x))
    return x[o].astype(np.uint32), y[o].astype(np.uint32), s[o]


def check_directed_symmetric(cx, cy, cs):
    a = undirected(cx, cy, cs)
    b = undirected(cy, cx, cs)
    assert all(np.array_equal(p, q) for p, q in zip(a, b)), "directed connection list is not symmetric"


def components_partition(comp_off, comp_read):
    comp_off = np.asarray(comp_off).astype(np.int64)
    return sorted(tuple(sorted(int(v) for v in comp_read[comp_off[i]:comp_off[i + 1]])) for i in range(comp_off.shape[0] - 1))


def tree_edges(tree_off, tx, ty):
    tree_off = np.asarray(tree_off).astype(np.int64)
    out = []
    for i in range(tree_off.shape[0] - 1):
        e = sorted((min(int(a), int(b)), max(int(a), int(b))) for a, b in zip(tx[tree_off[i]:tree_off[i + 1]], ty[tree_off[i]:tree_off[i + 1]]))
        out.append(tuple(e))
    return sorted(out)


def check_enrichment(ref, e, kmers_sorted):
    """Oracle.enrich-style result (oracle_lib.enrich / the CUDA path's mirror of it) against a ref_driver --enrich dump."""
    kmers_sorted = np.asarray(kmers_sorted, dtype=np.uint64)
    assert np.array_equal(e["core_id"], ref["core_id"]), "core (merged scaffold) survivor ids differ"
    if "core_kmers" in e:
        ck = np.concatenate([np.sort(kmers_sorted[np.asarray(c, dtype=np.int64)]) for c in e["core_kmers"]]) if len(e["core_kmers"]) else np.zeros(0, np.uint64)
        assert np.array_equal(ck, ref["core_kmer"]), "merged k-mer lists differ"
        assert np.array_equal(np.cumsum([0] + [len(c) for c in e["core_kmers"]]).astype(np.uint64), ref["core_kmer_off"])
    cr = np.concatenate(e["core_reads"]) if len(e["core_reads"]) else np.zeros(0, np.uint32)
    assert np.array_equal(cr, ref["core_read"]), "core members differ"
    if "purged_off" in e:
        assert np.array_equal(e["purged_off"], ref["purged_off"]) and np.array_equal(e["purged_read"], ref["purged_read"]), "purged inverted index differs"
    ex, ey, es = e["econn"]
    assert np.array_equal(ex, ref["econn_x"]) and np.array_equal(ey, ref["econn_y"]) and np.array_equal(es, ref["econn_score"]), "enrichment connections differ"
    assert np.array_equal(e["final_id"], ref["final_id"]), "final component ids differ"
    fr = np.concatenate(e["final_reads"]) if len(e["final_reads"]) else np.zeros(0, np.uint32)
    assert np.array_equal(fr, ref["final_read"]), "final components differ"
    assert np.array_equal(np.cumsum([0] + [len(c) for c in e["final_reads"]]).astype(np.uint64), ref["final_off"])


def enrichment_as_dump(e, kmers_sorted):
    """an Oracle.enrich-style result (exact_ref.enrich, oracle_lib.enrich) in the shape of a ref_driver --enrich dump, so that
    check_enrichment can judge another result with it"""
    kmers_sorted = np.asarray(kmers_sorted, dtype=np.uint64)
    cat = lambda parts, dt: np.concatenate([np.asarray(p, dtype=dt) for p in parts]) if len(parts) else np.zeros(0, dt)
    off = lambda parts: np.cumsum([0] + [len(p) for p in parts]).astype(np.uint64)
    ex, ey, es = e["econn"]
    return dict(core_id=np.asarray(e["core_id"], dtype=np.uint32), core_kmer=cat([np.sort(kmers_sorted[np.asarray(c, dtype=np.int64)]) for c in e["core_kmers"]], np.uint64),
                core_kmer_off=off(e["core_kmers"]), core_read=cat(e["core_reads"], np.uint32), purged_off=np.asarray(e["purged_off"], dtype=np.uint64),
                purged_read=np.asarray(e["purged_read"], dtype=np.uint32), econn_x=np.asarray(ex, dtype=np.uint32), econn_y=np.asarray(ey, dtype=np.uint32),
                econn_score=np.asarray(es, dtype=np.uint64), final_id=np.asarray(e["final_id"], dtype=np.uint32), final_read=cat(e["final_reads"], np.uint32),
                final_off=off(e["final_reads"]))
