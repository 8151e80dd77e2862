"""Independent exact reference of the hot path in plain numpy / scipy, int64 arithmetic throughout. Test infrastructure only.

It shares no code with the C oracle (oracle/hga_oracle.c) or the kernels, and unlike the oracle (O(sum of list^2) in Python-visible
loops) it scales to tens of Mbases, so it can judge the GPU in the regimes only large inputs reach. Read ids are 1-based.

  scan        uppercase ACGT input only (the rule for other bytes stays with the oracle tests): canonical k-mers of every window that
              lies inside one read, membership and id by bisection in the sorted set, hit position = window end (seq[pos - k:pos])
  index       stable argsort of the hit ids: reads ascending inside every list, one entry per occurrence
  pairs       A = reads x k-mers matrix of multiplicities (duplicate hits summed), S = A A^T, pairs x < y with score >= min_score;
              with pivots, the pairs with at least one pivot
  select      canonical order (score desc, x asc, y asc); fraction mode: n = int(2P * fraction) directed entries, s* = score of the
              pair that holds the n-th one, every pair above s* plus the first ceil(r / 2) ties in (x, y) order, r = n - 2 |above|;
              threshold mode: score > S
  components  connected components of the selected edges, label = smallest member id; a read without a selected edge is labelled
              with itself and is no listed component whatever min_size is (as union_find only sees the reads of some edge)
"""
import numpy as np
import scipy.sparse as sp
from scipy.sparse import csgraph

import datagen

_CODE = np.full(256, 255, dtype=np.uint8)
for _i, _c in enumerate(b"ACGT"):
    _CODE[_c] = _i


def scan(bases, read_off, k, kmers_sorted, chunk_bases=1 << 22):
    """-> (row_off uint64[n_reads + 1], kmer id uint32[E], window end uint32[E]) in (read, position) order"""
    codes = _CODE[np.frombuffer(bytes(bases), dtype=np.uint8)]
    if codes.shape[0] and codes.max() > 3:
        raise ValueError("exact_ref.scan takes uppercase ACGT input only")
    kmers_sorted = np.asarray(kmers_sorted, dtype=np.uint64)
    off = np.asarray(read_off, dtype=np.int64)
    n_reads = off.shape[0] - 1
    counts = np.zeros(n_reads, dtype=np.int64)
    kids, poss = [], []
    r0 = 0
    while r0 < n_reads:
        # a run of whole reads of about chunk_bases bases (at least one read)
        r1 = max(r0 + 1, int(np.searchsorted(off, off[r0] + chunk_bases, side="right")) - 1)
        r1 = min(r1, n_reads)
        seg = codes[off[r0]:off[r1]]
        km = datagen.canonical_kmers(seg, k)               # window starting at every position of the segment
        if km.shape[0]:
            start = np.arange(km.shape[0], dtype=np.int64)
            rel = off[r0:r1 + 1] - off[r0]
            read = np.searchsorted(rel, start, side="right") - 1
            inside = start + k <= rel[read + 1]
            idx = np.searchsorted(kmers_sorted, km)
            found = idx < kmers_sorted.shape[0]
            found[found] = kmers_sorted[idx[found]] == km[found]
            hit = inside & found
            read = read[hit]
            counts[r0:r1] = np.bincount(read, minlength=r1 - r0)
            kids.append(idx[hit].astype(np.uint32))
            poss.append((start[hit] + k - rel[read]).astype(np.uint32))
        r0 = r1
    row_off = np.zeros(n_reads + 1, dtype=np.uint64)
    np.cumsum(counts, out=row_off[1:])
    cat = lambda parts: np.concatenate(parts) if parts else np.zeros(0, dtype=np.uint32)
    return row_off, cat(kids), cat(poss)


def _rows(row_off):
    ro = np.asarray(row_off, dtype=np.int64)
    return np.repeat(np.arange(ro.shape[0] - 1, dtype=np.int64), np.diff(ro))


def index(row_off, kid, n_kmers):
    """-> (off uint64[n_kmers + 1], read id uint32[E]), reads ascending inside every list"""
    kid = np.asarray(kid, dtype=np.int64)
    order = np.argsort(kid, kind="stable")
    inv_off = np.zeros(n_kmers + 1, dtype=np.uint64)
    np.cumsum(np.bincount(kid, minlength=n_kmers), out=inv_off[1:])
    return inv_off, (_rows(row_off)[order] + 1).astype(np.uint32)


def incidence(row_off, kid, n_kmers):
    """reads x k-mers CSR matrix of multiplicities (int64; duplicate hits are summed)"""
    rows = _rows(row_off)
    n_reads = np.asarray(row_off).shape[0] - 1
    a = sp.coo_matrix((np.ones(rows.shape[0], dtype=np.int64), (rows, np.asarray(kid, dtype=np.int64))), shape=(n_reads, n_kmers))
    return a.tocsr()


def pairs(row_off, kid, n_kmers, min_score=1, pivots=None):
    """-> (x uint32, y uint32, score int64): x < y, ascending (x, y), score >= min_score; pivots (read ids): pairs touching one"""
    a = incidence(row_off, kid, n_kmers)
    s = sp.triu(a @ a.T, k=1).tocoo()
    x, y, sc = s.row.astype(np.int64) + 1, s.col.astype(np.int64) + 1, s.data.astype(np.int64)
    o = np.lexsort((y, x))
    return restrict(x[o].astype(np.uint32), y[o].astype(np.uint32), sc[o], min_score, pivots)


def restrict(x, y, score, min_score=1, pivots=None):
    """the pairs of a min_score = 1 result that a run with this min_score (and pivot subset) keeps"""
    keep = score >= max(int(min_score), 1)
    if pivots is not None:
        flag = np.zeros(int(max(x.max(initial=0), y.max(initial=0))) + 2, dtype=bool)
        pv = np.asarray(pivots, dtype=np.int64)
        flag[pv[pv < flag.shape[0]]] = True
        keep &= flag[x] | flag[y]
    return x[keep], y[keep], score[keep]


def select(x, y, score, fraction=0.15, score_threshold=0):
    """-> dict(n_directed, cut_score, x, y, score) with the selected pairs in (x, y) order"""
    x = np.asarray(x, dtype=np.int64); y = np.asarray(y, dtype=np.int64); score = np.asarray(score, dtype=np.int64)
    P = x.shape[0]
    if score_threshold > 0:
        keep = score > score_threshold
        n, cut = 2 * int(keep.sum()), int(score_threshold)
    else:
        n = min(int(2 * P * fraction), 2 * P)
        keep = np.zeros(P, dtype=bool)
        cut = 0
        if n > 0:
            desc = np.lexsort((y, x, -score))               # canonical order
            cut = int(score[desc[(n + 1) // 2 - 1]])          # the pair that holds the n-th directed entry
            above = score > cut
            quota = (n - 2 * int(above.sum()) + 1) // 2
            ties = np.nonzero(score == cut)[0]                # already in (x, y) order
            keep = above
            keep[ties[:quota]] = True
    return dict(n_directed=n, cut_score=cut, x=x[keep].astype(np.uint32), y=y[keep].astype(np.uint32), score=score[keep])


def components(n_reads, sel_x, sel_y, min_size):
    """-> dict(label uint32[n_reads] = smallest member id, comp_label / comp_size of the components of >= min_size reads, labels
    ascending). A read without a selected edge keeps its own id as label and is not listed."""
    ex = np.asarray(sel_x, dtype=np.int64) - 1
    ey = np.asarray(sel_y, dtype=np.int64) - 1
    g = sp.coo_matrix((np.ones(ex.shape[0], dtype=np.int8), (ex, ey)), shape=(n_reads, n_reads))
    _, comp = csgraph.connected_components(g, directed=False)
    first = np.full(comp.max() + 1 if n_reads else 0, n_reads, dtype=np.int64)
    np.minimum.at(first, comp, np.arange(n_reads, dtype=np.int64))
    label = (first[comp] + 1).astype(np.uint32)
    size = np.bincount(comp)
    big = np.nonzero(size >= max(int(min_size), 2))[0]
    o = np.argsort(first[big])
    return dict(label=label, comp_label=(first[big][o] + 1).astype(np.uint32), comp_size=size[big][o].astype(np.uint32))
