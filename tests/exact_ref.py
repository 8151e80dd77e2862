"""Independent exact reference of the hot path in plain numpy / scipy, int64 arithmetic throughout. Test infrastructure only.

It shares no code with the C oracle (oracle/hga_oracle.c) or the kernels, and unlike the oracle (O(sum of list^2) in Python-visible
loops) it scales to tens of Mbases, so it can judge the GPU in the regimes only large inputs reach. Read ids are 1-based.

  scan        canonical k-mers of every window that lies inside one read, membership and id by bisection in the sorted set, hit
              position = window end (seq[pos - k:pos]). A byte other than uppercase ACGT has code 0 on both strands (KmerIterator.cpp:56,62)
  count       the k-mer count's rule instead (jellyfish): ACGT and acgt are bases, a window holding any other byte is skipped

Inputs of many Gbases are built from a small library of distinct reads: a stream is a list of library indices, and since no window
crosses a read, hits and counts of the stream follow from those of the library (library_hits, stream_hits, library_counts,
stream_counts, spectrum). A library read may be periodic: tile(block)[:head] + tail, so that a read of 2^30 bases costs the
reference one period and its tail.
  index       stable argsort of the hit ids: reads ascending inside every list, one entry per occurrence
  pairs       A = reads x k-mers matrix of multiplicities (duplicate hits summed), S = A A^T, pairs x < y with score >= min_score;
              with pivots, the pairs with at least one pivot
  select      canonical order (score desc, x asc, y asc); fraction mode: n = int(2P * fraction) directed entries, s* = score of the
              pair that holds the n-th one, every pair above s* plus the first ceil(r / 2) ties in (x, y) order, r = n - 2 |above|;
              threshold mode: score > S
  components  connected components of the selected edges, label = smallest member id; a read without a selected edge is labelled
              with itself and is no listed component whatever min_size is (as union_find only sees the reads of some edge)

From the selection on, what run_clustering does to its engine state (ReadClusteringEngine.cpp), in the order it does it:

  scaffold list  the directed list union_find receives, built literally: fraction mode = the first n entries of the canonical order
              (score desc, min(x, y) asc, max(x, y) asc, x asc) over both directions of every pair; sc_score mode = what
              get_connections emits for the pivots ((pivot, other); a pair of two pivots in both directions), score > S, canonical
  union_find  sequential over the list in order; vertices = ids some edge touches; union by size, ties to y's root; a union is
              skipped when it would exceed max_size or join two restricted roots; a root inherits `restricted`; components of
              >= min_size vertices with the root first, spanning-tree edges in replay order
  merge       merge_components: element [0] survives with the sorted unique union of the members' k-mer lists and all their reads;
              every member goes into the removal list of every k-mer once per entry of its current list (the survivor's current
              list being the union); each inverted list of a k-mer with removals is then purged by the two-pointer walk that stops
              when the removal list runs out (purge_walk; vectorized in purge)
  connections get_connections on the current state: score(p, y) = sum over the entries k of p's list of the copies of y in the list
              of k, y != p, score >= min_score; a pivot that is no survivor keeps its own list with duplicates
  enrich      union_find(min_size, max_size) -> merge -> [second merge of caller-given clusters] -> cores = ids with >= min_size
              reads -> connections(cores, enrich_min), canonical -> union_find(min 2, restricted = cores) -> merge -> final ids
              with >= min_size reads
"""
import numpy as np
import scipy.sparse as sp
from scipy.sparse import csgraph

_FWD = np.zeros(256, dtype=np.uint64)          # scan rule: forward code, 0 for a byte other than ACGT
_REV = np.zeros(256, dtype=np.uint64)          # complement code, 0 for a byte other than ACGT too
_FOLD = np.full(256, 255, dtype=np.uint8)      # count rule: ACGT and acgt, 255 = not a base
for _i, _c in enumerate(b"ACGT"):
    _FWD[_c] = _i; _REV[_c] = 3 - _i
    _FOLD[_c] = _FOLD[_c + 32] = _i


def window_values(raw, k, rule="scan"):
    """canonical value of the window starting at every position of the bytes raw (uint8 array) -> (uint64[n - k + 1], valid bool[..]).
    rule "scan": every window is valid, a byte other than ACGT has code 0 on both strands; rule "count": ACGT and acgt are bases and a
    window holding any other byte is not valid"""
    raw = np.asarray(raw, dtype=np.uint8)
    n = raw.shape[0] - k + 1
    if n <= 0:
        return np.zeros(0, dtype=np.uint64), np.zeros(0, dtype=bool)
    if rule == "scan":
        f, r = _FWD[raw], _REV[raw]
        valid = np.ones(n, dtype=bool)
    else:
        c = _FOLD[raw]
        bad = c == 255
        f = np.where(bad, 0, c).astype(np.uint64)
        r = np.uint64(3) - f
        nb = np.concatenate([[0], np.cumsum(bad, dtype=np.int64)])
        valid = nb[k:] == nb[:n]
    fwd = np.zeros(n, dtype=np.uint64)
    rev = np.zeros(n, dtype=np.uint64)
    for j in range(k):
        fwd |= f[j:j + n] << np.uint64(2 * (k - 1 - j))
        rev |= r[j:j + n] << np.uint64(2 * j)
    return np.minimum(fwd, rev), valid


def scan(bases, read_off, k, kmers_sorted, chunk_bases=1 << 22):
    """-> (row_off uint64[n_reads + 1], kmer id uint32[E], window end uint32[E]) in (read, position) order"""
    codes = np.frombuffer(bases, dtype=np.uint8) if isinstance(bases, (bytes, bytearray)) else np.asarray(bases, dtype=np.uint8)
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
        km, _ = window_values(seg, k)                      # window starting at every position of the segment
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


# ---- scaffold stage, merge and enrichment (ReadClusteringEngine::run_clustering after the selection) ------------------------------

def canonical(x, y, score):
    """-> (x, y, score) of a directed list in the canonical order: score desc, min(x, y) asc, max(x, y) asc, x asc"""
    x = np.asarray(x, dtype=np.int64); y = np.asarray(y, dtype=np.int64); score = np.asarray(score, dtype=np.int64)
    o = np.lexsort((x, np.maximum(x, y), np.minimum(x, y), -score))
    return x[o], y[o], score[o]


def directed_fraction(x, y, score, n):
    """the list union_find receives in fraction mode: the first n entries of the canonical order over both directions of every pair"""
    x = np.asarray(x, dtype=np.int64); y = np.asarray(y, dtype=np.int64); score = np.asarray(score, dtype=np.int64)
    cx, cy, cs = canonical(np.concatenate([x, y]), np.concatenate([y, x]), np.concatenate([score, score]))
    return cx[:n], cy[:n], cs[:n]


def directed_pivots(x, y, score, pivots, sc_score):
    """the list union_find receives in sc_score mode: get_connections of every pivot emits (pivot, other), so a pair of two pivots
    is there in both directions and a pair with one pivot only as (pivot, other); the entries with score > sc_score, canonical"""
    x = np.asarray(x, dtype=np.int64); y = np.asarray(y, dtype=np.int64); score = np.asarray(score, dtype=np.int64)
    pv = np.zeros(int(max(x.max(initial=0), y.max(initial=0))) + 2, dtype=bool)
    p = np.asarray(pivots, dtype=np.int64)
    pv[p[p < pv.shape[0]]] = True
    fwd, bwd = pv[x], pv[y]                         # (x, y) is emitted by pivot x, (y, x) by pivot y
    dx = np.concatenate([x[fwd], y[bwd]]); dy = np.concatenate([y[fwd], x[bwd]]); ds = np.concatenate([score[fwd], score[bwd]])
    keep = ds > sc_score
    return canonical(dx[keep], dy[keep], ds[keep])


def union_find(ex, ey, min_size, max_size=-1, restricted=None):
    """The sequential union_find over a directed edge list in its given order. Only vertices some edge touches exist. A union
    skips when both roots are restricted or the merged size would exceed max_size; otherwise the smaller root joins the larger, ties
    to y's root, and the new root inherits `restricted`. -> (components of >= min_size vertices ordered by smallest member, each an
    int64 array with the root first and the other members ascending; the spanning-tree edges of each, in replay order)"""
    limit = (1 << 31) - 1 if max_size == -1 else int(max_size)
    ex = np.asarray(ex, dtype=np.int64).tolist(); ey = np.asarray(ey, dtype=np.int64).tolist()
    parent, size, tree = {}, {}, {}
    for v in ex + ey:
        parent[v] = v; size[v] = 1
    rest = {int(v) for v in (restricted if restricted is not None else ()) if int(v) in parent}

    def find(v):
        r = v
        while parent[r] != r:
            r = parent[r]
        while parent[v] != r:
            parent[v], v = r, parent[v]
        return r

    order = []
    for i, (x, y) in enumerate(zip(ex, ey)):
        px, py = find(x), find(y)
        if px == py or (px in rest and py in rest) or size[px] + size[py] > limit:
            continue
        big, small = (px, py) if size[px] > size[py] else (py, px)
        parent[small] = big
        size[big] += size[small]
        if small in rest:
            rest.add(big)
        order.append(i)
    verts = np.array(sorted(parent), dtype=np.int64)
    roots = np.array([find(int(v)) for v in verts], dtype=np.int64)
    comps, trees = [], []
    for r in np.unique(roots):
        if size[int(r)] < min_size:
            continue
        mem = verts[roots == r]
        comps.append(np.concatenate([[r], mem[mem != r]]))
    comps.sort(key=lambda c: int(c.min()))
    at = {int(c[0]): j for j, c in enumerate(comps)}
    trees = [([], []) for _ in comps]
    for i in order:
        j = at.get(find(ex[i]))
        if j is not None:
            trees[j][0].append(ex[i]); trees[j][1].append(ey[i])
    return comps, [(np.array(a, dtype=np.int64), np.array(b, dtype=np.int64)) for a, b in trees]


class State:
    """The engine state merge_components and get_connections work on. Ids 1..n_reads; id r starts as read r with its k-mer id list
    (sorted, one entry per hit) and contains read r. kl_id / kl_kmer: every (id, k-mer) list entry, sorted by (id, k-mer);
    owner[r - 1]: the id that contains read r; inv_off / inv_id: the inverted index, one ascending id list per k-mer."""

    def __init__(self, row_off, kid, n_kmers):
        self.n_reads = np.asarray(row_off).shape[0] - 1
        self.n_kmers = int(n_kmers)
        rows = _rows(row_off) + 1
        kid = np.asarray(kid, dtype=np.int64)
        o = np.lexsort((kid, rows))
        self.kl_id, self.kl_kmer = rows[o], kid[o]
        self.owner = np.arange(1, self.n_reads + 1, dtype=np.int64)
        self.inv_off, ids = index(row_off, kid, n_kmers)
        self.inv_off = self.inv_off.astype(np.int64)
        self.inv_id = ids.astype(np.int64)

    def copy(self):
        s = object.__new__(State)
        s.__dict__.update({k: (v.copy() if isinstance(v, np.ndarray) else v) for k, v in self.__dict__.items()})
        return s

    def kmers_of(self, i):
        lo, hi = np.searchsorted(self.kl_id, [i, i + 1])
        return self.kl_kmer[lo:hi]

    def ids(self, min_size):
        """ids that contain >= min_size reads, ascending"""
        cnt = np.bincount(self.owner, minlength=self.n_reads + 1)
        return np.nonzero(cnt >= min_size)[0].astype(np.int64)

    def reads_of(self, i):
        return np.nonzero(self.owner == i)[0].astype(np.int64) + 1

    def _inv_rows(self):
        return np.repeat(np.arange(self.n_kmers, dtype=np.int64), np.diff(self.inv_off))


def _entries(st, ids):
    """(id, k-mer) list entries of the given ids, duplicates included"""
    m = np.isin(st.kl_id, ids)
    return st.kl_id[m], st.kl_kmer[m]


def purge_walk(lst, removal):
    """the purge of one inverted list as the reference writes it: a two-pointer walk over the ascending list and the ascending removal
    list that ends when either runs out, keeping only what it copied"""
    removal = sorted(removal)
    out, i, j = [], 0, 0
    while i < len(removal) and j < len(lst):
        if removal[i] < lst[j]:
            i += 1
        elif lst[j] < removal[i]:
            out.append(lst[j]); j += 1
        else:
            i += 1; j += 1
    return out


def purge(inv_off, inv_id, rem_kmer, rem_id):
    """purge_walk of every list at once: k-mers with no removal entry keep their list; the others keep the entries below their largest
    removed id, minus the removal multiset. -> (off, id)"""
    inv_off = np.asarray(inv_off, dtype=np.int64); inv_id = np.asarray(inv_id, dtype=np.int64)
    n_kmers = inv_off.shape[0] - 1
    rem_kmer = np.asarray(rem_kmer, dtype=np.int64); rem_id = np.asarray(rem_id, dtype=np.int64)
    base = int(max(inv_id.max(initial=0), rem_id.max(initial=0))) + 1
    rows = np.repeat(np.arange(n_kmers, dtype=np.int64), np.diff(inv_off))
    R = np.full(n_kmers, -1, dtype=np.int64)
    np.maximum.at(R, rem_kmer, rem_id)
    lk, lc = np.unique(rows * base + inv_id, return_counts=True)
    rk, rc = np.unique(rem_kmer * base + rem_id, return_counts=True)
    at = np.searchsorted(rk, lk)
    hit = at < rk.shape[0]
    hit[hit] = rk[at[hit]] == lk[hit]
    r = np.zeros(lk.shape[0], dtype=np.int64)
    r[hit] = rc[at[hit]]
    k, e = lk // base, lk % base
    keep = np.where(R[k] < 0, lc, np.where(e < R[k], np.maximum(lc - r, 0), 0))
    off = np.zeros(n_kmers + 1, dtype=np.int64)
    np.add.at(off, k + 1, keep)
    return np.cumsum(off), np.repeat(e, keep)


def merge(st, comps):
    """merge_components: element [0] of every component of >= 2 ids survives with the sorted unique union of the members' k-mer lists
    and all their reads; every member is removed from every k-mer once per entry of its current list (the survivor's current list
    being the union), then every inverted list is purged (purge)."""
    comps = [np.asarray(c, dtype=np.int64) for c in comps if len(c) > 1]
    if not comps:
        return st
    mem = np.concatenate(comps)
    surv = np.concatenate([np.full(len(c), c[0], dtype=np.int64) for c in comps])
    mi, mk = _entries(st, mem)
    into = np.zeros(st.n_reads + 1, dtype=np.int64)
    into[mem] = surv
    u = np.unique(into[mi] * (st.n_kmers + 1) + mk)
    uid, ukm = u // (st.n_kmers + 1), u % (st.n_kmers + 1)
    is_surv = np.zeros(st.n_reads + 1, dtype=bool)
    is_surv[[c[0] for c in comps]] = True
    other = ~is_surv[mi]
    st.inv_off, st.inv_id = purge(st.inv_off, st.inv_id, np.concatenate([mk[other], ukm]), np.concatenate([mi[other], uid]))
    keep = ~is_surv[st.kl_id]
    kl_id = np.concatenate([st.kl_id[keep], uid]); kl_kmer = np.concatenate([st.kl_kmer[keep], ukm])
    o = np.lexsort((kl_kmer, kl_id))
    st.kl_id, st.kl_kmer = kl_id[o], kl_kmer[o]
    moved = into[st.owner]
    st.owner = np.where(moved != 0, moved, st.owner)
    return st


def connections(st, pivots, min_score):
    """get_connections on the current state: score(p, y) = sum over the entries k of p's k-mer list of the copies of y in the list of
    k, for y != p with score >= min_score. -> (x = pivot, y, score) in (x, y) order"""
    pivots = np.unique(np.asarray(pivots, dtype=np.int64))
    if pivots.shape[0] == 0:
        z = np.zeros(0, dtype=np.int64)
        return z, z, z
    pi, pk = _entries(st, pivots)
    a = sp.csr_matrix((np.ones(pi.shape[0], dtype=np.int64), (np.searchsorted(pivots, pi), pk)), shape=(pivots.shape[0], st.n_kmers))
    b = sp.csr_matrix((np.ones(st.inv_id.shape[0], dtype=np.int64), (st._inv_rows(), st.inv_id)), shape=(st.n_kmers, st.n_reads + 1))
    s = (a @ b).tocoo()
    x, y, sc = pivots[s.row], s.col.astype(np.int64), s.data.astype(np.int64)
    keep = (y != x) & (sc >= min_score)
    x, y, sc = x[keep], y[keep], sc[keep]
    o = np.lexsort((y, x))
    return x[o], y[o], sc[o]


def enrich(row_off, kid, n_kmers, ex, ey, min_size, enrich_min, max_size=-1, clusters=None):
    """run_clustering from the directed scaffold list (ex, ey) on: union_find(min_size, max_size), merge of the scaffold components,
    optionally a second merge of caller-given clusters of cores (the tail / spectral block's), cores = ids with >= min_size reads,
    connections(cores, enrich_min) in canonical order, union_find(min 2, restricted = cores), merge, final ids with >= min_size reads.
    -> dict with what hga_get_enrichment / hga_get_purged_index / hga_get_core_kmers return (in compare.check_enrichment's shape,
    final components ordered by smallest member, assignment[r - 1] = final id of read r or 0), plus the scaffold components, their
    spanning trees and the state right after the first merge"""
    scaffold, trees = union_find(ex, ey, min_size, max_size)
    st = merge(State(row_off, kid, n_kmers), scaffold)
    first = st.copy()
    if clusters is not None:
        st = merge(st, clusters)
    cores = st.ids(min_size)
    core_kmers = [st.kmers_of(c) for c in cores]
    core_reads = [st.reads_of(c) for c in cores]
    purged_off, purged_read = st.inv_off.copy(), st.inv_id.copy()
    cx, cy, cs = canonical(*connections(st, cores, enrich_min))
    ecomp, _ = union_find(cx, cy, 2, restricted=cores)
    merge(st, ecomp)
    final = st.ids(min_size)
    final_reads = [st.reads_of(f) for f in final]
    o = np.argsort([int(r[0]) for r in final_reads], kind="stable")
    final, final_reads = final[o], [final_reads[i] for i in o]
    assignment = np.zeros(st.n_reads, dtype=np.int64)
    for f, r in zip(final, final_reads):
        assignment[r - 1] = f
    return dict(core_id=cores, core_kmers=core_kmers, core_reads=core_reads, purged_off=purged_off, purged_read=purged_read,
                econn=(cx, cy, cs), final_id=final, final_reads=final_reads, assignment=assignment,
                scaffold=scaffold, trees=trees, first_merge=first)


# ---- streams built from a library of reads -----------------------------------------------------------------------------------

class LibRead:
    """a library read: tile(block)[:head] + tail (block None, head 0: the tail alone). bytes() materialises it."""

    def __init__(self, tail, block=None, head=0):
        self.tail = np.asarray(tail, dtype=np.uint8)
        self.block = None if block is None else np.asarray(block, dtype=np.uint8)
        self.head = int(head)

    def __len__(self):
        return self.head + self.tail.shape[0]

    def bytes(self):
        if not self.head:
            return self.tail
        reps = -(-self.head // self.block.shape[0])
        return np.concatenate([np.tile(self.block, reps)[:self.head], self.tail])

    def cyclic(self, k):
        """the bytes of every window of the periodic part (one period and k - 1 more)"""
        return np.concatenate([self.block, np.tile(self.block, -(-(k - 1) // self.block.shape[0]))[:k - 1]])

    def end_part(self, k):
        """(bytes of the windows that end in the tail, their first base in the read): k - 1 bases of context and the tail"""
        if not self.head:
            return self.tail, 0
        L = self.block.shape[0]
        c0 = max(self.head - (k - 1), 0)
        ctx = np.array([self.block[i % L] for i in range(c0, self.head)], dtype=np.uint8)
        return np.concatenate([ctx, self.tail]), c0

    def head_windows(self, k):
        """windows that lie inside the periodic part"""
        return max(self.head - k + 1, 0)


def library_hits(lib, k, kmers_sorted):
    """scan of every library read on its own -> list of (kmer id uint32[], window end uint32[]). The windows of a periodic read's
    head must hold no k-mer of the set (checked)."""
    out = []
    for r in lib:
        if r.head:
            v, _ = window_values(r.cyclic(k), k)
            at = np.searchsorted(kmers_sorted, v)
            assert not np.any(kmers_sorted[np.minimum(at, kmers_sorted.shape[0] - 1)] == v), "the periodic part of a read holds a k-mer of the set"
        part, p0 = r.end_part(k)
        _, kid, pos = scan(part, np.array([0, part.shape[0]], dtype=np.uint64), k, kmers_sorted)
        out.append((kid, (pos.astype(np.int64) + p0).astype(np.uint32)))
    return out


def stream_hits(lib_hits, order):
    """the scan of the stream whose reads are lib[order[0]], lib[order[1]], ... -> (row_off, kmer id, window end)"""
    order = np.asarray(order, dtype=np.int64)
    n = np.array([h[0].shape[0] for h in lib_hits], dtype=np.int64)
    row_off = np.zeros(order.shape[0] + 1, dtype=np.uint64)
    np.cumsum(n[order], out=row_off[1:])
    used = [i for i in order.tolist() if n[i]]
    cat = lambda j, dt: np.concatenate([lib_hits[i][j] for i in used]) if used else np.zeros(0, dtype=dt)
    return row_off, cat(0, np.uint32), cat(1, np.uint32)


def library_counts(lib, k):
    """canonical k-mer counts of every library read on its own (count rule) -> list of (k-mers ascending uint64, counts int64)"""
    out = []
    for r in lib:
        part, _ = r.end_part(k)
        v, ok = window_values(part, k, "count")
        vals, wts = [v[ok]], [np.ones(int(ok.sum()), dtype=np.int64)]
        if r.head:
            cv, cok = window_values(r.cyclic(k), k, "count")
            N, L = r.head_windows(k), r.block.shape[0]
            per = np.full(L, N // L, dtype=np.int64) + (np.arange(L) < N % L)      # windows of the head at cyclic position i
            vals.append(cv[cok]); wts.append(per[cok])
        out.append(_sum_by_value(np.concatenate(vals), np.concatenate(wts)))
    return out


def _sum_by_value(v, w):
    """(distinct values ascending, summed weights > 0)"""
    o = np.argsort(v, kind="stable")
    v, w = v[o], np.asarray(w, dtype=np.int64)[o]
    if v.shape[0] == 0:
        return v, w
    start = np.concatenate([[0], np.flatnonzero(v[1:] != v[:-1]) + 1])
    u, c = v[start], np.add.reduceat(w, start)
    keep = c > 0
    return u[keep], c[keep]


def stream_counts(lib_counts, order, min_count=1):
    """the counts of the stream lib[order[0]], lib[order[1]], ...: every library read's counts times its multiplicity, summed. ->
    (k-mers ascending uint64, counts int64 >= min_count)"""
    mult = np.bincount(np.asarray(order, dtype=np.int64), minlength=len(lib_counts))
    used = [i for i in range(len(lib_counts)) if mult[i] and lib_counts[i][0].shape[0]]
    if not used:
        return np.zeros(0, dtype=np.uint64), np.zeros(0, dtype=np.int64)
    u, c = _sum_by_value(np.concatenate([lib_counts[i][0] for i in used]), np.concatenate([lib_counts[i][1] * mult[i] for i in used]))
    keep = c >= max(int(min_count), 1)
    return u[keep], c[keep]


def spectrum(counts, n_bins):
    """-> (hist uint64[n_bins], n_windows, n_distinct, max_count) of exact counts, as hga_count_spectrum returns them"""
    c = np.asarray(counts, dtype=np.int64)
    hist = np.zeros(int(n_bins), dtype=np.uint64)
    if n_bins and c.shape[0]:
        hist[:] = np.bincount(np.minimum(c, n_bins) - 1, minlength=int(n_bins))
    return hist, int(c.sum()), int(c.shape[0]), int(c.max(initial=0))
