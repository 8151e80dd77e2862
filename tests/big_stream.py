"""Read streams past a boundary X (2^32 bases on the GPU) built from a small library of reads, and their exact reference through
exact_ref's library helpers. Test infrastructure only.

Layout (stream order), with D = the bases of the first `n_prefix` reads (odd, so that D is no multiple of 4):

    prefix fillers | fillers and the first half of the hit reads | pad | S (straddles X) | fillers, pad | E (empty) T (starts at X + D)
    | P (2^30 - 1 bases in the GPU layout, hits within 512 bases of its end) | the other half of the hit reads among fillers

  - fillers: n_filler random reads of about filler_len bases, repeated to pass X. The k-mer set is the discriminative k-mers of a
    diploid pair minus every k-mer of a filler window (cyclic: a filler repeated back to back adds none either), so fillers have no hit;
    with hits their copies would make the pair count grow quadratically. A pad is a filler prefix of the length that puts the next
    read where it belongs.
  - hit reads: long diploid reads (test_long_reads_above_both_size_thresholds), each once.
  - S and T are hit reads; P is a filler repeated to its length with a hit-bearing tail whose last window is a hit.
  - fillers, S, T and P's tail carry N runs and lowercase bytes, so a packing has exception runs on both sides of X.

The stream from read n_prefix on (the suffix) has E and T at exactly X in its own coordinates; the whole stream has S across X.
"""
import numpy as np

import datagen
import exact_ref

ACGT = np.frombuffer(b"ACGT", dtype=np.uint8)


def _sprinkle(rng, seq, n_runs):
    """n_runs N runs (1-40 bytes) and n_runs lowercase runs (1-300 bytes) at random places of an ASCII array (in place)"""
    L = seq.shape[0]
    for _ in range(n_runs):
        a = int(rng.integers(0, L)); seq[a:a + int(rng.integers(1, 41))] = ord("N")
        a = int(rng.integers(0, L)); b = a + int(rng.integers(1, 301))
        seq[a:b] = np.where((seq[a:b] >= 65) & (seq[a:b] <= 90) & (seq[a:b] != ord("N")), seq[a:b] + 32, seq[a:b])
    return seq


def layout(X, k=19, filler_len=1 << 20, n_filler=16, long_len=(1 << 30) - 1, genome=2_000_000, hit_reads=4000, n_prefix=3, seed=8100):
    """-> dict(lib = [exact_ref.LibRead], order = int64[], kmers sorted uint64, k, X, D, rows: S / E / T / P / suffix (first read of the
    suffix), genome pair a, b)"""
    rng = np.random.default_rng(seed)
    a = datagen.random_genome(genome, seed + 1)
    b = datagen.mutate(a, 0.01, seed + 2)
    fillers = []
    for i in range(n_filler):
        f = ACGT[rng.integers(0, 4, filler_len + 2 * int(rng.integers(0, 500)) + 1, dtype=np.uint8)]      # odd lengths
        fillers.append(_sprinkle(rng, f, 4))
    drop = np.unique(np.concatenate([exact_ref.window_values(exact_ref.LibRead(f, f, f.shape[0]).cyclic(k), k)[0] for f in fillers]))
    kmers = np.setdiff1d(datagen.discriminative_kmers([a, b], k), drop)
    hit = datagen.sample_reads(a, hit_reads, 5000, seed + 3, error_rate=0.02, length_sigma=0.5, min_len=500, max_len=40000) + \
        datagen.sample_reads(b, hit_reads, 5000, seed + 4, error_rate=0.02, length_sigma=0.5, min_len=500, max_len=40000)
    hit = [ACGT[hit[i]] for i in rng.permutation(len(hit))]
    S = _sprinkle(rng, ACGT[datagen.sample_reads(a, 1, 20000, seed + 5)[0]], 3)
    T = _sprinkle(rng, ACGT[datagen.sample_reads(b, 1, 20000, seed + 6)[0]], 3)
    # P's tail: 512 bases of a that end with a window of the set, with an N run and lowercase bytes
    va = datagen.canonical_kmers(a, k)
    ends = np.flatnonzero(np.isin(va, kmers)) + k
    e = int(ends[np.searchsorted(ends, 1000)])
    tail = ACGT[a[e - 512:e]].copy()
    tail[100:110] = ord("N"); tail[200:260] += 32
    lib = [exact_ref.LibRead(f) for f in fillers] + [exact_ref.LibRead(h) for h in hit]
    iS, iT, iE, iP = len(lib), len(lib) + 1, len(lib) + 2, len(lib) + 3
    lib += [exact_ref.LibRead(S), exact_ref.LibRead(T), exact_ref.LibRead(np.zeros(0, np.uint8)),
            exact_ref.LibRead(tail, fillers[0], long_len - tail.shape[0])]
    flen = [f.shape[0] for f in fillers]
    order, pos = [], 0

    def put(i):
        nonlocal pos
        order.append(i); pos += len(lib[i])

    def fill_to(target):
        """fillers, then a pad, so that the next read starts at target"""
        while target - pos > max(flen):
            put(int(rng.integers(0, n_filler)))
        need = target - pos
        assert need >= 0
        if need:
            j = int(np.argmax(flen))
            lib.append(exact_ref.LibRead(fillers[j][:need]))
            put(len(lib) - 1)

    for i in range(n_prefix):
        put(i % n_filler)
    D = pos
    half = len(hit) // 2
    first = n_filler + np.arange(half)
    s_at = X - S.shape[0] // 2
    # fillers with the first half of the hit reads at random places among them, up to S
    budget = s_at - pos - int(sum(len(lib[i]) for i in first)) - 2 * max(flen)
    fill = []
    while budget > 0:
        j = int(rng.integers(0, n_filler)); fill.append(j); budget -= flen[j]
    fill = np.array(fill, dtype=np.int64)
    mixed = np.concatenate([fill, first])[rng.permutation(fill.shape[0] + half)]
    for i in mixed.tolist():
        put(i)
    fill_to(s_at)
    rows = dict(S=len(order))
    put(iS)
    fill_to(X + D)
    rows["E"] = len(order); put(iE)
    rows["T"] = len(order); put(iT)
    rows["P"] = len(order); put(iP)
    for i in (n_filler + np.arange(half, len(hit))).tolist():
        put(i)
        if rng.random() < 0.01:
            put(int(rng.integers(0, n_filler)))
    rows["suffix"] = n_prefix
    return dict(lib=lib, order=np.array(order, dtype=np.int64), kmers=kmers, k=k, X=X, D=D, rows=rows, a=a, b=b)


def read_off(L, order=None):
    """read offsets of the stream (or of the reads `order` of it)"""
    o = L["order"] if order is None else order
    lens = np.array([len(r) for r in L["lib"]], dtype=np.uint64)
    off = np.zeros(o.shape[0] + 1, dtype=np.uint64)
    np.cumsum(lens[o], out=off[1:])
    return off


def materialise(L):
    """the stream's ASCII bytes (uint8) and read offsets"""
    off = read_off(L)
    out = np.empty(int(off[-1]), dtype=np.uint8)
    cache = {}
    for r, i in enumerate(L["order"].tolist()):
        if i not in cache:
            cache[i] = L["lib"][i].bytes()
        out[int(off[r]):int(off[r + 1])] = cache[i]
        if L["lib"][i].head:
            del cache[i]                                   # a long periodic read is needed once
    return out, off


def clip_runs(st, en, lo, hi):
    """exception runs of a stream clipped to the slice [lo, hi) and made relative to lo (what jf_occurrences does per file)"""
    st = np.asarray(st, dtype=np.uint64); en = np.asarray(en, dtype=np.uint64)
    s = np.maximum(st, np.uint64(lo)); e = np.minimum(en, np.uint64(hi))
    keep = e > s
    return s[keep] - np.uint64(lo), e[keep] - np.uint64(lo)
