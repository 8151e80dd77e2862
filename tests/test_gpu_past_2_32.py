"""GPU: scan, the stages after it and the k-mer count past 2^32 bases, and the entries' limits, against the exact reference.

The stream of about 5.4 Gbases is big_stream.layout with X = 2^32 (about 270 copies of 16 hit-free filler reads of ~1 Mbases, 40 Mbases
of diploid long reads each used once, half of them on each side of 2^32, a read across 2^32, an empty read and a read at exactly 2^32
in the stream that starts D bases in, a read of 2^30 - 1 bases past 2^32; N runs and lowercase bytes throughout). Its reference is
built from the library (exact_ref.library_hits / stream_hits / library_counts / stream_counts), which test_big_stream_cpu.py checks
against the direct reference on the same layout at X = 2^24. Every output is compared value for value; every test asserts what shows
that it reached its regime.

  - scan -> index -> pairs -> selection -> components, hga_scan (pipelined, 256 MB chunks) and hga_scan_device at an unaligned address
  - hga_scan_packed / hga_scan_packed_device, exception runs on both sides of 2^32, a slice at a first_base above 2^32
  - the read-length limit (reads shorter than 2^30 bases) on all four scan entries
  - hga_count_kmers[_packed] and hga_count_spectrum[_packed] with more than 2^32 windows, in key-range passes
  - one k-mer seen 2^32 - 1 times (the largest count the count returns) and more than that (HGA_E_OVERFLOW; the spectrum stays exact)
"""
import re
import time

import numpy as np
import pytest

import big_stream
import exact_ref
from test_gpu_exact_reference import _check_components, _check_hits, _check_index, _check_pairs, _check_selection

pytestmark = pytest.mark.gpu

HGA_E_ARG = 2
HGA_E_OVERFLOW = 5
X = 1 << 32


@pytest.fixture(scope="module")
def layout():
    return big_stream.layout(X)


@pytest.fixture(scope="module")
def big(layout):
    L = layout
    bases, off = big_stream.materialise(L)
    k, kmers, r = L["k"], L["kmers"], L["rows"]
    lib_hits = exact_ref.library_hits(L["lib"], k, kmers)
    B = dict(L=L, bases=bases, off=off, lib_hits=lib_hits, hits=exact_ref.stream_hits(lib_hits, L["order"]))
    B["pairs"] = exact_ref.pairs(B["hits"][0], B["hits"][1], len(kmers))
    # the regime: more than 2^32 bases, S across 2^32, E and T at D + 2^32 (at 2^32 in the suffix), P of 2^30 - 1 bases past 2^32
    # with hits in its last 512 bases, hit reads on both sides of 2^32
    D = L["D"]
    assert off[-1] > X + (1 << 30) and off[r["S"]] < X < off[r["S"] + 1] and off[r["E"]] == off[r["T"]] == X + D
    assert off[r["P"] + 1] - off[r["P"]] == (1 << 30) - 1 and off[r["P"]] > X
    ro = B["hits"][0].astype(np.int64)
    p_pos = B["hits"][2][ro[r["P"]]:ro[r["P"] + 1]].astype(np.int64)
    assert p_pos.shape[0] and p_pos.min() > (1 << 30) - 1 - 512
    rows_with_hits = np.flatnonzero(np.diff(ro))
    assert (off[rows_with_hits] < X).sum() > 1000 and (off[rows_with_hits] > X).sum() > 1000
    return B


def _device(arr, lead):
    """a device copy of a uint8 / uint64 host array starting `lead` bytes into a fresh buffer -> (buffer, address)"""
    import torch
    raw = np.ascontiguousarray(arr).view(np.uint8)
    buf = torch.empty(raw.shape[0] + lead + 64, dtype=torch.uint8, device="cuda")
    buf[lead:lead + raw.shape[0]].copy_(torch.from_numpy(raw))
    torch.cuda.synchronize()
    return buf, buf.data_ptr() + lead


def test_scan_to_components_past_2_32_ascii(big):
    """hga_scan of the whole stream (pipelined), every stage after it, and the suffix; then hga_scan_device of both from an address
    that is not 16-byte aligned"""
    import hga_b200
    import torch
    L, bases, off = big["L"], big["bases"], big["off"]
    k, kmers, r, D = L["k"], L["kmers"], L["rows"], L["D"]
    s0 = r["suffix"]
    off_s = off[s0:] - off[s0]
    hits_s = exact_ref.stream_hits(big["lib_hits"], L["order"][s0:])
    with hga_b200.Handle(kmers, k) as h:
        h.scan(bases, off)
        m = h.metrics()
        assert m["n_bases"] == off[-1] > X and m["n_bases"] > 2 * (256 << 20)          # more than two 256 MB chunks: pipelined
        _check_hits(h, big["hits"])
        h.build_index()
        _check_index(h, big["hits"], len(kmers))
        h.pair_count(min_score=1)
        _check_pairs(h, big["pairs"])
        sel = _check_selection(h, big["pairs"], fraction=0.15)
        _check_components(h, len(L["order"]), sel, 10)
        assert big["pairs"][0].shape[0] > 50_000
        h.scan(bases[D:], off_s)
        _check_hits(h, hits_s)
        lead = next(x for x in range(1, 16) if x % 16 and (x + D) % 16)
        buf, ptr = _device(bases, lead)
        d_off, d_off_ptr = _device(off, 0)
        d_off_s, d_off_s_ptr = _device(off_s, 0)
        h.scan_device(ptr, d_off_ptr, len(L["order"]), int(off[-1]))
        _check_hits(h, big["hits"])
        h.build_index()
        _check_index(h, big["hits"], len(kmers))
        h.pair_count(min_score=1)
        _check_pairs(h, big["pairs"])
        _check_components(h, len(L["order"]), _check_selection(h, big["pairs"], fraction=0.15), 10)
        h.scan_device(ptr + D, d_off_s_ptr, len(off_s) - 1, int(off_s[-1]))
        _check_hits(h, hits_s)
        del buf, d_off, d_off_s
        torch.cuda.empty_cache()


def test_packed_past_2_32(big):
    """hga_scan_packed of the whole stream and of a slice at first_base = D + 2^32 (no multiple of 4), and hga_scan_packed_device of
    both from an odd byte address"""
    import hga_b200
    import torch
    L, bases, off = big["L"], big["bases"], big["off"]
    k, kmers, r = L["k"], L["kmers"], L["rows"]
    packed, st, en = hga_b200.pack_bases(bases)
    assert (en < X).sum() > 100 and (st > X).sum() > 100, "exception runs on both sides of 2^32"
    t = r["T"]
    fb = int(off[t])
    assert fb > X and fb % 4
    off_t = off[t:] - off[t]
    cst, cen = big_stream.clip_runs(st, en, fb, int(off[-1]))
    hits_t = exact_ref.stream_hits(big["lib_hits"], L["order"][t:])
    with hga_b200.Handle(kmers, k) as h:
        h.scan_packed(packed, off, st, en)
        _check_hits(h, big["hits"])
        h.scan_packed(packed, off_t, cst, cen, first_base=fb)
        _check_hits(h, hits_t)
        buf, ptr = _device(packed, 3)
        d_off, d_off_ptr = _device(off, 0)
        d_st, d_st_ptr = _device(st, 0)
        d_en, d_en_ptr = _device(en, 0)
        h.scan_packed_device(ptr, 0, d_off_ptr, len(L["order"]), int(off[-1]), d_st_ptr, d_en_ptr, st.shape[0])
        _check_hits(h, big["hits"])
        d_off_t, d_off_t_ptr = _device(off_t, 0)
        d_cst, d_cst_ptr = _device(cst, 0)
        d_cen, d_cen_ptr = _device(cen, 0)
        h.scan_packed_device(ptr, fb, d_off_t_ptr, len(off_t) - 1, int(off_t[-1]), d_cst_ptr, d_cen_ptr, cst.shape[0])
        _check_hits(h, hits_t)
        del buf, d_off, d_st, d_en, d_off_t, d_cst, d_cen
        torch.cuda.empty_cache()


def _limit_case(L):
    """bases of a short read and a periodic read of 2^30 bases whose last window is a hit; read offsets that make them 2^30 - 1
    (the first base of the long read joins the short one) and 2^30 bases long; the reference hits of the valid split"""
    k, kmers = L["k"], L["kmers"]
    P = L["lib"][L["order"][L["rows"]["P"]]]
    short = L["lib"][L["order"][L["rows"]["S"]]].tail
    long_bad = exact_ref.LibRead(P.tail, P.block, (1 << 30) - P.tail.shape[0])
    lb = long_bad.bytes()
    bases = np.concatenate([short, lb])
    del lb
    n = short.shape[0]
    off_ok = np.array([0, n + 1, n + (1 << 30)], dtype=np.uint64)
    off_bad = np.array([0, n, n + (1 << 30)], dtype=np.uint64)
    lib_ok = [exact_ref.LibRead(bases[:n + 1]), exact_ref.LibRead(P.tail, np.roll(P.block, -1), (1 << 30) - 1 - P.tail.shape[0])]
    want = exact_ref.stream_hits(exact_ref.library_hits(lib_ok, k, kmers), np.array([0, 1]))
    ro = want[0].astype(np.int64)
    assert want[2][ro[1]:ro[2]].max() == (1 << 30) - 1, "a hit ends at the last base of the read of 2^30 - 1 bases"
    assert want[2][ro[1]:ro[2]].min() > (1 << 30) - 1 - 512
    return bases, off_ok, off_bad, want


def _refused(fn):
    import hga_b200
    with pytest.raises(hga_b200.HgaError) as e:
        fn()
    assert e.value.code == HGA_E_ARG and "2^30" in str(e.value), str(e.value)


def test_read_length_limit_on_every_scan_entry(layout):
    """a read of 2^30 - 1 bases scans exactly on every scan entry, hits at its last base included; a read of 2^30 bases fails with
    HGA_E_ARG and a message, and the same handle then scans the valid input exactly"""
    import hga_b200
    import torch
    L = layout
    bases, off_ok, off_bad, want = _limit_case(L)
    packed, st, en = hga_b200.pack_bases(bases)
    assert st.shape[0] > 0
    with hga_b200.Handle(L["kmers"], L["k"]) as h:
        h.scan(bases, off_ok)
        _check_hits(h, want)
        _refused(lambda: h.scan(bases, off_bad))
        h.scan(bases, off_ok)
        _check_hits(h, want)
        h.scan_packed(packed, off_ok, st, en)
        _check_hits(h, want)
        _refused(lambda: h.scan_packed(packed, off_bad, st, en))
        h.scan_packed(packed, off_ok, st, en)
        _check_hits(h, want)
        buf, ptr = _device(bases, 7)
        d_ok, d_ok_ptr = _device(off_ok, 0)
        d_bad, d_bad_ptr = _device(off_bad, 0)
        _refused(lambda: h.scan_device(ptr, d_bad_ptr, 2, int(off_bad[-1])))
        h.scan_device(ptr, d_ok_ptr, 2, int(off_ok[-1]))
        _check_hits(h, want)
        del buf
        pbuf, pptr = _device(packed, 1)
        d_st, d_st_ptr = _device(st, 0)
        d_en, d_en_ptr = _device(en, 0)
        _refused(lambda: h.scan_packed_device(pptr, 0, d_bad_ptr, 2, int(off_bad[-1]), d_st_ptr, d_en_ptr, st.shape[0]))
        h.scan_packed_device(pptr, 0, d_ok_ptr, 2, int(off_ok[-1]), d_st_ptr, d_en_ptr, st.shape[0])
        _check_hits(h, want)
        del pbuf, d_ok, d_bad, d_st, d_en
        torch.cuda.empty_cache()


def _passes(capfd):
    err = capfd.readouterr().err
    got = [int(v) for v in re.findall(r"(\d+) key-range passes", err)]
    assert got, err
    return got[-1]


def _same_counts(got, want):
    assert got[0].shape[0] == want[0].shape[0], f"{got[0].shape[0]} k-mers, want {want[0].shape[0]}"
    assert np.array_equal(got[0], want[0]), "k-mers differ"
    assert np.array_equal(got[1].astype(np.int64), want[1]), "counts differ"


def _same_spectrum(got, c, n_bins):
    hist, n_windows, n_distinct, max_count = exact_ref.spectrum(c, n_bins)
    assert (got[1], got[2], got[3]) == (n_windows, n_distinct, max_count)
    assert np.array_equal(got[0], hist)


def test_count_and_spectrum_past_2_32(big, capfd, monkeypatch):
    """hga_count_kmers / _packed with min_count 1 and 2, a packed slice counted in place at first_base = D + 2^32, and the spectra
    with n_bins 0 and 1000, in key-range passes over more than 2^32 windows"""
    import hga_b200
    monkeypatch.setenv("HGA_COUNT_STATS", "1")
    L, bases, off = big["L"], big["bases"], big["off"]
    k, r = L["k"], L["rows"]
    lib_counts = exact_ref.library_counts(L["lib"], k)
    want1 = exact_ref.stream_counts(lib_counts, L["order"], 1)
    c = want1[1]
    want2 = (want1[0][c >= 2], c[c >= 2])
    assert int(c.sum()) > X and c.min() == 1 and (c == 2).any() and ((c >= 100) & (c < 1000)).any()
    _same_counts(hga_b200.capi.count_kmers(bases, off, k, min_count=1), want1)
    assert _passes(capfd) > 1
    _same_counts(hga_b200.capi.count_kmers(bases, off, k, min_count=2), want2)
    assert _passes(capfd) > 1
    fp, fst, fen = hga_b200.pack_bases(bases, fold_case=True)
    assert (fen < X).sum() > 100 and (fst > X).sum() > 100
    _same_counts(hga_b200.capi.count_kmers_packed(fp, off, fst, fen, k, min_count=1), want1)
    assert _passes(capfd) > 1
    _same_counts(hga_b200.capi.count_kmers_packed(fp, off, fst, fen, k, min_count=2), want2)
    assert _passes(capfd) > 1
    t = r["T"]
    fb = int(off[t])
    assert fb > X and fb % 4
    cst, cen = big_stream.clip_runs(fst, fen, fb, int(off[-1]))
    _same_counts(hga_b200.capi.count_kmers_packed(fp, off[t:] - off[t], cst, cen, k, min_count=2, first_base=fb),
                 exact_ref.stream_counts(lib_counts, L["order"][t:], 2))
    _same_spectrum(hga_b200.capi.count_spectrum(bases, off, k, n_bins=1000), c, 1000)
    assert _passes(capfd) > 1
    _same_spectrum(hga_b200.capi.count_spectrum_packed(fp, off, fst, fen, k, n_bins=0), c, 0)
    _same_spectrum(hga_b200.capi.count_spectrum_packed(fp, off, fst, fen, k, n_bins=1000), c, 1000)
    assert _passes(capfd) > 1


def _poly_a(k, n_windows):
    """all-zero packed bases (poly-A) in reads shorter than 2^30 that hold n_windows windows of k bases in all"""
    per = (1 << 30) - 1
    lens = []
    left = n_windows
    while left > 0:
        w = min(left, per - k + 1)
        lens.append(w + k - 1)
        left -= w
    off = np.zeros(len(lens) + 1, dtype=np.uint64)
    np.cumsum(lens, out=off[1:])
    return np.zeros((int(off[-1]) + 3) // 4, dtype=np.uint8), off


def test_count_past_32_bits_poly_a(capfd, monkeypatch):
    """k-mer 0 (poly-A) seen exactly 2^32 - 1 times comes back with that count; seen 2^32 + 2^20 times, the count fails with
    HGA_E_OVERFLOW and a message that names the count, and the spectrum of the same input is exact. The key range is split down to the
    one k-mer (about 64 midpoint splits whatever k is); the time each call takes is printed"""
    import hga_b200
    monkeypatch.setenv("HGA_COUNT_STATS", "1")
    k = 25
    none = np.zeros(0, dtype=np.uint64)
    packed, off = _poly_a(k, (1 << 32) - 1)
    t0 = time.perf_counter()
    km, cnt = hga_b200.capi.count_kmers_packed(packed, off, none, none, k, min_count=1)
    t1 = time.perf_counter()
    assert km.tolist() == [0] and cnt.tolist() == [(1 << 32) - 1]
    passes = _passes(capfd)
    assert passes > 64
    big_n = (1 << 32) + (1 << 20)
    packed, off = _poly_a(k, big_n)
    t2 = time.perf_counter()
    with pytest.raises(hga_b200.HgaError) as e:
        hga_b200.capi.count_kmers_packed(packed, off, none, none, k, min_count=1)
    t3 = time.perf_counter()
    assert e.value.code == HGA_E_OVERFLOW and str(big_n) in str(e.value) and "A" * k in str(e.value), str(e.value)
    hist, n_windows, n_distinct, max_count = hga_b200.capi.count_spectrum_packed(packed, off, none, none, k, n_bins=1000)
    t4 = time.perf_counter()
    assert (n_windows, n_distinct, max_count) == (big_n, 1, big_n)
    assert hist[999] == 1 and not hist[:999].any()
    print(f"\npoly-A, k = {k}: count of 2^32 - 1 windows {t1 - t0:.1f} s ({passes} key-range passes), refused count of 2^32 + 2^20 "
          f"windows {t3 - t2:.1f} s, its spectrum {t4 - t3:.1f} s")
