"""GPU: the packed scan (hga_scan_packed / hga_scan_packed_device) gives what the ASCII scan gives, value for value, for every k, for
inputs full of exception bytes (N, lowercase, CR), for slices of larger buffers at any base / byte offset, in the pipelined host path,
after an overflow rerun and at tens of Mbases; every later stage agrees as well; bad arguments fail with HGA_E_ARG; the CLI, which
now packs while it loads, still exports what the oracle computes."""
import os
import subprocess

import numpy as np
import pytest

import datagen
import exact_ref

pytestmark = pytest.mark.gpu

HGA_E_ARG = 2
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EXE = os.path.join(ROOT, "hybrid-genome-assembler_b200", "categorization")


def _join(seqs):
    seqs = [s.encode() if isinstance(s, str) else s for s in seqs]
    off = np.zeros(len(seqs) + 1, dtype=np.uint64)
    np.cumsum([len(s) for s in seqs], out=off[1:])
    return b"".join(seqs), off


def _hits(h):
    return h.get_hits()


def _same(a, b, what):
    for x, y, name in zip(a, b, ("row offsets", "k-mer ids", "positions")):
        assert np.array_equal(x, y), f"{what}: {name} differ"


def _mess(rng, seq, n_runs=3):
    """N runs, lowercase stretches and single CR bytes in a read"""
    s = bytearray(seq.encode() if isinstance(seq, str) else seq)
    for _ in range(n_runs):
        if not s:
            break
        a = int(rng.integers(0, len(s))); L = int(rng.integers(1, 40))
        kind = int(rng.integers(0, 3))
        if kind == 0:
            s[a:a + L] = b"N" * len(s[a:a + L])
        elif kind == 1:
            s[a:a + L] = bytes(s[a:a + L]).lower()
        else:
            s[a] = 13
    return bytes(s)


def _scan_both(h, bases, off):
    """ASCII scan, then packed scan of the same bytes on the same handle; returns both hit sets"""
    import hga_b200
    h.scan(bases, off)
    a = _hits(h)
    packed, st, en = hga_b200.pack_bases(bases)
    h.scan_packed(packed, off, st, en)
    return a, _hits(h), len(st)


@pytest.mark.parametrize("k", [1, 2, 5, 15, 16, 17, 19, 21, 27, 31, 32])
def test_packed_equals_ascii_and_oracle_for_every_k(oracle, k):
    import hga_b200
    rng = np.random.default_rng(100 + k)
    g = datagen.random_genome(30000, 200 + k)
    reads = [datagen.to_ascii(r) for r in datagen.sample_reads(g, 300, 400, 300 + k, length_sigma=0.8, min_len=1)]
    reads += ["", datagen.to_ascii(g[:max(k - 1, 0)]), datagen.to_ascii(g[100:100 + k]), "", "N" * (k + 3), datagen.to_ascii(g[500:500 + k]).lower()]
    seqs = [_mess(rng, r, int(rng.integers(0, 4))) for r in reads]
    seqs = [seqs[i] for i in rng.permutation(len(seqs))]
    bases, off = _join(seqs)
    km = datagen.canonical_kmers(g, k)
    kmers = np.unique(km[rng.random(km.shape[0]) < 0.3])
    want = oracle.scan(bases, off, k, kmers)
    with hga_b200.Handle(kmers, k) as h:
        a, p, n_exc = _scan_both(h, bases, off)
    assert n_exc > 50
    _same(a, want, "ASCII vs oracle")
    _same(p, want, "packed vs oracle")
    assert p[1].shape[0] > 100


def test_dense_and_awkward_exceptions(oracle, monkeypatch):
    """an all-N read, an all-lowercase read, an exception every other base, runs across tiles, reads and pipeline chunks
    (HGA_SCAN_CHUNK_MB=1: the host copy travels in 1 Mbase chunks while the scan runs)"""
    import hga_b200
    k = 17
    rng = np.random.default_rng(5)
    g = datagen.random_genome(400_000, 6)
    reads = [datagen.to_ascii(r) for r in datagen.sample_reads(g, 1500, 2000, 7, length_sigma=0.5, min_len=1)]
    seqs = []
    for i, r in enumerate(reads):
        if i % 50 == 0:
            r = "N" * len(r)
        elif i % 50 == 1:
            r = r.lower()
        elif i % 50 == 2:
            r = "".join(c if j % 2 else "n" for j, c in enumerate(r))
        elif i % 7 == 3:
            r = r[:-5] + "NNNNN"                       # a run that continues into the next read
        elif i % 7 == 4:
            r = "N" * 700 + r + "N" * 700              # runs longer than a tile
        seqs.append(_mess(rng, r, 2))
    bases, off = _join(seqs)
    assert len(bases) > 2_200_000
    km = datagen.canonical_kmers(g, k)
    kmers = np.unique(km[rng.random(km.shape[0]) < 0.2])
    want = oracle.scan(bases, off, k, kmers)
    monkeypatch.setenv("HGA_SCAN_CHUNK_MB", "1")
    with hga_b200.Handle(kmers, k) as h:
        a, p, n_exc = _scan_both(h, bases, off)
        assert h.metrics()["h2d_ms"] > 0
    assert n_exc > 1000
    _same(a, want, "ASCII vs oracle")
    _same(p, want, "packed vs oracle")


def test_in_place_slices_host_and_device():
    """first_base 0..15 inside a larger host buffer; hga_scan_packed_device on a slice at byte offsets 0..3 of a device buffer"""
    import torch
    import hga_b200
    k = 21
    rng = np.random.default_rng(11)
    g = datagen.random_genome(50_000, 12)
    reads = [_mess(rng, datagen.to_ascii(r), 2) for r in datagen.sample_reads(g, 400, 300, 13, length_sigma=0.5, min_len=1)]
    bases, off = _join(reads)
    km = datagen.canonical_kmers(g, k)
    kmers = np.unique(km[rng.random(km.shape[0]) < 0.3])
    _, st, en = hga_b200.pack_bases(bases)
    assert len(st) > 100
    with hga_b200.Handle(kmers, k) as h:
        h.scan(bases, off)
        want = _hits(h)
        for fb in range(16):
            junk = _mess(rng, datagen.to_ascii(rng.integers(0, 4, fb + 37, dtype=np.uint8)), 2)
            full, _, _ = hga_b200.pack_bases(junk[:fb] + bases + junk[fb:])
            h.scan_packed(full, off, st, en, first_base=fb)
            _same(_hits(h), want, f"host first_base {fb}")
        d_off = torch.from_numpy(off.astype(np.int64)).cuda()
        d_st = torch.from_numpy(st.astype(np.int64)).cuda(); d_en = torch.from_numpy(en.astype(np.int64)).cuda()
        for byte_off in range(4):
            for sub in range(4):
                fb = 4 * 3 + sub
                full, _, _ = hga_b200.pack_bases(b"ACGTNACGTACGTnGA"[:fb] + bases + b"TTTT")
                buf = torch.zeros(len(full) + 64, dtype=torch.uint8, device="cuda")
                buf[byte_off:byte_off + len(full)].copy_(torch.from_numpy(full))
                torch.cuda.synchronize()
                h.scan_packed_device(buf.data_ptr() + byte_off, fb, d_off.data_ptr(), len(reads), len(bases), d_st.data_ptr(), d_en.data_ptr(), len(st))
                _same(_hits(h), want, f"device byte offset {byte_off}, first_base {fb}")
                del buf
        # no runs at all: the kernel never reads the run arrays (NULL pointers with n_exc = 0)
        clean = [datagen.to_ascii(r) for r in datagen.sample_reads(g, 300, 300, 14, min_len=1)]
        cb, co = _join(clean)
        h.scan(cb, co)
        want = _hits(h)
        cp, cs, ce = hga_b200.pack_bases(cb)
        assert len(cs) == 0
        h.scan_packed(cp, co, cs, ce)
        _same(_hits(h), want, "clean host")
        buf = torch.from_numpy(cp).cuda(); d_co = torch.from_numpy(co.astype(np.int64)).cuda()
        torch.cuda.synchronize()
        h.scan_packed_device(buf.data_ptr(), 0, d_co.data_ptr(), len(clean), len(cb), 0, 0, 0)
        _same(_hits(h), want, "clean device")


def test_scale_and_denser_rerun():
    """~38 Mbases of long reads judged by exact_ref (hit buffer sized from a count-only sample), then a denser packed scan on the same
    handle overflows the estimate from the first one's density and reruns with the exact count"""
    import hga_b200
    k = 21
    dense = datagen.random_genome(1_500_000, 7201)
    other = datagen.random_genome(1_500_000, 7202)
    kmers = np.unique(datagen.canonical_kmers(dense, k))
    first = datagen.sample_reads(dense, 2600, 5000, 7203, length_sigma=0.3, min_len=1000) + \
        datagen.sample_reads(other, 5000, 5000, 7204, length_sigma=0.3, min_len=1000)
    first = [datagen.to_ascii(first[i]) for i in np.random.default_rng(7205).permutation(len(first))]
    second = [datagen.to_ascii(r) for r in datagen.sample_reads(dense, 7600, 5000, 7206, length_sigma=0.3, min_len=1000)]
    b1, o1 = _join(first)
    b2, o2 = _join(second)
    h1 = exact_ref.scan(b1, o1, k, kmers)
    h2 = exact_ref.scan(b2, o2, k, kmers)
    assert len(b1) > 32 << 20 and len(b2) > 32 << 20
    with hga_b200.Handle(kmers, k) as h:
        p, s, e = hga_b200.pack_bases(b1)
        h.scan_packed(p, o1, s, e)
        _same(_hits(h), h1, "first packed scan")
        p, s, e = hga_b200.pack_bases(b2)
        h.scan_packed(p, o2, s, e)
        assert h.metrics()["scan_retries"] == 1, "the denser scan was meant to overflow its estimated hit buffer"
        _same(_hits(h), h2, "denser packed scan")


def _chain(h, read_off):
    out = {"hits": h.get_hits(), "sorted": h.get_hits(sorted_by_kmer_id=True)}
    h.build_index()
    out["index"] = h.get_index()
    h.pair_count(min_score=1)
    out["pairs"] = h.get_pairs()
    h.select_edges(fraction=0.15)
    out["selection"] = h.get_selection()
    h.components(min_size=5)
    out["components"] = h.get_components()
    h.enrich_full(read_off, min_size=5, enrichment_min_score=20)
    out["enrichment"] = h.get_enrichment()
    out["tail"] = h.get_tail_block()
    out["purged"] = h.get_purged_index()
    out["core_kmers"] = h.get_core_kmers()
    return out


def _equal(a, b, path="result"):
    if isinstance(a, dict):
        assert a.keys() == b.keys(), path
        for key in a:
            _equal(a[key], b[key], f"{path}.{key}")
    elif isinstance(a, (list, tuple)):
        assert len(a) == len(b), path
        for i, (x, y) in enumerate(zip(a, b)):
            _equal(x, y, f"{path}[{i}]")
    elif isinstance(a, np.ndarray):
        assert np.array_equal(a, b), path
    else:
        assert a == b, path


def test_later_stages_equal_after_packed_and_ascii_scans():
    """index, pairs, selection, components, hga_enrich_full with its tail block: value for value, from an ASCII scan and from a
    packed scan of reads with N runs and lowercase stretches"""
    import hga_b200
    k = 19
    rng = np.random.default_rng(21)
    a = datagen.random_genome(60000, 22)
    b = datagen.mutate(a, 0.03, 23)
    reads = datagen.sample_reads(a, 700, 1500, 24, error_rate=0.01, length_sigma=0.4) + datagen.sample_reads(b, 700, 1500, 25, error_rate=0.01, length_sigma=0.4)
    seqs = [_mess(rng, datagen.to_ascii(r), 2) for r in reads]
    bases, off = _join(seqs)
    kmers = datagen.discriminative_kmers([a, b], k)
    with hga_b200.Handle(kmers, k) as h:
        h.scan(bases, off)
        want = _chain(h, off)
    packed, st, en = hga_b200.pack_bases(bases)
    assert len(st) > 500
    with hga_b200.Handle(kmers, k) as h:
        h.scan_packed(packed, off, st, en)
        got = _chain(h, off)
    assert want["selection"]["x"].shape[0] > 100
    _equal(want, got)


def test_argument_errors_on_both_entries():
    import torch
    import hga_b200
    k = 11
    g = datagen.random_genome(5000, 31)
    bases, off = _join([datagen.to_ascii(g[i:i + 500]) for i in range(0, 5000, 500)])
    packed, _, _ = hga_b200.pack_bases(bases)
    kmers = np.unique(datagen.canonical_kmers(g, k))[:1000]
    n = len(bases)
    bad_runs = {"unsorted": ([100, 10], [110, 20]), "overlapping": ([10, 15], [20, 30]), "empty": ([10], [10]), "reversed": ([20], [10]),
                "out of range": ([n - 2], [n + 1])}
    with hga_b200.Handle(kmers, k) as h:
        d_p = torch.from_numpy(packed).cuda(); d_off = torch.from_numpy(off.astype(np.int64)).cuda()
        for name, (s, e) in bad_runs.items():
            s = np.array(s, dtype=np.uint64); e = np.array(e, dtype=np.uint64)
            with pytest.raises(hga_b200.HgaError) as x:
                h.scan_packed(packed, off, s, e)
            assert x.value.code == HGA_E_ARG, name
            d_s = torch.from_numpy(s.astype(np.int64)).cuda(); d_e = torch.from_numpy(e.astype(np.int64)).cuda()
            torch.cuda.synchronize()
            with pytest.raises(hga_b200.HgaError) as x:
                h.scan_packed_device(d_p.data_ptr(), 0, d_off.data_ptr(), len(off) - 1, n, d_s.data_ptr(), d_e.data_ptr(), len(s))
            assert x.value.code == HGA_E_ARG, name
            with pytest.raises(hga_b200.HgaError):
                h.get_hits()                                  # no scan result survives a refused scan
        shifted = off + np.uint64(4)
        with pytest.raises(hga_b200.HgaError) as x:
            h.scan_packed(packed, shifted, [], [])
        assert x.value.code == HGA_E_ARG and "read_off[0]" in str(x.value)
        d_sh = torch.from_numpy(shifted.astype(np.int64)).cuda()
        torch.cuda.synchronize()
        with pytest.raises(hga_b200.HgaError) as x:
            h.scan_packed_device(d_p.data_ptr(), 0, d_sh.data_ptr(), len(off) - 1, n, 0, 0, 0)
        assert x.value.code == HGA_E_ARG and "read_off[0]" in str(x.value)
        ro = off.astype(np.uint64)
        for args in ((0, 0, ro.ctypes.data, len(off) - 1, 0, 0, 0),                  # NULL packed
                     (packed.ctypes.data, 0, 0, len(off) - 1, 0, 0, 0),               # NULL read_off
                     (packed.ctypes.data, 0, ro.ctypes.data, len(off) - 1, 0, 0, 3)):  # NULL runs
            with pytest.raises(hga_b200.HgaError) as x:
                h.scan_packed_host_ptr(*args)
            assert x.value.code == HGA_E_ARG
        for args in ((0, 0, d_off.data_ptr(), len(off) - 1, n, 0, 0, 0),
                     (d_p.data_ptr(), 0, 0, len(off) - 1, n, 0, 0, 0),
                     (d_p.data_ptr(), 0, d_off.data_ptr(), len(off) - 1, n, 0, 0, 2)):
            with pytest.raises(hga_b200.HgaError) as x:
                h.scan_packed_device(*args)
            assert x.value.code == HGA_E_ARG
        h.scan_packed(packed, off, [], [])                    # the handle still works
        assert h.metrics()["n_bases"] == n


def _messy_case(tmp_path, seed):
    """diploid reads in two files: N runs, lowercase reads, CRLF line ends in one of them"""
    paths, kp = datagen.make_diploid_case(str(tmp_path / "c"), genome_size=30000, divergence=0.03, k=19, read_len=1200, coverage=12, seed=seed,
                                          error_rate=0.01, fmt="fastq", length_sigma=0.3)
    rng = np.random.default_rng(seed)
    for fi, p in enumerate(paths):
        lines = open(p, "rb").read().split(b"\n")
        for i in range(1, len(lines), 4):
            if lines[i]:
                if i % 13 == 1:
                    lines[i] = lines[i].lower()
                else:
                    lines[i] = _mess(rng, lines[i], 2).replace(b"\r", b"N")
        nl = b"\r\n" if fi == 1 else b"\n"
        open(p, "wb").write(nl.join(lines))
    return paths, kp


def test_cli_with_exceptions_exports_what_the_oracle_says(oracle, tmp_path):
    assert os.path.exists(EXE)
    paths, kp = _messy_case(tmp_path, 41)
    outdir = str(tmp_path / "out")
    r = subprocess.run([EXE] + paths + ["--kmers", kp, "-o", outdir, "--sc_min_size", "5", "--scaffolds-only"], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    rc, reads = oracle.load_reads(paths)
    assert rc == 0 and b"n" in reads["seq"] and b"N" in reads["seq"] and b"\r" in reads["seq"]
    kmers, k = oracle.load_kmers(kp)
    ref = oracle.run(reads["seq"], reads["seq_off"], k, kmers, fraction=0.15, min_size=5)
    co, cm, _, _, _ = ref["comp"]
    co = co.astype(np.int64)
    hdr_off = reads["hdr_off"].astype(np.int64)
    want = sorted(sorted(reads["hdr"][hdr_off[i - 1]:hdr_off[i]].decode() for i in cm[co[c]:co[c + 1]]) for c in range(len(co) - 1))
    got = []
    for f in sorted(os.listdir(outdir)):
        lines = open(os.path.join(outdir, f), newline="").read().split("\n")
        got.append(sorted(l[1:] for l in lines[0::4] if l))
    assert len(want) >= 2 and sorted(got) == want
    # the exported records are the input bytes (sequence views into the files, CR included)
    raw = b"".join(open(p, "rb").read() for p in paths)
    for f in os.listdir(outdir):
        data = open(os.path.join(outdir, f), "rb").read()
        for rec in data.split(b"\n@")[:20]:
            seq = rec.split(b"\n")[1]
            assert seq in raw


def test_cli_two_gpus_with_exceptions(tmp_path):
    import hga_b200
    if hga_b200.capi.device_count() < 2:
        pytest.skip("needs two GPUs")
    paths, kp = _messy_case(tmp_path, 43)
    outs = []
    for gpus in (1, 2):
        outdir = str(tmp_path / f"out{gpus}")
        r = subprocess.run([EXE] + paths + ["--kmers", kp, "-o", outdir, "--sc_min_size", "5", "--scaffolds-only", "--gpus", str(gpus)], capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
        outs.append({f: open(os.path.join(outdir, f), "rb").read() for f in sorted(os.listdir(outdir))})
    assert outs[0] == outs[1] and len(outs[0]) >= 2
