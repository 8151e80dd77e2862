"""GPU: the packed k-mer count (hga_count_kmers_packed on the case-folded packing) gives what hga_count_kmers gives on the ASCII bytes and
what exact counting gives, value for value and in order: for every k of the sweep and more, min_count 1..3, empty and short reads, N runs,
lowercase stretches and CR bytes, runs on read ends and on thread-span ends, slices starting inside a byte, forced key-range passes down
to a single over-budget k-mer, and tens of Mbases. Bad arguments fail with HGA_E_ARG. jf_occurrences, which now packs while it loads,
prints and exports what the ASCII counts pushed through the host functions give."""
import os
import subprocess

import numpy as np
import pytest

import datagen
from test_packed_count_cpu import count_reads, slice_runs
from test_sdk_selection_cpu import exact_counts

pytestmark = pytest.mark.gpu

HGA_E_ARG = 2
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EXE = os.path.join(ROOT, "hybrid-genome-assembler_b200", "jf_occurrences")


def _join(reads):
    reads = [r.encode() if isinstance(r, str) else r for r in reads]
    off = np.zeros(len(reads) + 1, dtype=np.uint64)
    np.cumsum([len(r) for r in reads], out=off[1:])
    return b"".join(reads), off


def _packed_slice(seq, first_base, rng):
    """seq packed (folded) first_base bases into a larger stream, as a caller slicing a file out of a packed buffer sees it"""
    import hga_b200
    pre = np.frombuffer(b"ACGTacgtN", dtype=np.uint8)[rng.integers(0, 9, first_base)].tobytes()
    stream = pre + seq + b"nACGT"
    packed, st, en = hga_b200.pack_bases(stream, fold_case=True)
    es, ee = slice_runs(st, en, first_base, first_base + len(seq))
    return packed, es, ee


def _both(seq, off, k, min_count, first_base=0, seed=0):
    import hga_b200
    packed, es, ee = _packed_slice(seq, first_base, np.random.default_rng(seed))
    got = hga_b200.capi.count_kmers_packed(packed, off, es, ee, k, min_count=min_count, first_base=first_base)
    want = hga_b200.capi.count_kmers(seq, off, k, min_count=min_count)
    return got, want


def _same(a, b):
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])


@pytest.mark.parametrize("k", [1, 2, 5, 11, 15, 16, 17, 19, 21, 31, 32])
def test_packed_count_equals_ascii_and_exact(k):
    reads = count_reads(k, k, n_reads=160)
    reads[20] = reads[20][:33] + "N" * 31 + reads[20][64:]                 # a run across a 32-window span end
    reads[21] = "acgt" * 8 + "N" + reads[21]
    seq, off = _join(reads)
    for i, min_count in enumerate((1, 2, 3)):
        first_base = (k + i) % 4 + 4 * i
        got, want = _both(seq, off, k, min_count, first_base, seed=k)
        _same(got, want)
        _same(got, exact_counts(seq, off, k, min_count))
        assert len(got[0]) > 0


def test_empty_short_and_exception_only_reads():
    import hga_b200
    for k in (1, 4, 19, 32):
        reads = ["", "ACG", "", "N" * 40, "acgtn" * 9, "A" * (k - 1), "\r", "T" * k, "ACGT" * 10 + "\r", "", "tttttttttttttttttttttttttttttttttt"]
        seq, off = _join(reads)
        for first_base in (0, 1, 2, 3):
            got, want = _both(seq, off, k, 1, first_base)
            _same(got, want)
            _same(got, exact_counts(seq, off, k, 1))
    # only empty reads / no reads
    assert len(hga_b200.capi.count_kmers_packed(np.zeros(4, np.uint8), np.zeros(4, np.uint64), [], [], 5, min_count=1)[0]) == 0
    assert len(hga_b200.capi.count_kmers_packed(np.zeros(4, np.uint8), np.zeros(1, np.uint64), [], [], 5, min_count=1)[0]) == 0


@pytest.mark.parametrize("k", [11, 19, 31])
def test_n_runs_lowercase_and_crlf_from_files(tmp_path, k):
    """reads as the CLI loader sees them: CRLF lines leave a CR at the end of every sequence"""
    rng = np.random.default_rng(100 + k)
    g = datagen.random_genome(30000, 200 + k)
    reads = [datagen.to_ascii(r) for r in datagen.sample_reads(g, 300, 400, 300 + k, error_rate=0.01, length_sigma=0.4)]
    out = []
    for j, r in enumerate(reads):
        a = int(rng.integers(0, max(len(r), 1)))
        if j % 3 == 0:
            r = r[:a] + r[a:a + 50].lower() + r[a + 50:]
        if j % 4 == 1:
            r = r[:a] + "N" * int(rng.integers(1, 30)) + r[a:]
        out.append(r + "\r" if j % 2 else r)
    seq, off = _join(out)
    for first_base in (0, 3, 4 * 1000 + 2):
        got, want = _both(seq, off, k, 2, first_base, seed=first_base)
        _same(got, want)
    _same(got, exact_counts(seq, off, k, 2))


def test_forced_key_range_passes_on_a_large_input():
    """~40 Mbases with N runs and lowercase stretches, a budget of 2^21 keys per pass (~30 key ranges; the range of the poly-A k-mer
    overflows and is halved down to that single value) and the single pass, packed and ASCII: all four identical"""
    import hga_b200
    rng = np.random.default_rng(78)
    g = datagen.random_genome(400000, 601)
    g[1000:51000] = 0
    reads = datagen.sample_reads(g, 4000, 10000, 602, error_rate=0.02, length_sigma=0.3, max_len=60000)
    seq = bytearray(b"".join(datagen.to_ascii(r).encode() for r in reads))
    off = np.zeros(len(reads) + 1, dtype=np.uint64)
    np.cumsum([len(r) for r in reads], out=off[1:])
    assert off[-1] > 30_000_000
    n = len(seq)
    for a in rng.integers(0, n - 3000, 400):
        seq[a:a + 2000] = bytes(seq[a:a + 2000]).lower()
    for a in rng.integers(0, n - 300, 400):
        L = int(rng.integers(1, 300))
        seq[a:a + L] = b"N" * L
    seq = bytes(seq)
    first_base = 3
    packed, es, ee = _packed_slice(seq, first_base, rng)
    one = hga_b200.capi.count_kmers_packed(packed, off, es, ee, 19, min_count=2, first_base=first_base)
    ascii_one = hga_b200.capi.count_kmers(seq, off, 19, min_count=2)
    os.environ["HGA_COUNT_CHUNK"] = str(1 << 21)
    try:
        multi = hga_b200.capi.count_kmers_packed(packed, off, es, ee, 19, min_count=2, first_base=first_base)
        ascii_multi = hga_b200.capi.count_kmers(seq, off, 19, min_count=2)
    finally:
        del os.environ["HGA_COUNT_CHUNK"]
    km, ct = one
    assert len(km) > 100000 and np.all(km[1:] > km[:-1]) and km[0] == 0 and ct[0] > (1 << 21)
    _same(one, ascii_one)
    _same(multi, ascii_multi)
    _same(one, multi)


def test_argument_errors():
    import hga_b200
    packed = np.zeros(64, dtype=np.uint8)
    cases = [
        (dict(read_off=[0, 100], st=[], en=[], k=0), "Kmer size"),
        (dict(read_off=[0, 100], st=[], en=[], k=33), "Kmer size"),
        (dict(read_off=[4, 100], st=[], en=[], k=19), "read_off[0] must be 0"),
        (dict(read_off=[0, 100], st=[10, 5], en=[12, 7], k=19), "exception run 1"),           # unsorted
        (dict(read_off=[0, 100], st=[10, 11], en=[12, 14], k=19), "exception run 1"),         # overlapping
        (dict(read_off=[0, 100], st=[90], en=[101], k=19), "exception run 0"),                # outside the read set
        (dict(read_off=[0, 100], st=[10], en=[10], k=19), "exception run 0"),                 # empty
    ]
    for a, what in cases:
        with pytest.raises(hga_b200.HgaError) as e:
            hga_b200.capi.count_kmers_packed(packed, a["read_off"], a["st"], a["en"], a["k"])
        assert e.value.code == HGA_E_ARG and what in str(e.value), (a, str(e.value))


# ---- jf_occurrences --------------------------------------------------------------------------------------------------------------
def _messy_files(tmp_path):
    g = datagen.random_genome(8000, 41)
    g2 = datagen.mutate(g, 0.03, 42)
    paths = []
    for i, hap in enumerate((g, g2, g)):
        rng = np.random.default_rng(50 + i)
        reads = [datagen.to_ascii(r) for r in datagen.sample_reads(hap, 120, 300, 60 + i, error_rate=0.01, length_sigma=0.3)]
        for j in range(len(reads)):
            a = int(rng.integers(0, len(reads[j])))
            if j % 3 == 0:
                reads[j] = reads[j][:a] + reads[j][a:a + 60].lower() + reads[j][a + 60:]
            if j % 5 == 2:
                reads[j] = reads[j][:a] + "N" * int(rng.integers(1, 20)) + reads[j][a:]
        p = str(tmp_path / f"r{i}.{'fq' if i == 0 else 'fa'}")
        (datagen.write_fastq if i == 0 else datagen.write_fasta)(p, reads, prefix=f"f{i}_", newline="\r\n" if i != 2 else "\n")
        paths.append(p)
    return paths


def _expected_stdout(oracle, paths, k, lower, upper, percent, seed):
    """what jf_occurrences prints and exports, from hga_count_kmers on the ASCII bytes of the same record stream (the record reader runs
    on across files, so a file is the records the stream attributes to it) and the host functions"""
    import hga_b200
    rc, allr = oracle.load_reads(paths)
    assert rc == 0
    first = np.concatenate([[0], np.cumsum(allr["f_records"])]).astype(np.int64)
    lines = []
    if k == 0:
        distinct = lambda kk: len(hga_b200.capi.count_kmers(allr["seq"], allr["seq_off"], kk, min_count=1)[0])
        k = 11
        previous = distinct(k)
        lines.append(f"k=11 : {previous} kmers")
        while k < 33 and k + 2 <= 32:
            count = distinct(k + 2)
            lines.append(f"k={k + 2} : {count} kmers")
            if abs(count - previous) / ((count + previous) / 2.0) < 0.1:
                break
            k += 2
            previous = count
    per_file = [hga_b200.capi.count_kmers(allr["seq"], allr["seq_off"][first[f]:first[f + 1] + 1], k, min_count=2) for f in range(len(first) - 1)]
    assert all(len(c[0]) > 0 for c in per_file)
    km, total, largest, files = hga_b200.capi.sdk_merge(per_file)
    t, o, u = hga_b200.capi.sdk_specificity(total, largest)
    lines.append(f"# k = {k}: upper specificity, occurrences, unique k-mers")
    lines += [f"{float(a):.2f} {int(b)} {int(c)}" for a, b, c in zip(t, o, u)]
    lines.append("Enter lower and upper bounds for exported kmers as well as percentage")
    sel, n_sel, n_disc = hga_b200.capi.sdk_select(total, files, lower, upper, percent, seed)
    lines.append(f"{n_disc} out of {n_sel} exported kmers are discriminative")
    return "\n".join(lines) + "\n", [datagen.kmer_to_str(v, k) for v in km[sel]], n_sel


@pytest.mark.parametrize("k", [0, 15, 21])
def test_cli_jf_occurrences_on_messy_multi_file_input(oracle, tmp_path, k):
    paths = _messy_files(tmp_path)
    out = str(tmp_path / "sdk.txt")
    args = [EXE] + paths + (["-k", str(k)] if k else []) + ["-o", out, "--seed", "7"]
    r = subprocess.run(args, input="2 9 0.5\n", capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    want_stdout, want_kmers, n_sel = _expected_stdout(oracle, paths, k, 2, 9, 0.5, 7)
    assert r.stdout == want_stdout
    assert open(out).read() == "".join(s + "\n" for s in want_kmers) and n_sel > 0
