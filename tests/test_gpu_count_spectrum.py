"""GPU: the k-mer spectrum (hga_count_spectrum on ASCII bytes, hga_count_spectrum_packed on the case-folded packing) equals the spectrum
of hga_count_kmers(min_count = 1) and of exact numpy counts: hist, n_windows, n_distinct and max_count, for every k of the sweep and
more, n_bins from 0 to past the bins a CTA keeps in shared memory, N runs, lowercase and CR bytes, empty and short reads, slices
starting inside a byte, and tens of Mbases with k-mers seen more than 65 536 times in one pass and in forced key-range passes (which cut
the same ranges as the count). jf_occurrences, whose k sweep now reads the spectrum, prints what the counts give."""
import os
import re
import subprocess

import numpy as np
import pytest

import datagen
from test_count_spectrum_cpu import np_spectrum, spectrum_reads
from test_gpu_packed_count import EXE, _expected_stdout, _join, _messy_files, _packed_slice
from test_sdk_selection_cpu import exact_counts

pytestmark = pytest.mark.gpu

CSRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "hybrid-genome-assembler_b200", "csrc")
SHARED_BINS = int(re.search(r"#define COUNT_SPECTRUM_SHARED_BINS (\d+)", open(os.path.join(CSRC, "hga_count.cu")).read()).group(1))


def _spectra(seq, off, k, n_bins, first_base=0, seed=0):
    """(packed spectrum of seq sliced first_base bases into a larger stream, ASCII spectrum of seq)"""
    import hga_b200
    packed, es, ee = _packed_slice(seq, first_base, np.random.default_rng(seed))
    return (hga_b200.capi.count_spectrum_packed(packed, off, es, ee, k, n_bins=n_bins, first_base=first_base),
            hga_b200.capi.count_spectrum(seq, off, k, n_bins=n_bins))


def _same(a, b):
    assert np.array_equal(a[0], b[0]) and tuple(int(v) for v in a[1:]) == tuple(int(v) for v in b[1:]), (a[1:], b[1:])


@pytest.mark.parametrize("k", [1, 2, 5, 11, 15, 16, 17, 19, 21, 31, 32])
def test_spectrum_equals_count_and_exact(k):
    import hga_b200
    reads = spectrum_reads(k, n_reads=160)
    reads[20] = reads[20][:33] + "N" * 31 + reads[20][64:]
    reads[21] = "acgt" * 8 + "N" + reads[21] + "\r"
    seq, off = _join(reads)
    _, wc = exact_counts(seq, off, k, 1)
    _, cc = hga_b200.capi.count_kmers(seq, off, k, min_count=1)
    for i, n_bins in enumerate((0, 1, 3, 10001)):
        want = np_spectrum(wc, n_bins)
        _same(want, np_spectrum(cc, n_bins))
        for got in _spectra(seq, off, k, n_bins, first_base=(k + i) % 4 + 4 * i, seed=k):
            _same(got, want)


def test_empty_short_and_exception_only_reads():
    import hga_b200
    for k in (1, 4, 19, 32):
        reads = ["", "ACG", "", "N" * 40, "acgtn" * 9, "A" * (k - 1), "\r", "T" * k, "ACGT" * 10 + "\r", "", "tttttttttttttttttttttttttttttttttt"]
        seq, off = _join(reads)
        for first_base in (0, 1, 2, 3):
            for got in _spectra(seq, off, k, 7, first_base):
                _same(got, np_spectrum(exact_counts(seq, off, k, 1)[1], 7))
    # no reads / only empty reads / no window at all: zeros
    zero = (np.zeros(5, np.uint64), 0, 0, 0)
    _same(hga_b200.capi.count_spectrum_packed(np.zeros(4, np.uint8), np.zeros(1, np.uint64), [], [], 5, n_bins=5), zero)
    _same(hga_b200.capi.count_spectrum_packed(np.zeros(4, np.uint8), np.zeros(4, np.uint64), [], [], 5, n_bins=5), zero)
    _same(hga_b200.capi.count_spectrum(b"", np.zeros(4, np.uint64), 5, n_bins=5), zero)
    _same(hga_b200.capi.count_spectrum(b"ACGN", np.array([0, 4], np.uint64), 5, n_bins=5), zero)


def _large_input():
    """~40 Mbases with N runs and lowercase stretches, plus reads that make k-mers seen far more often than a CTA's chunk of sorted
    positions: a 70 kbase poly-A read (> 65 536 windows of one k-mer), a tandem repeat, and 6000 copies of one 200-base read"""
    rng = np.random.default_rng(91)
    g = datagen.random_genome(400000, 701)
    reads = [datagen.to_ascii(r) for r in datagen.sample_reads(g, 4000, 10000, 702, error_rate=0.02, length_sigma=0.3, max_len=60000)]
    reads += ["A" * 70000, "ACGGT" * 20000] + [reads[7][:200]] * 6000
    seq = bytearray("".join(reads).encode())
    off = np.zeros(len(reads) + 1, dtype=np.uint64)
    np.cumsum([len(r) for r in reads], out=off[1:])
    assert off[-1] > 30_000_000
    for a in rng.integers(0, int(off[4000]) - 3000, 400):
        seq[a:a + 2000] = bytes(seq[a:a + 2000]).lower()
    for a in rng.integers(0, int(off[4000]) - 300, 400):
        L = int(rng.integers(1, 300))
        seq[a:a + L] = b"N" * L
    return bytes(seq), off


def test_large_input_one_pass_and_key_range_passes(capfd):
    import hga_b200
    seq, off = _large_input()
    k, n_bins, first_base = 19, 10001, 3
    assert n_bins > SHARED_BINS
    packed, es, ee = _packed_slice(seq, first_base, np.random.default_rng(5))
    _, cc = hga_b200.capi.count_kmers(seq, off, k, min_count=1)
    want = np_spectrum(cc, n_bins)
    assert want[3] > 65536 and want[0][SHARED_BINS:n_bins - 1].sum() > 0 and want[0][n_bins - 1] > 0 and want[2] > 10_000_000
    _same(hga_b200.capi.count_spectrum_packed(packed, off, es, ee, k, n_bins=n_bins, first_base=first_base), want)
    _same(hga_b200.capi.count_spectrum(seq, off, k, n_bins=n_bins), want)
    os.environ["HGA_COUNT_CHUNK"] = str(1 << 21)
    os.environ["HGA_COUNT_STATS"] = "1"
    try:
        capfd.readouterr()
        hga_b200.capi.count_kmers_packed(packed, off, es, ee, k, min_count=1, first_base=first_base)
        count_line = capfd.readouterr().err
        got = hga_b200.capi.count_spectrum_packed(packed, off, es, ee, k, n_bins=n_bins, first_base=first_base)
        spectrum_line = capfd.readouterr().err
        got_ascii = hga_b200.capi.count_spectrum(seq, off, k, n_bins=n_bins)
    finally:
        del os.environ["HGA_COUNT_CHUNK"], os.environ["HGA_COUNT_STATS"]
    _same(got, want)
    _same(got_ascii, want)
    m = re.fullmatch(r"hga_count_kmers_packed: (\d+) key-range passes \(\d+ ranges split\)\n", count_line)
    assert m and int(m.group(1)) > 10, count_line
    assert spectrum_line == count_line.replace("hga_count_kmers_packed:", "hga_count_spectrum_packed:")


def test_cli_k_sweep_under_key_range_passes(oracle, tmp_path):
    """jf_occurrences without -k: the sweep's distinct counts come from the spectrum, under forced key-range passes"""
    paths = _messy_files(tmp_path)
    out = str(tmp_path / "sdk.txt")
    r = subprocess.run([EXE] + paths + ["-o", out, "--seed", "7"], input="2 9 0.5\n", capture_output=True, text=True,
                       env=dict(os.environ, HGA_COUNT_CHUNK="4096"))
    assert r.returncode == 0, r.stderr
    want_stdout, want_kmers, n_sel = _expected_stdout(oracle, paths, 0, 2, 9, 0.5, 7)
    assert r.stdout == want_stdout
    assert open(out).read() == "".join(s + "\n" for s in want_kmers) and n_sel > 0
