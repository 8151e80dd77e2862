"""GPU: the SDK selection on the device (hga_sdk_count_packed / _specificity / _range) against the per-file hga_count_kmers_packed lists
pushed through the host functions (hga_host_sdk_merge / _specificity / _select), jf_occurrences on several files against the same
host path, and the 32-bit limit of a total merged over two files."""
import os
import re
import subprocess
import time

import numpy as np
import pytest

import datagen

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HGA_E_OVERFLOW = 5


def _clip(st, en, b0, b1):
    m = (en > b0) & (st < b1)
    return np.maximum(st[m], b0) - b0, np.minimum(en[m], b1) - b0


def _reference(hga_b200, packed, off, st, en, first, k, min_count, first_base):
    """per-file hga_count_kmers_packed (each file a slice counted in place) merged by hga_host_sdk_merge; st / en are the runs of the
    whole packed stream, the read set starts first_base bases into it"""
    per_file = []
    for f in range(len(first) - 1):
        r0, r1 = int(first[f]), int(first[f + 1])
        b0, b1 = int(off[r0]), int(off[r1])
        es, ee = _clip(st, en, np.uint64(first_base + b0), np.uint64(first_base + b1))
        per_file.append(hga_b200.capi.count_kmers_packed(packed, off[r0:r1 + 1] - off[r0], es, ee, k, min_count=min_count, first_base=first_base + b0))
    return hga_b200.capi.sdk_merge(per_file)


def _same_table(hga_b200, t, want, thresholds=(70, 85, 90, 95, 99, 100, 100.01)):
    got = t.range()
    assert t.n == len(want[0])
    for g, w in zip(got, want):
        assert np.array_equal(g, w)
    for g, w in zip(t.specificity(thresholds), hga_b200.capi.sdk_specificity(want[1], want[2], thresholds)):
        assert np.array_equal(g, w)
    km, total, _, files = want
    for lo, hi in ((2, 2), (3, 40), (40, 3), (0, 0xFFFFFFFF)):
        r = t.range(lo, hi)
        m = (total >= lo) & (total <= hi)
        assert np.array_equal(r[0], km[m]) and np.array_equal(r[3], files[m])
        for percent, seed in ((1.0, 0), (0.3, 5)):
            s_full = hga_b200.capi.sdk_select(total, files, lo, hi, percent, seed)
            s_rng = hga_b200.capi.sdk_select(r[1], r[3], lo, hi, percent, seed)
            assert np.array_equal(km[s_full[0]], r[0][s_rng[0]]) and s_full[1:] == s_rng[1:]


def test_sdk_on_the_device_equals_the_host_merge(capfd, monkeypatch):
    """about 40 Mbases in 4 files (N runs, lowercase stretches, CR bytes, an empty file), a slice 3 bases into a byte, min_count 1 and
    2; one pass, and key-range passes with a budget of 2^21 keys where the poly-A k-mer's range is split down to that single value"""
    import hga_b200
    rng = np.random.default_rng(91)
    g = datagen.random_genome(400000, 911)
    g[1000:41000] = 0                                                         # 40 kb of poly-A: one k-mer far beyond a budget of 2^21
    reads = [datagen.to_ascii(r) for r in datagen.sample_reads(g, 4000, 10000, 912, error_rate=0.02, length_sigma=0.3, max_len=60000)]
    for j in range(0, len(reads), 7):
        a = int(rng.integers(0, max(len(reads[j]) - 60, 1)))
        reads[j] = reads[j][:a] + reads[j][a:a + 50].lower() + "N" * int(rng.integers(1, 9)) + reads[j][a + 50:]
    for j in range(3, len(reads), 11):
        reads[j] = reads[j] + "\r"
    cuts = [0, 1300, 2400, 2400, len(reads)]                                  # file 2 is empty
    seq = "".join(reads).encode()
    off = np.zeros(len(reads) + 1, dtype=np.uint64)
    np.cumsum([len(r) for r in reads], out=off[1:])
    assert off[-1] > 35_000_000
    first_base = 4 * 1001 + 3
    packed, st, en = hga_b200.pack_bases((b"ACGTN" * 802)[:first_base] + seq + b"ACGT", fold_case=True)
    es, ee = _clip(st, en, np.uint64(first_base), np.uint64(first_base + len(seq)))
    first = np.array(cuts, dtype=np.uint64)
    k = 19
    monkeypatch.setenv("HGA_COUNT_STATS", "1")
    for chunk in (None, str(1 << 21)):
        if chunk:
            monkeypatch.setenv("HGA_COUNT_CHUNK", chunk)
        for min_count in (2, 1):
            want = _reference(hga_b200, packed, off, st, en, first, k, min_count, first_base)
            t0 = time.perf_counter()
            with hga_b200.capi.sdk_count_packed(packed, off, es, ee, k, first, min_count=min_count, first_base=first_base) as t:
                t1 = time.perf_counter()
                assert want[0][0] == 0 and want[3][0] == 3 and want[1][0] > (1 << 21)
                _same_table(hga_b200, t, want)
            if chunk:
                passes = [int(v) for v in re.findall(r"hga_sdk_count_packed: (\d+) key-range passes", capfd.readouterr().err)]
                assert passes and passes[-1] > 10
            print(f"\nsdk count, {int(off[-1])} bases in 4 files, chunk {chunk}, min_count {min_count}: {t1 - t0:.2f} s, {t.n} merged k-mers")


def test_cli_jf_occurrences_on_several_files(oracle, tmp_path):
    """jf_occurrences on 3 files with percent 1.0 and 0.3 (and --seed): the table, the summary line and the exported k-mers equal
    those of exact per-file counts pushed through hga_host_sdk_merge / _specificity / _select"""
    import hga_b200
    from test_sdk_selection_cpu import exact_counts
    exe = os.path.join(ROOT, "hybrid-genome-assembler_b200", "jf_occurrences")
    k = 17
    paths, _ = datagen.make_polyploid_case(str(tmp_path), genome_size=8000, divergence=0.03, k=k, read_len=400, coverage=8, seed=12, n_haplotypes=3,
                                           error_rate=0.01)
    per_file = []
    for p in paths:
        rc, rd = oracle.load_reads([p])
        per_file.append(exact_counts(rd["seq"], rd["seq_off"], k))
    km, total, largest, files = hga_b200.capi.sdk_merge(per_file)
    t, o, u = hga_b200.capi.sdk_specificity(total, largest)
    for percent, seed in ((1.0, 0), (0.3, 7)):
        out = str(tmp_path / f"sdk_{percent}.txt")
        r = subprocess.run([exe] + paths + ["-k", str(k), "-o", out, "--seed", str(seed)], input=f"3 20 {percent}\n", capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
        sel, n_sel, n_disc = hga_b200.capi.sdk_select(total, files, 3, 20, percent, seed)
        assert open(out).read() == "".join(datagen.kmer_to_str(v, k) + "\n" for v in km[sel]) and n_sel > 0
        want_stdout = (f"# k = {k}: upper specificity, occurrences, unique k-mers\n" + "".join(f"{a:.2f} {b} {c}\n" for a, b, c in zip(t, o, u))
                       + "Enter lower and upper bounds for exported kmers as well as percentage\n" + f"{n_disc} out of {n_sel} exported kmers are discriminative\n")
        assert r.stdout == want_stdout


def _poly_a_files(k, windows):
    """all-zero packed bases (poly-A): one file per entry of `windows`, each of reads shorter than 2^30 holding that many windows"""
    per = (1 << 30) - 1
    lens, first = [], [0]
    for n in windows:
        left = n
        while left > 0:
            w = min(left, per - k + 1)
            lens.append(w + k - 1)
            left -= w
        first.append(len(lens))
    off = np.zeros(len(lens) + 1, dtype=np.uint64)
    np.cumsum(lens, out=off[1:])
    return np.zeros((int(off[-1]) + 3) // 4, dtype=np.uint8), off, np.array(first, dtype=np.uint64)


def test_sdk_total_past_32_bits_poly_a():
    """poly-A in two files: totals of exactly 2^32 - 1 are accepted, a total of 2^32 fails with HGA_E_OVERFLOW (as hga_host_sdk_merge
    does) and leaves no handle"""
    import hga_b200
    k = 25
    none = np.zeros(0, dtype=np.uint64)
    packed, off, first = _poly_a_files(k, [1 << 31, (1 << 31) - 1])
    t0 = time.perf_counter()
    with hga_b200.capi.sdk_count_packed(packed, off, none, none, k, first, min_count=1) as t:
        got = t.range()
    t1 = time.perf_counter()
    assert got[0].tolist() == [0] and got[1].tolist() == [(1 << 32) - 1] and got[2].tolist() == [1 << 31] and got[3].tolist() == [2]
    packed, off, first = _poly_a_files(k, [1 << 31, 1 << 31])
    with pytest.raises(hga_b200.HgaError) as e:
        hga_b200.capi.sdk_count_packed(packed, off, none, none, k, first, min_count=1)
    t2 = time.perf_counter()
    assert e.value.code == HGA_E_OVERFLOW and "total count overflows 32 bits" in str(e.value), str(e.value)
    print(f"\npoly-A in 2 files, k = {k}: total 2^32 - 1 in {t1 - t0:.1f} s, refused total 2^32 in {t2 - t1:.1f} s")
