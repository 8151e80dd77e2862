"""CPU: the whole of hga_count_spectrum and hga_count_spectrum_packed (argument checks of csrc/hga_capi.cu + csrc/hga_count.cu with
count_spectrum_kernel, its launches, CUB calls and buffers) compiled for the host with the fake-CUDA harness of
test_kernel_bodies_on_host.py, against the spectrum of exact numpy counts and of hga_count_kmers(min_count = 1) from the same host
library. Runs longer than a thread's chunk of sorted positions take the galloping search; a range split down to one k-mer is added on
the host side. Argument errors are checked on the real library, which needs no GPU to refuse them. No GPU involved."""
import ctypes as C
import os
import re
import subprocess

import numpy as np
import pytest

from test_kernel_bodies_on_host import FAKE_CUDA, PRELUDE, _cut, _cut_macros
from test_packed_count_cpu import _KC, _p, _take, count_reads, hga, np_pack_folded, slice_runs  # noqa: F401  (hga: fixture)
from test_sdk_selection_cpu import exact_counts

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "hybrid-genome-assembler_b200", "csrc")
HGA_E_ARG = 2
CHUNK = int(re.search(r"#define COUNT_SPECTRUM_CHUNK (\d+)", open(os.path.join(CSRC, "hga_count.cu")).read()).group(1))


class _Spec(C.Structure):
    _fields_ = [("n_windows", C.c_uint64), ("n_distinct", C.c_uint64), ("max_count", C.c_uint64)]


SPECTRUM_ARGS = [C.c_int, C.c_int, C.c_char_p, C.c_void_p, C.c_uint64, C.c_uint32, C.c_void_p, C.c_void_p]
SPECTRUM_PACKED_ARGS = [C.c_int, C.c_int, C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint32, C.c_void_p, C.c_void_p]


@pytest.fixture(scope="module")
def host_spectrum(tmp_path_factory):
    """hga_count.cu as test_packed_count_cpu.py's host_count compiles it, plus both packed entries cut out of hga_capi.cu"""
    text = open(os.path.join(CSRC, "hga_count.cu")).read()
    capi = open(os.path.join(CSRC, "hga_capi.cu")).read()
    internal = open(os.path.join(CSRC, "hga_internal.cuh")).read()
    text = re.sub(r'#include\s+"hga_internal.cuh"\n', "", text)
    text = re.sub(r"#include\s+<cub/[^>]+>\n", "", text)
    text = re.sub(r"<<<[^;]*?>>>", "", text)
    devbuf = internal[internal.index("struct DevBuf {"):internal.index("struct PinBuf {")]
    entry = "\n".join([_cut(capi, r"^static int check_read_off"), _cut(capi, r"^static int check_exc_runs"),
                       'extern "C" {\n' + _cut(capi, r"^int hga_count_kmers_packed") + _cut(capi, r"^int hga_count_spectrum_packed") + '}\n'])
    d = tmp_path_factory.mktemp("host_spectrum")
    src, so = str(d / "spectrum_host.cpp"), str(d / "spectrum_host.so")
    open(src, "w").write(PRELUDE + FAKE_CUDA + _cut_macros(internal) + devbuf + text + entry)
    subprocess.run(["g++", "-std=c++17", "-O1", "-fPIC", "-shared", "-I", os.path.join(ROOT, "include"), "-o", so, src], check=True)
    lib = C.CDLL(so)
    lib.fake_last_error.restype = C.c_char_p
    lib.hga_count_spectrum.argtypes = SPECTRUM_ARGS
    lib.hga_count_spectrum_packed.argtypes = SPECTRUM_PACKED_ARGS
    lib.hga_count_kmers.argtypes = [C.c_int, C.c_int, C.c_char_p, C.c_void_p, C.c_uint64, C.c_uint32, C.c_void_p]
    return lib


def np_spectrum(counts, n_bins):
    """(hist, n_windows, n_distinct, max_count) of a list of counts"""
    c = np.asarray(counts, dtype=np.int64)
    hist = np.bincount(np.minimum(c, n_bins) - 1, minlength=n_bins).astype(np.uint64) if n_bins and len(c) else np.zeros(n_bins, np.uint64)
    return hist, int(c.sum()), len(c), int(c.max()) if len(c) else 0


def _join(reads):
    seq = "".join(reads).encode()
    off = np.zeros(len(reads) + 1, dtype=np.uint64)
    np.cumsum([len(r) for r in reads], out=off[1:])
    return seq, off


def _spectra(lib, reads, k, n_bins, first_base, rng):
    """the packed spectrum of the reads sliced first_base bases into a larger stream, and the ASCII spectrum of the same bytes"""
    seq, off = _join(reads)
    pre = np.frombuffer(b"ACGTacgN", dtype=np.uint8)[rng.integers(0, 8, first_base)].tobytes()
    packed, st, en = np_pack_folded(pre + seq + b"NNacgtTT")
    es, ee = slice_runs(st, en, first_base, first_base + len(seq))
    got = []
    for ascii_ in (False, True):
        hist = np.full(n_bins, 77, dtype=np.uint64)                 # the entries zero it
        sp = _Spec(5, 6, 7)
        if ascii_:
            rc = lib.hga_count_spectrum(0, k, seq, _p(off), len(reads), n_bins, _p(hist) if n_bins else None, C.byref(sp))
        else:
            rc = lib.hga_count_spectrum_packed(0, k, _p(packed), first_base, _p(off), len(reads), _p(es), _p(ee), len(es), n_bins, _p(hist) if n_bins else None,
                                               C.byref(sp))
        assert rc == 0, lib.fake_last_error()
        got.append((hist, sp.n_windows, sp.n_distinct, sp.max_count))
    return got, seq, off


def _same(a, b):
    assert np.array_equal(a[0], b[0]) and tuple(a[1:]) == tuple(b[1:]), (a, b)


def spectrum_reads(k, n_reads=120, long_run=600):
    """count_reads plus a poly-A read and a tandem repeat: runs of sorted keys far longer than a thread's chunk"""
    reads = count_reads(k, k, n_reads=n_reads, poly_a=long_run)
    reads.append("ACGGT" * (long_run // 5))
    return reads


@pytest.mark.parametrize("chunk", [None, "1024"])
@pytest.mark.parametrize("k", [1, 5, 11, 19, 31, 32])
def test_count_spectrum_on_host(host_spectrum, k, chunk):
    """one pass and forced key-range passes, slices starting 0..3 bases into a byte, n_bins 0..1000: hist, n_distinct, n_windows and
    max_count of both entries equal the spectrum of exact counts and of hga_count_kmers(min_count = 1)"""
    if chunk:
        os.environ["HGA_COUNT_CHUNK"] = chunk
    try:
        reads = spectrum_reads(k)
        seq, off = _join(reads)
        _, wc = exact_counts(seq, off, k, 1)
        assert (wc > 4 * CHUNK).sum() >= 2                               # runs that cross several chunks: the galloping path runs
        out = _KC()
        assert host_spectrum.hga_count_kmers(0, k, seq, _p(off), len(reads), 1, C.byref(out)) == 0, host_spectrum.fake_last_error()
        _, ac = _take(host_spectrum, out)
        for first_base in (0, 1, 2, 3, 149):
            for n_bins in (0, 1, 2, 5, 1000):
                got, _, _ = _spectra(host_spectrum, reads, k, n_bins, first_base, np.random.default_rng(first_base))
                want = np_spectrum(wc, n_bins)
                assert want[2] > 0 and want[1] == int(np.sum(wc))
                for g in got:
                    _same(g, want)
                    _same(g, np_spectrum(ac, n_bins))
    finally:
        os.environ.pop("HGA_COUNT_CHUNK", None)


def test_count_spectrum_on_host_splits_down_to_one_kmer(host_spectrum, capfd):
    """a budget of 256 keys and a poly-A read of 3000 bases: the range of A...A is split down to that single value, which the host adds
    to its bin with its exact count as max_count; the count and the spectrum cut the same ranges"""
    k = 19
    reads = count_reads(3, k, n_reads=30, poly_a=3000)
    seq, off = _join(reads)
    _, wc = exact_counts(seq, off, k, 1)
    assert wc.max() == 3000 - k + 1 > 256
    os.environ["HGA_COUNT_CHUNK"] = "256"
    os.environ["HGA_COUNT_STATS"] = "1"
    try:
        capfd.readouterr()
        out = _KC()
        assert host_spectrum.hga_count_kmers(0, k, seq, _p(off), len(reads), 1, C.byref(out)) == 0
        _take(host_spectrum, out)
        count_line = capfd.readouterr().err
        for n_bins in (0, 5, 2981, 2982, 2983, 5000):
            got, _, _ = _spectra(host_spectrum, reads, k, n_bins, 3, np.random.default_rng(3))
            lines = capfd.readouterr().err
            for g in got:
                _same(g, np_spectrum(wc, n_bins))
                assert g[3] == 3000 - k + 1
    finally:
        os.environ.pop("HGA_COUNT_CHUNK", None)
        os.environ.pop("HGA_COUNT_STATS", None)
    m = re.search(r"hga_count_kmers: (\d+) key-range passes \((\d+) ranges split\)", count_line)
    assert m and int(m.group(2)) > 0, count_line
    tail = count_line.split(": ", 1)[1]
    assert lines == f"hga_count_spectrum_packed: {tail}hga_count_spectrum: {tail}", (lines, count_line)


def test_count_spectrum_argument_errors(hga):
    """refused before any device is needed: HGA_E_ARG and a message, *out and hist zeroed"""
    lib = hga.load_library()
    lib.hga_count_spectrum.argtypes = SPECTRUM_ARGS
    lib.hga_count_spectrum_packed.argtypes = SPECTRUM_PACKED_ARGS
    packed = np.zeros(64, dtype=np.uint8)

    def packed_call(k, off, st, en, n_bins=3, hist=True, out=True):
        off = np.asarray(off, dtype=np.uint64); st = np.asarray(st, dtype=np.uint64); en = np.asarray(en, dtype=np.uint64)
        h = np.full(max(n_bins, 1), 9, dtype=np.uint64)
        sp = _Spec(1, 2, 3)
        rc = lib.hga_count_spectrum_packed(0, k, _p(packed), 0, _p(off), len(off) - 1, _p(st), _p(en), len(st), n_bins, _p(h) if hist else None,
                                           C.byref(sp) if out else None)
        if hist:
            assert not h[:n_bins].any()
        if out:
            assert (sp.n_windows, sp.n_distinct, sp.max_count) == (0, 0, 0)
        return rc, lib.hga_last_error().decode()

    def ascii_call(k, n_bins=3, hist=True, out=True):
        off = np.array([0, 8], dtype=np.uint64)
        h = np.full(max(n_bins, 1), 9, dtype=np.uint64)
        sp = _Spec(1, 2, 3)
        rc = lib.hga_count_spectrum(0, k, b"ACGTACGT", _p(off), 1, n_bins, _p(h) if hist else None, C.byref(sp) if out else None)
        if hist:
            assert not h[:n_bins].any()
        if out:
            assert (sp.n_windows, sp.n_distinct, sp.max_count) == (0, 0, 0)
        return rc, lib.hga_last_error().decode()

    for k in (0, 33):
        assert packed_call(k, [0, 100], [], [])[0] == HGA_E_ARG and "Kmer size" in packed_call(k, [0, 100], [], [])[1]
        rc, msg = ascii_call(k)
        assert rc == HGA_E_ARG and "Kmer size" in msg
    rc, msg = packed_call(19, [0, 100], [], [], out=False)
    assert rc == HGA_E_ARG and "hga_count_spectrum_packed: NULL argument" in msg
    rc, msg = packed_call(19, [0, 100], [], [], n_bins=4, hist=False)
    assert rc == HGA_E_ARG and "hga_count_spectrum_packed: NULL argument" in msg
    rc, msg = ascii_call(19, out=False)
    assert rc == HGA_E_ARG and "hga_count_spectrum: NULL argument" in msg
    rc, msg = ascii_call(19, n_bins=4, hist=False)
    assert rc == HGA_E_ARG and "hga_count_spectrum: NULL argument" in msg
    rc, msg = packed_call(19, [5, 100], [], [])
    assert rc == HGA_E_ARG and "hga_count_spectrum_packed: read_off[0] must be 0" in msg
    rc, msg = packed_call(19, [0, 100, 50], [], [])
    assert rc == HGA_E_ARG and "hga_count_spectrum_packed: read_off is not monotone" in msg
    for st, en in (([10, 5], [12, 7]), ([10, 11], [12, 14]), ([90], [101]), ([10], [10])):
        rc, msg = packed_call(19, [0, 100], st, en)
        assert rc == HGA_E_ARG and "hga_count_spectrum_packed: exception run" in msg, (st, en, msg)
