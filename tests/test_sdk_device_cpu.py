"""CPU: the whole of the device SDK selection (hga_sdk_count_packed / _specificity / _range of csrc/hga_count.cu, the argument checks and
entry cut out of csrc/hga_capi.cu) compiled for the host with the fake-CUDA harness of test_kernel_bodies_on_host.py, against the
per-file hga_count_kmers_packed of the same emulated build pushed through the real hga_host_sdk_merge / _specificity / _select of
libhga_b200.so, and against exact numpy counts per file. Run with HGA_EMU_ASAN=1 (and libasan preloaded) every emulated device
buffer is an exact-size malloc block, so AddressSanitizer sees any store past one. Test infrastructure only: the product never runs
this way."""
import ctypes as C
import os
import re
import subprocess

import numpy as np
import pytest

from test_kernel_bodies_on_host import FAKE_CUDA, PRELUDE, _cut, _cut_macros
from test_packed_count_cpu import count_reads, np_pack_folded, slice_runs
from test_sdk_selection_cpu import exact_counts

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "hybrid-genome-assembler_b200", "csrc")
HGA_E_ARG, HGA_E_OVERFLOW = 2, 5
CLI_THRESHOLDS = (70, 85, 90, 95, 99, 100, 100.01)
P = C.c_void_p


@pytest.fixture(scope="module")
def hga():
    import importlib
    importlib.import_module("hybrid-genome-assembler_b200.build").build()
    import hga_b200
    return hga_b200


class _KC(C.Structure):
    _fields_ = [("n", C.c_uint64), ("kmer", C.POINTER(C.c_uint64)), ("count", C.POINTER(C.c_uint32))]


class _SR(C.Structure):
    _fields_ = [("n", C.c_uint64), ("kmer", C.POINTER(C.c_uint64)), ("total", C.POINTER(C.c_uint32)), ("max", C.POINTER(C.c_uint32)),
                ("files", C.POINTER(C.c_uint32))]


def _set_types(lib):
    lib.hga_count_kmers_packed.argtypes = [C.c_int, C.c_int, P, C.c_uint64, P, C.c_uint64, P, P, C.c_uint64, C.c_uint32, P]
    lib.hga_sdk_count_packed.argtypes = [C.c_int, C.c_int, P, C.c_uint64, P, C.c_uint64, P, P, C.c_uint64, C.c_int, P, C.c_uint32, C.POINTER(C.c_void_p)]
    lib.hga_sdk_size.argtypes = [P, C.POINTER(C.c_uint64)]
    lib.hga_sdk_specificity.argtypes = [P, P, C.c_int, P, P, P, C.c_uint64, C.POINTER(C.c_uint64)]
    lib.hga_sdk_range.argtypes = [P, C.c_uint32, C.c_uint32, C.POINTER(_SR)]
    lib.hga_free_sdk_range.argtypes = [C.POINTER(_SR)]
    lib.hga_free_sdk_range.restype = None
    lib.hga_sdk_free.argtypes = [P]
    lib.hga_sdk_free.restype = None
    return lib


@pytest.fixture(scope="module")
def emu(tmp_path_factory):
    text = open(os.path.join(CSRC, "hga_count.cu")).read()
    capi = open(os.path.join(CSRC, "hga_capi.cu")).read()
    internal = open(os.path.join(CSRC, "hga_internal.cuh")).read()
    text = re.sub(r'#include\s+"hga_internal.cuh"\n', "", text)
    text = re.sub(r"#include\s+<cub/[^>]+>\n", "", text)
    text = re.sub(r"<<<[^;]*?>>>", "", text)
    devbuf = internal[internal.index("struct DevBuf {"):internal.index("struct PinBuf {")]
    asan = bool(os.environ.get("HGA_EMU_ASAN"))
    if asan:
        devbuf = devbuf.replace("size_t want = bytes + (bytes >> 4) + 256;", "size_t want = bytes;")
    entry = "\n".join([_cut(capi, r"^static int check_read_off"), _cut(capi, r"^static int check_exc_runs"),
                       'extern "C" {\n' + _cut(capi, r"^int hga_count_kmers_packed") + _cut(capi, r"^int hga_sdk_count_packed") + '}\n'])
    d = tmp_path_factory.mktemp("host_sdk")
    src, so = str(d / "sdk_host.cpp"), str(d / "sdk_host.so")
    open(src, "w").write(PRELUDE + FAKE_CUDA + _cut_macros(internal) + devbuf + text + entry)
    san = ["-fsanitize=address", "-fno-omit-frame-pointer", "-g"] if asan else []
    subprocess.run(["g++", "-std=c++17", "-O1", "-ffp-contract=off", "-fPIC", "-shared"] + san + ["-I", os.path.join(ROOT, "include"), "-o", so, src],
                   check=True)
    lib = _set_types(C.CDLL(so))
    lib.fake_last_error.restype = C.c_char_p
    return lib


def _p(a):
    return a.ctypes.data_as(P)


def _arr(ptr, n, dt):
    return np.ctypeslib.as_array(ptr, shape=(int(n),)).copy() if n else np.zeros(0, dt)


class Input:
    """reads cut into files, as one packed stream: the read set starts first_base bases into it"""

    def __init__(self, files, first_base, rng):
        self.files = files
        reads = [r for f in files for r in f]
        self.seq = "".join(reads).encode()
        self.off = np.zeros(len(reads) + 1, dtype=np.uint64)
        np.cumsum([len(r) for r in reads], out=self.off[1:])
        self.first = np.zeros(len(files) + 1, dtype=np.uint64)
        np.cumsum([len(f) for f in files], out=self.first[1:])
        pre = np.frombuffer(b"ACGTacgN", dtype=np.uint8)[rng.integers(0, 8, first_base)].tobytes()
        self.packed, st, en = np_pack_folded(pre + self.seq + b"NNacgtTT")
        self.first_base = first_base
        self.st, self.en = st, en
        self.es, self.ee = slice_runs(st, en, first_base, first_base + len(self.seq))

    def file_slice(self, f):
        r0, r1 = int(self.first[f]), int(self.first[f + 1])
        b0, b1 = int(self.off[r0]), int(self.off[r1])
        es, ee = slice_runs(self.st, self.en, self.first_base + b0, self.first_base + b1)
        return self.first_base + b0, (self.off[r0:r1 + 1] - np.uint64(b0)).astype(np.uint64), es, ee, r1 - r0


def per_file_counts(lib, inp, k, min_count):
    """emulated hga_count_kmers_packed of every file's slice, checked against exact numpy counts"""
    out = []
    for f in range(len(inp.files)):
        fb, off, es, ee, nr = inp.file_slice(f)
        kc = _KC()
        assert lib.hga_count_kmers_packed(0, k, _p(inp.packed), fb, _p(off), nr, _p(es), _p(ee), len(es), min_count, C.byref(kc)) == 0, lib.fake_last_error()
        km, ct = _arr(kc.kmer, kc.n, np.uint64), _arr(kc.count, kc.n, np.uint32)
        wk, wc = exact_counts("".join(inp.files[f]).encode(), off, k, min_count)
        assert np.array_equal(km, wk) and np.array_equal(ct, wc)
        out.append((km, ct))
    return out


class Sdk:
    def __init__(self, lib, inp, k, min_count):
        self.lib = lib
        h = C.c_void_p()
        self.rc = lib.hga_sdk_count_packed(0, k, _p(inp.packed), inp.first_base, _p(inp.off), len(inp.off) - 1, _p(inp.es), _p(inp.ee), len(inp.es),
                                           len(inp.files), _p(inp.first), min_count, C.byref(h))
        self.h = h.value
        if self.rc == 0:
            n = C.c_uint64()
            assert lib.hga_sdk_size(self.h, C.byref(n)) == 0
            self.n = n.value
        else:
            assert self.h is None

    def range(self, lower=0, upper=0xFFFFFFFF):
        r = _SR()
        assert self.lib.hga_sdk_range(self.h, lower, upper, C.byref(r)) == 0, self.lib.fake_last_error()
        got = (_arr(r.kmer, r.n, np.uint64), _arr(r.total, r.n, np.uint32), _arr(r.max, r.n, np.uint32), _arr(r.files, r.n, np.uint32))
        self.lib.hga_free_sdk_range(C.byref(r))
        return got

    def specificity(self, thresholds, capacity=None):
        thr = np.ascontiguousarray(thresholds, dtype=np.float64)
        n = C.c_uint64()
        rc = self.lib.hga_sdk_specificity(self.h, _p(thr), len(thr), None, None, None, 0, C.byref(n))
        if rc:
            return rc, self.lib.fake_last_error().decode()
        need = n.value
        cap = need if capacity is None else capacity
        ot = np.zeros(max(cap, 1)); oo = np.zeros(max(cap, 1), np.uint32); ou = np.zeros(max(cap, 1), np.uint64)
        assert self.lib.hga_sdk_specificity(self.h, _p(thr), len(thr), _p(ot), _p(oo), _p(ou), cap, C.byref(n)) == 0
        assert n.value == need
        m = min(cap, need)
        return 0, (ot[:m], oo[:m], ou[:m])

    def free(self):
        self.lib.hga_sdk_free(self.h)


def _split(reads, n_files, k):
    """n_files files; with 3 or more one of them is empty, with 5 one holds only a read of k bases (no k-mer seen twice)"""
    if n_files == 1:
        return [reads]
    cuts = np.linspace(0, len(reads), n_files + 1).astype(int)
    files = [reads[cuts[i]:cuts[i + 1]] for i in range(n_files)]
    if n_files >= 3:
        files[1] = []
    if n_files >= 5:
        files[3] = ["ACGTTGCAGGTCAACGTATCGGATCCTAGCTAGCATG"[:k]]
    return files


def _check_all(hga, lib, inp, k, min_count):
    per_file = per_file_counts(lib, inp, k, min_count)
    want = hga.capi.sdk_merge(per_file)
    s = Sdk(lib, inp, k, min_count)
    assert s.rc == 0, lib.fake_last_error()
    try:
        got = s.range()
        assert s.n == len(want[0])
        for g, w in zip(got, want):
            assert np.array_equal(g, w)
        rc, rows = s.specificity(CLI_THRESHOLDS)
        assert rc == 0
        for g, w in zip(rows, hga.capi.sdk_specificity(want[1], want[2], CLI_THRESHOLDS)):
            assert np.array_equal(g, w)
    finally:
        s.free()
    return want


@pytest.mark.parametrize("chunk", [None, "1024"])
@pytest.mark.parametrize("k", [1, 5, 11, 19, 31, 32])
def test_sdk_count_matches_per_file_counts_and_host_merge(hga, emu, k, chunk):
    """1 / 2 / 3 / 5 files (an empty one, one without a k-mer reaching min_count), slices 0..3 bases into a byte, min_count 1..3, one
    pass and forced key-range passes: the merged table is hga_host_sdk_merge of the per-file counts, and so is the specificity table"""
    if chunk:
        os.environ["HGA_COUNT_CHUNK"] = chunk
    try:
        for i, n_files in enumerate((1, 2, 3, 5)):
            reads = count_reads(k + n_files, k)
            for min_count in (1, 2, 3):
                first_base = (i + min_count) % 4 + (4 * 29 if min_count == 3 else 0)
                _check_all(hga, emu, Input(_split(reads, n_files, k), first_base, np.random.default_rng(first_base)), k, min_count)
    finally:
        os.environ.pop("HGA_COUNT_CHUNK", None)


def test_sdk_split_down_to_one_kmer_across_files(hga, emu):
    """a budget of 256 keys; A...A is in two files far beyond the budget and once (below min_count) in a third: its range is split down
    to the single value, whose merged entry comes from the per-file cursor snapshots"""
    k = 19
    reads = count_reads(3, k, n_reads=30)
    files = [reads[:10] + ["A" * 3000], reads[10:20] + ["A" * k], [], reads[20:] + ["A" * 2000, "a" * 500]]
    os.environ["HGA_COUNT_CHUNK"] = "256"
    try:
        for min_count in (2, 1):
            want = _check_all(hga, emu, Input(files, 3, np.random.default_rng(3)), k, min_count)
            assert want[0][0] == 0 and want[1][0] == 2982 + 1982 + 482 + (1 if min_count == 1 else 0) and want[3][0] == (2 if min_count == 2 else 3)
    finally:
        os.environ.pop("HGA_COUNT_CHUNK", None)


@pytest.fixture(scope="module")
def table(hga, emu):
    """three files and a poly-A total past 2^16 (the compacted tail of the specificity bins)"""
    k = 11
    reads = count_reads(7, k)
    inp = Input([reads[:50] + ["A" * 40000], reads[50:90], reads[90:] + ["A" * 30000]], 2, np.random.default_rng(2))
    want = hga.capi.sdk_merge(per_file_counts(emu, inp, k, 2))
    assert want[1].max() > 65536
    s = Sdk(emu, inp, k, 2)
    assert s.rc == 0
    yield s, want
    s.free()


def test_sdk_specificity_thresholds_and_capacity(hga, table):
    s, (km, total, largest, files) = table
    many = list(np.linspace(30, 100.5, 70))                                  # more than 64 bins: a smaller dense part, the rest in the tail
    for thr in (CLI_THRESHOLDS, (99, 70, 100.01, 70, 85, 99), (100.01,), many):
        rc, rows = s.specificity(thr)
        assert rc == 0
        want = hga.capi.sdk_specificity(total, largest, thr)
        for g, w in zip(rows, want):
            assert np.array_equal(g, w)
    full = s.specificity(CLI_THRESHOLDS)[1]
    for cap in (0, 1, 5):
        rc, rows = s.specificity(CLI_THRESHOLDS, capacity=cap)
        assert rc == 0 and all(np.array_equal(g, w[:cap]) for g, w in zip(rows, full))
    for thr in ((10, 20), (60, 99.5)):                                       # the first k-mer without a bin is named by its specificity
        rc, msg = s.specificity(thr)
        with pytest.raises(Exception) as e:
            hga.capi.sdk_specificity(total, largest, thr)
        want = re.search(r"no threshold above [0-9.]+", str(e.value)).group(0)
        assert rc == HGA_E_ARG and want in msg, (msg, want)


def test_sdk_range_and_selection(hga, table):
    s, (km, total, largest, files) = table
    for lo, hi in ((0, 0xFFFFFFFF), (2, 2), (3, 7), (7, 3), (int(total.max()), int(total.max())), (5, 0xFFFFFFFF)):
        got = s.range(lo, hi)
        m = (total >= lo) & (total <= hi)
        for g, w in zip(got, (km[m], total[m], largest[m], files[m])):
            assert np.array_equal(g, w)
        for percent, seed in ((1.0, 0), (0.3, 11), (0.3, 12)):
            sel_full, n_full, d_full = hga.capi.sdk_select(total, files, lo, hi, percent, seed)
            sel_r, n_r, d_r = hga.capi.sdk_select(got[1], got[3], lo, hi, percent, seed)
            assert np.array_equal(km[sel_full], got[0][sel_r]) and (n_full, d_full) == (n_r, d_r)


def test_sdk_empty_inputs(emu):
    """no reads, or reads without a window: an empty table, an empty specificity table and empty ranges"""
    for files in ([[]], [[], []], [["AC"], ["G"]]):
        s = Sdk(emu, Input(files, 1, np.random.default_rng(0)), 5, 2)
        assert s.rc == 0 and s.n == 0
        rc, rows = s.specificity(CLI_THRESHOLDS)
        assert rc == 0 and all(a.size == 0 for a in rows)
        assert all(a.size == 0 for a in s.range())
        s.free()


def test_sdk_count_argument_errors(hga):
    """checked before any device work, against the real library: HGA_E_ARG, a message and no handle"""
    lib = _set_types(hga.capi.load_library())
    packed = np.zeros(64, dtype=np.uint8)

    def call(k=19, off=(0, 50, 100), first=(0, 1, 2), st=(), en=(), n_files=None, first_null=False):
        off = np.asarray(off, dtype=np.uint64); first = np.asarray(first, dtype=np.uint64)
        st = np.asarray(st, dtype=np.uint64); en = np.asarray(en, dtype=np.uint64)
        h = C.c_void_p(12345)
        rc = lib.hga_sdk_count_packed(0, k, _p(packed), 0, _p(off), len(off) - 1, _p(st), _p(en), len(st), len(first) - 1 if n_files is None else n_files,
                                      None if first_null else _p(first), 2, C.byref(h))
        assert h.value is None
        return rc, lib.hga_last_error().decode()

    for k in (0, 33):
        rc, msg = call(k=k)
        assert rc == HGA_E_ARG and "Kmer size" in msg
    rc, msg = call(off=(5, 50, 100))
    assert rc == HGA_E_ARG and "read_off[0] must be 0" in msg
    rc, msg = call(off=(0, 100, 50))
    assert rc == HGA_E_ARG and "not monotone" in msg
    rc, msg = call(st=(90,), en=(101,))
    assert rc == HGA_E_ARG and "hga_sdk_count_packed: exception run" in msg
    rc, msg = call(n_files=0)
    assert rc == HGA_E_ARG and "n_files must be at least 1" in msg
    rc, msg = call(first_null=True)
    assert rc == HGA_E_ARG and "file_first_read is NULL" in msg
    for first in ((1, 1, 2), (0, 1, 1), (0, 1, 3)):
        rc, msg = call(first=first)
        assert rc == HGA_E_ARG and "must start at 0 and end at n_reads" in msg, first
    rc, msg = call(first=(0, 2, 1, 2))
    assert rc == HGA_E_ARG and "decreases at file 1" in msg
    rc = lib.hga_sdk_count_packed(0, 19, _p(packed), 0, None, 0, None, None, 0, 1, None, 2, None)
    assert rc == HGA_E_ARG


def test_sdk_handle_argument_errors(hga):
    lib = _set_types(hga.capi.load_library())
    n = C.c_uint64()
    assert lib.hga_sdk_size(None, C.byref(n)) == HGA_E_ARG
    thr = np.array(CLI_THRESHOLDS, dtype=np.float64)
    assert lib.hga_sdk_specificity(None, _p(thr), 7, None, None, None, 0, C.byref(n)) == HGA_E_ARG
    r = _SR()
    assert lib.hga_sdk_range(None, 0, 10, C.byref(r)) == HGA_E_ARG and r.n == 0
    lib.hga_sdk_free(None)
    lib.hga_free_sdk_range(None)
