"""CPU: the case-folded 2-bit packing of the k-mer count (hga_host_pack_bases_folded, and the folded mode of the CLI loader) against an
independent numpy packer, and the whole of hga_count_kmers_packed (argument checks of csrc/hga_capi.cu + csrc/hga_count.cu with its packed
emit kernel, launches, CUB calls and buffers) compiled for the host with the fake-CUDA harness of test_kernel_bodies_on_host.py, against
exact numpy counts and against hga_count_kmers on the ASCII bytes. No GPU involved."""
import ctypes as C
import os
import re
import subprocess

import numpy as np
import pytest

import datagen
from test_kernel_bodies_on_host import FAKE_CUDA, PRELUDE, _cut, _cut_macros
from test_sdk_selection_cpu import exact_counts

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "hybrid-genome-assembler_b200", "csrc")
HGA_E_ARG = 2


@pytest.fixture(scope="module")
def hga():
    import importlib
    importlib.import_module("hybrid-genome-assembler_b200.build").build()
    import hga_b200
    hga_b200.load_library()
    return hga_b200


def np_pack_folded(data):
    """independent folded packer: A/a 0, C/c 1, G/g 2, T/t 3, first base in the top bits; every other byte code 0 under maximal runs"""
    b = np.frombuffer(bytes(data), dtype=np.uint8) if not isinstance(data, np.ndarray) else data.astype(np.uint8)
    code = np.full(256, -1, dtype=np.int16)
    for chars in (b"ACGT", b"acgt"):
        for ch, v in zip(chars, range(4)):
            code[ch] = v
    c = code[b]
    exc = c < 0
    c = np.where(exc, 0, c).astype(np.uint8)
    n = b.shape[0]
    pad = np.zeros((n + 3) // 4 * 4, dtype=np.uint8)
    pad[:n] = c
    q = pad.reshape(-1, 4)
    packed = (q[:, 0] << 6) | (q[:, 1] << 4) | (q[:, 2] << 2) | q[:, 3]
    d = np.diff(np.concatenate([[False], exc, [False]]).astype(np.int8))
    return packed.astype(np.uint8), np.nonzero(d == 1)[0].astype(np.uint64), np.nonzero(d == -1)[0].astype(np.uint64)


def _check(hga, data, threads):
    p, s, e = hga.pack_bases(data, threads=threads, capacity=2, fold_case=True)
    rp, rs, re_ = np_pack_folded(data)
    assert np.array_equal(p, rp)
    assert np.array_equal(s, rs) and np.array_equal(e, re_)
    return len(s)


def _mixed(rng, n):
    """ACGT with lowercase stretches (the 8-byte fast path on mixed case), N runs, CR bytes and random bytes"""
    b = np.frombuffer(b"ACGTacgt", dtype=np.uint8)[rng.integers(0, 8, n)].copy()
    for _ in range(int(rng.integers(1, 30))):
        a = int(rng.integers(0, n)); L = int(rng.integers(1, 400))
        kind = int(rng.integers(0, 4))
        if kind == 0:
            b[a:a + L] = ord("N") if L % 2 else ord("n")
        elif kind == 1:
            b[a:a + L] = np.frombuffer(b"acgt", dtype=np.uint8)[rng.integers(0, 4, len(b[a:a + L]))]
        elif kind == 2:
            b[a] = 13
        else:
            b[a:a + L] = rng.integers(0, 256, len(b[a:a + L]), dtype=np.uint8)
    return b


@pytest.mark.parametrize("threads", [1, 2, 16])
@pytest.mark.parametrize("n", [0, 1, 3, 4, 5, 8, 9, 17, 64, 65, 1000, 4099])
def test_folded_pack_all_byte_values(hga, threads, n):
    rng = np.random.default_rng(7000 + 1000 * n + threads)
    _check(hga, rng.integers(0, 256, n, dtype=np.uint8), threads)
    # every byte whose bit-5-cleared form is A C G T, and its neighbours: only ACGTacgt are bases
    _check(hga, np.arange(256, dtype=np.uint8)[rng.permutation(256)][:n], threads)


@pytest.mark.parametrize("threads", [1, 2, 16])
@pytest.mark.parametrize("seed", range(6))
def test_folded_pack_mixed_case_with_runs(hga, threads, seed):
    rng = np.random.default_rng(seed)
    b = _mixed(rng, int(rng.integers(3000, 9000)))
    if seed % 2 == 0:
        b[:int(rng.integers(1, 40))] = ord("N")
    if seed % 3 == 0:
        b[-int(rng.integers(1, 40)):] = 13
    assert _check(hga, b, threads) > 0
    # the scan's packing of the same bytes differs exactly where lowercase acgt sit
    p, s, e = hga.pack_bases(b, threads=threads)
    assert len(s) >= _check(hga, b, threads)


@pytest.mark.parametrize("threads", [2, 16])
def test_folded_pack_runs_across_thread_seams(hga, threads):
    n = 4096
    b = bytearray(b"ACgt" * (n // 4))
    per = (n // 4 + threads - 1) // threads * 4
    b[per - 10:3 * per + 7] = b"N" * (3 * per + 17 - per)
    b[4 * per - 3:4 * per] = b"xyz"
    b[5 * per:5 * per + 2] = b"nn"
    b[6 * per - 1:6 * per + 1] = b"\r\r"
    _check(hga, bytes(b), threads)
    assert _check(hga, b"N" * 1001, threads) == 1
    assert _check(hga, b"acgtACGT" * 500, threads) == 0


def test_folded_pack_capacity_protocol(hga):
    lib = hga.load_library()
    data = b"aNa" * 50 + b"c"
    packed = np.zeros((len(data) + 3) // 4, dtype=np.uint8)
    st = np.zeros(10, dtype=np.uint64); en = np.zeros(10, dtype=np.uint64)
    n = C.c_uint64(7)
    ptr = C.cast(C.c_char_p(data), C.c_void_p)
    rc = lib.hga_host_pack_bases_folded(ptr, len(data), packed.ctypes.data_as(C.c_void_p), st.ctypes.data_as(C.c_void_p), en.ctypes.data_as(C.c_void_p), 10, C.byref(n), 1)
    assert rc == HGA_E_ARG and n.value == 50 and b"capacity" in lib.hga_last_error()
    assert lib.hga_host_pack_bases_folded(ptr, len(data), packed.ctypes.data_as(C.c_void_p), None, None, 0, C.byref(n), 4) == HGA_E_ARG and n.value == 50
    st = np.zeros(50, dtype=np.uint64); en = np.zeros(50, dtype=np.uint64)
    rc = lib.hga_host_pack_bases_folded(ptr, len(data), packed.ctypes.data_as(C.c_void_p), st.ctypes.data_as(C.c_void_p), en.ctypes.data_as(C.c_void_p), 50, C.byref(n), 3)
    assert rc == 0 and n.value == 50
    rp, rs, re_ = np_pack_folded(data)
    assert np.array_equal(packed, rp) and np.array_equal(st, rs) and np.array_equal(en, re_)
    rc = lib.hga_host_pack_bases_folded(C.cast(C.c_char_p(b"acgtTGCA"), C.c_void_p), 8, packed.ctypes.data_as(C.c_void_p), None, None, 0, C.byref(n), 0)
    assert rc == 0 and n.value == 0
    assert lib.hga_host_pack_bases_folded(None, 8, packed.ctypes.data_as(C.c_void_p), None, None, 0, C.byref(n), 0) == HGA_E_ARG


# ---- the CLI loader's folded mode --------------------------------------------------------------------------------------------------
HARNESS = r"""
#include "hga_host.h"
#include <cstdio>
// loads the reads ASCII and packed-folded, and writes the ASCII stream, the packed stream and the runs to <out>.{ascii,packed,runs}
int main(int argc, char **argv) {
    const std::string out = argv[1];
    const int threads = atoi(argv[2]);
    std::vector<std::string> paths(argv + 3, argv + argc);
    try {
        hga_host::SequenceRecords a(paths, threads), p(paths, threads, true, true);
        if (a.bases_size != p.bases_size || a.seq_off != p.seq_off) return 3;
        for (size_t i = 0; i < a.n_reads(); i++) if (a.sequence(i) != p.sequence(i)) return 4;
        FILE *f = fopen((out + ".ascii").c_str(), "wb"); fwrite(a.bases_data, 1, a.bases_size, f); fclose(f);
        f = fopen((out + ".packed").c_str(), "wb"); fwrite(p.packed_data, 1, (p.bases_size + 3) / 4, f); fclose(f);
        f = fopen((out + ".runs").c_str(), "wb");
        fwrite(p.exc_start.data(), 8, p.exc_start.size(), f); fwrite(p.exc_end.data(), 8, p.exc_end.size(), f); fclose(f);
    } catch (const std::exception &e) {
        printf("%s\n", e.what());
        return 2;
    }
    return 0;
}
"""


@pytest.fixture(scope="module")
def harness(tmp_path_factory):
    d = tmp_path_factory.mktemp("folded_harness")
    src = d / "harness.cpp"
    src.write_text(HARNESS)
    exe = str(d / "harness")
    subprocess.run(["g++", "-std=c++17", "-O2", "-I", os.path.join(ROOT, "include"), "-I", os.path.join(ROOT, "hybrid-genome-assembler_b200", "cli"),
                    str(src), "-o", exe, "-lpthread"], check=True)
    return exe


def _compare_loader(hga, harness, paths, tmp_path, threads):
    out = str(tmp_path / "dump")
    r = subprocess.run([harness, out, str(threads)] + paths, capture_output=True, text=True)
    if r.returncode == 2:
        return None                                     # the reader refuses this input in both modes alike (test_cli covers that)
    assert r.returncode == 0, (r.returncode, r.stdout)
    ascii_ = np.fromfile(out + ".ascii", dtype=np.uint8)
    packed = np.fromfile(out + ".packed", dtype=np.uint8)
    runs = np.fromfile(out + ".runs", dtype=np.uint64)
    p, s, e = hga.pack_bases(ascii_, threads=1, fold_case=True)
    assert np.array_equal(packed, p) and np.array_equal(runs, np.concatenate([s, e]))
    rp, rs, re_ = np_pack_folded(ascii_)
    assert np.array_equal(packed, rp) and np.array_equal(runs, np.concatenate([rs, re_]))
    return len(s)


@pytest.mark.parametrize("threads", [1, 2, 16])
@pytest.mark.parametrize("seed", range(12))
def test_folded_loader_on_mangled_inputs(hga, harness, tmp_path, seed, threads):
    from test_cli import _mangled_files
    _compare_loader(hga, harness, _mangled_files(tmp_path, seed), tmp_path, threads)


@pytest.mark.parametrize("threads", [1, 3, 16])
def test_folded_loader_with_lowercase_and_n_across_files(hga, harness, tmp_path, threads):
    g = datagen.random_genome(20000, 9)
    paths = []
    for i in range(3):
        reads = [datagen.to_ascii(r) for r in datagen.sample_reads(g, 60, 250, 90 + i, length_sigma=0.5, min_len=1)]
        reads = [r if j % 5 else "N" * len(r) for j, r in enumerate(reads)]
        reads = [r.lower() if j % 7 == 3 else r for j, r in enumerate(reads)]
        reads = [r[:10] + "NNNNNNN" + r[10:] if j % 3 == 1 else r for j, r in enumerate(reads)]
        p = str(tmp_path / f"r{i}.{'fq' if i % 2 else 'fa'}")
        (datagen.write_fastq if i % 2 else datagen.write_fasta)(p, reads, prefix=f"f{i}_", newline="\r\n" if i == 1 else "\n")
        paths.append(p)
    assert _compare_loader(hga, harness, paths, tmp_path, threads) > 10


# ---- the whole of hga_count_kmers_packed on the host -------------------------------------------------------------------------------
# hga_count.cu is compiled as test_kernel_bodies_on_host.py compiles it for hga_count_kmers; the argument checks and the entry itself are
# cut out of hga_capi.cu (check_read_off, check_exc_runs, hga_count_kmers_packed). Both entries are then in one host library.
@pytest.fixture(scope="module")
def host_count(tmp_path_factory):
    text = open(os.path.join(CSRC, "hga_count.cu")).read()
    capi = open(os.path.join(CSRC, "hga_capi.cu")).read()
    internal = open(os.path.join(CSRC, "hga_internal.cuh")).read()
    text = re.sub(r'#include\s+"hga_internal.cuh"\n', "", text)
    text = re.sub(r"#include\s+<cub/[^>]+>\n", "", text)
    text = re.sub(r"<<<[^;]*?>>>", "", text)
    devbuf = internal[internal.index("struct DevBuf {"):internal.index("struct PinBuf {")]
    entry = "\n".join([_cut(capi, r"^static int check_read_off"), _cut(capi, r"^static int check_exc_runs"),
                       'extern "C" {\n' + _cut(capi, r"^int hga_count_kmers_packed") + '}\n'])
    d = tmp_path_factory.mktemp("host_packed_count")
    src, so = str(d / "count_host.cpp"), str(d / "count_host.so")
    open(src, "w").write(PRELUDE + FAKE_CUDA + _cut_macros(internal) + devbuf + text + entry)
    subprocess.run(["g++", "-std=c++17", "-O1", "-fPIC", "-shared", "-I", os.path.join(ROOT, "include"), "-o", so, src], check=True)
    lib = C.CDLL(so)
    lib.fake_last_error.restype = C.c_char_p
    lib.hga_count_kmers_packed.argtypes = [C.c_int, C.c_int, C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint32, C.c_void_p]
    lib.hga_count_kmers.argtypes = [C.c_int, C.c_int, C.c_char_p, C.c_void_p, C.c_uint64, C.c_uint32, C.c_void_p]
    return lib


class _KC(C.Structure):
    _fields_ = [("n", C.c_uint64), ("kmer", C.POINTER(C.c_uint64)), ("count", C.POINTER(C.c_uint32))]


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def _take(lib, out):
    km = np.ctypeslib.as_array(out.kmer, shape=(max(out.n, 1),))[:out.n].copy() if out.n else np.zeros(0, np.uint64)
    ct = np.ctypeslib.as_array(out.count, shape=(max(out.n, 1),))[:out.n].copy() if out.n else np.zeros(0, np.uint32)
    lib.hga_free_kmer_counts(C.byref(out))
    return km, ct


def slice_runs(st, en, b0, b1):
    """the runs of a packed stream clipped to bases [b0, b1) and rebased to b0"""
    st = np.asarray(st, dtype=np.uint64); en = np.asarray(en, dtype=np.uint64)
    m = (en > np.uint64(b0)) & (st < np.uint64(b1))
    return (np.maximum(st[m], np.uint64(b0)) - np.uint64(b0)).astype(np.uint64), (np.minimum(en[m], np.uint64(b1)) - np.uint64(b0)).astype(np.uint64)


def count_reads(seed, k, n_reads=120, poly_a=0):
    """reads with N runs, lowercase stretches, CR bytes, an empty read, reads shorter than k and runs on read ends"""
    rng = np.random.default_rng(seed)
    g = datagen.random_genome(3000, 300 + seed)
    reads = [datagen.to_ascii(r) for r in datagen.sample_reads(g, n_reads, 150, 400 + seed, error_rate=0.01)]
    reads[1] = reads[1][:20] + "N" + reads[1][21:]
    reads[3] = reads[3].lower()
    reads[5] = ""
    reads[7] = reads[7][:max(k - 1, 0)]
    reads[8] = "NNN" + reads[8] + "nn"                                   # runs that touch both ends of a read
    reads[9] = reads[9][:40] + "\r"
    reads[10] = reads[10][:30].lower() + reads[10][30:60] + "ac" + "N" * 5
    for j in range(12, n_reads, 9):
        a = int(rng.integers(0, max(len(reads[j]), 1)))
        reads[j] = reads[j][:a] + reads[j][a:a + 25].lower() + reads[j][a + 25:]
    if poly_a:
        reads.append("A" * poly_a)
    return reads


def _run_both(lib, reads, k, min_count, first_base, prefix_rng):
    seq = "".join(reads).encode()
    off = np.zeros(len(reads) + 1, dtype=np.uint64)
    np.cumsum([len(r) for r in reads], out=off[1:])
    # the read set sits first_base bases into a larger stream, between foreign bases (an N run across the seam included)
    pre = np.frombuffer(b"ACGTacgN", dtype=np.uint8)[prefix_rng.integers(0, 8, first_base)].tobytes()
    stream = pre + seq + b"NNacgtTT"
    packed, st, en = np_pack_folded(stream)
    es, ee = slice_runs(st, en, first_base, first_base + len(seq))
    out = _KC()
    rc = lib.hga_count_kmers_packed(0, k, _p(packed), first_base, _p(off), len(reads), _p(es), _p(ee), len(es), min_count, C.byref(out))
    assert rc == 0, lib.fake_last_error()
    got = _take(lib, out)
    out = _KC()
    assert lib.hga_count_kmers(0, k, seq, _p(off), len(reads), min_count, C.byref(out)) == 0, lib.fake_last_error()
    return got, _take(lib, out), exact_counts(seq, off, k, min_count)


@pytest.mark.parametrize("chunk", [None, "1024"])
@pytest.mark.parametrize("k", [1, 5, 11, 19, 31, 32])
def test_count_kmers_packed_on_host(host_count, k, chunk):
    """one pass and forced key-range passes, slices starting 0..3 bases into a byte, min_count 1..3: the k-mers, counts and order of
    hga_count_kmers on the ASCII bytes and of exact counting"""
    if chunk:
        os.environ["HGA_COUNT_CHUNK"] = chunk
    try:
        for first_base in (0, 1, 2, 3, 4 * 37 + 1):
            for min_count in (1, 2, 3):
                (km, ct), (ak, ac), (wk, wc) = _run_both(host_count, count_reads(k, k), k, min_count, first_base, np.random.default_rng(first_base))
                assert np.array_equal(km, wk) and np.array_equal(ct, wc) and len(km) > 0
                assert np.array_equal(km, ak) and np.array_equal(ct, ac)
    finally:
        os.environ.pop("HGA_COUNT_CHUNK", None)


def test_count_kmers_packed_on_host_splits_down_to_one_kmer(host_count):
    """a budget of 256 keys and a poly-A read of 3000 bases: the range of A...A overflows and is split down to that single value"""
    os.environ["HGA_COUNT_CHUNK"] = "256"
    try:
        (km, ct), (ak, ac), (wk, wc) = _run_both(host_count, count_reads(3, 19, n_reads=30, poly_a=3000), 19, 2, 3, np.random.default_rng(3))
    finally:
        os.environ.pop("HGA_COUNT_CHUNK", None)
    assert km[0] == 0 and ct[0] > 256
    assert np.array_equal(km, wk) and np.array_equal(ct, wc) and np.array_equal(km, ak) and np.array_equal(ct, ac)


def test_count_kmers_packed_argument_errors(hga):
    """checked before any device is needed: HGA_E_ARG and a message"""
    lib = hga.load_library()
    lib.hga_count_kmers_packed.argtypes = [C.c_int, C.c_int, C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint32, C.c_void_p]
    packed = np.zeros(64, dtype=np.uint8)

    def call(k, off, st, en):
        off = np.asarray(off, dtype=np.uint64); st = np.asarray(st, dtype=np.uint64); en = np.asarray(en, dtype=np.uint64)
        out = _KC()
        rc = lib.hga_count_kmers_packed(0, k, _p(packed), 0, _p(off), len(off) - 1, _p(st), _p(en), len(st), 2, C.byref(out))
        return rc, lib.hga_last_error().decode()

    for k in (0, 33):
        rc, msg = call(k, [0, 100], [], [])
        assert rc == HGA_E_ARG and "Kmer size" in msg
    rc, msg = call(19, [5, 100], [], [])
    assert rc == HGA_E_ARG and "read_off[0] must be 0" in msg
    rc, msg = call(19, [0, 100, 50], [], [])
    assert rc == HGA_E_ARG and "not monotone" in msg
    for st, en in (([10, 5], [12, 7]), ([10, 11], [12, 14]), ([90], [101]), ([10], [10])):
        rc, msg = call(19, [0, 100], st, en)
        assert rc == HGA_E_ARG and "hga_count_kmers_packed: exception run" in msg, (st, en, msg)
