"""CPU: the 2-bit packer hga_host_pack_bases against an independent numpy packer, and the packing loader of the `categorization` CLI
(cli/hga_host.h, packed mode) against the packer run on the ASCII loader's buffer. No GPU involved."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def hga():
    import importlib
    importlib.import_module("hybrid-genome-assembler_b200.build").build()
    import hga_b200
    hga_b200.load_library()
    return hga_b200


def np_pack(data):
    """independent packer: A0 C1 G2 T3, first base in the top bits; everything else code 0 under maximal half-open runs"""
    b = np.frombuffer(bytes(data), dtype=np.uint8) if not isinstance(data, np.ndarray) else data.astype(np.uint8)
    code = np.full(256, -1, dtype=np.int16)
    for ch, v in zip(b"ACGT", range(4)):
        code[ch] = v
    c = code[b]
    exc = c < 0
    c = np.where(exc, 0, c).astype(np.uint8)
    n = b.shape[0]
    pad = np.zeros((n + 3) // 4 * 4, dtype=np.uint8)
    pad[:n] = c
    q = pad.reshape(-1, 4)
    packed = (q[:, 0] << 6) | (q[:, 1] << 4) | (q[:, 2] << 2) | q[:, 3]
    e = np.concatenate([[False], exc, [False]]).astype(np.int8)
    d = np.diff(e)
    return packed.astype(np.uint8), np.nonzero(d == 1)[0].astype(np.uint64), np.nonzero(d == -1)[0].astype(np.uint64)


def _check(hga, data, threads):
    p, s, e = hga.pack_bases(data, threads=threads, capacity=2)
    rp, rs, re_ = np_pack(data)
    assert np.array_equal(p, rp)
    assert np.array_equal(s, rs) and np.array_equal(e, re_)
    return len(s)


@pytest.mark.parametrize("threads", [1, 2, 16])
@pytest.mark.parametrize("n", [0, 1, 2, 3, 4, 5, 7, 8, 9, 15, 16, 17, 63, 64, 65, 1000, 4099])
def test_pack_all_byte_values(hga, threads, n):
    rng = np.random.default_rng(1000 * n + threads)
    _check(hga, rng.integers(0, 256, n, dtype=np.uint8), threads)


@pytest.mark.parametrize("threads", [1, 2, 16])
@pytest.mark.parametrize("seed", range(6))
def test_pack_mostly_acgt_with_runs(hga, threads, seed):
    """clean stretches (the 8-byte fast path) with N runs, lowercase stretches, CR bytes and single odd bytes, runs at the start and
    at the end of the stream, lengths not divisible by 4"""
    rng = np.random.default_rng(seed)
    n = int(rng.integers(3000, 9000))
    b = np.frombuffer(b"ACGT", dtype=np.uint8)[rng.integers(0, 4, n)].copy()
    for _ in range(int(rng.integers(1, 30))):
        a = int(rng.integers(0, n)); L = int(rng.integers(1, 400))
        kind = int(rng.integers(0, 4))
        if kind == 0:
            b[a:a + L] = ord("N")
        elif kind == 1:
            b[a:a + L] = np.frombuffer(b"acgt", dtype=np.uint8)[rng.integers(0, 4, len(b[a:a + L]))]
        elif kind == 2:
            b[a] = 13
        else:
            b[a:a + L] = rng.integers(0, 256, len(b[a:a + L]), dtype=np.uint8)
    if seed % 2 == 0:
        b[:int(rng.integers(1, 40))] = ord("n")
    if seed % 3 == 0:
        b[-int(rng.integers(1, 40)):] = ord("N")
    assert _check(hga, b, threads) > 0


@pytest.mark.parametrize("threads", [2, 16])
def test_pack_runs_across_thread_seams(hga, threads):
    """one run covering many thread ranges, and runs that end / start exactly at a seam, join into maximal runs"""
    n = 4096
    b = bytearray(b"ACGT" * (n // 4))
    per = (n // 4 + threads - 1) // threads * 4
    b[per - 10:3 * per + 7] = b"N" * (3 * per + 17 - per)
    b[4 * per - 3:4 * per] = b"xyz"                       # ends exactly at a seam
    b[5 * per:5 * per + 2] = b"nn"                        # starts exactly at a seam
    b[6 * per - 1:6 * per + 1] = b"\r\r"                  # straddles a seam by one byte each side
    _check(hga, bytes(b), threads)
    assert _check(hga, b"N" * 1001, threads) == 1


def test_pack_capacity_protocol(hga):
    """too few run slots: HGA_E_ARG and the exact number needed; nothing else is required of the call"""
    lib = hga.load_library()
    data = b"ANA" * 50 + b"C"
    packed = np.zeros((len(data) + 3) // 4, dtype=np.uint8)
    st = np.zeros(10, dtype=np.uint64); en = np.zeros(10, dtype=np.uint64)
    n = C.c_uint64(7)
    rc = lib.hga_host_pack_bases(C.cast(C.c_char_p(data), C.c_void_p), len(data), packed.ctypes.data_as(C.c_void_p), st.ctypes.data_as(C.c_void_p),
                                 en.ctypes.data_as(C.c_void_p), 10, C.byref(n), 1)
    assert rc == 2 and n.value == 50 and b"capacity" in lib.hga_last_error()
    rc = lib.hga_host_pack_bases(C.cast(C.c_char_p(data), C.c_void_p), len(data), packed.ctypes.data_as(C.c_void_p), None, None, 0, C.byref(n), 4)
    assert rc == 2 and n.value == 50
    st = np.zeros(50, dtype=np.uint64); en = np.zeros(50, dtype=np.uint64)
    rc = lib.hga_host_pack_bases(C.cast(C.c_char_p(data), C.c_void_p), len(data), packed.ctypes.data_as(C.c_void_p), st.ctypes.data_as(C.c_void_p),
                                 en.ctypes.data_as(C.c_void_p), 50, C.byref(n), 3)
    assert rc == 0 and n.value == 50
    rp, rs, re_ = np_pack(data)
    assert np.array_equal(packed, rp) and np.array_equal(st, rs) and np.array_equal(en, re_)
    # a clean stream needs no run slots at all
    rc = lib.hga_host_pack_bases(C.cast(C.c_char_p(b"ACGTTGCA"), C.c_void_p), 8, packed.ctypes.data_as(C.c_void_p), None, None, 0, C.byref(n), 0)
    assert rc == 0 and n.value == 0
    assert lib.hga_host_pack_bases(None, 8, packed.ctypes.data_as(C.c_void_p), None, None, 0, C.byref(n), 0) == 2


HARNESS = r"""
#include "hga_host.h"
#include <cstdio>
// loads the reads twice, ASCII and packed, and writes the ASCII stream, the packed stream and the runs to <out>.{ascii,packed,runs}
int main(int argc, char **argv) {
    const std::string out = argv[1];
    const int threads = atoi(argv[2]);
    std::vector<std::string> paths(argv + 3, argv + argc);
    try {
        hga_host::SequenceRecords a(paths, threads), p(paths, threads, true);
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
    d = tmp_path_factory.mktemp("harness")
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
    p, s, e = hga.pack_bases(ascii_, threads=1)
    assert np.array_equal(packed, p)
    assert np.array_equal(runs, np.concatenate([s, e]))
    rp, rs, re_ = np_pack(ascii_)
    assert np.array_equal(packed, rp) and np.array_equal(runs, np.concatenate([rs, re_]))
    return len(s)


@pytest.mark.parametrize("threads", [1, 2, 16])
@pytest.mark.parametrize("seed", range(24))
def test_packed_loader_on_mangled_inputs(hga, harness, tmp_path, seed, threads):
    """the mangled multi-file inputs of the record-reader fuzz (CRLF, format switches, empty headers, lowercase bytes)"""
    from test_cli import _mangled_files
    _compare_loader(hga, harness, _mangled_files(tmp_path, seed), tmp_path, threads)


@pytest.mark.parametrize("threads", [1, 3, 16])
def test_packed_loader_with_n_runs_across_reads_and_files(hga, harness, tmp_path, threads):
    import datagen
    g = datagen.random_genome(20000, 7)
    paths = []
    for i in range(3):
        reads = [datagen.to_ascii(r) for r in datagen.sample_reads(g, 60, 250, 70 + i, length_sigma=0.5, min_len=1)]
        reads = [r if j % 5 else "N" * len(r) for j, r in enumerate(reads)]                     # whole reads of N: runs across read ends
        reads = [r.lower() if j % 7 == 3 else r for j, r in enumerate(reads)]
        reads = [r[:10] + "NNNNNNN" + r[10:] if j % 3 == 1 else r for j, r in enumerate(reads)]
        p = str(tmp_path / f"r{i}.{'fq' if i % 2 else 'fa'}")
        (datagen.write_fastq if i % 2 else datagen.write_fasta)(p, reads, prefix=f"f{i}_", newline="\r\n" if i == 1 else "\n")
        paths.append(p)
    assert _compare_loader(hga, harness, paths, tmp_path, threads) > 10
