"""ctypes binding of libhga_b200.so — one Python method per C-ABI entry point of include/hga_b200.h."""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None

u64p = C.POINTER(C.c_uint64)
u32p = C.POINTER(C.c_uint32)


class HgaError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"hga_b200 error {code}: {msg}")
        self.code = code


class _Hits(C.Structure):
    _fields_ = [("n_reads", C.c_uint64), ("n_hits", C.c_uint64), ("row_off", u64p), ("kmer_id", u32p), ("pos", u32p)]


class _Index(C.Structure):
    _fields_ = [("n_kmers", C.c_uint64), ("n_entries", C.c_uint64), ("off", u64p), ("read_id", u32p)]


class _Pairs(C.Structure):
    _fields_ = [("n_pairs", C.c_uint64), ("n_increments", C.c_uint64), ("x", u32p), ("y", u32p), ("score", u32p)]


class _Selection(C.Structure):
    _fields_ = [("n_directed", C.c_uint64), ("cut_score", C.c_uint64), ("n_selected", C.c_uint64), ("x", u32p), ("y", u32p), ("score", u32p)]


class _Components(C.Structure):
    _fields_ = [("n_reads", C.c_uint64), ("read_id_first", C.c_uint32), ("label", u32p), ("n_components", C.c_uint64),
                ("comp_label", u32p), ("comp_size", u32p)]


class _Enrichment(C.Structure):
    _fields_ = [("n_cores", C.c_uint64), ("core_id", u32p), ("core_off", u64p), ("core_read", u32p),
                ("n_connections", C.c_uint64), ("conn_x", u32p), ("conn_y", u32p), ("conn_score", u32p),
                ("n_final", C.c_uint64), ("final_id", u32p), ("final_off", u64p), ("final_read", u32p),
                ("n_reads", C.c_uint64), ("read_id_first", C.c_uint32), ("assignment", u32p)]


class _TailBlock(C.Structure):
    _fields_ = [("ran", C.c_int), ("n_scaffold_cores", C.c_uint64), ("n_connections", C.c_uint64), ("conn_x", u32p), ("conn_y", u32p), ("conn_score", u64p),
                ("n_clusters", C.c_uint64), ("cluster_off", u64p), ("cluster_member", u32p)]


class _CoreKmers(C.Structure):
    _fields_ = [("n_cores", C.c_uint64), ("off", u64p), ("kmer_id", u32p)]


class Metrics(C.Structure):
    _fields_ = [(n, C.c_double) for n in ("table_build_ms", "h2d_ms", "scan_ms", "index_ms", "pair_ms", "select_ms", "components_ms", "exchange_ms")] + \
               [(n, C.c_uint64) for n in ("n_bases", "n_reads", "n_hits", "n_pairs", "n_increments", "n_selected", "n_components", "table_bytes",
                                          "filter_bytes", "pair_retries", "heavy_pivots", "kernel_launches", "table_overflow_keys", "mid_pivots", "n_candidates")] + \
               [("enrich_ms", C.c_double)] + [(n, C.c_uint64) for n in ("n_cores", "n_enrich_connections", "n_final_components", "redo_pivots")] + \
               [("enrich_phase_ms", C.c_double * 6), ("scan_retries", C.c_uint64)]

    def as_dict(self):
        return {n: (list(getattr(self, n)) if n == "enrich_phase_ms" else getattr(self, n)) for n, _ in self._fields_}


# every symbol include/hga_b200.h declares (tests check the .so exports exactly these)
EXPORTS = ["hga_last_error", "hga_version", "hga_device_count", "hga_init", "hga_host_alloc", "hga_host_free", "hga_create", "hga_destroy", "hga_set_stream",
           "hga_scan", "hga_scan_device", "hga_host_pack_bases", "hga_host_pack_bases_folded", "hga_scan_packed", "hga_scan_packed_device", "hga_get_hits", "hga_build_index", "hga_get_index", "hga_pair_count", "hga_get_pairs", "hga_select_edges",
           "hga_get_selection", "hga_components", "hga_get_components", "hga_enrich", "hga_enrich_ex", "hga_enrich_full", "hga_get_tail_block", "hga_count_kmers", "hga_count_kmers_packed", "hga_count_spectrum", "hga_count_spectrum_packed", "hga_free_kmer_counts", "hga_host_sdk_merge", "hga_host_sdk_specificity", "hga_host_sdk_select", "hga_sdk_count_packed", "hga_sdk_size", "hga_sdk_specificity", "hga_sdk_range", "hga_free_sdk_range", "hga_sdk_free", "hga_get_enrichment", "hga_get_purged_index", "hga_get_core_kmers", "hga_spectral_clustering", "hga_host_tail_connections", "hga_host_sym_eigen",
           "hga_metrics", "hga_comm_unique_id", "hga_comm_init", "hga_comm_gather_root"]


def library_path():
    return os.path.join(_HERE, "libhga_b200.so")


def load_library():
    """Loads the in-tree CUDA library. Fails loudly when it has not been built: there is no fallback."""
    global _LIB
    if _LIB is None:
        path = library_path()
        if not os.path.exists(path):
            raise HgaError(-1, f"{path} is missing: run `python hybrid-genome-assembler_b200/build.py` (no CPU fallback exists)")
        lib = C.CDLL(path)
        lib.hga_last_error.restype = C.c_char_p
        lib.hga_version.restype = C.c_char_p
        lib.hga_create.argtypes = [C.c_int, C.c_int, C.c_void_p, C.c_uint64, C.POINTER(C.c_void_p)]
        lib.hga_destroy.argtypes = [C.c_void_p]
        lib.hga_destroy.restype = None
        lib.hga_set_stream.argtypes = [C.c_void_p, C.c_void_p]
        lib.hga_scan.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint32]
        lib.hga_scan_device.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint32]
        lib.hga_host_pack_bases.argtypes = [C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.POINTER(C.c_uint64), C.c_int]
        lib.hga_host_pack_bases_folded.argtypes = lib.hga_host_pack_bases.argtypes
        lib.hga_scan_packed.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint32]
        lib.hga_scan_packed_device.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64, C.c_uint64, C.c_void_p, C.c_void_p, C.c_uint64,
                                               C.c_uint32]
        lib.hga_get_hits.argtypes = [C.c_void_p, C.c_int, C.POINTER(_Hits)]
        lib.hga_build_index.argtypes = [C.c_void_p]
        lib.hga_get_index.argtypes = [C.c_void_p, C.POINTER(_Index)]
        lib.hga_pair_count.argtypes = [C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint64]
        lib.hga_get_pairs.argtypes = [C.c_void_p, C.POINTER(_Pairs)]
        lib.hga_select_edges.argtypes = [C.c_void_p, C.c_double, C.c_uint32]
        lib.hga_get_selection.argtypes = [C.c_void_p, C.POINTER(_Selection)]
        lib.hga_components.argtypes = [C.c_void_p, C.c_int]
        lib.hga_get_components.argtypes = [C.c_void_p, C.POINTER(_Components)]
        lib.hga_enrich.argtypes = [C.c_void_p, C.c_int, C.c_uint32]
        lib.hga_enrich_ex.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_uint32]
        lib.hga_enrich_full.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_uint32, C.c_uint32, C.c_int, C.c_void_p]
        lib.hga_get_tail_block.argtypes = [C.c_void_p, C.POINTER(_TailBlock)]
        lib.hga_get_enrichment.argtypes = [C.c_void_p, C.POINTER(_Enrichment)]
        lib.hga_get_purged_index.argtypes = [C.c_void_p, C.POINTER(_Index)]
        lib.hga_get_core_kmers.argtypes = [C.c_void_p, C.POINTER(_CoreKmers)]
        lib.hga_metrics.argtypes = [C.c_void_p, C.POINTER(Metrics)]
        lib.hga_comm_unique_id.argtypes = [C.c_void_p]
        lib.hga_comm_init.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_uint64]
        lib.hga_comm_gather_root.argtypes = [C.c_void_p]
        lib.hga_host_alloc.argtypes = [C.POINTER(C.c_void_p), C.c_size_t]
        lib.hga_host_free.argtypes = [C.c_void_p]
        lib.hga_device_count.argtypes = [C.POINTER(C.c_int)]
        _LIB = lib
    return _LIB


def _check(rc):
    if rc != 0:
        raise HgaError(rc, load_library().hga_last_error().decode())


def _arr(ptr, n, dtype):
    if n == 0:
        return np.zeros(0, dtype=dtype)
    return np.ctypeslib.as_array(ptr, shape=(int(n),)).astype(dtype, copy=True)


def _host_bytes(bases):
    """(keep-alive object, pointer, length) of host bytes given as bytes / bytearray / uint8 array"""
    if isinstance(bases, np.ndarray):
        b = np.ascontiguousarray(bases, dtype=np.uint8)
        return b, b.ctypes.data_as(C.c_void_p), b.shape[0]
    b = bytes(bases)
    return b, C.cast(C.c_char_p(b), C.c_void_p), len(b)


def pack_bases(bases, threads=0, capacity=64, fold_case=False):
    """hga_host_pack_bases: ASCII bases -> (packed uint8[(n + 3) // 4], exc_start uint64[], exc_end uint64[]), the input of Handle.scan_packed.
    Codes A0 C1 G2 T3, four bases per byte, first base in the most significant bits; every byte other than uppercase ACGT is code 0 under
    a maximal exception run [start, end). Starts with `capacity` runs and retries once with the exact count.
    fold_case=True (hga_host_pack_bases_folded): the case-folded packing count_kmers_packed takes; lowercase acgt are packed as their
    bases and only bytes outside ACGTacgt are exceptions."""
    lib = load_library()
    pack = lib.hga_host_pack_bases_folded if fold_case else lib.hga_host_pack_bases
    keep, ptr, n = _host_bytes(bases)
    packed = np.zeros((n + 3) // 4, dtype=np.uint8)
    n_exc = C.c_uint64()
    while True:
        cap = max(int(capacity), 1)
        st = np.zeros(cap, dtype=np.uint64); en = np.zeros(cap, dtype=np.uint64)
        rc = pack(ptr, n, packed.ctypes.data_as(C.c_void_p), st.ctypes.data_as(C.c_void_p), en.ctypes.data_as(C.c_void_p), cap, C.byref(n_exc),
                  int(threads))
        if rc == 2 and n_exc.value > cap:
            capacity = n_exc.value
            continue
        _check(rc)
        del keep
        return packed, st[:n_exc.value].copy(), en[:n_exc.value].copy()


def spectral_clustering(conn_x, conn_y, conn_score, dims=16):
    """Host-side spectral clustering of scaffold components (hga_spectral_clustering). Returns the clusters as a list of uint32
    arrays of component ids (element [0] = the member closest to the cluster centre); empty clusters are kept."""
    lib = load_library()
    x = np.ascontiguousarray(conn_x, dtype=np.uint32); y = np.ascontiguousarray(conn_y, dtype=np.uint32)
    s = np.ascontiguousarray(conn_score, dtype=np.uint64)
    n = x.shape[0]
    out = np.zeros(2 * n + 1, dtype=np.uint32)
    off = np.zeros(max(dims, 2) + 2, dtype=np.uint64)
    n_comp = C.c_uint64(); n_cl = C.c_uint64()
    lib.hga_spectral_clustering.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_int, C.c_void_p, C.c_void_p, C.POINTER(C.c_uint64),
                                            C.POINTER(C.c_uint64)]
    _check(lib.hga_spectral_clustering(x.ctypes.data_as(C.c_void_p), y.ctypes.data_as(C.c_void_p), s.ctypes.data_as(C.c_void_p), n, int(dims),
                                       out.ctypes.data_as(C.c_void_p), off.ctypes.data_as(C.c_void_p), C.byref(n_comp), C.byref(n_cl)))
    o = off.astype(np.int64)
    return [out[o[i]:o[i + 1]].copy() for i in range(n_cl.value)]


def host_sym_eigen(a):
    """eigenvalues (ascending) and eigenvectors (columns) of a symmetric matrix with the library's own solver"""
    lib = load_library()
    a = np.ascontiguousarray(a, dtype=np.float64)
    n = a.shape[0]
    val = np.zeros(n, dtype=np.float64); vec = np.zeros((n, n), dtype=np.float64)
    lib.hga_host_sym_eigen.argtypes = [C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
    _check(lib.hga_host_sym_eigen(n, a.ctypes.data_as(C.c_void_p), val.ctypes.data_as(C.c_void_p), vec.ctypes.data_as(C.c_void_p)))
    return val, vec


class _KmerCounts(C.Structure):
    _fields_ = [("n", C.c_uint64), ("kmer", u64p), ("count", u32p)]


def count_kmers(bases, read_off, k, min_count=2, device=0):
    """hga_count_kmers: exact canonical k-mer counts of a read set on the GPU (the jellyfish step of the SDK selection). Returns
    (k-mers ascending, counts) of the k-mers that occur at least min_count times."""
    lib = load_library()
    lib.hga_count_kmers.argtypes = [C.c_int, C.c_int, C.c_char_p, C.c_void_p, C.c_uint64, C.c_uint32, C.POINTER(_KmerCounts)]
    lib.hga_free_kmer_counts.argtypes = [C.POINTER(_KmerCounts)]
    lib.hga_free_kmer_counts.restype = None
    ro = np.ascontiguousarray(read_off, dtype=np.uint64)
    out = _KmerCounts()
    _check(lib.hga_count_kmers(int(device), int(k), bytes(bases), ro.ctypes.data_as(C.c_void_p), ro.shape[0] - 1, int(min_count), C.byref(out)))
    try:
        return _arr(out.kmer, out.n, np.uint64), _arr(out.count, out.n, np.uint32)
    finally:
        lib.hga_free_kmer_counts(C.byref(out))


def count_kmers_packed(packed, read_off, exc_start, exc_end, k, min_count=2, first_base=0, device=0):
    """hga_count_kmers_packed: count_kmers from the case-folded packing (pack_bases(..., fold_case=True)). The read set is bases
    first_base + read_off[..] of `packed` (read_off[0] == 0); exc_start / exc_end are the exception runs relative to first_base. Returns
    what count_kmers returns on the ASCII bytes."""
    lib = load_library()
    lib.hga_count_kmers_packed.argtypes = [C.c_int, C.c_int, C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint32,
                                           C.POINTER(_KmerCounts)]
    lib.hga_free_kmer_counts.argtypes = [C.POINTER(_KmerCounts)]
    lib.hga_free_kmer_counts.restype = None
    keep, ptr, _ = _host_bytes(packed)
    ro = np.ascontiguousarray(read_off, dtype=np.uint64)
    st = np.ascontiguousarray(exc_start, dtype=np.uint64); en = np.ascontiguousarray(exc_end, dtype=np.uint64)
    out = _KmerCounts()
    _check(lib.hga_count_kmers_packed(int(device), int(k), ptr, int(first_base), ro.ctypes.data_as(C.c_void_p), ro.shape[0] - 1, st.ctypes.data_as(C.c_void_p),
                                      en.ctypes.data_as(C.c_void_p), st.shape[0], int(min_count), C.byref(out)))
    del keep
    try:
        return _arr(out.kmer, out.n, np.uint64), _arr(out.count, out.n, np.uint32)
    finally:
        lib.hga_free_kmer_counts(C.byref(out))


class _KmerSpectrum(C.Structure):
    _fields_ = [("n_windows", C.c_uint64), ("n_distinct", C.c_uint64), ("max_count", C.c_uint64)]


def count_spectrum(bases, read_off, k, n_bins=0, device=0):
    """hga_count_spectrum: the k-mer spectrum of count_kmers(.., min_count=1) without materialising the k-mers. Returns (hist, n_windows,
    n_distinct, max_count): hist[c - 1] = distinct k-mers seen exactly c times, the last of the n_bins entries those seen n_bins times or more."""
    lib = load_library()
    lib.hga_count_spectrum.argtypes = [C.c_int, C.c_int, C.c_char_p, C.c_void_p, C.c_uint64, C.c_uint32, C.c_void_p, C.POINTER(_KmerSpectrum)]
    ro = np.ascontiguousarray(read_off, dtype=np.uint64)
    hist = np.zeros(int(n_bins), dtype=np.uint64)
    out = _KmerSpectrum()
    _check(lib.hga_count_spectrum(int(device), int(k), bytes(bases), ro.ctypes.data_as(C.c_void_p), ro.shape[0] - 1, int(n_bins), hist.ctypes.data_as(C.c_void_p),
                                  C.byref(out)))
    return hist, out.n_windows, out.n_distinct, out.max_count


def count_spectrum_packed(packed, read_off, exc_start, exc_end, k, n_bins=0, first_base=0, device=0):
    """hga_count_spectrum_packed: count_spectrum from the case-folded packing, with the read set and runs of count_kmers_packed"""
    lib = load_library()
    lib.hga_count_spectrum_packed.argtypes = [C.c_int, C.c_int, C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint32,
                                              C.c_void_p, C.POINTER(_KmerSpectrum)]
    keep, ptr, _ = _host_bytes(packed)
    ro = np.ascontiguousarray(read_off, dtype=np.uint64)
    st = np.ascontiguousarray(exc_start, dtype=np.uint64); en = np.ascontiguousarray(exc_end, dtype=np.uint64)
    hist = np.zeros(int(n_bins), dtype=np.uint64)
    out = _KmerSpectrum()
    _check(lib.hga_count_spectrum_packed(int(device), int(k), ptr, int(first_base), ro.ctypes.data_as(C.c_void_p), ro.shape[0] - 1, st.ctypes.data_as(C.c_void_p),
                                         en.ctypes.data_as(C.c_void_p), st.shape[0], int(n_bins), hist.ctypes.data_as(C.c_void_p), C.byref(out)))
    del keep
    return hist, out.n_windows, out.n_distinct, out.max_count


def sdk_merge(per_file):
    """hga_host_sdk_merge: per_file = [(k-mers ascending, counts), ...] -> (k-mers, total count, largest per-file count, files holding it)"""
    lib = load_library()
    P = C.c_void_p
    lib.hga_host_sdk_merge.argtypes = [C.c_int, P, P, P, P, P, P, P, C.POINTER(C.c_uint64)]
    off = np.zeros(len(per_file) + 1, dtype=np.uint64)
    np.cumsum([len(kc[0]) for kc in per_file], out=off[1:])
    km = np.ascontiguousarray(np.concatenate([np.asarray(kc[0], dtype=np.uint64) for kc in per_file]) if per_file else np.zeros(0, np.uint64))
    ct = np.ascontiguousarray(np.concatenate([np.asarray(kc[1], dtype=np.uint32) for kc in per_file]) if per_file else np.zeros(0, np.uint32))
    cap = max(int(off[-1]), 1)
    ok = np.zeros(cap, dtype=np.uint64); ot = np.zeros(cap, dtype=np.uint32); om = np.zeros(cap, dtype=np.uint32); of = np.zeros(cap, dtype=np.uint32)
    n = C.c_uint64()
    _check(lib.hga_host_sdk_merge(len(per_file), off.ctypes.data_as(P), km.ctypes.data_as(P), ct.ctypes.data_as(P), ok.ctypes.data_as(P), ot.ctypes.data_as(P),
                                  om.ctypes.data_as(P), of.ctypes.data_as(P), C.byref(n)))
    return ok[:n.value], ot[:n.value], om[:n.value], of[:n.value]


SDK_THRESHOLDS = (70, 85, 90, 95, 99, 100, 100.01)      # jellyfish_occurrences.cpp:47


def sdk_specificity(total, largest, thresholds=SDK_THRESHOLDS):
    """hga_host_sdk_specificity: rows (upper specificity, total count, number of distinct k-mers), ordered like the reference's nested map"""
    lib = load_library()
    P = C.c_void_p
    lib.hga_host_sdk_specificity.argtypes = [C.c_uint64, P, P, P, C.c_int, P, P, P, C.c_uint64, C.POINTER(C.c_uint64)]
    t = np.ascontiguousarray(total, dtype=np.uint32); m = np.ascontiguousarray(largest, dtype=np.uint32)
    thr = np.ascontiguousarray(thresholds, dtype=np.float64)
    n = C.c_uint64()
    _check(lib.hga_host_sdk_specificity(t.shape[0], t.ctypes.data_as(P), m.ctypes.data_as(P), thr.ctypes.data_as(P), thr.shape[0], None, None, None, 0, C.byref(n)))
    cap = max(n.value, 1)
    ot = np.zeros(cap, dtype=np.float64); oo = np.zeros(cap, dtype=np.uint32); ou = np.zeros(cap, dtype=np.uint64)
    _check(lib.hga_host_sdk_specificity(t.shape[0], t.ctypes.data_as(P), m.ctypes.data_as(P), thr.ctypes.data_as(P), thr.shape[0], ot.ctypes.data_as(P),
                                        oo.ctypes.data_as(P), ou.ctypes.data_as(P), cap, C.byref(n)))
    return ot[:n.value], oo[:n.value], ou[:n.value]


def sdk_select(total, files, lower, upper, percent=1.0, seed=0):
    """hga_host_sdk_select: mask of the k-mers with lower <= total <= upper (each kept with probability percent), and how many of the
    selected ones are present in exactly one file"""
    lib = load_library()
    P = C.c_void_p
    lib.hga_host_sdk_select.argtypes = [C.c_uint64, P, P, C.c_uint32, C.c_uint32, C.c_double, C.c_uint64, P, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]
    t = np.ascontiguousarray(total, dtype=np.uint32); f = np.ascontiguousarray(files, dtype=np.uint32)
    sel = np.zeros(max(t.shape[0], 1), dtype=np.uint8)
    ns = C.c_uint64(); nd = C.c_uint64()
    _check(lib.hga_host_sdk_select(t.shape[0], t.ctypes.data_as(P), f.ctypes.data_as(P), int(lower), int(upper), float(percent), int(seed), sel.ctypes.data_as(P),
                                   C.byref(ns), C.byref(nd)))
    return sel[:t.shape[0]].astype(bool), int(ns.value), int(nd.value)


class _SdkRange(C.Structure):
    _fields_ = [("n", C.c_uint64), ("kmer", u64p), ("total", u32p), ("max", u32p), ("files", u32p)]


def _sdk_lib():
    lib = load_library()
    P = C.c_void_p
    lib.hga_sdk_count_packed.argtypes = [C.c_int, C.c_int, P, C.c_uint64, P, C.c_uint64, P, P, C.c_uint64, C.c_int, P, C.c_uint32, C.POINTER(C.c_void_p)]
    lib.hga_sdk_size.argtypes = [P, C.POINTER(C.c_uint64)]
    lib.hga_sdk_specificity.argtypes = [P, P, C.c_int, P, P, P, C.c_uint64, C.POINTER(C.c_uint64)]
    lib.hga_sdk_range.argtypes = [P, C.c_uint32, C.c_uint32, C.POINTER(_SdkRange)]
    lib.hga_free_sdk_range.argtypes = [C.POINTER(_SdkRange)]
    lib.hga_free_sdk_range.restype = None
    lib.hga_sdk_free.argtypes = [P]
    lib.hga_sdk_free.restype = None
    return lib


class SdkTable:
    """The merged k-mer table of sdk_count_packed, held in device memory until close() (or the end of a `with` block)."""

    def __init__(self, ptr):
        self._p = ptr
        n = C.c_uint64()
        _check(_sdk_lib().hga_sdk_size(self._p, C.byref(n)))
        self.n = int(n.value)

    def specificity(self, thresholds=SDK_THRESHOLDS):
        """hga_sdk_specificity: the rows of sdk_specificity on the merged table (upper specificity, total count, number of k-mers)"""
        lib = _sdk_lib()
        P = C.c_void_p
        thr = np.ascontiguousarray(thresholds, dtype=np.float64)
        n = C.c_uint64()
        _check(lib.hga_sdk_specificity(self._p, thr.ctypes.data_as(P), thr.shape[0], None, None, None, 0, C.byref(n)))
        cap = max(n.value, 1)
        ot = np.zeros(cap, dtype=np.float64); oo = np.zeros(cap, dtype=np.uint32); ou = np.zeros(cap, dtype=np.uint64)
        _check(lib.hga_sdk_specificity(self._p, thr.ctypes.data_as(P), thr.shape[0], ot.ctypes.data_as(P), oo.ctypes.data_as(P), ou.ctypes.data_as(P), cap,
                                       C.byref(n)))
        return ot[:n.value], oo[:n.value], ou[:n.value]

    def range(self, lower=0, upper=0xFFFFFFFF):
        """hga_sdk_range: (k-mers ascending, total, largest per-file count, files) of the entries with lower <= total <= upper"""
        lib = _sdk_lib()
        out = _SdkRange()
        _check(lib.hga_sdk_range(self._p, int(lower), int(upper), C.byref(out)))
        try:
            return (_arr(out.kmer, out.n, np.uint64), _arr(out.total, out.n, np.uint32), _arr(out.max, out.n, np.uint32),
                    _arr(out.files, out.n, np.uint32))
        finally:
            lib.hga_free_sdk_range(C.byref(out))

    def close(self):
        if self._p:
            _sdk_lib().hga_sdk_free(self._p)
            self._p = None

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def __del__(self):
        self.close()


def sdk_count_packed(packed, read_off, exc_start, exc_end, k, file_first_read, min_count=2, first_base=0, device=0):
    """hga_sdk_count_packed: the read set of count_kmers_packed cut into files (file f = reads file_first_read[f] ..
    file_first_read[f + 1]), every file counted with min_count and the files merged on the GPU. Returns an SdkTable holding what
    sdk_merge returns on the per-file count_kmers_packed lists."""
    lib = _sdk_lib()
    P = C.c_void_p
    keep, ptr, _ = _host_bytes(packed)
    ro = np.ascontiguousarray(read_off, dtype=np.uint64)
    st = np.ascontiguousarray(exc_start, dtype=np.uint64); en = np.ascontiguousarray(exc_end, dtype=np.uint64)
    ff = np.ascontiguousarray(file_first_read, dtype=np.uint64)
    out = C.c_void_p()
    _check(lib.hga_sdk_count_packed(int(device), int(k), ptr, int(first_base), ro.ctypes.data_as(P), ro.shape[0] - 1, st.ctypes.data_as(P), en.ctypes.data_as(P),
                                    st.shape[0], ff.shape[0] - 1, ff.ctypes.data_as(P), int(min_count), C.byref(out)))
    del keep
    return SdkTable(out.value)


def host_tail_connections(row_off, kmer_id, pos, read_len, avg_read_length, comp_off, comp_member, tree_off, tree_x, tree_y, purged_off, purged_read,
                          amplification_min_score=40, read_id_first=1):
    """Host-side tail connections between scaffold components (hga_host_tail_connections). Rows must be sorted by (kmer_id, pos)."""
    lib = load_library()
    a = [np.ascontiguousarray(row_off, dtype=np.uint64), np.ascontiguousarray(kmer_id, dtype=np.uint32), np.ascontiguousarray(pos, dtype=np.uint32),
         np.ascontiguousarray(read_len, dtype=np.uint32), np.ascontiguousarray(comp_off, dtype=np.uint64), np.ascontiguousarray(comp_member, dtype=np.uint32),
         np.ascontiguousarray(tree_off, dtype=np.uint64), np.ascontiguousarray(tree_x, dtype=np.uint32), np.ascontiguousarray(tree_y, dtype=np.uint32),
         np.ascontiguousarray(purged_off, dtype=np.uint64), np.ascontiguousarray(purged_read, dtype=np.uint32)]
    n_reads = a[0].shape[0] - 1
    n_comp = a[4].shape[0] - 1
    cap = max(1, n_comp * (n_comp - 1) // 2)
    ox = np.zeros(cap, dtype=np.uint32); oy = np.zeros(cap, dtype=np.uint32); osc = np.zeros(cap, dtype=np.uint64)
    n = C.c_uint64()
    P = C.c_void_p
    lib.hga_host_tail_connections.argtypes = [C.c_uint64, P, P, P, P, C.c_uint64, C.c_uint32, C.c_uint64, P, P, P, P, P, P, P, C.c_uint32, P, P, P, C.POINTER(C.c_uint64)]
    ptr = [x.ctypes.data_as(P) for x in a]
    _check(lib.hga_host_tail_connections(n_reads, ptr[0], ptr[1], ptr[2], ptr[3], int(avg_read_length), int(read_id_first), n_comp, ptr[4], ptr[5], ptr[6], ptr[7],
                                         ptr[8], ptr[9], ptr[10], int(amplification_min_score), ox.ctypes.data_as(P), oy.ctypes.data_as(P), osc.ctypes.data_as(P),
                                         C.byref(n)))
    return ox[:n.value].copy(), oy[:n.value].copy(), osc[:n.value].copy()


def device_count():
    n = C.c_int(0)
    _check(load_library().hga_device_count(C.byref(n)))
    return n.value


def comm_unique_id():
    buf = (C.c_ubyte * 128)()
    _check(load_library().hga_comm_unique_id(buf))
    return bytes(buf)


class Handle:
    """One GPU-resident k-mer table + the stage results of the most recent run (hga_handle)."""

    def __init__(self, kmers, k, device=0):
        self.lib = load_library()
        kmers = np.ascontiguousarray(kmers, dtype=np.uint64)
        self.k = int(k)
        self.n_kmers = int(kmers.shape[0])
        self._h = C.c_void_p()
        _check(self.lib.hga_create(int(device), self.k, kmers.ctypes.data_as(C.c_void_p), self.n_kmers, C.byref(self._h)))

    def close(self):
        if getattr(self, "_h", None) is not None and self._h:
            self.lib.hga_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def set_stream(self, cuda_stream_ptr):
        _check(self.lib.hga_set_stream(self._h, C.c_void_p(cuda_stream_ptr or 0)))

    def comm_init(self, unique_id: bytes, rank, nranks, n_reads_total):
        buf = (C.c_ubyte * 128).from_buffer_copy(unique_id)
        _check(self.lib.hga_comm_init(self._h, buf, int(rank), int(nranks), int(n_reads_total)))

    def comm_gather_root(self):
        """collective: rank 0's handle becomes a complete single-GPU handle (hga_enrich* then runs there)"""
        _check(self.lib.hga_comm_gather_root(self._h))

    # -- stages ------------------------------------------------------------------------------------------
    def scan(self, bases, read_off, read_id_base=1):
        """bases: bytes / bytearray / uint8 array (host); read_off: uint64[n_reads+1]."""
        read_off = np.ascontiguousarray(read_off, dtype=np.uint64)
        n_reads = read_off.shape[0] - 1
        if isinstance(bases, np.ndarray):
            b = np.ascontiguousarray(bases, dtype=np.uint8)
            ptr = b.ctypes.data_as(C.c_void_p)
        else:
            b = bases
            ptr = C.cast(C.c_char_p(bytes(b)) if not isinstance(b, bytes) else C.c_char_p(b), C.c_void_p)
        _check(self.lib.hga_scan(self._h, ptr, read_off.ctypes.data_as(C.c_void_p), n_reads, int(read_id_base)))

    def scan_host_ptr(self, bases_ptr, read_off_ptr, n_reads, read_id_base=1):
        _check(self.lib.hga_scan(self._h, C.c_void_p(bases_ptr), C.c_void_p(read_off_ptr), int(n_reads), int(read_id_base)))

    def scan_device(self, d_bases_ptr, d_read_off_ptr, n_reads, n_bases, read_id_base=1):
        _check(self.lib.hga_scan_device(self._h, C.c_void_p(d_bases_ptr), C.c_void_p(d_read_off_ptr), int(n_reads), int(n_bases), int(read_id_base)))

    def scan_packed(self, packed, read_off, exc_start, exc_end, first_base=0, read_id_base=1):
        """packed: uint8 array / bytes (host), bases first_base + read_off[..] of it; exc_start / exc_end: the exception runs relative to
        first_base (pack_bases gives them for first_base = 0)."""
        read_off = np.ascontiguousarray(read_off, dtype=np.uint64)
        st = np.ascontiguousarray(exc_start, dtype=np.uint64); en = np.ascontiguousarray(exc_end, dtype=np.uint64)
        if st.shape != en.shape:
            raise ValueError("exc_start and exc_end differ in length")
        keep, ptr, _ = _host_bytes(packed)
        _check(self.lib.hga_scan_packed(self._h, ptr, int(first_base), read_off.ctypes.data_as(C.c_void_p), read_off.shape[0] - 1,
                                        st.ctypes.data_as(C.c_void_p), en.ctypes.data_as(C.c_void_p), st.shape[0], int(read_id_base)))
        del keep

    def scan_packed_host_ptr(self, packed_ptr, first_base, read_off_ptr, n_reads, exc_start_ptr, exc_end_ptr, n_exc, read_id_base=1):
        _check(self.lib.hga_scan_packed(self._h, C.c_void_p(packed_ptr), int(first_base), C.c_void_p(read_off_ptr), int(n_reads), C.c_void_p(exc_start_ptr),
                                        C.c_void_p(exc_end_ptr), int(n_exc), int(read_id_base)))

    def scan_packed_device(self, d_packed_ptr, first_base, d_read_off_ptr, n_reads, n_bases, d_exc_start_ptr, d_exc_end_ptr, n_exc, read_id_base=1):
        _check(self.lib.hga_scan_packed_device(self._h, C.c_void_p(d_packed_ptr), int(first_base), C.c_void_p(d_read_off_ptr), int(n_reads), int(n_bases),
                                               C.c_void_p(d_exc_start_ptr), C.c_void_p(d_exc_end_ptr), int(n_exc), int(read_id_base)))

    def get_hits(self, sorted_by_kmer_id=False):
        out = _Hits()
        _check(self.lib.hga_get_hits(self._h, 1 if sorted_by_kmer_id else 0, C.byref(out)))
        return _arr(out.row_off, out.n_reads + 1, np.uint64), _arr(out.kmer_id, out.n_hits, np.uint32), _arr(out.pos, out.n_hits, np.uint32)

    def build_index(self):
        _check(self.lib.hga_build_index(self._h))

    def get_index(self):
        out = _Index()
        _check(self.lib.hga_get_index(self._h, C.byref(out)))
        return _arr(out.off, out.n_kmers + 1, np.uint64), _arr(out.read_id, out.n_entries, np.uint32)

    def pair_count(self, min_score=1, pivots=None):
        if pivots is None:
            _check(self.lib.hga_pair_count(self._h, int(min_score), None, 0))
        else:
            pv = np.ascontiguousarray(pivots, dtype=np.uint32)
            n = pv.shape[0]
            if n == 0:                     # the empty subset: a non-NULL pointer with n = 0 (NULL would mean "all reads")
                pv = np.zeros(1, dtype=np.uint32)
            _check(self.lib.hga_pair_count(self._h, int(min_score), pv.ctypes.data_as(C.c_void_p), n))

    def get_pairs(self):
        out = _Pairs()
        _check(self.lib.hga_get_pairs(self._h, C.byref(out)))
        n = out.n_pairs
        return _arr(out.x, n, np.uint32), _arr(out.y, n, np.uint32), _arr(out.score, n, np.uint32), int(out.n_increments)

    def select_edges(self, fraction=0.15, score_threshold=0):
        _check(self.lib.hga_select_edges(self._h, float(fraction), int(score_threshold)))

    def get_selection(self):
        out = _Selection()
        _check(self.lib.hga_get_selection(self._h, C.byref(out)))
        n = out.n_selected
        return dict(n_directed=int(out.n_directed), cut_score=int(out.cut_score), x=_arr(out.x, n, np.uint32), y=_arr(out.y, n, np.uint32),
                    score=_arr(out.score, n, np.uint32))

    def components(self, min_size=30):
        _check(self.lib.hga_components(self._h, int(min_size)))

    def get_components(self):
        out = _Components()
        _check(self.lib.hga_get_components(self._h, C.byref(out)))
        return dict(read_id_first=int(out.read_id_first), label=_arr(out.label, out.n_reads, np.uint32),
                    comp_label=_arr(out.comp_label, out.n_components, np.uint32), comp_size=_arr(out.comp_size, out.n_components, np.uint32))

    def enrich(self, min_size=30, enrichment_min_score=20, max_size=-1):
        if max_size == -1:
            _check(self.lib.hga_enrich(self._h, int(min_size), int(enrichment_min_score)))
        else:
            _check(self.lib.hga_enrich_ex(self._h, int(min_size), int(max_size), int(enrichment_min_score)))

    def enrich_full(self, read_off, min_size=30, enrichment_min_score=20, max_size=-1, tail_amplification_min_score=40, spectral_dims=16):
        """hga_enrich_full: merge + enrichment INCLUDING the tail / spectral block (run_clustering :764-794). read_off as given to scan()."""
        ro = np.ascontiguousarray(read_off, dtype=np.uint64)
        _check(self.lib.hga_enrich_full(self._h, int(min_size), int(max_size), int(enrichment_min_score), int(tail_amplification_min_score), int(spectral_dims),
                                        ro.ctypes.data_as(C.c_void_p)))

    def get_tail_block(self):
        out = _TailBlock()
        _check(self.lib.hga_get_tail_block(self._h, C.byref(out)))
        off = _arr(out.cluster_off, out.n_clusters + 1, np.uint64) if out.n_clusters else np.zeros(1, dtype=np.uint64)
        mem = _arr(out.cluster_member, int(off[-1]), np.uint32)
        return dict(ran=bool(out.ran), n_scaffold_cores=int(out.n_scaffold_cores), conn_x=_arr(out.conn_x, out.n_connections, np.uint32),
                    conn_y=_arr(out.conn_y, out.n_connections, np.uint32), conn_score=_arr(out.conn_score, out.n_connections, np.uint64),
                    clusters=[mem[int(off[i]):int(off[i + 1])] for i in range(len(off) - 1)])

    def get_enrichment(self):
        out = _Enrichment()
        _check(self.lib.hga_get_enrichment(self._h, C.byref(out)))
        nc, nf = out.n_cores, out.n_final
        core_off = _arr(out.core_off, nc + 1, np.uint64); final_off = _arr(out.final_off, nf + 1, np.uint64)
        return dict(core_id=_arr(out.core_id, nc, np.uint32), core_off=core_off, core_read=_arr(out.core_read, int(core_off[-1]) if nc else 0, np.uint32),
                    conn_x=_arr(out.conn_x, out.n_connections, np.uint32), conn_y=_arr(out.conn_y, out.n_connections, np.uint32),
                    conn_score=_arr(out.conn_score, out.n_connections, np.uint32),
                    final_id=_arr(out.final_id, nf, np.uint32), final_off=final_off, final_read=_arr(out.final_read, int(final_off[-1]) if nf else 0, np.uint32),
                    read_id_first=int(out.read_id_first), assignment=_arr(out.assignment, out.n_reads, np.uint32))

    def get_purged_index(self):
        out = _Index()
        _check(self.lib.hga_get_purged_index(self._h, C.byref(out)))
        return _arr(out.off, out.n_kmers + 1, np.uint64), _arr(out.read_id, out.n_entries, np.uint32)

    def get_core_kmers(self):
        out = _CoreKmers()
        _check(self.lib.hga_get_core_kmers(self._h, C.byref(out)))
        off = _arr(out.off, out.n_cores + 1, np.uint64)
        return off, _arr(out.kmer_id, int(off[-1]), np.uint32)

    def metrics(self):
        m = Metrics()
        _check(self.lib.hga_metrics(self._h, C.byref(m)))
        return m.as_dict()
