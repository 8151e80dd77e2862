"""CPU: the bodies of the kernels written after this round's GPU minutes were spent (count_emit / count_flag of csrc/hga_count.cu,
enr_merge2_keys / enr_purge2 of csrc/hga_enrich.cu), compiled FOR THE HOST and run as one thread with a one-thread grid: the text of
each kernel is cut out of the .cu file at test time (nothing is copied into the repo), `__global__`, `blockIdx`, `atomicMax`, ... are
defined away in a few lines, and the results are compared with numpy. This checks the arithmetic and the indexing of the kernel
code itself; it says nothing about launches, CUB calls or buffers - the GPU tests (tests/test_zy_gpu_tail_block.py) do that.
Test infrastructure only: the product never runs this way."""
import ctypes as C
import os
import re
import subprocess

import numpy as np
import pytest

import datagen
from test_second_merge_rule import second_merge_rule
from test_sdk_selection_cpu import exact_counts

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "hybrid-genome-assembler_b200", "csrc")

PRELUDE = r"""
#include <cstdint>
#include <algorithm>
#define __global__
#define __device__
#define __host__
#define __forceinline__ inline
#define __restrict__
struct Dim { unsigned x, y, z; };
static Dim blockIdx{0, 0, 0}, threadIdx{0, 0, 0}, blockDim{1, 1, 1}, gridDim{1, 1, 1};
static inline uint32_t atomicMax(uint32_t *p, uint32_t v) { uint32_t o = *p; if (v > o) *p = v; return o; }
using std::max; using std::min;
"""


def _cut(text, start_pattern):
    """the source of one function / template / constant, from its first line to the closing brace at column 0"""
    m = re.search(start_pattern, text, flags=re.M)
    assert m, start_pattern
    end = text.index("\n}\n", m.start()) + 3
    return text[m.start():end]


@pytest.fixture(scope="module")
def host_kernels(tmp_path_factory):
    count = open(os.path.join(CSRC, "hga_count.cu")).read()
    enrich = open(os.path.join(CSRC, "hga_enrich.cu")).read()
    parts = [PRELUDE,
             re.search(r"^constexpr unsigned long long COUNT_SENTINEL.*$", count, flags=re.M).group(0),
             _cut(count, r"^__device__ __forceinline__ int count_base_code"),
             _cut(count, r"^__device__ __forceinline__ unsigned long long count_window_key"),
             _cut(count, r"^__global__ void count_emit_kernel"),
             _cut(count, r"^__global__ void count_flag_kernel"),
             _cut(enrich, r"^__global__ void enr_merge2_keys_kernel"),
             _cut(enrich, r"^template<bool FILL>\n__global__ void enr_purge2_kernel"),
             r"""
extern "C" {
void run_count_emit(const char *bases, const uint64_t *read_off, uint64_t n_reads, int k, uint64_t p0, uint64_t p1, unsigned long long *out) {
    count_emit_kernel(bases, read_off, n_reads, k, p0, p1, out);
}
void run_count_flag(const unsigned long long *keys, const uint32_t *cnt, uint64_t n, uint32_t min_count, uint8_t *flag) { count_flag_kernel(keys, cnt, n, min_count, flag); }
void run_merge2_keys(const uint64_t *ukeys, uint64_t n, const uint32_t *map, const uint32_t *surv_old, const uint32_t *surv_new, uint32_t *R2, uint64_t *out) {
    enr_merge2_keys_kernel(ukeys, n, map, surv_old, surv_new, R2, out);
}
void run_purge2_count(const uint32_t *p_off, const uint32_t *p_row, uint32_t n_slots, const uint32_t *R2, const uint8_t *once, uint32_t *cnt) {
    enr_purge2_kernel<false>(p_off, p_row, n_slots, R2, once, cnt, nullptr, nullptr);
}
void run_purge2_fill(const uint32_t *p_off, const uint32_t *p_row, uint32_t n_slots, const uint32_t *R2, const uint8_t *once, const uint32_t *out_off, uint32_t *out_row) {
    enr_purge2_kernel<true>(p_off, p_row, n_slots, R2, once, nullptr, out_off, out_row);
}
}
"""]
    d = tmp_path_factory.mktemp("host_kernels")
    src, so = str(d / "k.cpp"), str(d / "k.so")
    open(src, "w").write("\n".join(parts))
    subprocess.run(["g++", "-std=c++17", "-O1", "-fPIC", "-shared", "-o", so, src], check=True)
    return C.CDLL(so)


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


@pytest.mark.parametrize("k", [1, 5, 19, 31, 32])
def test_count_emit_and_flag_bodies(host_kernels, k):
    g = datagen.random_genome(1500, 10 + k)
    reads = [datagen.to_ascii(r) for r in datagen.sample_reads(g, 60, 120, 20 + k, error_rate=0.02)]
    reads[2] = reads[2][:30] + "N" + reads[2][31:]
    reads[4] = reads[4].lower()
    reads[6] = reads[6][:max(k - 1, 0)]
    reads[8] = ""
    reads[9] = ""
    seq = "".join(reads).encode()
    off = np.zeros(len(reads) + 1, dtype=np.uint64)
    np.cumsum([len(r) for r in reads], out=off[1:])
    n = len(seq)
    out = np.zeros(n, dtype=np.uint64)
    # two chunks, as hga_count_kmers launches them
    host_kernels.run_count_emit(seq, _p(off), C.c_uint64(len(reads)), k, C.c_uint64(0), C.c_uint64(n // 3), _p(out))
    tail = np.zeros(n - n // 3, dtype=np.uint64)
    host_kernels.run_count_emit(seq, _p(off), C.c_uint64(len(reads)), k, C.c_uint64(n // 3), C.c_uint64(n), _p(tail))
    out[n // 3:] = tail
    keys, cnt = np.unique(out, return_counts=True)                 # sort + run-length encode
    flag = np.zeros(len(keys), dtype=np.uint8)
    host_kernels.run_count_flag(_p(keys), _p(cnt.astype(np.uint32)), C.c_uint64(len(keys)), 2, _p(flag))
    wk, wc = exact_counts(seq, off, k, 2)
    assert np.array_equal(keys[flag.astype(bool)], wk) and np.array_equal(cnt[flag.astype(bool)].astype(np.uint32), wc)
    assert keys[-1] == np.uint64(0xFFFFFFFFFFFFFFFF) or k == 1     # windows over read ends / N produce the sentinel, which sorts last
    if k < 32:
        assert int(keys[:-1].max()) < (1 << (2 * k))               # ... also when only 2k bits are sorted


def test_second_merge_bodies_match_the_rule(host_kernels):
    """random purged index + unions + clusters: enr_merge2_keys_kernel and enr_purge2_kernel (count and fill) against the numpy rule
    that tests/test_second_merge_rule.py pins against the reference"""
    rng = np.random.default_rng(5)
    for trial in range(20):
        n_rows, n_slots, n_cores = 400, 300, int(rng.integers(3, 12))
        surv = np.sort(rng.choice(n_rows, n_cores, replace=False)).astype(np.uint32)          # survivor rows, ascending
        unions = [np.sort(rng.choice(n_slots, int(rng.integers(5, 120)), replace=False)) for _ in range(n_cores)]
        # purged lists: rows outside every core (here: any non-survivor row) and stale survivor copies, ascending, with duplicates
        lists = []
        for s in range(n_slots):
            e = rng.choice(n_rows, int(rng.integers(0, 12)))
            holders = [c for c in range(n_cores) if s in set(unions[c].tolist())]
            stale = [int(surv[c]) for c in holders for _ in range(int(rng.integers(0, 3)))]
            e = [int(v) for v in e if v not in set(surv.tolist())] + stale
            lists.append(np.sort(np.array(e, dtype=np.uint32)))
        p_off = np.zeros(n_slots + 1, dtype=np.uint32)
        np.cumsum([len(l) for l in lists], out=p_off[1:])
        p_row = np.concatenate(lists).astype(np.uint32) if p_off[-1] else np.zeros(1, np.uint32)
        # clusters over the cores: a few multi-member ones, singletons, and cores in no cluster
        perm = rng.permutation(n_cores)
        clusters, i = [], 0
        while i < n_cores - 1:
            sz = int(rng.integers(1, 4))
            clusters.append([int(surv[c]) for c in perm[i:i + sz]])
            i += sz
        # host glue as in hga_enrich_run: into / multi / new numbering / map / flags
        index_of = {int(s): c for c, s in enumerate(surv)}
        into = list(range(n_cores)); multi = [0] * n_cores
        for cl in clusters:
            if len(cl) < 2:
                continue
            for s in cl:
                into[index_of[s]] = index_of[cl[0]]; multi[index_of[s]] = 1
        new_idx, surv_new = [0] * n_cores, []
        for c in range(n_cores):
            if into[c] == c:
                new_idx[c] = len(surv_new); surv_new.append(int(surv[c]))
        cmap = np.array([new_idx[into[c]] | (multi[c] << 31) for c in range(n_cores)], dtype=np.uint32)
        once = np.zeros(n_rows + 1, dtype=np.uint8)
        for c in range(n_cores):
            if multi[c]:
                once[surv[c]] = 1
        ukeys = np.concatenate([(np.uint64(c) << np.uint64(32)) | unions[c].astype(np.uint64) for c in range(n_cores)])
        R2 = np.zeros(n_slots + 1, dtype=np.uint32)
        rel = np.zeros(len(ukeys), dtype=np.uint64)
        host_kernels.run_merge2_keys(_p(ukeys), C.c_uint64(len(ukeys)), _p(cmap), _p(surv), _p(np.array(surv_new + [0], dtype=np.uint32)), _p(R2), _p(rel))
        new_keys = np.unique(rel)                                                             # sort + unique
        cnt = np.zeros(n_slots + 1, dtype=np.uint32)
        host_kernels.run_purge2_count(_p(p_off), _p(p_row), n_slots, _p(R2), _p(once), _p(cnt))
        out_off = np.zeros(n_slots + 1, dtype=np.uint32)
        np.cumsum(cnt[:n_slots], out=out_off[1:])
        out_row = np.zeros(max(int(out_off[-1]), 1), dtype=np.uint32)
        host_kernels.run_purge2_fill(_p(p_off), _p(p_row), n_slots, _p(R2), _p(once), _p(out_off), _p(out_row))
        # the rule (rows as ids: first_id = 0)
        ids, want_unions, want_off, want_rows = second_merge_rule(surv.astype(np.int64), [u.astype(np.int64) for u in unions], p_off.astype(np.uint64),
                                                                  p_row[:p_off[-1]], clusters)
        assert ids.tolist() == surv_new
        assert np.array_equal(out_off.astype(np.uint64), want_off) and np.array_equal(out_row[:out_off[-1]], want_rows)
        got_unions = [np.sort((new_keys[(new_keys >> np.uint64(32)) == np.uint64(c)] & np.uint64(0xFFFFFFFF)).astype(np.int64)) for c in range(len(surv_new))]
        assert all(np.array_equal(a, b) for a, b in zip(got_unions, want_unions))


# ---- the whole of hga_count_kmers (kernels + launches + CUB calls + buffers) on the host -----------------------------------------
# csrc/hga_count.cu is self-contained apart from DevBuf and the error macros: its text is compiled for the host against a few lines
# that stand in for the CUDA runtime (malloc / memcpy) and for the five CUB entry points it calls (std algorithms honouring the
# two-phase temp-storage protocol and, for the radix sorts, ONLY the requested bit range), with `<<<...>>>` launches turned into
# plain calls of the one-thread grid.
FAKE_CUDA = r"""
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <numeric>
#include <vector>
#include "hga_b200.h"
typedef int cudaError_t;
typedef void *cudaStream_t;
enum { cudaSuccess = 0 };
enum cudaMemcpyKind { cudaMemcpyHostToDevice, cudaMemcpyDeviceToHost, cudaMemcpyDeviceToDevice };
enum cudaDeviceAttr { cudaDevAttrMultiProcessorCount };
static inline cudaError_t cudaGetDeviceCount(int *n) { *n = 1; return 0; }
static inline cudaError_t cudaSetDevice(int) { return 0; }
static inline cudaError_t cudaGetLastError() { return 0; }
static inline const char *cudaGetErrorString(cudaError_t) { return "fake"; }
static inline cudaError_t cudaDeviceGetAttribute(int *v, cudaDeviceAttr, int) { *v = 2; return 0; }
static inline cudaError_t cudaMalloc(void **p, size_t n) { *p = std::malloc(n ? n : 1); return *p ? 0 : 2; }
static inline cudaError_t cudaFree(void *p) { std::free(p); return 0; }
static inline cudaError_t cudaMemsetAsync(void *d, int v, size_t n, cudaStream_t) { std::memset(d, v, n); return 0; }
static inline unsigned long long atomicAdd(unsigned long long *p, unsigned long long v) { unsigned long long o = *p; *p += v; return o; }
static inline cudaError_t cudaMemcpy(void *d, const void *s, size_t n, cudaMemcpyKind) { std::memmove(d, s, n); return 0; }
static inline cudaError_t cudaMemcpyAsync(void *d, const void *s, size_t n, cudaMemcpyKind, cudaStream_t) { std::memmove(d, s, n); return 0; }
static inline cudaError_t cudaStreamSynchronize(cudaStream_t) { return 0; }
static char g_err[512];
void hga_set_error(const char *fmt, ...) { va_list ap; va_start(ap, fmt); vsnprintf(g_err, sizeof g_err, fmt, ap); va_end(ap); }
extern "C" const char *fake_last_error() { return g_err; }
namespace cub {
template<typename K> static inline unsigned long long bits_of(K k, int b0, int b1) { return b1 - b0 >= 64 ? (unsigned long long) k : (((unsigned long long) k >> b0) & ((1ull << (b1 - b0)) - 1)); }
struct DeviceRadixSort {
    template<typename K> static cudaError_t SortKeys(void *tmp, size_t &bytes, const K *in, K *out, unsigned long long n, int b0, int b1, cudaStream_t) {
        if (!tmp) { bytes = 1; return 0; }
        std::vector<K> v(in, in + n);
        std::stable_sort(v.begin(), v.end(), [&](K a, K b) { return bits_of(a, b0, b1) < bits_of(b, b0, b1); });
        std::copy(v.begin(), v.end(), out);
        return 0;
    }
    template<typename K, typename V> static cudaError_t SortPairs(void *tmp, size_t &bytes, const K *kin, K *kout, const V *vin, V *vout, unsigned long long n, int b0, int b1, cudaStream_t) {
        if (!tmp) { bytes = 1; return 0; }
        std::vector<size_t> o(n);
        std::iota(o.begin(), o.end(), (size_t) 0);
        std::stable_sort(o.begin(), o.end(), [&](size_t a, size_t b) { return bits_of(kin[a], b0, b1) < bits_of(kin[b], b0, b1); });
        std::vector<K> k2(n); std::vector<V> v2(n);
        for (size_t i = 0; i < n; i++) { k2[i] = kin[o[i]]; v2[i] = vin[o[i]]; }
        std::copy(k2.begin(), k2.end(), kout); std::copy(v2.begin(), v2.end(), vout);
        return 0;
    }
    template<typename K, typename V> static cudaError_t SortPairsDescending(void *tmp, size_t &bytes, const K *kin, K *kout, const V *vin, V *vout, unsigned long long n, int b0, int b1, cudaStream_t) {
        if (!tmp) { bytes = 1; return 0; }
        std::vector<size_t> o(n);
        std::iota(o.begin(), o.end(), (size_t) 0);
        std::stable_sort(o.begin(), o.end(), [&](size_t a, size_t b) { return bits_of(kin[a], b0, b1) > bits_of(kin[b], b0, b1); });
        std::vector<K> k2(n); std::vector<V> v2(n);
        for (size_t i = 0; i < n; i++) { k2[i] = kin[o[i]]; v2[i] = vin[o[i]]; }
        std::copy(k2.begin(), k2.end(), kout); std::copy(v2.begin(), v2.end(), vout);
        return 0;
    }
};
struct DeviceRunLengthEncode {
    template<typename K, typename L, typename N> static cudaError_t Encode(void *tmp, size_t &bytes, const K *in, K *uniq, L *len, N *runs, unsigned long long n, cudaStream_t) {
        if (!tmp) { bytes = 1; return 0; }
        unsigned long long r = 0;
        for (unsigned long long i = 0; i < n;) { unsigned long long j = i; while (j < n && in[j] == in[i]) j++; uniq[r] = in[i]; len[r] = (L) (j - i); r++; i = j; }
        *runs = (N) r;
        return 0;
    }
};
struct DeviceReduce {
    template<typename K, typename V, typename N, typename Op> static cudaError_t ReduceByKey(void *tmp, size_t &bytes, const K *kin, K *uniq, const V *vin, V *agg, N *runs, Op op, int n, cudaStream_t) {
        if (!tmp) { bytes = 1; return 0; }
        std::vector<K> ku; std::vector<V> va;                    // in and out may alias in the caller: build first, then write
        for (int i = 0; i < n;) { int j = i + 1; V a = vin[i]; while (j < n && kin[j] == kin[i]) { a = op(a, vin[j]); j++; } ku.push_back(kin[i]); va.push_back(a); i = j; }
        std::copy(ku.begin(), ku.end(), uniq); std::copy(va.begin(), va.end(), agg);
        *runs = (N) ku.size();
        return 0;
    }
};
struct DeviceSelect {
    template<typename T, typename F, typename N> static cudaError_t Flagged(void *tmp, size_t &bytes, const T *in, const F *flag, T *out, N *nsel, unsigned long long n, cudaStream_t) {
        if (!tmp) { bytes = 1; return 0; }
        unsigned long long m = 0;
        for (unsigned long long i = 0; i < n; i++) if (flag[i]) out[m++] = in[i];
        *nsel = (N) m;
        return 0;
    }
    template<typename T, typename N> static cudaError_t Unique(void *tmp, size_t &bytes, const T *in, T *out, N *nsel, unsigned long long n, cudaStream_t) {
        if (!tmp) { bytes = 1; return 0; }
        unsigned long long m = 0;
        for (unsigned long long i = 0; i < n; i++) if (i == 0 || in[i] != in[i - 1]) out[m++] = in[i];
        *nsel = (N) m;
        return 0;
    }
};
struct DeviceScan {
    template<typename I, typename O> static cudaError_t ExclusiveSum(void *tmp, size_t &bytes, const I *in, O *out, unsigned long long n, cudaStream_t) {
        if (!tmp) { bytes = 1; return 0; }
        O acc = 0;
        for (unsigned long long i = 0; i < n; i++) { const O v = (O) in[i]; out[i] = acc; acc += v; }
        return 0;
    }
};
}
"""


@pytest.fixture(scope="module")
def host_count_kmers(tmp_path_factory):
    text = open(os.path.join(CSRC, "hga_count.cu")).read()
    internal = open(os.path.join(CSRC, "hga_internal.cuh")).read()
    text = re.sub(r'#include\s+"hga_internal.cuh"\n', "", text)
    text = re.sub(r"#include\s+<cub/[^>]+>\n", "", text)
    text = re.sub(r"<<<[^;]*?>>>", "", text)                              # kernel<<<grid, block, smem, stream>>>(args) -> kernel(args)
    macros = _cut_macros(internal)
    devbuf = internal[internal.index("struct DevBuf {"):internal.index("struct PinBuf {")]
    if os.environ.get("HGA_EMU_ASAN"):
        devbuf = devbuf.replace("size_t want = bytes + (bytes >> 4) + 256;", "size_t want = bytes;")
    d = tmp_path_factory.mktemp("host_count")
    src, so = str(d / "count_host.cpp"), str(d / "count_host.so")
    open(src, "w").write(PRELUDE + FAKE_CUDA + macros + devbuf + text)
    san = ["-fsanitize=address", "-fno-omit-frame-pointer", "-g"] if os.environ.get("HGA_EMU_ASAN") else []
    subprocess.run(["g++", "-std=c++17", "-O1", "-fPIC", "-shared"] + san + ["-I", os.path.join(ROOT, "include"), "-o", so, src], check=True)
    return C.CDLL(so)


def _cut_macros(internal):
    a = internal.index("#define HGA_CUDA(call)")
    b = internal.index("while (0)", internal.index("#define HGA_TRY(call)")) + len("while (0)")
    return internal[a:b] + "\n"


class _KC(C.Structure):
    _fields_ = [("n", C.c_uint64), ("kmer", C.POINTER(C.c_uint64)), ("count", C.POINTER(C.c_uint32))]


@pytest.mark.parametrize("k,chunk", [(19, None), (19, "1024"), (11, "256"), (32, "700"), (5, "4096")])
def test_count_kmers_orchestration_on_host(host_count_kmers, k, chunk):
    g = datagen.random_genome(3000, 300 + k)
    reads = [datagen.to_ascii(r) for r in datagen.sample_reads(g, 120, 150, 400 + k, error_rate=0.01)]
    reads[1] = reads[1][:20] + "N" + reads[1][21:]
    reads[3] = reads[3].lower()
    reads[5] = ""
    seq = ("XXXX" + "".join(reads)).encode()                     # the first read does not start at offset 0
    off = np.zeros(len(reads) + 1, dtype=np.uint64)
    np.cumsum([len(r) for r in reads], out=off[1:])
    off += np.uint64(4)
    if chunk:
        os.environ["HGA_COUNT_CHUNK"] = chunk
    try:
        for min_count in (1, 2, 3):
            out = _KC()
            rc = host_count_kmers.hga_count_kmers(0, k, seq, _p(off), C.c_uint64(len(reads)), C.c_uint32(min_count), C.byref(out))
            assert rc == 0, C.c_char_p(host_count_kmers.fake_last_error()).value
            km = np.ctypeslib.as_array(out.kmer, shape=(max(out.n, 1),))[:out.n].copy()
            ct = np.ctypeslib.as_array(out.count, shape=(max(out.n, 1),))[:out.n].copy()
            host_count_kmers.hga_free_kmer_counts(C.byref(out))
            wk, wc = exact_counts(seq[4:], off - np.uint64(4), k, min_count)
            assert np.array_equal(km, wk) and np.array_equal(ct, wc) and len(km) > 0
    finally:
        os.environ.pop("HGA_COUNT_CHUNK", None)


# ---- the whole of hga_enrich_run, tail / spectral block included, on the host ----------------------------------------------------
# csrc/hga_enrich.cu + csrc/hga_internal.cuh compiled for the host like hga_count.cu above, linked with the REAL host stages
# (csrc/hga_tails.cpp, csrc/hga_spectral.cpp). The handle's "device" state (selected edges, inverted index keyed by slot = kmer_id,
# hits) is filled from the C oracle; hga_get_hits / hga_export_index (csrc/hga_capi.cu, GPU-verified) are stood in for by a few
# lines. What runs is the product's own source for: the root replay and its GPU pre-filter, the unions, both purges, the spanning
# forest, the glue around the host stages, the second merge, the enrichment connections and the final merge.
FAKE_CUDA_MORE = r"""
typedef void *cudaEvent_t;
static inline cudaError_t cudaEventCreate(cudaEvent_t *e) { *e = nullptr; return 0; }
static inline cudaError_t cudaEventDestroy(cudaEvent_t) { return 0; }
static inline cudaError_t cudaEventRecord(cudaEvent_t, cudaStream_t) { return 0; }
static inline cudaError_t cudaEventSynchronize(cudaEvent_t) { return 0; }
static inline cudaError_t cudaEventElapsedTime(float *ms, cudaEvent_t, cudaEvent_t) { *ms = 0; return 0; }
static inline cudaError_t cudaMallocHost(void **p, size_t n) { *p = std::malloc(n ? n : 1); return *p ? 0 : 2; }
static inline cudaError_t cudaFreeHost(void *p) { std::free(p); return 0; }
static inline unsigned atomicCAS(unsigned *p, unsigned cmp, unsigned v) { unsigned o = *p; if (o == cmp) *p = v; return o; }
static inline unsigned __umulhi(unsigned a, unsigned b) { return (unsigned) (((unsigned long long) a * b) >> 32); }
static inline unsigned __brev(unsigned x) { unsigned r = 0; for (int i = 0; i < 32; i++) r |= ((x >> i) & 1u) << (31 - i); return r; }
"""

EMU_HARNESS = r"""
static struct { std::vector<uint64_t> row_off, idx_off; std::vector<uint32_t> kid, pos, idx_read; } g_emu;
int hga_comm_size(const hga_handle *) { return 1; }
extern "C" int hga_get_hits(hga_handle *h, int sorted_by_kmer_id, hga_hits *out) {
    if (!sorted_by_kmer_id) return HGA_E_ARG;
    out->n_reads = h->n_reads; out->n_hits = g_emu.kid.size(); out->row_off = g_emu.row_off.data(); out->kmer_id = g_emu.kid.data(); out->pos = g_emu.pos.data();
    return HGA_OK;
}
int hga_export_index(hga_handle *h, const uint32_t *d_off, const uint32_t *d_row, uint64_t E, hga_index *out) {
    const uint64_t K = h->n_kmers;                             // emulation: slot == kmer_id
    g_emu.idx_off.assign(K + 1, 0); g_emu.idx_read.assign(E + 1, 0);
    for (uint64_t k = 0; k <= K; k++) g_emu.idx_off[k] = d_off[k];
    for (uint64_t i = 0; i < E; i++) g_emu.idx_read[i] = d_row[i] + h->inc_row_first_id;
    out->n_kmers = K; out->n_entries = E; out->off = g_emu.idx_off.data(); out->read_id = g_emu.idx_read.data();
    return HGA_OK;
}
static hga_handle *g_h = nullptr;
static std::vector<uint32_t> g_core_kmer;
static std::vector<uint64_t> g_core_koff;
static hga_index g_purged;
extern "C" int emu_enrich(uint64_t n_reads, uint64_t n_kmers, const uint64_t *row_off, const uint32_t *kid, const uint32_t *pos, const uint64_t *inv_off,
                          const uint32_t *inv_read, uint64_t M, const uint32_t *sel_x, const uint32_t *sel_y, const uint32_t *sel_score, const uint64_t *read_off,
                          int min_size, uint32_t min_score, uint32_t amp, int dims, int with_tail, int max_size, const uint8_t *pivot_flag) {
    delete g_h;
    hga_handle *h = g_h = new hga_handle();
    std::memset(&h->metrics, 0, sizeof h->metrics);
    h->n_kmers = n_kmers; h->n_reads = n_reads; h->inc_rows = n_reads; h->inc_row_first_id = 1; h->read_id_base = 1; h->sm_count = 2;
    h->index_keys = (uint32_t) n_kmers; h->n_hits = row_off[n_reads]; h->inc_entries = inv_off[n_kmers];
    h->have_scan = h->have_index = h->have_selection = true;
    g_emu.row_off.assign(row_off, row_off + n_reads + 1); g_emu.kid.assign(kid, kid + row_off[n_reads]); g_emu.pos.assign(pos, pos + row_off[n_reads]);
    if (h->d_inv_off.ensure((n_kmers + 1) * 4) || h->d_inv_row.ensure((inv_off[n_kmers] + 1) * 4) || h->d_sel_key.ensure((M + 1) * 8) || h->d_sel_score.ensure((M + 1) * 4)) return -1;
    if (h->d_row_off.ensure((n_reads + 1) * 8) || h->d_hit_slot.ensure((row_off[n_reads] + 1) * 4)) return -1;      // the hits by read (slot == kmer_id): the tail amplification reads them
    std::memcpy(h->d_row_off.p, row_off, (n_reads + 1) * 8);
    std::memcpy(h->d_hit_slot.p, kid, row_off[n_reads] * 4);
    for (uint64_t k = 0; k <= n_kmers; k++) h->d_inv_off.as<uint32_t>()[k] = (uint32_t) inv_off[k];
    for (uint64_t i = 0; i < inv_off[n_kmers]; i++) h->d_inv_row.as<uint32_t>()[i] = inv_read[i] - 1;
    for (uint64_t i = 0; i < M; i++) { h->d_sel_key.as<uint64_t>()[i] = ((uint64_t) (sel_x[i] - 1) << 32) | (sel_y[i] - 1); h->d_sel_score.as<uint32_t>()[i] = sel_score[i]; }
    h->n_selected = M;
    if (pivot_flag) {                                            // --sc_score: the pairs come from a pivot subset
        if (h->d_pivot_flag.ensure(n_reads + 1)) return -1;
        std::memcpy(h->d_pivot_flag.p, pivot_flag, n_reads);
        h->pair_subset = true;
    }
    TailParams tail{read_off, amp, dims};
    const int rc = hga_enrich_run(h, min_size, max_size, min_score, with_tail ? &tail : nullptr);
    if (rc != HGA_OK) return rc;
    // what hga_get_core_kmers / hga_get_purged_index return (slot == kmer_id here)
    const uint64_t C = h->enrich.core_id.size();
    g_core_kmer.assign(h->n_core_kmers + 1, 0);
    for (uint64_t i = 0; i < h->n_core_kmers; i++) g_core_kmer[i] = (uint32_t) h->d_enr_keys.as<uint64_t>()[i];
    g_core_koff.assign(C + 1, 0);
    for (uint64_t c = 0; c <= C; c++) g_core_koff[c] = h->d_enr_core_koff.as<unsigned long long>()[c];
    return hga_export_index(h, h->d_purged_off.as<uint32_t>(), h->d_purged_row.as<uint32_t>(), h->n_purged, &g_purged);
}
extern "C" int emu_rerun(const uint64_t *read_off, int min_size, uint32_t min_score, uint32_t amp, int dims, int with_tail) {
    hga_handle *h = g_h;                                         // the SAME handle again (buffers, swapped purged arrays and all)
    TailParams tail{read_off, amp, dims};
    const int rc = hga_enrich_run(h, min_size, -1, min_score, with_tail ? &tail : nullptr);
    if (rc != HGA_OK) return rc;
    const uint64_t C = h->enrich.core_id.size();
    g_core_kmer.assign(h->n_core_kmers + 1, 0);
    for (uint64_t i = 0; i < h->n_core_kmers; i++) g_core_kmer[i] = (uint32_t) h->d_enr_keys.as<uint64_t>()[i];
    g_core_koff.assign(C + 1, 0);
    for (uint64_t c = 0; c <= C; c++) g_core_koff[c] = h->d_enr_core_koff.as<unsigned long long>()[c];
    return hga_export_index(h, h->d_purged_off.as<uint32_t>(), h->d_purged_row.as<uint32_t>(), h->n_purged, &g_purged);
}
struct EmuOut {
    uint64_t n_cores; const uint32_t *core_id; const uint64_t *core_off; const uint32_t *core_read; const uint64_t *core_koff; const uint32_t *core_kmer;
    uint64_t n_conn; const uint32_t *cx, *cy, *cs; uint64_t n_final; const uint32_t *final_id; const uint64_t *final_off; const uint32_t *final_read;
    uint64_t n_kmers; const uint64_t *purged_off; const uint32_t *purged_read; int ran; uint64_t n_scaffold_cores; uint64_t n_tconn; const uint32_t *tx, *ty; const uint64_t *ts;
    uint64_t n_clusters; const uint64_t *cl_off; const uint32_t *cl_member;
};
extern "C" void emu_out(EmuOut *o) {
    const EnrichResult &r = g_h->enrich;
    o->n_cores = r.core_id.size(); o->core_id = r.core_id.data(); o->core_off = r.core_off.data(); o->core_read = r.core_read.data();
    o->core_koff = g_core_koff.data(); o->core_kmer = g_core_kmer.data();
    o->n_conn = r.conn_x.size(); o->cx = r.conn_x.data(); o->cy = r.conn_y.data(); o->cs = r.conn_score.data();
    o->n_final = r.final_id.size(); o->final_id = r.final_id.data(); o->final_off = r.final_off.data(); o->final_read = r.final_read.data();
    o->n_kmers = g_purged.n_kmers; o->purged_off = g_purged.off; o->purged_read = g_purged.read_id;
    o->ran = r.tail_block_ran; o->n_scaffold_cores = r.n_scaffold_cores; o->n_tconn = r.tconn_x.size(); o->tx = r.tconn_x.data(); o->ty = r.tconn_y.data(); o->ts = r.tconn_score.data();
    o->n_clusters = r.cluster_off.empty() ? 0 : r.cluster_off.size() - 1; o->cl_off = r.cluster_off.data(); o->cl_member = r.cluster_member.data();
}
"""


class _EmuOut(C.Structure):
    _u32, _u64 = C.POINTER(C.c_uint32), C.POINTER(C.c_uint64)
    _fields_ = [("n_cores", C.c_uint64), ("core_id", _u32), ("core_off", _u64), ("core_read", _u32), ("core_koff", _u64), ("core_kmer", _u32),
                ("n_conn", C.c_uint64), ("cx", _u32), ("cy", _u32), ("cs", _u32), ("n_final", C.c_uint64), ("final_id", _u32), ("final_off", _u64), ("final_read", _u32),
                ("n_kmers", C.c_uint64), ("purged_off", _u64), ("purged_read", _u32), ("ran", C.c_int), ("n_scaffold_cores", C.c_uint64), ("n_tconn", C.c_uint64),
                ("tx", _u32), ("ty", _u32), ("ts", _u64), ("n_clusters", C.c_uint64), ("cl_off", _u64), ("cl_member", _u32)]


@pytest.fixture(scope="module")
def host_enrich(tmp_path_factory):
    internal = open(os.path.join(CSRC, "hga_internal.cuh")).read()
    internal = internal.replace("#include <cuda_runtime.h>\n", "").replace("#pragma once\n", "")
    if os.environ.get("HGA_EMU_ASAN"):
        # no allocation slack under the sanitizer: a kernel that writes one element past what was asked for must be seen
        assert "size_t want = bytes + (bytes >> 4) + 256;" in internal
        internal = internal.replace("size_t want = bytes + (bytes >> 4) + 256;", "size_t want = bytes;").replace("size_t want = bytes + 64;", "size_t want = bytes;")
    internal = internal.replace('#include "../../include/hga_b200.h"', '#include "hga_b200.h"')
    text = open(os.path.join(CSRC, "hga_enrich.cu")).read()
    text = re.sub(r'#include\s+"hga_internal.cuh"\n', "", text)
    text = re.sub(r"#include\s+<cub/[^>]+>\n", "", text)
    text = re.sub(r"<<<[^;]*?>>>", "", text)
    fake = FAKE_CUDA.replace("void hga_set_error(const char *fmt, ...) {", "void hga_set_error_unused(const char *fmt, ...) {")
    d = tmp_path_factory.mktemp("host_enrich")
    src, so = str(d / "enrich_host.cpp"), str(d / "enrich_host.so")
    open(src, "w").write(PRELUDE + "#include <string>\n" + fake + FAKE_CUDA_MORE + internal + text + EMU_HARNESS)
    err = str(d / "err.cpp")
    open(err, "w").write('#include <cstdarg>\n#include <cstdio>\nstatic char g[512];\nvoid hga_set_error(const char *fmt, ...) { va_list ap; va_start(ap, fmt); vsnprintf(g, sizeof g, fmt, ap); va_end(ap); }\n'
                         'extern "C" const char *emu_last_error() { return g; }\n')
    # HGA_EMU_ASAN=1 (with LD_PRELOAD=libasan.so): the emulated "device" buffers are malloc blocks, so AddressSanitizer sees every
    # out-of-bounds kernel access and every use of a reallocated buffer
    san = ["-fsanitize=address", "-fno-omit-frame-pointer"] if os.environ.get("HGA_EMU_ASAN") else []
    subprocess.run(["g++", "-std=c++17", "-O1", "-g", "-ffp-contract=off", "-fPIC", "-shared"] + san + ["-I", os.path.join(ROOT, "include"), "-o", so, src, err,
                    os.path.join(CSRC, "hga_tails.cpp"), os.path.join(CSRC, "hga_spectral.cpp")], check=True)
    lib = C.CDLL(so)
    lib.emu_last_error.restype = C.c_char_p
    return lib


def _emu_run(lib, oracle, c, with_tail, max_size=-1, sc_score=0):
    res = oracle.run(c["bases"], c["seq_off"], c["k"], c["kmers"], fraction=c["fraction"], min_size=c["min_size"], sc_score=sc_score)
    n = len(c["seq_off"]) - 1
    ro = res["row_off"].astype(np.int64)
    rows = np.repeat(np.arange(n), np.diff(ro))
    o = np.lexsort((res["hit_pos"], res["hit_kid"], rows))
    kid, pos = np.ascontiguousarray(res["hit_kid"][o], dtype=np.uint32), np.ascontiguousarray(res["hit_pos"][o], dtype=np.uint32)
    sx, sy, ss = res["conn"]
    m = res["cut_n"]
    lo, hi = np.minimum(sx[:m], sy[:m]).astype(np.uint64), np.maximum(sx[:m], sy[:m]).astype(np.uint64)
    key, first = np.unique((lo << np.uint64(32)) | hi, return_index=True)                    # unordered selected edges in (x, y) order
    sel_x, sel_y = (key >> np.uint64(32)).astype(np.uint32), (key & np.uint64(0xFFFFFFFF)).astype(np.uint32)
    sel_s = np.ascontiguousarray(ss[:m][first], dtype=np.uint32)
    row_off = np.ascontiguousarray(res["row_off"], dtype=np.uint64); inv_off = np.ascontiguousarray(res["inv_off"], dtype=np.uint64)
    inv_read = np.ascontiguousarray(res["inv_read"], dtype=np.uint32); read_off = np.ascontiguousarray(c["seq_off"], dtype=np.uint64)
    pivot = None
    if sc_score:
        pivot = np.ascontiguousarray(np.diff(res["row_off"].astype(np.int64)) >= sc_score, dtype=np.uint8)
    rc = lib.emu_enrich(C.c_uint64(n), C.c_uint64(len(c["kmers"])), _p(row_off), _p(kid), _p(pos), _p(inv_off), _p(inv_read), C.c_uint64(len(key)), _p(sel_x), _p(sel_y),
                        _p(sel_s), _p(read_off), c["min_size"], C.c_uint32(c["enrich"]), C.c_uint32(40), 16, int(with_tail), int(max_size), _p(pivot) if pivot is not None else None)
    assert rc == 0, lib.emu_last_error()
    return _emu_collect(lib)


def _emu_collect(lib):
    out = _EmuOut()
    lib.emu_out(C.byref(out))

    def arr(p, k, dt):
        return np.ctypeslib.as_array(p, shape=(max(int(k), 1),))[:int(k)].astype(dt) if k else np.zeros(0, dt)
    co = arr(out.core_off, out.n_cores + 1, np.int64); fo = arr(out.final_off, out.n_final + 1, np.int64); ko = arr(out.core_koff, out.n_cores + 1, np.int64)
    cr = arr(out.core_read, co[-1], np.uint32); fr = arr(out.final_read, fo[-1], np.uint32); ck = arr(out.core_kmer, ko[-1], np.uint32)
    po = arr(out.purged_off, out.n_kmers + 1, np.uint64)
    clo = arr(out.cl_off, out.n_clusters + 1, np.int64) if out.n_clusters else np.zeros(1, np.int64)
    clm = arr(out.cl_member, clo[-1], np.uint32)
    e = dict(core_id=arr(out.core_id, out.n_cores, np.uint32), core_kmers=[ck[ko[i]:ko[i + 1]] for i in range(len(ko) - 1)],
             core_reads=[cr[co[i]:co[i + 1]] for i in range(len(co) - 1)], purged_off=po, purged_read=arr(out.purged_read, po[-1], np.uint32),
             econn=(arr(out.cx, out.n_conn, np.uint32), arr(out.cy, out.n_conn, np.uint32), arr(out.cs, out.n_conn, np.uint64)),
             final_id=arr(out.final_id, out.n_final, np.uint32), final_reads=[fr[fo[i]:fo[i + 1]] for i in range(len(fo) - 1)])
    t = dict(ran=bool(out.ran), n_scaffold_cores=int(out.n_scaffold_cores), conn_x=arr(out.tx, out.n_tconn, np.uint32), conn_y=arr(out.ty, out.n_tconn, np.uint32),
             conn_score=arr(out.ts, out.n_tconn, np.uint64), clusters=[clm[clo[i]:clo[i + 1]] for i in range(len(clo) - 1)])
    return e, t


@pytest.mark.parametrize("name", ["enrich_short", "enrich_long"])
def test_enrich_run_on_host_without_the_block(host_enrich, oracle, name):
    """sanity of the emulation itself: the GPU-verified path (hga_enrich) reproduces the reference's golden dump when run this way"""
    import compare
    import golden_util
    c = golden_util.load_case(name)
    e, t = _emu_run(host_enrich, oracle, c, with_tail=False)
    compare.check_enrichment(c["ref"], e, c["kmers"])
    assert not t["ran"]


@pytest.mark.parametrize("name", ["full_short", "full_long"])
def test_enrich_full_on_host_matches_the_reference(host_enrich, oracle, name):
    """hga_enrich_full's own source, run on the host, against the real reference's --full dump: tail connections, clusters, state after
    the second merge, enrichment connections, final components"""
    import compare
    import golden_util
    c = golden_util.load_case(name)
    ref = c["ref"]
    e, t = _emu_run(host_enrich, oracle, c, with_tail=True)
    assert t["ran"] and t["n_scaffold_cores"] == ref["merged_scaffolds"]
    assert np.array_equal(t["conn_x"], ref["tconn_x"]) and np.array_equal(t["conn_y"], ref["tconn_y"]) and np.array_equal(t["conn_score"], ref["tconn_score"])
    so = ref["spectral_off"].astype(np.int64)
    want = [(ref["spectral_member"][so[i]:so[i + 1]].tolist(), int(ref["spectral_first"][i])) for i in range(len(so) - 1)]
    assert sorted((sorted(cl.tolist()), int(cl[0])) for cl in t["clusters"]) == want
    compare.check_enrichment(ref, e, c["kmers"])


LIVE_CASES = {
    "wrapping_k17": (dict(genome_size=80000, divergence=0.02, k=17, read_len=2500, coverage=12, seed=61, error_rate=0.04, length_sigma=0.5), 5),
    "short_k19": (dict(genome_size=40000, divergence=0.03, k=19, read_len=200, coverage=24, seed=77, error_rate=0.005, fmt="fastq"), 30),
    "long_k21": (dict(genome_size=60000, divergence=0.03, k=21, read_len=1800, coverage=12, seed=78, error_rate=0.02, length_sigma=0.4), 5),
}


@pytest.mark.parametrize("name", list(LIVE_CASES))
def test_enrich_full_on_host_live_against_the_reference(host_enrich, oracle, ref_driver, tmp_path, name):
    import compare
    import refdump
    kw, ms = LIVE_CASES[name]
    paths, kp = datagen.make_diploid_case(str(tmp_path), **kw)
    ref = refdump.run_ref(ref_driver, paths, kp, enrich=20, full=True, min_size=ms)
    assert ref["scaffold_components"] > 2
    rc, reads = oracle.load_reads(paths)
    kmers, k = oracle.load_kmers(kp)
    c = dict(bases=reads["seq"], seq_off=reads["seq_off"], k=k, kmers=kmers, fraction=0.15, min_size=ms, enrich=20)
    e, t = _emu_run(host_enrich, oracle, c, with_tail=True)
    assert np.array_equal(t["conn_x"], ref["tconn_x"]) and np.array_equal(t["conn_y"], ref["tconn_y"]) and np.array_equal(t["conn_score"], ref["tconn_score"])
    compare.check_enrichment(ref, e, kmers)


def test_enrich_full_on_host_with_a_size_limit(host_enrich, oracle, ref_driver, tmp_path):
    """--sc_max_size together with the tail / spectral block: the scaffold components and their spanning forest come from the sequential
    replay of ALL selected edges under the size limit (:457), more and smaller components reach the block"""
    import compare
    import refdump
    kw, ms = LIVE_CASES["long_k21"]
    paths, kp = datagen.make_diploid_case(str(tmp_path), **kw)
    ref = refdump.run_ref(ref_driver, paths, kp, enrich=20, full=True, min_size=ms, max_size=40)
    free = refdump.run_ref(ref_driver, paths, kp, enrich=20, full=True, min_size=ms, dump=False)
    assert ref["scaffold_components"] > free["scaffold_components"] > 2
    rc, reads = oracle.load_reads(paths)
    kmers, k = oracle.load_kmers(kp)
    c = dict(bases=reads["seq"], seq_off=reads["seq_off"], k=k, kmers=kmers, fraction=0.15, min_size=ms, enrich=20)
    e, t = _emu_run(host_enrich, oracle, c, with_tail=True, max_size=40)
    assert t["ran"] and t["n_scaffold_cores"] == ref["merged_scaffolds"]
    assert np.array_equal(t["conn_x"], ref["tconn_x"]) and np.array_equal(t["conn_y"], ref["tconn_y"]) and np.array_equal(t["conn_score"], ref["tconn_score"])
    compare.check_enrichment(ref, e, kmers)


def test_enrich_full_on_host_with_sc_score(host_enrich, oracle, ref_driver, tmp_path):
    """--sc_score S together with the block: connections from a pivot subset, kept when score > S (:749-752)"""
    import compare
    import refdump
    kw, ms = LIVE_CASES["long_k21"]
    paths, kp = datagen.make_diploid_case(str(tmp_path), **kw)
    ref = refdump.run_ref(ref_driver, paths, kp, enrich=20, full=True, min_size=ms, sc_score=350)
    assert ref["scaffold_components"] > 2
    rc, reads = oracle.load_reads(paths)
    kmers, k = oracle.load_kmers(kp)
    c = dict(bases=reads["seq"], seq_off=reads["seq_off"], k=k, kmers=kmers, fraction=0.15, min_size=ms, enrich=20)
    e, t = _emu_run(host_enrich, oracle, c, with_tail=True, sc_score=350)
    assert t["ran"] and t["n_scaffold_cores"] == ref["merged_scaffolds"]
    assert np.array_equal(t["conn_x"], ref["tconn_x"]) and np.array_equal(t["conn_y"], ref["tconn_y"]) and np.array_equal(t["conn_score"], ref["tconn_score"])
    compare.check_enrichment(ref, e, kmers)


def test_enrich_on_host_same_handle_again(host_enrich, oracle):
    """full -> plain -> full on ONE handle: the buffers a run leaves behind (the swapped purged arrays, the survivor table with its
    second half, the relabelled unions) do not leak into the next run"""
    import compare
    import golden_util
    c = golden_util.load_case("full_long")
    e1, t1 = _emu_run(host_enrich, oracle, c, with_tail=True)
    read_off = np.ascontiguousarray(c["seq_off"], dtype=np.uint64)
    assert host_enrich.emu_rerun(_p(read_off), c["min_size"], C.c_uint32(c["enrich"]), C.c_uint32(40), 16, 0) == 0, host_enrich.emu_last_error()
    e2, t2 = _emu_collect(host_enrich)
    assert not t2["ran"] and len(e2["core_id"]) == c["ref"]["merged_scaffolds"] > len(e1["core_id"])
    assert host_enrich.emu_rerun(_p(read_off), c["min_size"], C.c_uint32(c["enrich"]), C.c_uint32(40), 16, 1) == 0, host_enrich.emu_last_error()
    e3, t3 = _emu_collect(host_enrich)
    compare.check_enrichment(c["ref"], e3, c["kmers"])
    assert t3["ran"] and all(np.array_equal(a, b) for a, b in zip(t1["clusters"], t3["clusters"]))


# ---- the k-mer table build (csrc/hga_table.cu) on the host --------------------------------------------------------------------------
# The table layout is a function of the k-mer array (bucket sort, one thread per bucket, sorted overflow region); the scan's lookup relies on three
# invariants nothing checks at run time: (i) a key sits in its home bucket and every SECTOR between its start sector and its own sector (going round the
# bucket) is full, so a lookup that goes sector by sector and stops at a sector with an empty slot never stops early; (ii) a key that is not in its
# bucket sits in the overflow region, which is sorted (bisection); (iii) the filter word of every key has the key's bits set.
TABLE_HARNESS = r"""
extern "C" int emu_table(int k, const uint64_t *kmers, uint64_t n, double load, uint64_t *stats) {
    static hga_handle hh;
    hga_handle *h = &hh;
    h->k = k; h->n_kmers = n; h->sm_count = 2; h->stream = nullptr;
    char buf[32];
    snprintf(buf, sizeof buf, "%g", load);
    if (load > 0) setenv("HGA_TABLE_LOAD", buf, 1); else unsetenv("HGA_TABLE_LOAD");
    int rc = hga_table_build(h, kmers);
    unsetenv("HGA_TABLE_LOAD");
    if (rc != HGA_OK) return rc;
    const KmerTable &t = h->table;
    uint64_t in_main = 0, in_over = 0, bad = 0;
    for (uint64_t i = 0; i < n; i++) {
        const uint64_t key = kmers[i];
        const uint32_t s = t.kid_slot[i];
        if (s >= t.n_slots || t.keys[s] != key || t.slot_kid[s] != (uint32_t) i) { bad |= 1; continue; }
        const uint32_t hb = hga_bits_hash(key, t.geom);
        const uint32_t B = hga_locality_from_min(hga_minimizer(key, hb, t.geom));
        if ((t.filter[(size_t) hga_scale(B, t.n_blocks) * 8 + hga_bits_word(hb)] & hga_bits_mask(hb)) != hga_bits_mask(hb)) bad |= 2;
        const uint32_t home = hga_scale(B, t.n_buckets) * HGA_BUCKET_SLOTS, start_sec = hga_start_sector(hb);
        const uint32_t n_sec = HGA_BUCKET_SLOTS / HGA_SECTOR_SLOTS;
        if (s < t.n_main) {
            in_main++;
            if (s / HGA_BUCKET_SLOTS != home / HGA_BUCKET_SLOTS) { bad |= 4; continue; }
            const uint32_t my_sec = (s - home) / HGA_SECTOR_SLOTS;
            for (uint32_t step = 0; (start_sec + step) % n_sec != my_sec; step++)            // every sector before the key's own is full
                for (uint32_t j = 0; j < HGA_SECTOR_SLOTS; j++)
                    if (t.keys[home + ((start_sec + step) % n_sec) * HGA_SECTOR_SLOTS + j] == HGA_EMPTY_KEY) bad |= 8;
        } else {
            in_over++;
            for (uint32_t j = 0; j < HGA_BUCKET_SLOTS; j++) if (t.keys[home + j] == HGA_EMPTY_KEY) bad |= 16;   // its bucket is full
            const uint32_t q = s - t.n_main;
            if (q >= t.n_over_keys) bad |= 32;
        }
    }
    for (uint32_t q = 1; q < t.n_over_keys; q++) if (t.keys[t.n_main + q - 1] >= t.keys[t.n_main + q]) bad |= 64;   // sorted, no duplicates
    for (uint32_t q = t.n_over_keys; q < t.n_over; q++) if (t.keys[t.n_main + q] != HGA_EMPTY_KEY) bad |= 128;
    uint64_t used = 0;
    for (uint32_t s = 0; s < t.n_slots; s++) used += t.keys[s] != HGA_EMPTY_KEY;
    if (used != n) bad |= 256;
    if (t.n_slots % HGA_BUCKET_SLOTS) bad |= 512;
    stats[0] = in_main; stats[1] = in_over; stats[2] = bad; stats[3] = t.n_slots; stats[4] = t.n_over_keys;
    return HGA_OK;
}
"""


@pytest.fixture(scope="module")
def host_table(tmp_path_factory):
    internal = open(os.path.join(CSRC, "hga_internal.cuh")).read()
    internal = internal.replace("#include <cuda_runtime.h>\n", "").replace("#pragma once\n", "")
    internal = internal.replace('#include "../../include/hga_b200.h"', '#include "hga_b200.h"')
    text = open(os.path.join(CSRC, "hga_table.cu")).read()
    text = re.sub(r'#include\s+"hga_internal.cuh"\n', "", text)
    text = re.sub(r"#include\s+<cub/[^>]+>\n", "", text)
    text = re.sub(r"<<<[^;]*?>>>", "", text)
    fake = FAKE_CUDA.replace("void hga_set_error(const char *fmt, ...) {", "void hga_set_error_unused(const char *fmt, ...) {")
    more = FAKE_CUDA_MORE + r"""
static inline unsigned atomicOr(unsigned *p, unsigned v) { unsigned o = *p; *p |= v; return o; }
static inline int atomicOr(int *p, int v) { int o = *p; *p |= v; return o; }
static inline unsigned atomicAdd(unsigned *p, unsigned v) { unsigned o = *p; *p += v; return o; }
"""
    d = tmp_path_factory.mktemp("host_table")
    src, so = str(d / "table_host.cpp"), str(d / "table_host.so")
    open(src, "w").write(PRELUDE + "#include <string>\n" + fake + more + internal + text + TABLE_HARNESS)
    err = str(d / "err.cpp")
    open(err, "w").write('#include <cstdarg>\n#include <cstdio>\nstatic char g[512];\nvoid hga_set_error(const char *fmt, ...) { va_list ap; va_start(ap, fmt); vsnprintf(g, sizeof g, fmt, ap); va_end(ap); }\n'
                         'extern "C" const char *emu_last_error() { return g; }\n')
    subprocess.run(["g++", "-std=c++17", "-O1", "-g", "-fPIC", "-shared", "-I", os.path.join(ROOT, "include"), "-o", so, src, err], check=True)
    lib = C.CDLL(so)
    lib.emu_last_error.restype = C.c_char_p
    return lib


@pytest.mark.parametrize("k,load", [(19, 0.0), (19, 0.9), (15, 0.9), (31, 0.9), (8, 0.0)])
def test_table_layout_and_filter_invariants_on_host(host_table, k, load):
    """load 0.9 (HGA_TABLE_LOAD) fills buckets, so that start sectors wrap round, sectors fill up and keys spill into the overflow region"""
    g1 = datagen.random_genome(60000, 600 + k)
    g2 = datagen.mutate(g1, 0.03, 700 + k)
    kmers = np.ascontiguousarray(datagen.discriminative_kmers([g1, g2], k), dtype=np.uint64)
    assert len(kmers) > 100
    stats = np.zeros(8, dtype=np.uint64)
    try:
        rc = host_table.emu_table(k, _p(kmers), C.c_uint64(len(kmers)), C.c_double(load), _p(stats))
    finally:
        os.environ.pop("HGA_TABLE_LOAD", None)
    assert rc == 0, host_table.emu_last_error()
    assert int(stats[2]) == 0, f"table invariants violated (bit mask {int(stats[2])})"
    assert int(stats[0]) + int(stats[1]) == len(kmers)
    if load >= 0.9 and k >= 15:
        assert int(stats[1]) > 0, "the dense table was meant to exercise the overflow region"
