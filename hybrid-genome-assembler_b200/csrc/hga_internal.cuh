// Internal declarations shared by the CUDA translation units of libhga_b200.so (sm_100a only).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include <cstdarg>
#include <cstdlib>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

#include "../../include/hga_b200.h"

// ------------------------------------------------------------------------------------------------
// error plumbing
// ------------------------------------------------------------------------------------------------
void hga_set_error(const char *fmt, ...);

#define HGA_CUDA(call)                                                                                          \
    do {                                                                                                        \
        cudaError_t _e = (call);                                                                                \
        if (_e != cudaSuccess) {                                                                                \
            hga_set_error("%s:%d: %s failed: %s", __FILE__, __LINE__, #call, cudaGetErrorString(_e));           \
            return HGA_E_CUDA;                                                                                  \
        }                                                                                                       \
    } while (0)

#define HGA_TRY(call)                   \
    do {                                \
        int _rc = (call);               \
        if (_rc != HGA_OK) return _rc;  \
    } while (0)

// ------------------------------------------------------------------------------------------------
// device / pinned buffers that only grow
// ------------------------------------------------------------------------------------------------
struct DevBuf {
    void *p = nullptr;
    size_t cap = 0;
    int ensure(size_t bytes) {
        if (bytes <= cap) return HGA_OK;
        if (p) cudaFree(p);
        p = nullptr; cap = 0;
        size_t want = bytes + (bytes >> 4) + 256;   // a little slack so repeated runs do not realloc
        cudaError_t e = cudaMalloc(&p, want);
        if (e != cudaSuccess) {
            hga_set_error("cudaMalloc(%zu) failed: %s", want, cudaGetErrorString(e));
            cudaGetLastError();
            return HGA_E_NOMEM;
        }
        cap = want;
        return HGA_OK;
    }
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
    template<typename T> T *as() const { return reinterpret_cast<T *>(p); }
};

struct PinBuf {
    void *p = nullptr;
    size_t cap = 0;
    int ensure(size_t bytes) {
        if (bytes <= cap) return HGA_OK;
        if (p) cudaFreeHost(p);
        p = nullptr; cap = 0;
        size_t want = bytes + 64;
        cudaError_t e = cudaMallocHost(&p, want);
        if (e != cudaSuccess) {
            hga_set_error("cudaMallocHost(%zu) failed: %s", want, cudaGetErrorString(e));
            cudaGetLastError();
            return HGA_E_NOMEM;
        }
        cap = want;
        return HGA_OK;
    }
    void release() { if (p) cudaFreeHost(p); p = nullptr; cap = 0; }
    template<typename T> T *as() const { return reinterpret_cast<T *>(p); }
};

// ------------------------------------------------------------------------------------------------
// k-mer membership structures (device)
//
// Everything the scan computes per window is STRAND SYMMETRIC and needs neither the canonical k-mer value nor a 64-bit
// compare: with F the forward k-mer and R its reverse complement,
//   bit hash   hb(x) = g(F) + g(R),  g(v) = (hi(v) * ca + lo(v)) * cb   (ca / cb shift the bits above the k-mer out, so the scan
//              feeds raw 32-bit pieces of its packed streams)
//   minimizer  Mc(x) = min over ALL m-mers of the k-mer of min(h(m-mer), h(revcomp m-mer)),  h(y) = y * cm + C4
// Runs of ~(W + 1) / 2 consecutive windows of a read share Mc (W = k - m + 1 m-mers per window), so their filter probes fall into
// the same 32 B block and coalesce inside a warp, and their keys share a 128 B bucket. m is chosen from the size of the set
// (4^m / 2 >= 3 n: unrelated loci must not share a minimizer VALUE) with W <= HGA_MIN_W; when k leaves no room for that
// (k < HGA_MIN_K_FOR_MIN, or k - 16 + 1 > HGA_MIN_W) a mix of hb takes Mc's place (no locality, still correct).
//
//   filter    : blocked Bloom filter over the canonical keys; block = 32 B (8 words) selected by Mc, word + 3 bits inside the
//               block selected by hb. Sized to stay L2 resident: measured on B200 (profiles/r2c), a filter of <= 48 MB is served
//               from L2 while 10 Gbases stream through, 64 MB is not (26.9 -> 37.6 -> 59.2 ms at 48 / 64 / 96 MB).
//   key table : canonical keys, u64, buckets of 32 (256 B) selected by Mc. Inside the bucket a key starts at the 32 B SECTOR
//               picked by hb and goes round the bucket's eight sectors; a lookup reads one sector per step (one 256-bit load)
//               and stops at a match or at a sector with an empty slot: 96 % of the lookups end in the first step (load 1/4).
//               Keys that find their bucket full (0.1 %) go to the overflow region, a sorted array searched by bisection,
//               consulted only after eight full sectors. The layout is a function of the k-mer array (hga_table.cu): no insertion races. The internal k-mer id ("slot") is the index of the key in the
//               (main | overflow) array; slot_kid maps it to the caller's id.
// ------------------------------------------------------------------------------------------------
#define HGA_MIN_W 8
#define HGA_MIN_K_FOR_MIN 12
#define HGA_BUCKET_SLOTS 32      // two 128 B lines of u64 keys
#define HGA_SECTOR_SLOTS 4       // one 32 B sector

struct KmerGeom {
    int k = 0;
    int use_min = 0;      // 1: locality from the minimizer, 0: from the bit hash
    int m = 0;            // m-mer length (<= 16)
    int W = 0;            // m-mers per window = k - m + 1 (2 .. HGA_MIN_W)
    uint32_t cm = 0;      // HGA_C1 << (32 - 2m)
    uint32_t mtop = 0;    // the top 2m bits of a word
    uint32_t ca = 0, cb = 0;   // g(v) = (hi * ca + lo) * cb
};

struct KmerTable {
    uint64_t *keys = nullptr;       // n_slots (main region, then overflow region)
    uint32_t *slot_kid = nullptr;   // n_slots
    uint32_t *kid_slot = nullptr;   // n_kmers
    uint32_t *filter = nullptr;     // n_blocks * 8 words
    uint32_t n_buckets = 0;         // main region: n_buckets * HGA_BUCKET_SLOTS slots
    uint32_t n_main = 0;            // slots in the main region
    uint32_t n_over = 0;            // slots in the overflow region (0: none; else a multiple of HGA_BUCKET_SLOTS)
    uint32_t n_over_keys = 0;       // keys in the overflow region: a SORTED array (binary search), HGA_EMPTY_KEY padding behind it
    uint32_t n_blocks = 0;
    uint32_t n_slots = 0;           // n_main + n_over
    uint32_t slot_bits = 0;         // ceil(log2(n_slots))
    KmerGeom geom;
};

#define HGA_EMPTY_KEY 0xFFFFFFFFFFFFFFFFull
#define HGA_C1 0x9E3779B1u
#define HGA_C2 0x85EBCA77u
#define HGA_C3 0xC2B2AE3Du
#define HGA_C4 0x27D4EB2Fu

static inline KmerGeom hga_make_geom(int k, uint64_t n_kmers) {
    KmerGeom g;
    g.k = k;
    if (k > 16) { g.ca = HGA_C3 << (64 - 2 * k); g.cb = HGA_C1; }
    else { g.ca = 0; g.cb = HGA_C1 << (32 - 2 * k); }
    if (k < HGA_MIN_K_FOR_MIN || k - 16 + 1 > HGA_MIN_W) return g;
    g.use_min = 1;
    int m = 4;
    while (m < 16 && (1ull << (2 * m - 1)) < 3 * n_kmers) m++;      // 4^m / 2 >= 3 n
    if (m < k - HGA_MIN_W + 1) m = k - HGA_MIN_W + 1;                // W <= HGA_MIN_W
    if (m > 16) m = 16;
    if (m > k - 1) m = k - 1;                                         // W >= 2
    g.m = m; g.W = k - m + 1;
    g.cm = HGA_C1 << (32 - 2 * m);
    g.mtop = m == 16 ? 0xFFFFFFFFu : ~(0xFFFFFFFFu >> (2 * m));
    return g;
}

__host__ __device__ __forceinline__ uint32_t hga_scale(uint32_t h, uint32_t n) {
#ifdef __CUDA_ARCH__
    return __umulhi(h, n);
#else
    return (uint32_t) (((uint64_t) h * n) >> 32);
#endif
}

// reverse complement of a k-mer held in the low 2k bits (codes A0 C1 G2 T3)
__host__ __device__ __forceinline__ uint64_t hga_revcomp64(uint64_t x, int k) {
#ifdef __CUDA_ARCH__
    x = __brevll(x);
#else
    x = ((x >> 1) & 0x5555555555555555ull) | ((x & 0x5555555555555555ull) << 1);
    x = ((x >> 2) & 0x3333333333333333ull) | ((x & 0x3333333333333333ull) << 2);
    x = ((x >> 4) & 0x0F0F0F0F0F0F0F0Full) | ((x & 0x0F0F0F0F0F0F0F0Full) << 4);
    x = ((x >> 8) & 0x00FF00FF00FF00FFull) | ((x & 0x00FF00FF00FF00FFull) << 8);
    x = ((x >> 16) & 0x0000FFFF0000FFFFull) | ((x & 0x0000FFFF0000FFFFull) << 16);
    x = (x >> 32) | (x << 32);
#endif
    x = ((x >> 1) & 0x5555555555555555ull) | ((x & 0x5555555555555555ull) << 1);   // bits reversed -> 2-bit groups reversed
    return (~x) >> (64 - 2 * k);
}

// one strand's share of the bit hash: v = an oriented k-mer value
__host__ __device__ __forceinline__ uint32_t hga_strand_hash(uint32_t hi, uint32_t lo, const KmerGeom &g) { return (hi * g.ca + lo) * g.cb; }
// strand-symmetric hash of the k-mer x (either orientation): picks the word and the two bits inside a filter block and the
// start sector inside a key bucket
__host__ __device__ __forceinline__ uint32_t hga_bits_hash(uint64_t x, const KmerGeom &g) {
    const uint64_t r = hga_revcomp64(x, g.k);
    return hga_strand_hash((uint32_t) (x >> 32), (uint32_t) x, g) + hga_strand_hash((uint32_t) (r >> 32), (uint32_t) r, g);
}
__host__ __device__ __forceinline__ uint32_t hga_bits_word(uint32_t h) { return h >> 29; }
// the three bit positions a key sets inside its filter word (3 bits: 9.1 % of the windows of config 4 pass the 48 MB filter, 2 bits: 10.0 %)
// come from the HIGH half of hb * C2: its low bits are well mixed, so a wrapping shift takes a bit position straight from the register (no
// mask is ever built by the scan)
__host__ __device__ __forceinline__ uint32_t hga_bits_pos(uint32_t hb) { return hga_scale(hb, HGA_C2); }
__host__ __device__ __forceinline__ uint32_t hga_bits_mask(uint32_t hb) {
    const uint32_t v = hga_bits_pos(hb);
    return (1u << (v & 31)) | (1u << ((v >> 5) & 31)) | (1u << ((v >> 10) & 31));
}
#ifdef __CUDACC__
__device__ __forceinline__ bool hga_bits_test(uint32_t word, uint32_t hb) {
    const uint32_t v = hga_bits_pos(hb);
    return (__funnelshift_r(word, 0u, v) & __funnelshift_r(word, 0u, v >> 5) & __funnelshift_r(word, 0u, v >> 10) & 1u) != 0;
}
#endif
// start sector of a key inside its bucket, from the bit hash: keys spread evenly, 95 % of the lookups end in their first sector
__host__ __device__ __forceinline__ uint32_t hga_start_sector(uint32_t hb) { return (hb >> 16) & (HGA_BUCKET_SLOTS / HGA_SECTOR_SLOTS - 1); }
// when there is no minimizer: the locality value is a mix of the bit hash
__host__ __device__ __forceinline__ uint32_t hga_mix_bits(uint32_t hb) { return (hb ^ (hb >> 15)) * HGA_C3; }

// multi-GPU partition of the table slots (and with them of the inverted lists): whole 32-slot buckets round robin, so that the hits of
// a minimizer run keep neighbouring list numbers at their owner (the locality the pair counter's list walks live on)
__host__ __device__ __forceinline__ uint32_t hga_owner_of_slot(uint32_t slot, uint32_t G) { return (slot / HGA_BUCKET_SLOTS) % G; }
__host__ __device__ __forceinline__ uint32_t hga_list_of_slot(uint32_t slot, uint32_t G) { return (slot / HGA_BUCKET_SLOTS) / G * HGA_BUCKET_SLOTS + slot % HGA_BUCKET_SLOTS; }

// hashed m-mer: x = any word whose LOW 2m bits are the m-mer (cm shifts the rest out)
__host__ __device__ __forceinline__ uint32_t hga_mmer_hash(uint32_t x, uint32_t cm) { return x * cm + HGA_C4; }

// Mc from the k-mer VALUE (table build; scan windows that contain a non-ACGT byte, whose two strands are not reverse
// complements of each other). x and its reverse complement give the same result.
__host__ __device__ __forceinline__ uint32_t hga_minimizer(uint64_t x, uint32_t hb, const KmerGeom &g) {
    if (!g.use_min) return hga_mix_bits(hb);
    const uint64_t r = hga_revcomp64(x, g.k);
    uint32_t mn = 0xFFFFFFFFu;
    for (int o = 0; o < g.W; o++) {
        const uint32_t hf = hga_mmer_hash((uint32_t) (x >> (2 * o)), g.cm), hr = hga_mmer_hash((uint32_t) (r >> (2 * o)), g.cm);
        const uint32_t h = hf < hr ? hf : hr;
        mn = h < mn ? h : mn;
    }
    return mn;
}
// the minimum of W hashes is biased towards small values; the multiply carries its low bits up into the bits hga_scale uses
__host__ __device__ __forceinline__ uint32_t hga_locality_from_min(uint32_t mn) { return mn * HGA_C2; }

// ------------------------------------------------------------------------------------------------
// the handle
// ------------------------------------------------------------------------------------------------
struct hga_comm;   // NCCL state, hga_comm.cu

// host-side result of hga_enrich (small: cores, enrichment connections, final membership)
struct EnrichResult {
    std::vector<uint32_t> core_id, core_read;           // survivor ids ascending; members ascending inside a core
    std::vector<uint64_t> core_off;
    std::vector<uint32_t> conn_x, conn_y, conn_score;   // directed (core survivor -> partner), canonical order
    std::vector<uint32_t> final_id, final_read, assignment;
    std::vector<uint64_t> final_off;
    // tail / spectral block (hga_enrich_full): what it saw and what it merged
    bool tail_block_ran = false;                        // more than two scaffold components (:768)
    uint64_t n_scaffold_cores = 0;                      // cores before the merge of the spectral clusters
    std::vector<uint32_t> tconn_x, tconn_y;             // tail connections, x < y, canonical order (all, not only score > 5)
    std::vector<uint64_t> tconn_score;
    std::vector<uint32_t> cluster_member;               // spectral clusters, element [0] of a cluster = the surviving id; empty clusters dropped
    std::vector<uint64_t> cluster_off;
};

// hga_enrich_full: the parameters of the tail / spectral block (:768-777)
struct TailParams {
    const uint64_t *read_off;       // HOST, n_reads + 1, as given to hga_scan
    uint32_t amplification_min_score;
    int spectral_dims;
};

struct hga_handle {
    int device = 0;
    int k = 0;
    uint64_t n_kmers = 0;
    cudaStream_t own_stream = nullptr;
    cudaStream_t copy_stream = nullptr;   // H2D of the bases, overlapped with the scan (hga_scan)
    cudaStream_t stream = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr, ev2 = nullptr, ev3 = nullptr;   // stage timer, nested (exchange) timer
    int sm_count = 148;

    // table
    KmerTable table;
    DevBuf d_keys, d_slot_kid, d_kid_slot, d_filter;

    // scan results (rows = reads of this rank's shard)
    uint64_t n_reads = 0, n_bases = 0, n_hits = 0;
    uint32_t read_id_base = 1;
    DevBuf d_bases, d_read_off;           // staging for hga_scan (host entry)
    DevBuf d_row_off;                     // u64[n_reads+1]
    DevBuf d_hit_slot, d_hit_pos;         // u32[E]
    DevBuf d_pos_tmp;                     // positions in tile-completion order until hga_get_hits moves them (hga_scan_finish_positions)
    uint64_t scan_tiles = 0;
    double scan_density = 0;              // hits per base of the previous scan on this handle (sizes the next one's hit buffers)
    bool pos_pending = false;
    DevBuf d_tile_state, d_tile_dir, d_scan_scalars;
    DevBuf d_exc, d_exc_dir;              // packed scans: exception runs (host entry: starts then ends), first run touching each tile
    bool have_scan = false;

    // row space of the inverted index, pairs and components (this GPU's reads; ALL reads with a communicator)
    uint64_t inc_rows = 0;                // number of rows
    uint32_t inc_row_first_id = 1;        // read id of row 0
    uint64_t inc_entries = 0;             // entries of the inverted index
    DevBuf d_x_slot, d_x_row;             // exchange staging (multi-GPU)
    DevBuf d_g_kid, d_g_row_off;          // multi-GPU: by-row incidence of ALL rows restricted to this rank's k-mers (list number per hit, u64 row offsets)
    bool index_by_kid = false;            // multi-GPU (name kept): the inverted index holds the lists of this rank's share of the table: slot s belongs to
                                          // rank (s / 32) mod G and is list ((s / 32) / G) * 32 + s mod 32 there (hga_owner_of_slot / hga_list_of_slot)
    uint32_t index_keys = 0;              // number of lists in the inverted index: n_slots, or the owner's share of them with a communicator

    // inverted index
    DevBuf d_inv_off;                     // u32[index_keys + 1] (the incidence held by one GPU has < 2^32 entries)
    DevBuf d_inv_row;                     // u32[inc_entries]: ROW numbers (0-based), ascending inside a list
    DevBuf d_sort_a, d_sort_b, d_sort_tmp;
    DevBuf d_index_tmp, d_index_goff;     // rows sorted by slot group, group offsets (index_local_sort_kernel)
    bool have_index = false;

    // pairs
    uint64_t n_pairs = 0, n_increments = 0;
    DevBuf d_pair_key, d_pair_score;      // u64 key = (x_row << 32 | y_row), u32 score; sorted by key
    DevBuf d_pair_key2, d_pair_score2, d_pair_scalars, d_heavy_list, d_mid_list, d_redo_list, d_heavy_tab, d_pivot_flag, d_pivot_order, d_pivot_rows;
    uint64_t pair_capacity = 0;
    uint64_t pair_rows = 0;               // rows of the by-read incidence the pair counter walks (this rank's pivots with a communicator)
    uint32_t pair_pivot_mul = 1, pair_pivot_add = 0;   // local row t is global row t * mul + add (rank, rank + G, ...)
    bool have_pairs = false;
    uint32_t pair_min_score = 1;
    bool pair_subset = false;             // the pairs come from a pivot subset (d_pivot_flag marks the pivots)

    // selection
    uint64_t sel_n_directed = 0, sel_cut = 0, n_selected = 0;
    DevBuf d_hist, d_sel_key, d_sel_score, d_sel_scalars;
    bool have_selection = false;

    // components
    DevBuf d_parent, d_comp_size, d_comp_label, d_comp_scalars;
    uint64_t n_components = 0;
    bool have_components = false;

    // merge + enrichment (hga_enrich.cu)
    DevBuf d_enr_parent, d_enr_core_of, d_enr_surv, d_enr_R, d_enr_scalars, d_enr_keys, d_enr_keys2, d_enr_core_koff, d_purged_off, d_purged_row;
    DevBuf d_purged2_off, d_purged2_row;  // second purge (merge of the spectral clusters); swapped into d_purged_* when it ran
    uint64_t n_purged = 0, n_core_kmers = 0;
    EnrichResult enrich;
    bool have_enrichment = false;

    // host mirrors for hga_get_*
    PinBuf h_row_off, h_kid, h_pos, h_inv_off, h_inv_read, h_px, h_py, h_ps, h_sx, h_sy, h_ss, h_label, h_clabel, h_csize, h_scalars;
    DevBuf d_export_a, d_export_b, d_export_c;

    hga_metrics_t metrics;
    hga_comm *comm = nullptr;
    hga_comm *comm_parked = nullptr;      // rank 0 after hga_comm_gather_root: the communicator, detached (destroyed with the handle)
    uint64_t n_reads_total = 0;           // over all ranks (== n_reads without a comm)
};

// stage launchers (each in its own .cu)
int hga_table_build(hga_handle *h, const uint64_t *host_kmers);
// A packed scan (hga_scan_packed*): d_bases / h_bases point at the byte that holds the first base, `sub` bases into it (0..3).
struct ScanPackedInput {
    uint32_t sub;
    const uint64_t *d_exc_start, *d_exc_end;  // device, n_exc each (the host entry's runs are copied there first: h_exc_* != nullptr)
    const uint64_t *h_exc_start, *h_exc_end;
    uint64_t n_exc;
};
// h_bases != nullptr: the bases are still on the host; the run copies them (in chunks, overlapped with the scan when large)
// packed == nullptr: ASCII bases, one byte each
// check != nullptr: a device entry of that name; its read lengths (and, packed, read_off[0] and the runs) are checked on the GPU and a violation
// fails with HGA_E_ARG (the host entries check their input before they call this)
int hga_scan_run(hga_handle *h, const char *d_bases, const uint64_t *d_read_off, uint64_t n_reads, uint64_t n_bases, const char *h_bases,
                 const ScanPackedInput *packed = nullptr, const char *check = nullptr);
int hga_scan_finish_positions(hga_handle *h);
// the k-mer count behind hga_count_kmers[_packed] and hga_count_spectrum[_packed] (csrc/hga_count.cu), arguments already checked.
// packed == nullptr: ASCII `bases`, read set bases[read_off[0] .. read_off[n_reads]). Otherwise the case-folded packing, bases
// first_base + read_off[0 .. n_reads] (read_off[0] == 0) and the exception runs relative to first_base.
// spec == nullptr: the counts >= min_count into *out. Otherwise the spectrum is ADDED to *spec and hist[0 .. n_bins) (zeroed by the caller).
int hga_count_run(const char *who, int device, int k, const char *bases, const uint8_t *packed, uint64_t first_base, const uint64_t *read_off,
                  uint64_t n_reads, const uint64_t *exc_start, const uint64_t *exc_end, uint64_t n_exc, uint32_t min_count, hga_kmer_counts_t *out,
                  hga_kmer_spectrum_t *spec, uint32_t n_bins, uint64_t *hist);
int hga_sdk_run(const char *who, int device, int k, const uint8_t *packed, uint64_t first_base, const uint64_t *read_off, uint64_t n_reads,
                const uint64_t *exc_start, const uint64_t *exc_end, uint64_t n_exc, int n_files, const uint64_t *file_first, uint32_t min_count, hga_sdk **out);
int hga_index_run(hga_handle *h);
int hga_build_lists(hga_handle *h, const uint32_t *d_keys, const uint64_t *d_row_off, uint64_t n_rows, uint64_t E, uint32_t n_keys);
int hga_pairs_run(hga_handle *h, uint32_t min_score, const uint32_t *pivots, uint64_t n_pivots);
int hga_select_run(hga_handle *h, double fraction, uint32_t score_threshold);
int hga_cc_run(hga_handle *h, int min_size);
// tail == nullptr: without the tail / spectral block (hga_enrich, hga_enrich_ex)
int hga_enrich_run(hga_handle *h, int min_size, int max_size, uint32_t min_score, const TailParams *tail);
// CSR by index key (off u32[keys + 1], rows) -> CSR by the caller's kmer_id with read ids, in the pinned export buffers (hga_capi.cu)
int hga_export_index(hga_handle *h, const uint32_t *d_off, const uint32_t *d_row, uint64_t E, hga_index *out);

// multi-GPU hooks (hga_comm.cu); all are no-ops / never called without a communicator
int hga_comm_build_owner_index(hga_handle *h);
int hga_comm_exchange_partials(hga_handle *h, uint64_t n, uint64_t *out_n);
int hga_comm_reduce_partials_packed(hga_handle *h, uint64_t n, uint64_t *out_n, bool *reduced);
int hga_comm_allgather_u64(hga_handle *h, uint64_t mine, std::vector<uint64_t> &all);
int hga_comm_allgatherv(hga_handle *h, const void *d_mine, void *d_all, const std::vector<uint64_t> &counts, int elem_bytes);
int hga_comm_allreduce_u64_sum(hga_handle *h, uint64_t *d_buf, size_t n);
int hga_comm_allreduce_u32_min(hga_handle *h, uint32_t *d_buf, size_t n);
int hga_comm_allreduce_u32_max(hga_handle *h, uint32_t *d_buf, size_t n);
int hga_comm_rank(const hga_handle *h);
int hga_comm_size(const hga_handle *h);
void hga_comm_destroy(hga_handle *h);

static inline uint32_t hga_ceil_log2(uint64_t n) {
    uint32_t b = 0;
    while (b < 63 && (1ull << b) < n) b++;
    return b;
}

struct StageTimer {
    hga_handle *h;
    double *slot;
    cudaEvent_t a, b;
    StageTimer(hga_handle *hh, double *s, bool nested = false) : h(hh), slot(s), a(nested ? hh->ev2 : hh->ev0), b(nested ? hh->ev3 : hh->ev1) {
        cudaEventRecord(a, h->stream);
    }
    void stop() {
        cudaEventRecord(b, h->stream);
        cudaEventSynchronize(b);
        float ms = 0.f;
        cudaEventElapsedTime(&ms, a, b);
        *slot = ms;
    }
};

// HGA_TRACE=1: sub-stage times on stderr (CUDA events on the stage's stream; the dump synchronises, so a traced run is for reading,
// not for quoting)
struct Trace {
    bool on;
    cudaStream_t s;
    std::vector<std::pair<const char *, cudaEvent_t>> ev;
    explicit Trace(hga_handle *h) : on(getenv("HGA_TRACE") != nullptr), s(h->stream) { mark("begin"); }
    void mark(const char *name) {
        if (!on) return;
        cudaEvent_t e;
        cudaEventCreate(&e);
        cudaEventRecord(e, s);
        ev.emplace_back(name, e);
    }
    void dump(const char *stage, int rank) {
        if (!on || ev.empty()) return;
        cudaEventSynchronize(ev.back().second);
        std::string line = "[hga trace r" + std::to_string(rank) + " " + stage + "]";
        for (size_t i = 1; i < ev.size(); i++) {
            float ms = 0.f;
            cudaEventElapsedTime(&ms, ev[i - 1].second, ev[i].second);
            char buf[96];
            snprintf(buf, sizeof(buf), " %s=%.2f", ev[i].first, ms);
            line += buf;
        }
        fprintf(stderr, "%s\n", line.c_str());
        for (auto &p : ev) cudaEventDestroy(p.second);
        ev.clear();
    }
};

#define HGA_STR2(x) #x
#define HGA_STR(x) HGA_STR2(x)
