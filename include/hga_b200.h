/*
 * hga_b200.h — C-ABI of the B200-native `categorization` hot path.
 *
 * The reference (matuszelenak/Hybrid-Genome-Assembler) has no FFI; the seam this library replaces is the set
 * of protected stage functions of ReadClusteringEngine (paths relative to /root/reference/src):
 *
 *   hga_create           <- load_text_file_kmers' set + KmerIndex           read_clustering.cpp:18-33,
 *                                                                           clustering/ReadClusteringEngine.cpp:237-241
 *   hga_scan[_device]    <- construct_indices, per-read half                clustering/ReadClusteringEngine.cpp:246-277
 *   hga_scan_packed[_device]   the same from 2-bit packed bases (hga_host_pack_bases packs on the host)
 *                           (KmerIterator semantics: common/KmerIterator.cpp:23-76)
 *   hga_build_index      <- construct_indices, kmer_component_index half    clustering/ReadClusteringEngine.cpp:262-269,282-284
 *   hga_pair_count       <- get_connections / get_all_connections           clustering/ReadClusteringEngine.cpp:301-339
 *   hga_select_edges     <- the 15 % slice / --sc_score filter              clustering/ReadClusteringEngine.cpp:748-756
 *   hga_components       <- union_find(edges, {}, min, -1)                  clustering/ReadClusteringEngine.cpp:424-489, call :763
 *   hga_host_tail_connections <- get_core_component_connections             clustering/ReadClusteringEngine.cpp:491-651
 *   hga_spectral_clustering <- spectral_clustering(connections, dims)       clustering/ReadClusteringEngine.cpp:653-697, lib/clustering/ (all files)
 *   hga_enrich           <- merge_components(scaffolds), get_connections(cores, min), union_find(conns, cores, 2, -1),
 *                           merge_components, get_component_ids             clustering/ReadClusteringEngine.cpp:349-422, :764, :785-794
 *   hga_count_kmers / hga_host_sdk_* <- jellyfish + JellyfishOccurrenceReader (the --kmers file)          occurrences/ (all files), jellyfish_occurrences.cpp
 *   hga_count_kmers_packed     the same count from case-folded 2-bit packed bases (hga_host_pack_bases_folded packs on the host)
 *   hga_count_spectrum[_packed]  the k-mer spectrum of that count (distinct k-mers per count) without materialising the k-mers
 *   hga_sdk_*            the per-file counts merged on the GPU, with the specificity table and the count-range export of hga_host_sdk_*
 *   hga_enrich_full      <- the same plus the tail / spectral block in between (second merge_components)     :764-794
 *
 * Conventions
 *   - every function returns 0 on success, non-zero on failure; hga_last_error() gives the message
 *     (thread-local). The reference signals errors by uncaught C++ exceptions (std::terminate).
 *   - plain pointers and sizes only. Inputs are caller-owned HOST buffers unless the name says _device.
 *   - results stay in HBM between stages; hga_get_* copies them into library-owned pinned host buffers that
 *     remain valid until the next call that produces the same result, or hga_destroy. hga_enrich / hga_enrich_ex / hga_enrich_full and
 *     hga_comm_gather_root use the same buffers as scratch: they invalidate what hga_get_hits, hga_get_index and hga_get_selection
 *     returned before (call those again afterwards if their results are still needed).
 *   - read ids are 1-based and global (SequenceRecordIterator.h:82): row r of a scan has id read_id_base + r.
 *   - kmer_id = index into the array given to hga_create (the reference's KmerID is an arbitrary bijection,
 *     so parity is by k-mer VALUE).
 *   - one handle per GPU; a handle is not thread-safe. There is NO CPU fallback: every entry point fails
 *     with an error if no CUDA device is usable.
 */
#ifndef HGA_B200_H
#define HGA_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct hga_handle hga_handle;

#define HGA_OK 0
#define HGA_E_CUDA 1        /* CUDA runtime / no device */
#define HGA_E_ARG 2         /* bad argument (k > 32 mirrors KmerIterator.cpp:24-26) */
#define HGA_E_STATE 3       /* stage called out of order */
#define HGA_E_NOMEM 4
#define HGA_E_OVERFLOW 5    /* a 32-bit pair score, entry count or k-mer count overflowed */
#define HGA_E_NCCL 6
#define HGA_E_DUPLICATE 7   /* duplicate k-mer handed to hga_create */

const char *hga_last_error(void);
/* library + build identification, e.g. "hga_b200 0.1 sm_100a" */
const char *hga_version(void);
int hga_device_count(int *count);
/* Optional: create the CUDA context of `device` ahead of time. The one-off driver / context start-up takes seconds on a cold
 * machine; a host can run this on a second thread while it reads its input files (the CLI does). */
int hga_init(int device);

/* Pinned host memory helpers (H2D from pinned buffers runs at PCIe speed). */
int hga_host_alloc(void **ptr, size_t bytes);
int hga_host_free(void *ptr);

/* Table of canonical discriminative k-mers on `device` (open-addressing key table + blocked Bloom pre-filter,
 * built by CUDA kernels). kmers must be canonical (min(forward, reverse-complement) in the 2-bit code
 * A0 C1 G2 T3) and unique. 1 <= k <= 32. */
int hga_create(int device, int k, const uint64_t *kmers, uint64_t n_kmers, hga_handle **out);
void hga_destroy(hga_handle *h);
/* Run every kernel of this handle on an existing CUDA stream (cudaStream_t passed as void*); NULL restores
 * the handle's own stream. Lets a caller bracket stages with its own CUDA events. */
int hga_set_stream(hga_handle *h, void *cuda_stream);

/* Scan: 2-bit pack + canonical k-mer windows + membership -> hits in (read, position) order.
 * bases  : the reads' sequence bytes back to back (no separators), ASCII as in the file
 * read_off[n_reads+1] : byte offset of every read in `bases`
 * Any byte other than 'A','C','G','T' follows the reference rule (code 0 on BOTH strands).
 * hga_scan copies the host buffers to the GPU inside the call; hga_scan_device takes device pointers. d_bases may have any
 * alignment (a read set can start anywhere inside a larger buffer): the scan loads the aligned 16-byte blocks that hold the bases.
 * Every read must be shorter than 2^30 bases, on every scan entry (hga_scan, hga_scan_device, hga_scan_packed, hga_scan_packed_device):
 * a longer read fails with HGA_E_ARG and a message, and leaves no scan result. The host entries check read_off before they copy; the
 * device entries check it on the GPU (the last read ends at n_bases). The stream itself may be longer than 2^32 bases. */
int hga_scan(hga_handle *h, const char *bases, const uint64_t *read_off, uint64_t n_reads, uint32_t read_id_base);
int hga_scan_device(hga_handle *h, const char *d_bases, const uint64_t *d_read_off, uint64_t n_reads, uint64_t n_bases,
                    uint32_t read_id_base);

/* Packed bases: the same scan from 2-bit codes, a quarter of the bytes on the wire and in HBM. Results (hits and every later stage) are
 * identical to an ASCII scan of the same bytes.
 *   codes      : A0 C1 G2 T3, four bases per byte, the first base in the most significant bits: base i of a buffer is
 *                (packed[i >> 2] >> (6 - 2 * (i & 3))) & 3
 *   exceptions : every byte other than uppercase A C G T (lowercase, N, '\r', ...) has code 0 on BOTH strands in the reference, which two
 *                bits cannot express. Such bases travel as half-open runs [exc_start[j], exc_end[j]): sorted, non-overlapping,
 *                non-empty, in the coordinates of read_off. The packer writes code 0 under a run; the scan ignores the codes there.
 * hga_host_pack_bases: host arithmetic, no GPU. Packs n_bases ASCII bytes; packed needs (n_bases + 3) / 4 bytes. Writes the maximal
 *   exception runs of the whole stream. If more than exc_capacity runs are needed: HGA_E_ARG and *n_exc = the number needed (retry with
 *   that capacity). threads <= 0: automatic. */
int hga_host_pack_bases(const char *bases, uint64_t n_bases, uint8_t *packed, uint64_t *exc_start, uint64_t *exc_end,
                        uint64_t exc_capacity, uint64_t *n_exc, int threads);
/* hga_host_pack_bases_folded: the same with the case-folded packing that hga_count_kmers_packed takes (jellyfish's rule): lowercase
 *   a c g t are packed as their bases, and only bytes outside A C G T a c g t are covered by exception runs. */
int hga_host_pack_bases_folded(const char *bases, uint64_t n_bases, uint8_t *packed, uint64_t *exc_start, uint64_t *exc_end,
                               uint64_t exc_capacity, uint64_t *n_exc, int threads);
/* The read set = bases first_base + read_off[0 .. n_reads] of `packed` (read_off[0] == 0, the same rules as for ASCII), so a slice of
 * a larger packed buffer is scanned in place; the exception runs are relative to first_base and lie inside [0, read_off[n_reads]).
 * The host entry copies only the bytes that hold the read set and checks read_off and the runs (HGA_E_ARG with a message). The device
 * entry takes device pointers (d_packed at any byte address) and checks read_off[0], the read lengths and the runs on the GPU: HGA_E_ARG,
 * no hits. */
int hga_scan_packed(hga_handle *h, const uint8_t *packed, uint64_t first_base, const uint64_t *read_off, uint64_t n_reads,
                    const uint64_t *exc_start, const uint64_t *exc_end, uint64_t n_exc, uint32_t read_id_base);
int hga_scan_packed_device(hga_handle *h, const uint8_t *d_packed, uint64_t first_base, const uint64_t *d_read_off, uint64_t n_reads,
                           uint64_t n_bases, const uint64_t *d_exc_start, const uint64_t *d_exc_end, uint64_t n_exc, uint32_t read_id_base);

typedef struct {
    uint64_t n_reads;          /* rows scanned */
    uint64_t n_hits;           /* E */
    const uint64_t *row_off;   /* n_reads + 1 */
    const uint32_t *kmer_id;   /* E, position order inside a row (sorted by kmer_id if requested) */
    const uint32_t *pos;       /* E, KmerIterator::position_in_sequence = window start + k */
} hga_hits;
/* sorted_by_kmer_id != 0: each row ordered by (kmer_id, pos) like ReadComponent::discriminative_kmer_ids */
int hga_get_hits(hga_handle *h, int sorted_by_kmer_id, hga_hits *out);

/* Inverted index by k-mer. With a communicator attached this includes the all-to-all by k-mer owner. */
int hga_build_index(hga_handle *h);
typedef struct {
    uint64_t n_kmers;
    uint64_t n_entries;
    const uint64_t *off;       /* n_kmers + 1, indexed by kmer_id */
    const uint32_t *read_id;   /* n_entries, ascending inside a list, one entry per occurrence */
} hga_index;
int hga_get_index(hga_handle *h, hga_index *out);

/* score(x,y) = sum_k mult_x(k) * mult_y(k) for every unordered read pair sharing a k-mer.
 * pivots == NULL: all reads (get_all_connections); else only pairs with at least one endpoint in pivots
 * (get_connections over a component list). A non-NULL pointer with n_pivots == 0 is the EMPTY subset: no pairs, as get_connections({}).
 * Pairs with score < min_score are dropped. Scores are 32-bit: a score above 2^32 - 1 (possible only when two reads have more than
 * 65 535 hits each) fails with HGA_E_OVERFLOW. With a communicator an input with a read of more than 65 535 hits fails with it
 * up front, since the reduction of partial scores does not check for a carry. */
int hga_pair_count(hga_handle *h, uint32_t min_score, const uint32_t *pivots, uint64_t n_pivots);
typedef struct {
    uint64_t n_pairs;          /* unordered pairs, x < y, ordered by (x, y) */
    uint64_t n_increments;     /* sum_k occ(k)*(occ(k)-1)/2 over the processed lists (work measure) */
    const uint32_t *x, *y, *score;
} hga_pairs;
int hga_get_pairs(hga_handle *h, hga_pairs *out);

typedef struct {
    uint64_t n_directed;       /* n = (size_t)(2P * fraction), the reference's slice length */
    uint64_t cut_score;        /* s*: score of the last directed edge inside the slice (0 if n == 0) */
    uint64_t n_selected;       /* unordered edges selected under the canonical tie order */
    const uint32_t *x, *y, *score;
} hga_selection;
/* score_threshold == 0: fraction slice under the canonical order (score desc, x asc, y asc);
 * score_threshold  > 0: keep score > score_threshold (--sc_score). */
int hga_select_edges(hga_handle *h, double fraction, uint32_t score_threshold);
int hga_get_selection(hga_handle *h, hga_selection *out);

typedef struct {
    uint64_t n_reads;          /* labels cover read ids read_id_first .. read_id_first + n_reads - 1 */
    uint32_t read_id_first;
    const uint32_t *label;     /* smallest read id of the read's component (itself when isolated) */
    uint64_t n_components;     /* components with size >= min_size */
    const uint32_t *comp_label;/* their labels, ascending */
    const uint32_t *comp_size;
} hga_components_t;
int hga_components(hga_handle *h, int min_size);
int hga_get_components(hga_handle *h, hga_components_t *out);

/* Merge of the scaffold components + enrichment (SURVEY §8f-1): everything run_clustering does after the scaffold union_find
 * EXCEPT the tail / spectral block (:768-777), i.e. the reference's path when it has at most two scaffold components or no strong
 * tail connection. Needs hga_scan, hga_build_index and hga_select_edges on this handle (single GPU).
 *   cores          : the components of the selected edges with >= min_size reads, identified by the SURVIVOR the reference's
 *                    sequential union_find would end with under the canonical edge order (element [0], :366)
 *   purged index   : kmer_component_index after merge_components (:395-419), including its truncation at the largest removed id
 *   connections    : get_connections(cores, enrichment_min_score) on the merged state, directed core -> partner, canonical order
 *   final          : components after union_find(connections, restricted = cores, 2, -1) + merge; id = surviving component id */
int hga_enrich(hga_handle *h, int min_size, uint32_t enrichment_min_score);
/* the same with --sc_max_size: a scaffold union is skipped when the merged component would exceed max_size reads (union_find,
 * :426, :457; -1 = no limit). The limit makes the components depend on the edge order, so they come from the sequential replay
 * of ALL selected edges on the host, not from hga_components (whose labels ignore the limit). */
int hga_enrich_ex(hga_handle *h, int min_size, int max_size, uint32_t enrichment_min_score);
typedef struct {
    uint64_t n_cores;
    const uint32_t *core_id;       /* n_cores, ascending */
    const uint64_t *core_off;      /* n_cores + 1 */
    const uint32_t *core_read;     /* member read ids, ascending inside a core */
    uint64_t n_connections;
    const uint32_t *conn_x, *conn_y, *conn_score;
    uint64_t n_final;
    const uint32_t *final_id;      /* ordered by the smallest member */
    const uint64_t *final_off;     /* n_final + 1 */
    const uint32_t *final_read;    /* ascending inside a component */
    uint64_t n_reads;              /* assignment covers read ids read_id_first .. read_id_first + n_reads - 1 */
    uint32_t read_id_first;
    const uint32_t *assignment;    /* final component id of the read, 0 = in no exported component */
} hga_enrichment_t;
int hga_get_enrichment(hga_handle *h, hga_enrichment_t *out);
/* the purged inverted index (same layout as hga_get_index) and the merged k-mer id list of every core (off[n_cores + 1]) */
int hga_get_purged_index(hga_handle *h, hga_index *out);
typedef struct {
    uint64_t n_cores;
    const uint64_t *off;
    const uint32_t *kmer_id;       /* unique inside a core, unordered */
} hga_core_kmers_t;
int hga_get_core_kmers(hga_handle *h, hga_core_kmers_t *out);

/* The same INCLUDING the tail / spectral block (SURVEY §8f-2, run_clustering :768-777), i.e. everything run_clustering does after
 * the scaffold union_find. When the scaffold merge leaves more than two cores: the engine state after the merge (hits, spanning
 * trees of the replayed union_find) goes to the host stages of hga_host_tail_connections - whose amplification step
 * (get_connections(tail, min) through the purged index) runs on the GPU, the purged index stays there - and, for the connections
 * with score > 5 (:770), to hga_spectral_clustering; the clusters are merged by a SECOND merge_components on the GPU (unique unions
 * of the members' merged k-mer lists, second purge of the already purged index with the same truncation rule: the removal list
 * of a k-mer holds every member of a multi-member cluster that lists it plus the cluster's survivor); enrichment, restricted
 * union_find and the final merge then run on that state. With at most two cores, or no strong tail connection, the result is
 * hga_enrich_ex's. read_off: HOST array of n_reads + 1 offsets as given to hga_scan (read lengths for the spanning-tree
 * distances; avg_read_length = total bases / reads, SequenceRecordIterator.cpp:64). hga_get_enrichment, hga_get_purged_index and
 * hga_get_core_kmers then describe the state after the second merge. */
int hga_enrich_full(hga_handle *h, int min_size, int max_size, uint32_t enrichment_min_score, uint32_t tail_amplification_min_score,
                    int spectral_dims, const uint64_t *read_off);
typedef struct {
    int ran;                       /* 1: more than two scaffold components, the block ran (:768) */
    uint64_t n_scaffold_cores;     /* cores before the merge of the spectral clusters */
    uint64_t n_connections;        /* all tail connections (score > 0), x < y, canonical order */
    const uint32_t *conn_x, *conn_y;
    const uint64_t *conn_score;
    uint64_t n_clusters;           /* non-empty spectral clusters; element [0] = the id that survives the merge */
    const uint64_t *cluster_off;   /* n_clusters + 1 */
    const uint32_t *cluster_member;
} hga_tail_block_t;
int hga_get_tail_block(hga_handle *h, hga_tail_block_t *out);

/* Spectral clustering of scaffold components from their tail connections (HOST arithmetic, no GPU involved; first piece of SURVEY
 * §8f-2): spectral_clustering(connections, dims) of clustering/ReadClusteringEngine.cpp:653-697 with lib/clustering's
 * SpectralClustering / ClusterRotate / Evrot. connections in the order the caller wants the affinity matrix built in (the
 * reference: its sorted tail connections with score > 5, :770). Output: the component ids cluster by cluster (out_component,
 * capacity 2 * n_conn; element [0] of a cluster is the member closest to the cluster centre = the surviving id in
 * merge_components) and the cluster boundaries (out_cluster_off, capacity dims + 1; empty clusters are kept). */
int hga_spectral_clustering(const uint32_t *conn_x, const uint32_t *conn_y, const uint64_t *conn_score, uint64_t n_conn, int dims,
                            uint32_t *out_component, uint64_t *out_cluster_off, uint64_t *out_n_components, uint64_t *out_n_clusters);

/* The symmetric eigen-solver hga_spectral_clustering uses (Householder tridiagonalisation + implicit QL), exposed so that it can be
 * checked against an independent implementation: a = n x n row major; val[n] ascending; vec = eigenvectors in columns, row major. */
int hga_host_sym_eigen(int n, const double *a, double *val, double *vec);

/* Tail connections between scaffold components (HOST arithmetic, no GPU involved; second piece of SURVEY §8f-2):
 * get_core_component_connections(components_and_trees) of clustering/ReadClusteringEngine.cpp:594-651 (spanning-tree tails :510-581,
 * approximate_read_overlap :491-508, amplify_component :583-592, accumulate_kmer_ids :340-346) on the engine state after
 * merge_components(scaffold components).
 *   row_off / kmer_id / pos : hits by read, every row sorted by (kmer_id, pos) (hga_get_hits(h, 1, ..)); read_len per read
 *   comp_off / comp_member  : the scaffold components, element [0] = the surviving id; tree_off / tree_x / tree_y their spanning trees
 *   purged_off / purged_read: the purged inverted index by kmer_id (hga_get_purged_index)
 * Output (capacity n_comp * (n_comp - 1) / 2): connections x < y with score > 0 in canonical order (score desc, x asc, y asc). */
int hga_host_tail_connections(uint64_t n_reads, const uint64_t *row_off, const uint32_t *kmer_id, const uint32_t *pos, const uint32_t *read_len,
                              uint64_t avg_read_length, uint32_t read_id_first, uint64_t n_comp, const uint64_t *comp_off, const uint32_t *comp_member,
                              const uint64_t *tree_off, const uint32_t *tree_x, const uint32_t *tree_y, const uint64_t *purged_off,
                              const uint32_t *purged_read, uint32_t amplification_min_score, uint32_t *out_x, uint32_t *out_y, uint64_t *out_score,
                              uint64_t *out_n);

/* SDK selection (SURVEY §8f-4): what produces the --kmers file. jellyfish_occurrences.cpp shells out to jellyfish per read file
 * (occurrences/run_jellyfish.sh, JellyfishOccurrenceReader.cpp:16-38), merges the sorted dumps and exports the k-mers whose total
 * count lies in a range (:63-134).
 *   hga_count_kmers  : the counting on the GPU, no handle needed: the canonical k-mers of `bases` (windows with a byte other than
 *                      A C G T a c g t skipped, as jellyfish does) that occur at least min_count times (2 = the two-pass
 *                      Bloom-counter filter of run_jellyfish.sh without its false positives), ascending, with exact 32-bit
 *                      counts: a k-mer seen more than 2^32 - 1 times fails the call with HGA_E_OVERFLOW and a message that
 *                      names it and its count (hga_count_spectrum reports such a count exactly).
 *                      The arrays are malloc'ed by the library: release them with hga_free_kmer_counts.
 *   hga_host_sdk_*   : the reader's host arithmetic on those lists (files back to back: file f = [file_off[f], file_off[f + 1])).
 *                      merge: out arrays need room for file_off[n_files] entries. specificity: rows (threshold, total count,
 *                      number of k-mers), *out_n = rows needed. select: lower <= total <= upper, kept with probability percent
 *                      (seeded; percent >= 1 keeps all); n_discriminative = selected k-mers present in exactly one file. */
typedef struct {
    uint64_t n;
    const uint64_t *kmer;
    const uint32_t *count;
} hga_kmer_counts_t;
int hga_count_kmers(int device, int k, const char *bases, const uint64_t *read_off, uint64_t n_reads, uint32_t min_count, hga_kmer_counts_t *out);
/* hga_count_kmers_packed: the same counts from the case-folded packing of hga_host_pack_bases_folded, identical to hga_count_kmers on
 *   the ASCII bytes (same k-mers, counts and order). The read set and the runs follow hga_scan_packed's rules: bases first_base +
 *   read_off[0 .. n_reads] of `packed` with read_off[0] == 0, every read shorter than 2^30 bases, runs relative to first_base, sorted,
 *   non-empty, non-overlapping, inside [0, read_off[n_reads]). Only the bytes that hold the read set are copied. Bad input: HGA_E_ARG
 *   with a message. */
int hga_count_kmers_packed(int device, int k, const uint8_t *packed, uint64_t first_base, const uint64_t *read_off, uint64_t n_reads,
                           const uint64_t *exc_start, const uint64_t *exc_end, uint64_t n_exc, uint32_t min_count, hga_kmer_counts_t *out);
void hga_free_kmer_counts(hga_kmer_counts_t *c);
/* hga_count_spectrum[_packed]: the k-mer spectrum of the same count, computed on the GPU without materialising the k-mers (what
 *   `jellyfish histo` / `stats` print; the k sweep of jf_occurrences reads n_distinct). Host memory is O(n_bins) whatever the input. */
typedef struct {
    uint64_t n_windows;    /* windows counted (k bases inside one read, all A C G T a c g t) = the sum of all counts */
    uint64_t n_distinct;   /* distinct canonical k-mers = hga_count_kmers(.., min_count = 1, ..).n */
    uint64_t max_count;    /* largest count of any k-mer, exact (not clipped at 2^32 - 1); 0 when there is no window */
} hga_kmer_spectrum_t;
/* hist: caller-owned, n_bins entries (NULL allowed when n_bins == 0). hist[c - 1] = distinct k-mers seen exactly c times for
 * 1 <= c < n_bins; hist[n_bins - 1] = those seen n_bins times or more. Same k-mer rule, read-set rules and checks as hga_count_kmers /
 * hga_count_kmers_packed (the packed spectrum too takes reads shorter than 2^30 bases only); nothing is allocated for the caller.
 * No count is clipped: a k-mer seen more than 2^32 - 1 times is counted exactly. */
int hga_count_spectrum(int device, int k, const char *bases, const uint64_t *read_off, uint64_t n_reads,
                       uint32_t n_bins, uint64_t *hist, hga_kmer_spectrum_t *out);
int hga_count_spectrum_packed(int device, int k, const uint8_t *packed, uint64_t first_base, const uint64_t *read_off, uint64_t n_reads,
                              const uint64_t *exc_start, const uint64_t *exc_end, uint64_t n_exc,
                              uint32_t n_bins, uint64_t *hist, hga_kmer_spectrum_t *out);
int hga_host_sdk_merge(int n_files, const uint64_t *file_off, const uint64_t *kmer, const uint32_t *count, uint64_t *out_kmer, uint32_t *out_total,
                       uint32_t *out_max, uint32_t *out_files, uint64_t *out_n);
int hga_host_sdk_specificity(uint64_t n, const uint32_t *total, const uint32_t *max, const double *thresholds, int n_thresholds, double *out_threshold,
                             uint32_t *out_occurrences, uint64_t *out_unique, uint64_t capacity, uint64_t *out_n);
int hga_host_sdk_select(uint64_t n, const uint32_t *total, const uint32_t *files, uint32_t lower, uint32_t upper, double percent, uint64_t seed,
                        uint8_t *out_selected, uint64_t *out_n_selected, uint64_t *out_n_discriminative);
/* hga_sdk_*: the merge, the specificity table and the count-range export on the GPU; the merged table stays in HBM, so host memory
 *   does not grow with the number of distinct k-mers (only hga_sdk_range's result does).
 *   hga_sdk_count_packed: file f = reads [file_first_read[f], file_first_read[f + 1]) of the read set of hga_count_kmers_packed
 *     (same packing, read-set and run rules). Every file is counted with min_count (the filter applies per file, before the merge)
 *     and the files are merged: the handle holds what hga_host_sdk_merge returns on the per-file hga_count_kmers_packed lists.
 *     file_first_read: n_files + 1 entries, [0] == 0, non-decreasing, [n_files] == n_reads (a file without reads is allowed).
 *     A per-file count above 2^32 - 1 fails with HGA_E_OVERFLOW and hga_count_kmers_packed's message; so does a total above
 *     2^32 - 1. On failure *out is NULL and no device memory is held. The handle owns device memory on `device` until hga_sdk_free.
 *   hga_sdk_size: the number of merged k-mers.
 *   hga_sdk_specificity: the rows, row order, errors and capacity protocol of hga_host_sdk_specificity on the merged table.
 *   hga_sdk_range: the merged entries with lower <= total <= upper, ascending (empty when lower > upper), in arrays malloc'ed by the
 *     library (release with hga_free_sdk_range). hga_host_sdk_select on it, with the same lower, upper, percent and seed, selects the
 *     same k-mers as on the whole merged table: it draws only for in-range k-mers. */
typedef struct hga_sdk hga_sdk;
typedef struct {
    uint64_t n;
    const uint64_t *kmer;
    const uint32_t *total, *max, *files;
} hga_sdk_range_t;
int hga_sdk_count_packed(int device, int k, const uint8_t *packed, uint64_t first_base, const uint64_t *read_off, uint64_t n_reads,
                         const uint64_t *exc_start, const uint64_t *exc_end, uint64_t n_exc, int n_files, const uint64_t *file_first_read,
                         uint32_t min_count, hga_sdk **out);
int hga_sdk_size(const hga_sdk *s, uint64_t *n_kmers);
int hga_sdk_specificity(const hga_sdk *s, const double *thresholds, int n_thresholds, double *out_threshold, uint32_t *out_occurrences,
                        uint64_t *out_unique, uint64_t capacity, uint64_t *out_n);
int hga_sdk_range(const hga_sdk *s, uint32_t lower, uint32_t upper, hga_sdk_range_t *out);
void hga_free_sdk_range(hga_sdk_range_t *r);
void hga_sdk_free(hga_sdk *s);

/* Per-stage device time (CUDA events on the handle's stream) and counters of the most recent run. */
typedef struct {
    double table_build_ms, h2d_ms, scan_ms, index_ms, pair_ms, select_ms, components_ms, exchange_ms;
    uint64_t n_bases, n_reads, n_hits, n_pairs, n_increments, n_selected, n_components;
    uint64_t table_bytes, filter_bytes, pair_retries, heavy_pivots;
    uint64_t kernel_launches;  /* kernels of this library launched on this handle since creation */
    uint64_t table_overflow_keys; /* keys that did not fit their locality chain (stored in the overflow region) */
    uint64_t mid_pivots;       /* pivot rows whose partner set overflowed the per-warp accumulator (tier 2) */
    uint64_t n_candidates;     /* windows that passed the membership filter in the last scan (hits + false positives) */
    double enrich_ms;          /* hga_enrich, host replay of the union_find roots included */
    uint64_t n_cores, n_enrich_connections, n_final_components;
    uint64_t redo_pivots;      /* pivot rows redone by the second pass of pair-count tier 1 (1024-entry accumulator) */
    /* wall time of the stages of hga_enrich* under the reference's own timer labels (ReadClusteringEngine.cpp:765-791):
     * [0] Merging of initial components, [1] Calculation of tail connections, [2] Spectral clustering, [3] Merging of scaffold
     * components, [4] Calculation of enrichment connections, [5] Merging into core components ([1]..[3]: 0 when the block did not run) */
    double enrich_phase_ms[6];
    uint64_t scan_retries;     /* reruns of the last scan with the exact hit count after its estimated hit buffer overflowed */
} hga_metrics_t;
int hga_metrics(hga_handle *h, hga_metrics_t *out);

/* Multi-GPU (one handle per rank/GPU). The 128-byte id comes from hga_comm_unique_id on rank 0 and is
 * distributed by the caller (torch.distributed broadcast, a file, ...). After hga_comm_init:
 *   hga_build_index   routes (kmer, read) incidences to the k-mer's owner rank (whole buckets of the k-mer table dealt round robin; the table
 *                     layout is a function of the k-mer array, the same on every rank) with one all-to-all; nothing is replicated:
 *                     hga_get_index on a rank returns the lists of ITS k-mers (every other list empty),
 *   hga_pair_count    counts partial scores over the owned lists and reduces them at the owner of x, x mod nranks (all-to-all):
 *                     every unordered pair ends up on exactly one rank,
 *   hga_select_edges  all-reduces the score histogram,
 *   hga_components    iterates union-find with all-reduce(min) on the label array.
 * n_reads_total = number of reads over all ranks (rows are global: rank shards are contiguous id ranges). */
int hga_comm_unique_id(void *id128);
int hga_comm_init(hga_handle *h, const void *id128, int rank, int nranks, uint64_t n_reads_total);
/* Collective, after hga_components on every rank: rank 0's handle becomes a complete single-GPU handle (hits and selected edges of all
 * ranks gathered over NCCL, by-slot inverted index rebuilt, communicator detached), on which hga_enrich / hga_enrich_ex / hga_enrich_full
 * and every hga_get_* except hga_get_pairs work as on one GPU: the stages after the scaffold union_find (run_clustering,
 * ReadClusteringEngine.cpp:764-794) run on rank 0. The other ranks' handles are left as they are and must not enter another collective.
 * Without a communicator: no-op. */
int hga_comm_gather_root(hga_handle *h);

#ifdef __cplusplus
}
#endif
#endif
