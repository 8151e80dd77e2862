// C-ABI entry points of libhga_b200.so (see include/hga_b200.h for the reference seams they replace).
#include "hga_internal.cuh"

#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>

static thread_local char g_err[1024] = "";

void hga_set_error(const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

namespace {

__global__ void slots_to_kids_kernel(const uint32_t *__restrict__ slot, const uint32_t *__restrict__ slot_kid, uint64_t n, uint32_t *out) {
    for (uint64_t i = blockIdx.x * (uint64_t) blockDim.x + threadIdx.x; i < n; i += (uint64_t) gridDim.x * blockDim.x) out[i] = slot_kid[slot[i]];
}

__global__ void row_kid_keys_kernel(const uint64_t *__restrict__ row_off, uint64_t n_rows, const uint32_t *__restrict__ kid, uint64_t *out_key) {
    const uint64_t warps = ((uint64_t) gridDim.x * blockDim.x) >> 5;
    const uint64_t w = (blockIdx.x * (uint64_t) blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    for (uint64_t r = w; r < n_rows; r += warps) {
        const uint64_t a = row_off[r], b = row_off[r + 1];
        for (uint64_t i = a + lane; i < b; i += 32) out_key[i] = (r << 32) | kid[i];
    }
}

__global__ void low32_kernel(const uint64_t *__restrict__ key, uint64_t n, uint32_t *out) {
    for (uint64_t i = blockIdx.x * (uint64_t) blockDim.x + threadIdx.x; i < n; i += (uint64_t) gridDim.x * blockDim.x) out[i] = (uint32_t) key[i];
}

// G == 0: the index is keyed by table slot. G > 0 (multi-GPU): this rank holds the lists of the slots it owns (hga_owner_of_slot) under
// their list numbers (hga_list_of_slot), and every other k-mer's list is empty here
__global__ void kid_list_len_kernel(const uint32_t *__restrict__ kid_slot, uint32_t G, uint32_t me, const uint32_t *__restrict__ inv_off, uint64_t n_kmers, unsigned long long *len) {
    for (uint64_t i = blockIdx.x * (uint64_t) blockDim.x + threadIdx.x; i <= n_kmers; i += (uint64_t) gridDim.x * blockDim.x) {
        if (i == n_kmers) { len[i] = 0; continue; }
        uint32_t s = kid_slot[i];
        if (G) { if (hga_owner_of_slot(s, G) != me) { len[i] = 0; continue; } s = hga_list_of_slot(s, G); }
        len[i] = inv_off[s + 1] - inv_off[s];
    }
}

__global__ void kid_list_copy_kernel(const uint32_t *__restrict__ kid_slot, uint32_t G, uint32_t me, const uint32_t *__restrict__ inv_off, const uint32_t *__restrict__ inv_row,
                                     const unsigned long long *__restrict__ out_off, uint64_t n_kmers, uint32_t first_id, uint32_t *out) {
    const uint64_t warps = ((uint64_t) gridDim.x * blockDim.x) >> 5;
    const uint64_t w = (blockIdx.x * (uint64_t) blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    for (uint64_t kid = w; kid < n_kmers; kid += warps) {
        uint32_t s = kid_slot[kid];
        if (G) { if (hga_owner_of_slot(s, G) != me) continue; s = hga_list_of_slot(s, G); }
        const uint64_t a = inv_off[s], b = inv_off[s + 1], o = out_off[kid];
        for (uint64_t i = lane; i < b - a; i += 32) out[o + i] = inv_row[a + i] + first_id;
    }
}

__global__ void split_keys_kernel(const uint64_t *__restrict__ key, uint64_t n, uint32_t first_id, uint32_t *x, uint32_t *y) {
    for (uint64_t i = blockIdx.x * (uint64_t) blockDim.x + threadIdx.x; i < n; i += (uint64_t) gridDim.x * blockDim.x) {
        const uint64_t k = key[i];
        x[i] = (uint32_t) (k >> 32) + first_id; y[i] = (uint32_t) k + first_id;
    }
}

__global__ void add_u32_kernel(const uint32_t *__restrict__ in, uint64_t n, uint32_t add, uint32_t *out) {
    for (uint64_t i = blockIdx.x * (uint64_t) blockDim.x + threadIdx.x; i < n; i += (uint64_t) gridDim.x * blockDim.x) out[i] = in[i] + add;
}

inline int grid_for(const hga_handle *h, uint64_t n, int per_block = 256) {
    return (int) std::max<uint64_t>(1, std::min<uint64_t>((n + per_block - 1) / per_block, (uint64_t) h->sm_count * 16));
}

int use_device(hga_handle *h) {
    HGA_CUDA(cudaSetDevice(h->device));
    return HGA_OK;
}

}  // namespace

extern "C" {

const char *hga_last_error(void) { return g_err; }
const char *hga_version(void) { return "hga_b200 0.1 (sm_100a, CUDA " HGA_STR(CUDART_VERSION) ")"; }

int hga_device_count(int *count) {
    HGA_CUDA(cudaGetDeviceCount(count));
    return HGA_OK;
}

int hga_init(int device) {
    HGA_CUDA(cudaSetDevice(device));
    HGA_CUDA(cudaFree(nullptr));
    return HGA_OK;
}

int hga_host_alloc(void **ptr, size_t bytes) {
    HGA_CUDA(cudaMallocHost(ptr, bytes ? bytes : 1));
    return HGA_OK;
}
int hga_host_free(void *ptr) {
    HGA_CUDA(cudaFreeHost(ptr));
    return HGA_OK;
}

int hga_create(int device, int k, const uint64_t *kmers, uint64_t n_kmers, hga_handle **out) {
    if (!out) { hga_set_error("hga_create: out is NULL"); return HGA_E_ARG; }
    *out = nullptr;
    if (k < 1 || k > 32) { hga_set_error("Kmer size is too big (k=%d; KmerIterator supports k <= 32)", k); return HGA_E_ARG; }
    if (n_kmers && !kmers) { hga_set_error("hga_create: kmers is NULL"); return HGA_E_ARG; }
    int n_dev = 0;
    cudaError_t e = cudaGetDeviceCount(&n_dev);
    if (e != cudaSuccess || n_dev == 0) {
        hga_set_error("no usable CUDA device (%s); this library has no CPU path", e == cudaSuccess ? "device count is 0" : cudaGetErrorString(e));
        cudaGetLastError();
        return HGA_E_CUDA;
    }
    if (device < 0 || device >= n_dev) { hga_set_error("device %d out of range (%d devices)", device, n_dev); return HGA_E_ARG; }
    HGA_CUDA(cudaSetDevice(device));
    cudaDeviceProp prop;
    HGA_CUDA(cudaGetDeviceProperties(&prop, device));
    if (prop.major < 10) { hga_set_error("device %d is sm_%d%d; this library is built for sm_100a (B200) only", device, prop.major, prop.minor); return HGA_E_CUDA; }
    hga_handle *h = new hga_handle();
    memset(&h->metrics, 0, sizeof(h->metrics));
    h->device = device; h->k = k; h->n_kmers = n_kmers; h->sm_count = prop.multiProcessorCount;
    cudaError_t e1 = cudaStreamCreateWithFlags(&h->own_stream, cudaStreamNonBlocking);
    if (cudaStreamCreateWithFlags(&h->copy_stream, cudaStreamNonBlocking) != cudaSuccess) { h->copy_stream = nullptr; cudaGetLastError(); }
    cudaError_t e2 = cudaEventCreate(&h->ev0), e3 = cudaEventCreate(&h->ev1), e4 = cudaEventCreate(&h->ev2), e5 = cudaEventCreate(&h->ev3);
    if (e1 != cudaSuccess || e2 != cudaSuccess || e3 != cudaSuccess || e4 != cudaSuccess || e5 != cudaSuccess) { hga_set_error("stream/event creation failed"); delete h; return HGA_E_CUDA; }
    h->stream = h->own_stream;
    int rc = hga_table_build(h, kmers);
    if (rc != HGA_OK) { hga_destroy(h); return rc; }
    *out = h;
    return HGA_OK;
}

void hga_destroy(hga_handle *h) {
    if (!h) return;
    cudaSetDevice(h->device);
    cudaDeviceSynchronize();
    hga_comm_destroy(h);
    DevBuf *dev[] = {&h->d_keys, &h->d_slot_kid, &h->d_kid_slot, &h->d_filter, &h->d_bases, &h->d_read_off, &h->d_row_off, &h->d_hit_slot, &h->d_hit_pos, &h->d_pos_tmp,
                     &h->d_tile_state, &h->d_tile_dir, &h->d_scan_scalars, &h->d_exc, &h->d_exc_dir, &h->d_x_slot, &h->d_x_row, &h->d_g_kid, &h->d_g_row_off, &h->d_inv_off, &h->d_inv_row, &h->d_sort_a,
                     &h->d_index_tmp, &h->d_index_goff, &h->d_sort_b, &h->d_sort_tmp, &h->d_pair_key, &h->d_pair_score, &h->d_pair_key2, &h->d_pair_score2, &h->d_pair_scalars,
                     &h->d_heavy_list, &h->d_mid_list, &h->d_redo_list, &h->d_heavy_tab, &h->d_pivot_flag, &h->d_pivot_order, &h->d_pivot_rows, &h->d_hist, &h->d_sel_key, &h->d_sel_score, &h->d_sel_scalars, &h->d_parent,
                     &h->d_comp_size, &h->d_comp_label, &h->d_comp_scalars, &h->d_export_a, &h->d_export_b, &h->d_export_c, &h->d_enr_parent, &h->d_enr_core_of,
                     &h->d_enr_surv, &h->d_enr_R, &h->d_enr_scalars, &h->d_enr_keys, &h->d_enr_keys2, &h->d_enr_core_koff, &h->d_purged_off, &h->d_purged_row, &h->d_purged2_off, &h->d_purged2_row};
    for (DevBuf *b : dev) b->release();
    PinBuf *pin[] = {&h->h_row_off, &h->h_kid, &h->h_pos, &h->h_inv_off, &h->h_inv_read, &h->h_px, &h->h_py, &h->h_ps, &h->h_sx, &h->h_sy, &h->h_ss,
                     &h->h_label, &h->h_clabel, &h->h_csize, &h->h_scalars};
    for (PinBuf *b : pin) b->release();
    if (h->ev0) cudaEventDestroy(h->ev0);
    if (h->ev1) cudaEventDestroy(h->ev1);
    if (h->ev2) cudaEventDestroy(h->ev2);
    if (h->ev3) cudaEventDestroy(h->ev3);
    if (h->own_stream) cudaStreamDestroy(h->own_stream);
    if (h->copy_stream) cudaStreamDestroy(h->copy_stream);
    delete h;
}

int hga_set_stream(hga_handle *h, void *cuda_stream) {
    if (!h) { hga_set_error("NULL handle"); return HGA_E_ARG; }
    h->stream = cuda_stream ? (cudaStream_t) cuda_stream : h->own_stream;
    return HGA_OK;
}

int hga_scan_device(hga_handle *h, const char *d_bases, const uint64_t *d_read_off, uint64_t n_reads, uint64_t n_bases, uint32_t read_id_base) {
    if (!h) { hga_set_error("NULL handle"); return HGA_E_ARG; }
    if ((n_bases && !d_bases) || !d_read_off) { hga_set_error("hga_scan_device: NULL buffer"); return HGA_E_ARG; }
    HGA_TRY(use_device(h));
    h->read_id_base = read_id_base;
    return hga_scan_run(h, d_bases, d_read_off, n_reads, n_bases, nullptr, nullptr, "hga_scan_device");
}

int hga_scan(hga_handle *h, const char *bases, const uint64_t *read_off, uint64_t n_reads, uint32_t read_id_base) {
    if (!h) { hga_set_error("NULL handle"); return HGA_E_ARG; }
    if (!read_off) { hga_set_error("hga_scan: read_off is NULL"); return HGA_E_ARG; }
    HGA_TRY(use_device(h));
    const uint64_t n_bases = read_off[n_reads];
    if (read_off[0] != 0) { hga_set_error("hga_scan: read_off[0] must be 0"); return HGA_E_ARG; }
    if (n_bases && !bases) { hga_set_error("hga_scan: bases is NULL"); return HGA_E_ARG; }
    for (uint64_t i = 0; i < n_reads; i++) {
        if (read_off[i + 1] < read_off[i]) { hga_set_error("hga_scan: read_off is not monotone at read %llu", (unsigned long long) i); return HGA_E_ARG; }
        if (read_off[i + 1] - read_off[i] >= (1ull << 30)) { hga_set_error("hga_scan: read %llu has 2^30 bases or more (reads must be shorter than 2^30 bases)", (unsigned long long) i); return HGA_E_ARG; }
    }
    HGA_TRY(h->d_bases.ensure(n_bases + 64));
    HGA_TRY(h->d_read_off.ensure((n_reads + 1) * 8));
    h->metrics.h2d_ms = 0;
    HGA_CUDA(cudaMemcpyAsync(h->d_read_off.p, read_off, (n_reads + 1) * 8, cudaMemcpyHostToDevice, h->stream));
    h->read_id_base = read_id_base;
    return hga_scan_run(h, h->d_bases.as<char>(), h->d_read_off.as<uint64_t>(), n_reads, n_bases, bases);
}

// read_off of a host entry: read_off[0] == 0, monotone, no read of 2^30 bases or more
static int check_read_off(const char *who, const uint64_t *read_off, uint64_t n_reads) {
    if (read_off[0] != 0) { hga_set_error("%s: read_off[0] must be 0", who); return HGA_E_ARG; }
    for (uint64_t i = 0; i < n_reads; i++) {
        if (read_off[i + 1] < read_off[i]) { hga_set_error("%s: read_off is not monotone at read %llu", who, (unsigned long long) i); return HGA_E_ARG; }
        if (read_off[i + 1] - read_off[i] >= (1ull << 30)) { hga_set_error("%s: read %llu has 2^30 bases or more (reads must be shorter than 2^30 bases)", who, (unsigned long long) i); return HGA_E_ARG; }
    }
    return HGA_OK;
}

// exception runs of a packed host entry: sorted, non-empty, non-overlapping, inside [0, n_bases)
static int check_exc_runs(const char *who, const uint64_t *exc_start, const uint64_t *exc_end, uint64_t n_exc, uint64_t n_bases) {
    if (n_exc && (!exc_start || !exc_end)) { hga_set_error("%s: exception runs are NULL", who); return HGA_E_ARG; }
    for (uint64_t i = 0; i < n_exc; i++) {
        if (exc_start[i] >= exc_end[i] || exc_end[i] > n_bases || (i && exc_start[i] < exc_end[i - 1])) {
            hga_set_error("%s: exception run %llu [%llu, %llu) is empty, out of order, overlaps its predecessor or lies outside [0, %llu)", who,
                          (unsigned long long) i, (unsigned long long) exc_start[i], (unsigned long long) exc_end[i], (unsigned long long) n_bases);
            return HGA_E_ARG;
        }
    }
    return HGA_OK;
}

int hga_scan_packed(hga_handle *h, const uint8_t *packed, uint64_t first_base, const uint64_t *read_off, uint64_t n_reads, const uint64_t *exc_start,
                    const uint64_t *exc_end, uint64_t n_exc, uint32_t read_id_base) {
    if (!h) { hga_set_error("NULL handle"); return HGA_E_ARG; }
    if (!read_off) { hga_set_error("hga_scan_packed: read_off is NULL"); return HGA_E_ARG; }
    HGA_TRY(use_device(h));
    HGA_TRY(check_read_off("hga_scan_packed", read_off, n_reads));
    const uint64_t n_bases = read_off[n_reads];
    if (n_bases && !packed) { hga_set_error("hga_scan_packed: packed is NULL"); return HGA_E_ARG; }
    HGA_TRY(check_exc_runs("hga_scan_packed", exc_start, exc_end, n_exc, n_bases));
    // only the bytes that hold the read set travel; on the device they start at an aligned buffer, first_base % 4 bases into its first byte
    const uint32_t sub = (uint32_t) (first_base & 3);
    const uint64_t n_bytes = n_bases ? (sub + n_bases + 3) / 4 : 0;
    HGA_TRY(h->d_bases.ensure(n_bytes + 64));
    HGA_TRY(h->d_read_off.ensure((n_reads + 1) * 8));
    HGA_TRY(h->d_exc.ensure(n_exc * 16 + 16));
    h->metrics.h2d_ms = 0;
    HGA_CUDA(cudaMemcpyAsync(h->d_read_off.p, read_off, (n_reads + 1) * 8, cudaMemcpyHostToDevice, h->stream));
    h->read_id_base = read_id_base;
    ScanPackedInput in;
    in.sub = sub;
    in.d_exc_start = h->d_exc.as<uint64_t>(); in.d_exc_end = in.d_exc_start + n_exc;
    in.h_exc_start = exc_start; in.h_exc_end = exc_end; in.n_exc = n_exc;
    return hga_scan_run(h, h->d_bases.as<char>(), h->d_read_off.as<uint64_t>(), n_reads, n_bases, n_bytes ? reinterpret_cast<const char *>(packed + first_base / 4) : nullptr,
                        &in);
}

int hga_count_kmers_packed(int device, int k, const uint8_t *packed, uint64_t first_base, const uint64_t *read_off, uint64_t n_reads, const uint64_t *exc_start,
                           const uint64_t *exc_end, uint64_t n_exc, uint32_t min_count, hga_kmer_counts_t *out) {
    if (!out) { hga_set_error("hga_count_kmers_packed: NULL argument"); return HGA_E_ARG; }
    out->n = 0; out->kmer = nullptr; out->count = nullptr;
    if (!read_off) { hga_set_error("hga_count_kmers_packed: read_off is NULL"); return HGA_E_ARG; }
    if (k < 1 || k > 32) { hga_set_error("Kmer size is too big or too small (k = %d)", k); return HGA_E_ARG; }
    HGA_TRY(check_read_off("hga_count_kmers_packed", read_off, n_reads));
    const uint64_t n_bases = read_off[n_reads];
    if (n_bases && !packed) { hga_set_error("hga_count_kmers_packed: packed is NULL"); return HGA_E_ARG; }
    HGA_TRY(check_exc_runs("hga_count_kmers_packed", exc_start, exc_end, n_exc, n_bases));
    return hga_count_run("hga_count_kmers_packed", device, k, nullptr, packed, first_base, read_off, n_reads, exc_start, exc_end, n_exc, min_count, out, nullptr, 0, nullptr);
}

int hga_sdk_count_packed(int device, int k, const uint8_t *packed, uint64_t first_base, const uint64_t *read_off, uint64_t n_reads, const uint64_t *exc_start,
                         const uint64_t *exc_end, uint64_t n_exc, int n_files, const uint64_t *file_first_read, uint32_t min_count, hga_sdk **out) {
    if (!out) { hga_set_error("hga_sdk_count_packed: NULL argument"); return HGA_E_ARG; }
    *out = nullptr;
    if (!read_off) { hga_set_error("hga_sdk_count_packed: read_off is NULL"); return HGA_E_ARG; }
    if (k < 1 || k > 32) { hga_set_error("Kmer size is too big or too small (k = %d)", k); return HGA_E_ARG; }
    HGA_TRY(check_read_off("hga_sdk_count_packed", read_off, n_reads));
    const uint64_t n_bases = read_off[n_reads];
    if (n_bases && !packed) { hga_set_error("hga_sdk_count_packed: packed is NULL"); return HGA_E_ARG; }
    HGA_TRY(check_exc_runs("hga_sdk_count_packed", exc_start, exc_end, n_exc, n_bases));
    if (n_files < 1 || !file_first_read) { hga_set_error("hga_sdk_count_packed: %s", n_files < 1 ? "n_files must be at least 1" : "file_first_read is NULL"); return HGA_E_ARG; }
    if (file_first_read[0] != 0 || file_first_read[n_files] != n_reads) {
        hga_set_error("hga_sdk_count_packed: file_first_read must start at 0 and end at n_reads (%llu)", (unsigned long long) n_reads);
        return HGA_E_ARG;
    }
    for (int f = 0; f < n_files; f++)
        if (file_first_read[f + 1] < file_first_read[f]) { hga_set_error("hga_sdk_count_packed: file_first_read decreases at file %d", f); return HGA_E_ARG; }
    return hga_sdk_run("hga_sdk_count_packed", device, k, packed, first_base, read_off, n_reads, exc_start, exc_end, n_exc, n_files, file_first_read, min_count, out);
}

int hga_count_spectrum_packed(int device, int k, const uint8_t *packed, uint64_t first_base, const uint64_t *read_off, uint64_t n_reads, const uint64_t *exc_start,
                              const uint64_t *exc_end, uint64_t n_exc, uint32_t n_bins, uint64_t *hist, hga_kmer_spectrum_t *out) {
    if (out) std::memset(out, 0, sizeof *out);
    if (hist && n_bins) std::memset(hist, 0, (size_t) n_bins * 8);
    if (!out || (n_bins && !hist)) { hga_set_error("hga_count_spectrum_packed: NULL argument"); return HGA_E_ARG; }
    if (!read_off) { hga_set_error("hga_count_spectrum_packed: read_off is NULL"); return HGA_E_ARG; }
    if (k < 1 || k > 32) { hga_set_error("Kmer size is too big or too small (k = %d)", k); return HGA_E_ARG; }
    HGA_TRY(check_read_off("hga_count_spectrum_packed", read_off, n_reads));
    const uint64_t n_bases = read_off[n_reads];
    if (n_bases && !packed) { hga_set_error("hga_count_spectrum_packed: packed is NULL"); return HGA_E_ARG; }
    HGA_TRY(check_exc_runs("hga_count_spectrum_packed", exc_start, exc_end, n_exc, n_bases));
    return hga_count_run("hga_count_spectrum_packed", device, k, nullptr, packed, first_base, read_off, n_reads, exc_start, exc_end, n_exc, 0, nullptr, out, n_bins, hist);
}

int hga_scan_packed_device(hga_handle *h, const uint8_t *d_packed, uint64_t first_base, const uint64_t *d_read_off, uint64_t n_reads, uint64_t n_bases,
                           const uint64_t *d_exc_start, const uint64_t *d_exc_end, uint64_t n_exc, uint32_t read_id_base) {
    if (!h) { hga_set_error("NULL handle"); return HGA_E_ARG; }
    if ((n_bases && !d_packed) || !d_read_off) { hga_set_error("hga_scan_packed_device: NULL buffer"); return HGA_E_ARG; }
    if (n_exc && (!d_exc_start || !d_exc_end)) { hga_set_error("hga_scan_packed_device: exception runs are NULL"); return HGA_E_ARG; }
    if (n_exc > n_bases) { hga_set_error("hga_scan_packed_device: %llu exception runs for %llu bases", (unsigned long long) n_exc, (unsigned long long) n_bases); return HGA_E_ARG; }
    HGA_TRY(use_device(h));
    h->read_id_base = read_id_base;
    ScanPackedInput in;
    in.sub = (uint32_t) (first_base & 3);
    in.d_exc_start = d_exc_start; in.d_exc_end = d_exc_end; in.h_exc_start = in.h_exc_end = nullptr; in.n_exc = n_exc;
    return hga_scan_run(h, reinterpret_cast<const char *>(d_packed + first_base / 4), d_read_off, n_reads, n_bases, nullptr, &in, "hga_scan_packed_device");
}

int hga_get_hits(hga_handle *h, int sorted_by_kmer_id, hga_hits *out) {
    if (!h || !out) { hga_set_error("NULL argument"); return HGA_E_ARG; }
    if (!h->have_scan) { hga_set_error("hga_get_hits: no scan result"); return HGA_E_STATE; }
    HGA_TRY(use_device(h));
    const uint64_t E = h->n_hits, R = h->n_reads;
    HGA_TRY(h->d_export_a.ensure((E + 1) * 4));
    uint32_t *d_kid = h->d_export_a.as<uint32_t>();
    HGA_TRY(hga_scan_finish_positions(h));
    const uint32_t *d_pos = h->d_hit_pos.as<uint32_t>();
    if (E) {
        slots_to_kids_kernel<<<grid_for(h, E), 256, 0, h->stream>>>(h->d_hit_slot.as<uint32_t>(), h->table.slot_kid, E, d_kid);
        h->metrics.kernel_launches++;
        if (sorted_by_kmer_id) {
            // stable sort of (row << 32 | kmer_id): positions stay ascending inside equal keys
            HGA_TRY(h->d_export_b.ensure((E + 1) * 8 * 2));
            HGA_TRY(h->d_export_c.ensure((E + 1) * 4));
            uint64_t *k_in = h->d_export_b.as<uint64_t>(), *k_out = k_in + (E + 1);
            row_kid_keys_kernel<<<grid_for(h, R * 32), 256, 0, h->stream>>>(h->d_row_off.as<uint64_t>(), R, d_kid, k_in);
            size_t tmp = 0;
            const int bits = 32 + (int) std::max<uint32_t>(hga_ceil_log2(R + 1), 1);
            HGA_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, tmp, k_in, k_out, d_pos, h->d_export_c.as<uint32_t>(), E, 0, bits, h->stream));
            HGA_TRY(h->d_sort_tmp.ensure(tmp + 16));
            HGA_CUDA(cub::DeviceRadixSort::SortPairs(h->d_sort_tmp.p, tmp, k_in, k_out, d_pos, h->d_export_c.as<uint32_t>(), E, 0, bits, h->stream));
            low32_kernel<<<grid_for(h, E), 256, 0, h->stream>>>(k_out, E, d_kid);
            d_pos = h->d_export_c.as<uint32_t>();
            h->metrics.kernel_launches += 8;
        }
        HGA_CUDA(cudaGetLastError());
    }
    HGA_TRY(h->h_row_off.ensure((R + 1) * 8));
    HGA_TRY(h->h_kid.ensure((E + 1) * 4));
    HGA_TRY(h->h_pos.ensure((E + 1) * 4));
    HGA_CUDA(cudaMemcpyAsync(h->h_row_off.p, h->d_row_off.p, (R + 1) * 8, cudaMemcpyDeviceToHost, h->stream));
    if (E) {
        HGA_CUDA(cudaMemcpyAsync(h->h_kid.p, d_kid, E * 4, cudaMemcpyDeviceToHost, h->stream));
        HGA_CUDA(cudaMemcpyAsync(h->h_pos.p, d_pos, E * 4, cudaMemcpyDeviceToHost, h->stream));
    }
    HGA_CUDA(cudaStreamSynchronize(h->stream));
    out->n_reads = R; out->n_hits = E;
    out->row_off = h->h_row_off.as<uint64_t>(); out->kmer_id = h->h_kid.as<uint32_t>(); out->pos = h->h_pos.as<uint32_t>();
    return HGA_OK;
}

int hga_build_index(hga_handle *h) {
    if (!h) { hga_set_error("NULL handle"); return HGA_E_ARG; }
    HGA_TRY(use_device(h));
    return hga_index_run(h);
}

// CSR by table slot (off u32[n_slots + 1], rows) -> CSR by the caller's kmer_id with read ids, in the pinned export buffers
static int export_index(hga_handle *h, const uint32_t *d_off, const uint32_t *d_row, uint64_t E, hga_index *out) {
    const uint64_t K = h->n_kmers;
    HGA_TRY(h->d_export_a.ensure((K + 2) * 8 * 2));
    HGA_TRY(h->d_export_b.ensure((E + 1) * 4));
    unsigned long long *len = h->d_export_a.as<unsigned long long>(), *off = len + (K + 2);
    const uint32_t *kid_slot = h->table.kid_slot;
    const uint32_t G = h->index_by_kid ? (uint32_t) hga_comm_size(h) : 0u, me = (uint32_t) hga_comm_rank(h);
    kid_list_len_kernel<<<grid_for(h, K + 1), 256, 0, h->stream>>>(kid_slot, G, me, d_off, K, len);
    size_t tmp = 0;
    HGA_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, tmp, len, off, K + 1, h->stream));
    HGA_TRY(h->d_sort_tmp.ensure(tmp + 16));
    HGA_CUDA(cub::DeviceScan::ExclusiveSum(h->d_sort_tmp.p, tmp, len, off, K + 1, h->stream));
    if (K) kid_list_copy_kernel<<<grid_for(h, K * 32), 256, 0, h->stream>>>(kid_slot, G, me, d_off, d_row, off, K,
                                                                          h->inc_row_first_id, h->d_export_b.as<uint32_t>());
    h->metrics.kernel_launches += 4;
    HGA_CUDA(cudaGetLastError());
    HGA_TRY(h->h_inv_off.ensure((K + 1) * 8));
    HGA_TRY(h->h_inv_read.ensure((E + 1) * 4));
    HGA_CUDA(cudaMemcpyAsync(h->h_inv_off.p, off, (K + 1) * 8, cudaMemcpyDeviceToHost, h->stream));
    if (E) HGA_CUDA(cudaMemcpyAsync(h->h_inv_read.p, h->d_export_b.p, E * 4, cudaMemcpyDeviceToHost, h->stream));
    HGA_CUDA(cudaStreamSynchronize(h->stream));
    out->n_kmers = K; out->n_entries = h->h_inv_off.as<uint64_t>()[K];
    out->off = h->h_inv_off.as<uint64_t>(); out->read_id = h->h_inv_read.as<uint32_t>();
    return HGA_OK;
}

int hga_get_index(hga_handle *h, hga_index *out) {
    if (!h || !out) { hga_set_error("NULL argument"); return HGA_E_ARG; }
    if (!h->have_index) { hga_set_error("hga_get_index: no index"); return HGA_E_STATE; }
    HGA_TRY(use_device(h));
    return export_index(h, h->d_inv_off.as<uint32_t>(), h->d_inv_row.as<uint32_t>(), h->inc_entries, out);
}

int hga_enrich(hga_handle *h, int min_size, uint32_t enrichment_min_score) {
    if (!h) { hga_set_error("NULL handle"); return HGA_E_ARG; }
    HGA_TRY(use_device(h));
    return hga_enrich_run(h, min_size, -1, enrichment_min_score, nullptr);
}

int hga_enrich_ex(hga_handle *h, int min_size, int max_size, uint32_t enrichment_min_score) {
    if (!h) { hga_set_error("NULL handle"); return HGA_E_ARG; }
    HGA_TRY(use_device(h));
    return hga_enrich_run(h, min_size, max_size, enrichment_min_score, nullptr);
}

int hga_enrich_full(hga_handle *h, int min_size, int max_size, uint32_t enrichment_min_score, uint32_t tail_amplification_min_score, int spectral_dims,
                    const uint64_t *read_off) {
    if (!h || !read_off) { hga_set_error("NULL argument"); return HGA_E_ARG; }
    if (spectral_dims < 2) { hga_set_error("hga_enrich_full: spectral_dims must be >= 2"); return HGA_E_ARG; }
    HGA_TRY(use_device(h));
    const TailParams tail{read_off, tail_amplification_min_score, spectral_dims};
    return hga_enrich_run(h, min_size, max_size, enrichment_min_score, &tail);
}

int hga_get_tail_block(hga_handle *h, hga_tail_block_t *out) {
    if (!h || !out) { hga_set_error("NULL argument"); return HGA_E_ARG; }
    if (!h->have_enrichment) { hga_set_error("hga_get_tail_block: no enrichment result"); return HGA_E_STATE; }
    const EnrichResult &r = h->enrich;
    out->ran = r.tail_block_ran ? 1 : 0;
    out->n_scaffold_cores = r.n_scaffold_cores;
    out->n_connections = r.tconn_x.size(); out->conn_x = r.tconn_x.data(); out->conn_y = r.tconn_y.data(); out->conn_score = r.tconn_score.data();
    out->n_clusters = r.cluster_off.empty() ? 0 : r.cluster_off.size() - 1; out->cluster_off = r.cluster_off.data(); out->cluster_member = r.cluster_member.data();
    return HGA_OK;
}

int hga_get_enrichment(hga_handle *h, hga_enrichment_t *out) {
    if (!h || !out) { hga_set_error("NULL argument"); return HGA_E_ARG; }
    if (!h->have_enrichment) { hga_set_error("hga_get_enrichment: no enrichment result"); return HGA_E_STATE; }
    const EnrichResult &r = h->enrich;
    out->n_cores = r.core_id.size(); out->core_id = r.core_id.data(); out->core_off = r.core_off.data(); out->core_read = r.core_read.data();
    out->n_connections = r.conn_x.size(); out->conn_x = r.conn_x.data(); out->conn_y = r.conn_y.data(); out->conn_score = r.conn_score.data();
    out->n_final = r.final_id.size(); out->final_id = r.final_id.data(); out->final_off = r.final_off.data(); out->final_read = r.final_read.data();
    out->n_reads = r.assignment.size(); out->read_id_first = h->inc_row_first_id; out->assignment = r.assignment.data();
    return HGA_OK;
}

int hga_get_purged_index(hga_handle *h, hga_index *out) {
    if (!h || !out) { hga_set_error("NULL argument"); return HGA_E_ARG; }
    if (!h->have_enrichment) { hga_set_error("hga_get_purged_index: no enrichment result"); return HGA_E_STATE; }
    HGA_TRY(use_device(h));
    return export_index(h, h->d_purged_off.as<uint32_t>(), h->d_purged_row.as<uint32_t>(), h->n_purged, out);
}

int hga_get_core_kmers(hga_handle *h, hga_core_kmers_t *out) {
    if (!h || !out) { hga_set_error("NULL argument"); return HGA_E_ARG; }
    if (!h->have_enrichment) { hga_set_error("hga_get_core_kmers: no enrichment result"); return HGA_E_STATE; }
    HGA_TRY(use_device(h));
    const uint64_t n = h->n_core_kmers, C = h->enrich.core_id.size();
    HGA_TRY(h->d_export_a.ensure((n + 1) * 4 * 2));
    uint32_t *d_slot = h->d_export_a.as<uint32_t>(), *d_kid = d_slot + (n + 1);
    HGA_TRY(h->h_kid.ensure((n + 1) * 4));
    HGA_TRY(h->h_row_off.ensure((C + 2) * 8));
    if (n) {
        low32_kernel<<<grid_for(h, n), 256, 0, h->stream>>>(h->d_enr_keys.as<uint64_t>(), n, d_slot);
        slots_to_kids_kernel<<<grid_for(h, n), 256, 0, h->stream>>>(d_slot, h->table.slot_kid, n, d_kid);
        h->metrics.kernel_launches += 2;
        HGA_CUDA(cudaGetLastError());
        HGA_CUDA(cudaMemcpyAsync(h->h_kid.p, d_kid, n * 4, cudaMemcpyDeviceToHost, h->stream));
    }
    HGA_CUDA(cudaMemcpyAsync(h->h_row_off.p, h->d_enr_core_koff.p, (C + 1) * 8, cudaMemcpyDeviceToHost, h->stream));
    HGA_CUDA(cudaStreamSynchronize(h->stream));
    out->n_cores = C; out->off = h->h_row_off.as<uint64_t>(); out->kmer_id = h->h_kid.as<uint32_t>();
    return HGA_OK;
}

int hga_pair_count(hga_handle *h, uint32_t min_score, const uint32_t *pivots, uint64_t n_pivots) {
    if (!h) { hga_set_error("NULL handle"); return HGA_E_ARG; }
    if (n_pivots && !pivots) { hga_set_error("hga_pair_count: pivots is NULL"); return HGA_E_ARG; }
    HGA_TRY(use_device(h));
    return hga_pairs_run(h, min_score, pivots, n_pivots);
}

static int export_pairs(hga_handle *h, const uint64_t *d_key, const uint32_t *d_score, uint64_t n, PinBuf &hx, PinBuf &hy, PinBuf &hs) {
    HGA_TRY(h->d_export_a.ensure((n + 1) * 4 * 2));
    uint32_t *dx = h->d_export_a.as<uint32_t>(), *dy = dx + (n + 1);
    HGA_TRY(hx.ensure((n + 1) * 4)); HGA_TRY(hy.ensure((n + 1) * 4)); HGA_TRY(hs.ensure((n + 1) * 4));
    if (n) {
        split_keys_kernel<<<grid_for(h, n), 256, 0, h->stream>>>(d_key, n, h->inc_row_first_id, dx, dy);
        h->metrics.kernel_launches++;
        HGA_CUDA(cudaGetLastError());
        HGA_CUDA(cudaMemcpyAsync(hx.p, dx, n * 4, cudaMemcpyDeviceToHost, h->stream));
        HGA_CUDA(cudaMemcpyAsync(hy.p, dy, n * 4, cudaMemcpyDeviceToHost, h->stream));
        HGA_CUDA(cudaMemcpyAsync(hs.p, d_score, n * 4, cudaMemcpyDeviceToHost, h->stream));
    }
    HGA_CUDA(cudaStreamSynchronize(h->stream));
    return HGA_OK;
}

int hga_get_pairs(hga_handle *h, hga_pairs *out) {
    if (!h || !out) { hga_set_error("NULL argument"); return HGA_E_ARG; }
    if (!h->have_pairs) { hga_set_error("hga_get_pairs: no pairs"); return HGA_E_STATE; }
    HGA_TRY(use_device(h));
    HGA_TRY(export_pairs(h, h->d_pair_key.as<uint64_t>(), h->d_pair_score.as<uint32_t>(), h->n_pairs, h->h_px, h->h_py, h->h_ps));
    out->n_pairs = h->n_pairs; out->n_increments = h->n_increments;
    out->x = h->h_px.as<uint32_t>(); out->y = h->h_py.as<uint32_t>(); out->score = h->h_ps.as<uint32_t>();
    return HGA_OK;
}

int hga_select_edges(hga_handle *h, double fraction, uint32_t score_threshold) {
    if (!h) { hga_set_error("NULL handle"); return HGA_E_ARG; }
    if (!(fraction >= 0.0 && fraction <= 1.0)) { hga_set_error("hga_select_edges: fraction must be in [0, 1]"); return HGA_E_ARG; }
    HGA_TRY(use_device(h));
    return hga_select_run(h, fraction, score_threshold);
}

int hga_get_selection(hga_handle *h, hga_selection *out) {
    if (!h || !out) { hga_set_error("NULL argument"); return HGA_E_ARG; }
    if (!h->have_selection) { hga_set_error("hga_get_selection: no selection"); return HGA_E_STATE; }
    HGA_TRY(use_device(h));
    HGA_TRY(export_pairs(h, h->d_sel_key.as<uint64_t>(), h->d_sel_score.as<uint32_t>(), h->n_selected, h->h_sx, h->h_sy, h->h_ss));
    out->n_directed = h->sel_n_directed; out->cut_score = h->sel_cut; out->n_selected = h->n_selected;
    out->x = h->h_sx.as<uint32_t>(); out->y = h->h_sy.as<uint32_t>(); out->score = h->h_ss.as<uint32_t>();
    return HGA_OK;
}

int hga_components(hga_handle *h, int min_size) {
    if (!h) { hga_set_error("NULL handle"); return HGA_E_ARG; }
    HGA_TRY(use_device(h));
    return hga_cc_run(h, min_size);
}

int hga_get_components(hga_handle *h, hga_components_t *out) {
    if (!h || !out) { hga_set_error("NULL argument"); return HGA_E_ARG; }
    if (!h->have_components) { hga_set_error("hga_get_components: no components"); return HGA_E_STATE; }
    HGA_TRY(use_device(h));
    const uint64_t n = h->inc_rows, nc = h->n_components;
    const uint32_t *label = h->d_parent.as<uint32_t>() + (n + 1);
    HGA_TRY(h->d_export_a.ensure((n + nc + 2) * 4));
    uint32_t *d_l = h->d_export_a.as<uint32_t>(), *d_c = d_l + (n + 1);
    if (n) add_u32_kernel<<<grid_for(h, n), 256, 0, h->stream>>>(label, n, h->inc_row_first_id, d_l);
    if (nc) add_u32_kernel<<<grid_for(h, nc), 256, 0, h->stream>>>(h->d_comp_label.as<uint32_t>(), nc, h->inc_row_first_id, d_c);
    h->metrics.kernel_launches += 2;
    HGA_CUDA(cudaGetLastError());
    HGA_TRY(h->h_label.ensure((n + 1) * 4)); HGA_TRY(h->h_clabel.ensure((nc + 1) * 4)); HGA_TRY(h->h_csize.ensure((nc + 1) * 4));
    if (n) HGA_CUDA(cudaMemcpyAsync(h->h_label.p, d_l, n * 4, cudaMemcpyDeviceToHost, h->stream));
    if (nc) {
        HGA_CUDA(cudaMemcpyAsync(h->h_clabel.p, d_c, nc * 4, cudaMemcpyDeviceToHost, h->stream));
        HGA_CUDA(cudaMemcpyAsync(h->h_csize.p, h->d_comp_size.p, nc * 4, cudaMemcpyDeviceToHost, h->stream));
    }
    HGA_CUDA(cudaStreamSynchronize(h->stream));
    out->n_reads = n; out->read_id_first = h->inc_row_first_id;
    out->label = h->h_label.as<uint32_t>(); out->n_components = nc;
    out->comp_label = h->h_clabel.as<uint32_t>(); out->comp_size = h->h_csize.as<uint32_t>();
    return HGA_OK;
}

int hga_metrics(hga_handle *h, hga_metrics_t *out) {
    if (!h || !out) { hga_set_error("NULL argument"); return HGA_E_ARG; }
    *out = h->metrics;
    return HGA_OK;
}

}  // extern "C"

int hga_export_index(hga_handle *h, const uint32_t *d_off, const uint32_t *d_row, uint64_t E, hga_index *out) { return export_index(h, d_off, d_row, E, out); }
