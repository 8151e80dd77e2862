// Inverted index (k-mer -> rows) from the by-read incidence.
// Replaces the kmer_component_index half of construct_indices
// (clustering/ReadClusteringEngine.cpp:262-269 push_back per occurrence, :282-284 sort of every list).
//
// A stable LSD radix sort of (slot, row) pairs by slot keeps rows ascending inside every list because the
// incidence is already ordered by row; offsets come from run boundaries of the sorted keys.
#include "hga_internal.cuh"

#include <cub/device/device_radix_sort.cuh>

namespace {

// one warp per row: out_row[row_off[r] .. row_off[r+1]) = r
__global__ void expand_rows_kernel(const uint64_t *__restrict__ row_off, uint64_t n_rows, uint32_t *__restrict__ out_row) {
    const uint64_t warps = ((uint64_t) gridDim.x * blockDim.x) >> 5;
    const uint64_t w = (blockIdx.x * (uint64_t) blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    for (uint64_t r = w; r < n_rows; r += warps) {
        const uint64_t a = row_off[r], b = row_off[r + 1];
        for (uint64_t i = a + lane; i < b; i += 32) out_row[i] = (uint32_t) r;
    }
}

// inv_off[s] = first position whose key is >= s (keys sorted ascending)
__global__ void run_offsets_kernel(const uint32_t *__restrict__ keys, uint64_t n, uint32_t n_slots, uint32_t *__restrict__ inv_off) {
    uint64_t i = blockIdx.x * (uint64_t) blockDim.x + threadIdx.x;
    const uint64_t stride = (uint64_t) gridDim.x * blockDim.x;
    for (; i <= n; i += stride) {
        const uint32_t cur = (i < n) ? keys[i] : n_slots;          // sentinel closes the tail
        const int64_t prev = (i == 0) ? -1 : (int64_t) keys[i - 1];
        for (int64_t s = prev + 1; s <= (int64_t) cur; s++) inv_off[s] = (uint32_t) i;
    }
}

// goff[g] = first position whose group (key >> shift) is >= g, g = 0 .. n_groups (keys sorted ascending by group)
__global__ void group_offsets_kernel(const uint32_t *__restrict__ keys, uint64_t n, uint32_t n_groups, int shift, uint32_t *__restrict__ goff) {
    uint64_t i = blockIdx.x * (uint64_t) blockDim.x + threadIdx.x;
    const uint64_t stride = (uint64_t) gridDim.x * blockDim.x;
    for (; i <= n; i += stride) {
        const uint32_t cur = (i < n) ? (keys[i] >> shift) : n_groups;
        const int64_t prev = (i == 0) ? -1 : (int64_t) (keys[i - 1] >> shift);
        for (int64_t g = prev + 1; g <= (int64_t) cur; g++) goff[g] = (uint32_t) i;
    }
}

// The last radix pass done locally. The (slot, row) pairs arrive sorted by GROUP = slot >> L (L <= 5: a group is at most one key
// bucket, a few hundred entries, contiguous) and in row order inside a group. One warp per group: a counting sort over the low L
// bits (lane s keeps the counter of slot s of the group in shared memory), stable because the entries of a step are ranked by lane
// (__match_any_sync) and the steps run in order. Writes the rows of every list ascending AND the list offsets (what run_offsets_kernel
// needed another pass over the sorted keys for). Reads 8 B, writes 4 B per entry, all inside one ~1 KB window per warp.
// lanes holding the same 5-bit key (idle lanes pass k >= 32 and get an empty mask back): five ballots instead of __match_any_sync
__device__ __forceinline__ uint32_t same_key_lanes(uint32_t k) {
    uint32_t peers = __ballot_sync(0xFFFFFFFFu, k < 32u);
    #pragma unroll
    for (int b = 0; b < 5; b++) {
        const uint32_t bal = __ballot_sync(0xFFFFFFFFu, (k >> b) & 1u);
        peers &= ((k >> b) & 1u) ? bal : ~bal;
    }
    return k < 32u ? peers : 0u;
}

#define IDX_WARPS 8
#define IDX_REG 8                                // entries per lane kept in registers
__global__ void __launch_bounds__(IDX_WARPS * 32) index_local_sort_kernel(const uint32_t *__restrict__ keys, const uint32_t *__restrict__ rows,
                                                                            const uint32_t *__restrict__ goff, uint32_t n_groups, int L, uint32_t n_entries,
                                                                            uint32_t *__restrict__ inv_off, uint32_t *__restrict__ inv_row) {
    __shared__ uint32_t s_cnt[IDX_WARPS][32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint32_t *cnt = s_cnt[warp];
    const uint32_t mask = (1u << L) - 1, lt = (1u << lane) - 1;
    const uint64_t warps = ((uint64_t) gridDim.x * blockDim.x) >> 5;
    for (uint64_t g = (blockIdx.x * (uint64_t) blockDim.x + threadIdx.x) >> 5; g < n_groups; g += warps) {
        const uint32_t lo = __ldg(&goff[g]), hi = __ldg(&goff[g + 1]);
        const uint32_t n = hi - lo;
        // groups of up to IDX_REG * 32 entries (all but repeats) are loaded ONCE, all loads in flight together, and sorted from registers;
        // larger ones re-read their entries in the second sweep
        uint32_t kk[IDX_REG], rr[IDX_REG];
        const bool in_regs = n <= IDX_REG * 32;
        if (in_regs) {
            #pragma unroll
            for (int u = 0; u < IDX_REG; u++) {
                const uint32_t i = lo + u * 32 + lane;
                const bool valid = i < hi;
                kk[u] = valid ? (__ldg(&keys[i]) & mask) : 32u + lane;                 // idle lanes: keys of their own
                rr[u] = valid ? __ldg(&rows[i]) : 0u;
            }
        }
        cnt[lane] = 0;
        __syncwarp();
        // counts: one shared-memory increment per entry (the hardware serialises equal slots)
        if (in_regs) {
            #pragma unroll
            for (int u = 0; u < IDX_REG; u++)
                if (kk[u] < 32u) atomicAdd(&cnt[kk[u]], 1u);
        } else {
            for (uint32_t i = lo + lane; i < hi; i += 32) atomicAdd(&cnt[__ldg(&keys[i]) & mask], 1u);
        }
        __syncwarp();
        // exclusive prefix over the group's slots -> list offsets
        const uint32_t c = cnt[lane];
        uint32_t incl = c;
        #pragma unroll
        for (int d = 1; d < 32; d <<= 1) { const uint32_t t = __shfl_up_sync(0xFFFFFFFFu, incl, d); if (lane >= d) incl += t; }
        const uint32_t start = lo + incl - c;
        if ((uint32_t) lane <= mask) inv_off[(g << L) + lane] = start;
        __syncwarp();
        cnt[lane] = start;                                                             // now: where the next entry of slot `lane` goes
        __syncwarp();
        if (in_regs) {
            #pragma unroll
            for (int u = 0; u < IDX_REG; u++) {
                if ((uint32_t) u * 32 < n) {
                    const bool valid = kk[u] < 32u;
                    const uint32_t peers = same_key_lanes(kk[u]);
                    uint32_t at = 0;
                    if (valid) at = cnt[kk[u]] + __popc(peers & lt);
                    __syncwarp();
                    if (valid) {
                        inv_row[at] = rr[u];
                        if ((peers & lt) == 0) cnt[kk[u]] += __popc(peers);
                    }
                    __syncwarp();
                }
            }
        } else {
            for (uint32_t base = lo; base < hi; base += 32) {
                const uint32_t i = base + lane;
                const bool valid = i < hi;
                const uint32_t k = valid ? (__ldg(&keys[i]) & mask) : 32u + lane;
                const uint32_t r = valid ? __ldg(&rows[i]) : 0u;
                const uint32_t peers = same_key_lanes(k);
                uint32_t at = 0;
                if (valid) at = cnt[k] + __popc(peers & lt);
                __syncwarp();
                if (valid) {
                    inv_row[at] = r;
                    if ((peers & lt) == 0) cnt[k] += __popc(peers);
                }
                __syncwarp();
            }
        }
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) inv_off[(size_t) n_groups << L] = n_entries;
}

}  // namespace

// Inverted lists from the by-row incidence (CSR: d_row_off u64[n_rows + 1], d_keys u32[E], keys < n_keys, n_keys a multiple of 32 or L = 0
// is used). On return h->d_inv_off[0 .. n_keys] / h->d_inv_row hold the lists, rows ascending inside a list. d_keys is left untouched (the
// pair counter walks it as the by-row incidence).
int hga_build_lists(hga_handle *h, const uint32_t *d_keys, const uint64_t *d_row_off, uint64_t n_rows, uint64_t E, uint32_t n_keys) {
    HGA_TRY(h->d_sort_b.ensure((E + 1) * 4));     // the row of every pair, expanded from the row offsets
    uint32_t *d_rows = h->d_sort_b.as<uint32_t>();
    if (E > 0) {
        const int blocks = (int) std::min<uint64_t>((n_rows * 32 + 255) / 256, (uint64_t) h->sm_count * 32);
        expand_rows_kernel<<<blocks, 256, 0, h->stream>>>(d_row_off, n_rows, d_rows);
        h->metrics.kernel_launches++;
        HGA_CUDA(cudaGetLastError());
    }
    HGA_TRY(h->d_inv_off.ensure(((size_t) n_keys + 2) * 4));
    HGA_TRY(h->d_inv_row.ensure((E + 4) * 4));
    HGA_TRY(h->d_sort_a.ensure((E + 1) * 4));     // sorted keys
    uint32_t *inv_off = h->d_inv_off.as<uint32_t>();
    if (E == 0) {
        HGA_CUDA(cudaMemsetAsync(inv_off, 0, ((size_t) n_keys + 1) * 4, h->stream));
        return HGA_OK;
    }
    size_t tmp_bytes = 0;
    const int end_bit = (int) std::max<uint32_t>(hga_ceil_log2(n_keys), 1);
    // Radix passes are 8 bits wide. When leaving the low L <= 5 bits out saves a whole pass (config 4: 28 bits = 4 passes, 23 = 3), the
    // sort runs over the GROUP bits only and index_local_sort_kernel finishes the order inside the groups.
    int L = 0;
    if (end_bit > 8 && (end_bit - 1) % 8 < 5 && n_keys % 32 == 0) L = 5;
    uint32_t *d_sorted_rows = h->d_inv_row.as<uint32_t>();
    if (L) { HGA_TRY(h->d_index_tmp.ensure((E + 1) * 4)); d_sorted_rows = h->d_index_tmp.as<uint32_t>(); }
    HGA_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, tmp_bytes, d_keys, h->d_sort_a.as<uint32_t>(), d_rows, d_sorted_rows, E, L, end_bit, h->stream));
    HGA_TRY(h->d_sort_tmp.ensure(tmp_bytes + 16));
    HGA_CUDA(cub::DeviceRadixSort::SortPairs(h->d_sort_tmp.p, tmp_bytes, d_keys, h->d_sort_a.as<uint32_t>(), d_rows, d_sorted_rows, E, L, end_bit, h->stream));
    h->metrics.kernel_launches += (uint64_t) (end_bit - L + 7) / 8 + 2;   // CUB: histogram + onesweep passes
    const int oblocks = (int) std::min<uint64_t>((E + 256) / 256, (uint64_t) h->sm_count * 16);
    if (L) {
        const uint32_t n_groups = n_keys >> L;
        HGA_TRY(h->d_index_goff.ensure(((size_t) n_groups + 2) * 4));
        group_offsets_kernel<<<oblocks, 256, 0, h->stream>>>(h->d_sort_a.as<uint32_t>(), E, n_groups, L, h->d_index_goff.as<uint32_t>());
        const int lblocks = (int) std::max<uint64_t>(1, std::min<uint64_t>(((uint64_t) n_groups + IDX_WARPS - 1) / IDX_WARPS, (uint64_t) h->sm_count * 8));
        index_local_sort_kernel<<<lblocks, IDX_WARPS * 32, 0, h->stream>>>(h->d_sort_a.as<uint32_t>(), d_sorted_rows, h->d_index_goff.as<uint32_t>(), n_groups, L,
                                                                          (uint32_t) E, inv_off, h->d_inv_row.as<uint32_t>());
        h->metrics.kernel_launches += 2;
    } else {
        run_offsets_kernel<<<oblocks, 256, 0, h->stream>>>(h->d_sort_a.as<uint32_t>(), E, n_keys, inv_off);
        h->metrics.kernel_launches++;
    }
    HGA_CUDA(cudaGetLastError());
    return HGA_OK;
}

int hga_index_run(hga_handle *h) {
    if (!h->have_scan) { hga_set_error("hga_build_index: no scan result"); return HGA_E_STATE; }
    h->have_index = h->have_pairs = h->have_selection = h->have_components = false;
    const uint32_t n_slots = h->table.n_slots;

    if (h->comm && hga_comm_size(h) > 1) {
        // sharded reads: all-to-all by k-mer owner into a PARTITIONED index (hga_comm.cu)
        StageTimer timer(h, &h->metrics.index_ms);
        HGA_TRY(hga_comm_build_owner_index(h));
        timer.stop();
        h->have_index = true;
        return HGA_OK;
    }
    h->inc_rows = h->n_reads;
    h->pair_rows = h->n_reads; h->pair_pivot_mul = 1; h->pair_pivot_add = 0;
    h->index_by_kid = false; h->index_keys = n_slots;
    h->inc_row_first_id = h->read_id_base;
    h->inc_entries = h->n_hits;
    const uint64_t E = h->inc_entries;
    if (E >= (1ull << 32)) { hga_set_error("incidence of %llu entries exceeds the 32-bit per-GPU limit", (unsigned long long) E); return HGA_E_OVERFLOW; }

    StageTimer timer(h, &h->metrics.index_ms);
    HGA_TRY(hga_build_lists(h, h->d_hit_slot.as<uint32_t>(), h->d_row_off.as<uint64_t>(), h->inc_rows, E, n_slots));
    timer.stop();
    h->have_index = true;
    return HGA_OK;
}
