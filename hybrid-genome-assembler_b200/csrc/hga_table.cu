// Device construction of the discriminative k-mer membership structures (layout: hga_internal.cuh).
// Replaces std::unordered_set<Kmer>::contains + KmerIndex of the reference
// (clustering/ReadClusteringEngine.cpp:237-241, :251, :263).
#include "hga_internal.cuh"

#include <cub/device/device_radix_sort.cuh>

#include <cstdlib>

namespace {

// The table layout is a FUNCTION of the k-mer array (no insertion races): every rank of a multi-GPU job builds the same table from the
// same array, so a slot number means the same k-mer everywhere and the inverted index can be partitioned by slot (hga_comm.cu).
//   1. table_bucket_kernel: filter bits (an OR: order free) and the home bucket of every k-mer;
//   2. stable radix sort of the k-mer numbers by bucket: inside a bucket the k-mers stand in kmer_id order;
//   3. table_place_kernel: one thread per bucket places its k-mers in that order (first free slot from the start sector, going round);
//      k-mers whose bucket is full are listed;
//   4. the listed k-mers, sorted by value, form the overflow region (a sorted array, looked up by binary search: 0.1 % of the keys).

__global__ void table_bucket_kernel(const uint64_t *__restrict__ kmers, uint64_t n, KmerTable t, uint32_t *__restrict__ bucket_of, uint32_t *__restrict__ idx, int *flags) {
    uint64_t i = blockIdx.x * (uint64_t) blockDim.x + threadIdx.x;
    const uint64_t stride = (uint64_t) gridDim.x * blockDim.x;
    for (; i < n; i += stride) {
        const unsigned long long key = kmers[i];
        idx[i] = (uint32_t) i;
        if (key == HGA_EMPTY_KEY) { atomicOr(flags, 2); bucket_of[i] = t.n_buckets; continue; }   // never a canonical k-mer
        const uint32_t hb = hga_bits_hash(key, t.geom);
        const uint32_t B = hga_locality_from_min(hga_minimizer(key, hb, t.geom));
        atomicOr(&t.filter[(size_t) hga_scale(B, t.n_blocks) * 8 + hga_bits_word(hb)], hga_bits_mask(hb));
        bucket_of[i] = hga_scale(B, t.n_buckets);
    }
}

// boff[b] = first position of the ascending bucket numbers with value >= b, b = 0 .. n_buckets
__global__ void table_bucket_offsets_kernel(const uint32_t *__restrict__ sorted_bucket, uint64_t n, uint32_t n_buckets, uint32_t *__restrict__ boff) {
    uint64_t i = blockIdx.x * (uint64_t) blockDim.x + threadIdx.x;
    const uint64_t stride = (uint64_t) gridDim.x * blockDim.x;
    for (; i <= n; i += stride) {
        const int64_t cur = (i < n) ? (int64_t) min(sorted_bucket[i], n_buckets) : (int64_t) n_buckets;
        const int64_t prev = (i == 0) ? -1 : (int64_t) min(sorted_bucket[i - 1], n_buckets);
        for (int64_t b = prev + 1; b <= cur; b++) boff[b] = (uint32_t) i;
    }
}

__global__ void table_place_kernel(const uint64_t *__restrict__ kmers, const uint32_t *__restrict__ sorted_idx, const uint32_t *__restrict__ boff, KmerTable t,
                                   uint32_t *over_list, unsigned int *over_count, int *flags) {
    unsigned long long *keys = reinterpret_cast<unsigned long long *>(t.keys);
    for (uint32_t b = blockIdx.x * blockDim.x + threadIdx.x; b < t.n_buckets; b += gridDim.x * blockDim.x) {
        const uint32_t home = b * HGA_BUCKET_SLOTS;
        for (uint32_t p = boff[b]; p < boff[b + 1]; p++) {
            const uint32_t i = sorted_idx[p];
            const unsigned long long key = kmers[i];
            const uint32_t start = hga_start_sector(hga_bits_hash(key, t.geom)) * HGA_SECTOR_SLOTS;
            bool done = false;
            for (uint32_t j = 0; j < HGA_BUCKET_SLOTS && !done; j++) {
                const uint32_t slot = home + ((start + j) & (HGA_BUCKET_SLOTS - 1));
                const unsigned long long cur = keys[slot];                 // this thread is the bucket's only writer
                if (cur == HGA_EMPTY_KEY) { keys[slot] = key; t.kid_slot[i] = slot; done = true; }
                else if (cur == key) { atomicOr(flags, 1); t.kid_slot[i] = slot; done = true; }   // duplicate
            }
            if (!done) over_list[atomicAdd(over_count, 1u)] = i;
        }
    }
}

__global__ void table_gather_keys_kernel(const uint64_t *__restrict__ kmers, const uint32_t *__restrict__ list, uint32_t n_list, uint64_t *__restrict__ out) {
    for (uint32_t q = blockIdx.x * blockDim.x + threadIdx.x; q < n_list; q += gridDim.x * blockDim.x) out[q] = kmers[list[q]];
}

// overflow region = the listed k-mers in ascending order (then HGA_EMPTY_KEY padding, which sorts last)
__global__ void table_place_over_kernel(const uint64_t *__restrict__ sorted_keys, const uint32_t *__restrict__ sorted_kid, uint32_t n_list, KmerTable t, int *flags) {
    for (uint32_t q = blockIdx.x * blockDim.x + threadIdx.x; q < n_list; q += gridDim.x * blockDim.x) {
        t.keys[t.n_main + q] = sorted_keys[q];
        t.kid_slot[sorted_kid[q]] = t.n_main + q;
        if (q > 0 && sorted_keys[q - 1] == sorted_keys[q]) atomicOr(flags, 1);
    }
}

__global__ void table_slot_kid_kernel(const uint32_t *__restrict__ kid_slot, uint64_t n, uint32_t *slot_kid) {
    for (uint64_t i = blockIdx.x * (uint64_t) blockDim.x + threadIdx.x; i < n; i += (uint64_t) gridDim.x * blockDim.x) slot_kid[kid_slot[i]] = (uint32_t) i;
}

}  // namespace

int hga_table_build(hga_handle *h, const uint64_t *host_kmers) {
    const uint64_t n = h->n_kmers;
    if (n >= (1ull << 29)) { hga_set_error("too many k-mers (%llu): the slot id space is 32 bit", (unsigned long long) n); return HGA_E_ARG; }
    // filter: 16 bits per key, at most 48 MB so that it stays L2 resident (see hga_internal.cuh). HGA_TABLE_LOAD sets the key table's load
    // factor (0.25) so that tests can fill buckets and reach the overflow region with small sets
    const double bits_per_key = 16.0, max_mb = 48.0;
    double load = 0.25;
    if (const char *e = getenv("HGA_TABLE_LOAD")) load = std::min(0.9, std::max(0.05, atof(e)));
    uint64_t n_blocks = (uint64_t) (n * bits_per_key / 256.0) + 64;
    const uint64_t max_blocks = (uint64_t) (max_mb * 1024 * 1024 / 32);
    if (n_blocks > max_blocks) n_blocks = max_blocks;

    KmerTable &t = h->table;
    t.geom = hga_make_geom(h->k, n);
    t.n_buckets = (uint32_t) ((uint64_t) (n / load) / HGA_BUCKET_SLOTS + 1);
    t.n_main = t.n_buckets * HGA_BUCKET_SLOTS;
    t.n_over = 0;
    t.n_blocks = (uint32_t) n_blocks;
    HGA_TRY(h->d_keys.ensure((size_t) t.n_main * 8));
    HGA_TRY(h->d_kid_slot.ensure((size_t) (n + 1) * 4));
    HGA_TRY(h->d_filter.ensure((size_t) n_blocks * 32));
    t.keys = h->d_keys.as<uint64_t>();
    t.kid_slot = h->d_kid_slot.as<uint32_t>();
    t.filter = h->d_filter.as<uint32_t>();

    DevBuf d_in, d_flags, d_over, d_bk, d_tmp;
    HGA_TRY(d_in.ensure((size_t) (n + 1) * 8));
    HGA_TRY(d_over.ensure((size_t) (n + 1) * 4));
    HGA_TRY(d_flags.ensure(16));
    HGA_TRY(d_bk.ensure((size_t) (n + 1) * 4 * 4 + ((size_t) t.n_buckets + 2) * 4));   // bucket | idx | sorted bucket | sorted idx | bucket offsets
    uint32_t *bucket_of = d_bk.as<uint32_t>(), *idx = bucket_of + (n + 1), *sorted_bucket = idx + (n + 1), *sorted_idx = sorted_bucket + (n + 1), *boff = sorted_idx + (n + 1);
    int *d_fl = d_flags.as<int>();
    unsigned int *d_cnt = reinterpret_cast<unsigned int *>(d_fl + 1);
    StageTimer timer(h, &h->metrics.table_build_ms);
    HGA_CUDA(cudaMemcpyAsync(d_in.p, host_kmers, n * 8, cudaMemcpyHostToDevice, h->stream));
    HGA_CUDA(cudaMemsetAsync(t.keys, 0xff, (size_t) t.n_main * 8, h->stream));
    HGA_CUDA(cudaMemsetAsync(t.filter, 0, (size_t) n_blocks * 32, h->stream));
    HGA_CUDA(cudaMemsetAsync(d_flags.p, 0, 16, h->stream));
    HGA_CUDA(cudaMemsetAsync(t.kid_slot, 0, (size_t) (n + 1) * 4, h->stream));
    int blocks = (int) std::max<uint64_t>(1, std::min<uint64_t>((n + 255) / 256, (uint64_t) h->sm_count * 16));
    if (n) {
        table_bucket_kernel<<<blocks, 256, 0, h->stream>>>(d_in.as<uint64_t>(), n, t, bucket_of, idx, d_fl);
        size_t tmp_bytes = 0;
        const int bits = (int) std::max<uint32_t>(hga_ceil_log2((uint64_t) t.n_buckets + 1), 1);
        HGA_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, tmp_bytes, bucket_of, sorted_bucket, idx, sorted_idx, n, 0, bits, h->stream));
        HGA_TRY(d_tmp.ensure(tmp_bytes + 16));
        HGA_CUDA(cub::DeviceRadixSort::SortPairs(d_tmp.p, tmp_bytes, bucket_of, sorted_bucket, idx, sorted_idx, n, 0, bits, h->stream));
        table_bucket_offsets_kernel<<<blocks, 256, 0, h->stream>>>(sorted_bucket, n, t.n_buckets, boff);
        const int pblocks = (int) std::max<uint32_t>(1, std::min<uint32_t>((t.n_buckets + 127) / 128, (uint32_t) h->sm_count * 16));
        table_place_kernel<<<pblocks, 128, 0, h->stream>>>(d_in.as<uint64_t>(), sorted_idx, boff, t, d_over.as<uint32_t>(), d_cnt, d_fl);
        h->metrics.kernel_launches += 6;
        HGA_CUDA(cudaGetLastError());
    }
    int host_flags[2] = {0, 0};
    HGA_CUDA(cudaMemcpyAsync(host_flags, d_flags.p, 8, cudaMemcpyDeviceToHost, h->stream));
    HGA_CUDA(cudaStreamSynchronize(h->stream));
    const uint32_t n_list = (uint32_t) host_flags[1];
    if (n_list > 0) {
        // grow the key array by the overflow region (main region preserved): the listed k-mers in ascending order, padded to whole buckets
        const uint32_t n_over = (n_list + HGA_BUCKET_SLOTS - 1) / HGA_BUCKET_SLOTS * HGA_BUCKET_SLOTS;
        DevBuf grown, d_ok;
        HGA_TRY(grown.ensure(((size_t) t.n_main + n_over) * 8));
        HGA_TRY(d_ok.ensure((size_t) n_list * (8 + 8 + 4) + 64));
        uint64_t *ok_in = d_ok.as<uint64_t>(), *ok_out = ok_in + n_list;
        uint32_t *kid_out = reinterpret_cast<uint32_t *>(ok_out + n_list);
        HGA_CUDA(cudaMemcpyAsync(grown.p, t.keys, (size_t) t.n_main * 8, cudaMemcpyDeviceToDevice, h->stream));
        HGA_CUDA(cudaMemsetAsync(grown.as<uint64_t>() + t.n_main, 0xff, (size_t) n_over * 8, h->stream));
        HGA_CUDA(cudaStreamSynchronize(h->stream));
        h->d_keys.release();
        h->d_keys = grown;
        t.keys = h->d_keys.as<uint64_t>();
        t.n_over = n_over;
        const int oblocks = (int) std::min<uint32_t>((n_list + 255) / 256, (uint32_t) h->sm_count * 16);
        table_gather_keys_kernel<<<oblocks, 256, 0, h->stream>>>(d_in.as<uint64_t>(), d_over.as<uint32_t>(), n_list, ok_in);
        size_t tmp_bytes = 0;
        HGA_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, tmp_bytes, ok_in, ok_out, d_over.as<uint32_t>(), kid_out, n_list, 0, 64, h->stream));
        HGA_TRY(d_tmp.ensure(tmp_bytes + 16));
        HGA_CUDA(cub::DeviceRadixSort::SortPairs(d_tmp.p, tmp_bytes, ok_in, ok_out, d_over.as<uint32_t>(), kid_out, n_list, 0, 64, h->stream));
        table_place_over_kernel<<<oblocks, 256, 0, h->stream>>>(ok_out, kid_out, n_list, t, d_fl);
        h->metrics.kernel_launches += 4;
        HGA_CUDA(cudaGetLastError());
        HGA_CUDA(cudaMemcpyAsync(host_flags, d_flags.p, 4, cudaMemcpyDeviceToHost, h->stream));
        HGA_CUDA(cudaStreamSynchronize(h->stream));
        d_ok.release();
    }
    t.n_over_keys = n_list;
    t.n_slots = t.n_main + t.n_over;
    t.slot_bits = hga_ceil_log2(t.n_slots);
    HGA_TRY(h->d_slot_kid.ensure((size_t) t.n_slots * 4));
    t.slot_kid = h->d_slot_kid.as<uint32_t>();
    HGA_CUDA(cudaMemsetAsync(t.slot_kid, 0xff, (size_t) t.n_slots * 4, h->stream));
    if (n) {
        table_slot_kid_kernel<<<blocks, 256, 0, h->stream>>>(t.kid_slot, n, t.slot_kid);
        h->metrics.kernel_launches++;
        HGA_CUDA(cudaGetLastError());
    }
    timer.stop();
    d_in.release(); d_flags.release(); d_over.release(); d_bk.release(); d_tmp.release();
    if (host_flags[0] & 2) { hga_set_error("k-mer value 0xFFFFFFFFFFFFFFFF is not a canonical k-mer"); return HGA_E_ARG; }
    if (host_flags[0] & 1) { hga_set_error("duplicate k-mer in the set handed to hga_create"); return HGA_E_DUPLICATE; }
    h->metrics.table_bytes = (uint64_t) t.n_slots * 8;
    h->metrics.filter_bytes = n_blocks * 32;
    h->metrics.table_overflow_keys = n_list;
    return HGA_OK;
}
