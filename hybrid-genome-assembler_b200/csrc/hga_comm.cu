// Multi-GPU exchanges over NCCL (NVLink 5 / NVSwitch), one handle per rank.
//
// The reference has no distributed path; SURVEY.md §8(e) defines this one. Reads shard by contiguous read-id ranges (each rank
// scans its own shard against a replicated k-mer table); the inverted index is PARTITIONED by k-mer owner and the pair scores
// are reduced at the owner of x:
//   1. the table layout is a function of the k-mer array (hga_table.cu), so a slot number means the same k-mer on every rank: whole
//      32-slot buckets are dealt round robin, owner(slot) = (slot / 32) mod G, list number at the owner = (slot / 32) / G * 32 + slot mod 32
//      (the hits of a minimizer run keep neighbouring list numbers: the pair counter's locality survives the partition);
//   2. ALL-TO-ALL 1 (grouped ncclSend / ncclRecv): the u32 list numbers of a source's hits go to their owners in row order, together
//      with one count per row and owner; the rows themselves do not travel. The sources arrive in rank order = global row order, so
//      the owner's by-row incidence is the received stream + an exclusive scan of the counts, and the single-GPU list builder
//      (hga_build_lists) gives its inverted lists with rows ascending. Nothing is replicated: a rank holds E / G incidence entries;
//   3. every rank runs the single-GPU pair kernels over ALL rows as pivots, each row restricted to the hits of the rank's own
//      lists (y > x, list tails only): PARTIAL scores, work = the increments of the owned lists = 1 / G of the total;
//   4. ALL-TO-ALL 2: partial (x, y, score) records, packed into one u64 when they fit, go to owner(x) = x mod G, where one radix sort
//      by (x, y) and a segmented sum give the final scores: every unordered pair ends up on exactly one rank, in canonical order;
//   5. hga_comm_gather_root: for the stages after the scaffold union_find, rank 0 gathers every rank's hits and selected edges and
//      becomes a complete single-GPU handle.
// Edge selection needs two small all-reduces (score histograms) and an all-gather of the tie keys; components iterate
// union-find with all-reduce(min) over the replicated label array.
//
// libnccl is bound at run time (dlopen) so that the library loads on machines without NCCL and shares the copy a
// host process (e.g. torch) has already loaded.
#include "hga_internal.cuh"

#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>
#include <cub/device/device_reduce.cuh>
#include <cub/iterator/transform_input_iterator.cuh>
#include <dlfcn.h>
#include <nccl.h>

struct hga_comm {
    ncclComm_t comm = nullptr;
    int rank = 0, size = 1;
    DevBuf d_small;       // counts / scratch
    DevBuf d_stage;       // padded all-gather staging
    DevBuf d_rows;        // per-row lengths / destinations of the by-read exchange
};

namespace {

struct NcclApi {
    void *lib = nullptr;
    ncclResult_t (*GetUniqueId)(ncclUniqueId *) = nullptr;
    ncclResult_t (*CommInitRank)(ncclComm_t *, int, ncclUniqueId, int) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    ncclResult_t (*AllReduce)(const void *, void *, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*AllGather)(const void *, void *, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*Broadcast)(const void *, void *, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*Send)(const void *, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*Recv)(void *, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*GroupStart)() = nullptr;
    ncclResult_t (*GroupEnd)() = nullptr;
    const char *(*GetErrorString)(ncclResult_t) = nullptr;
};

NcclApi g_nccl;

int load_nccl() {
    if (g_nccl.lib) return HGA_OK;
    void *lib = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
    if (!lib) lib = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
    if (!lib) { hga_set_error("libnccl.so.2 could not be loaded: %s", dlerror()); return HGA_E_NCCL; }
#define HGA_SYM(field, name)                                                                  \
    g_nccl.field = reinterpret_cast<decltype(g_nccl.field)>(dlsym(lib, name));                \
    if (!g_nccl.field) { hga_set_error("libnccl: symbol %s missing", name); return HGA_E_NCCL; }
    HGA_SYM(GetUniqueId, "ncclGetUniqueId");
    HGA_SYM(CommInitRank, "ncclCommInitRank");
    HGA_SYM(CommDestroy, "ncclCommDestroy");
    HGA_SYM(AllReduce, "ncclAllReduce");
    HGA_SYM(AllGather, "ncclAllGather");
    HGA_SYM(Broadcast, "ncclBroadcast");
    HGA_SYM(Send, "ncclSend");
    HGA_SYM(Recv, "ncclRecv");
    HGA_SYM(GroupStart, "ncclGroupStart");
    HGA_SYM(GroupEnd, "ncclGroupEnd");
    HGA_SYM(GetErrorString, "ncclGetErrorString");
#undef HGA_SYM
    g_nccl.lib = lib;
    return HGA_OK;
}

#define HGA_NCCL(call)                                                                                                  \
    do {                                                                                                                \
        ncclResult_t _r = (call);                                                                                       \
        if (_r != ncclSuccess) {                                                                                        \
            hga_set_error("%s:%d: %s failed: %s", __FILE__, __LINE__, #call, g_nccl.GetErrorString(_r));                \
            return HGA_E_NCCL;                                                                                          \
        }                                                                                                               \
    } while (0)

// per hit: list number at the owner + owner; per row and owner: the number of the row's hits that go there (cnt[g * n_rows + r]).
// One warp per row. The rows themselves do not travel: a source sends its list numbers in row order and one count per row, and the
// owner rebuilds the row offsets from the counts of all sources in rank order = global row order.
__global__ void pack_lists_kernel(const uint64_t *__restrict__ row_off, uint64_t n_rows, const uint32_t *__restrict__ slot, uint32_t G,
                                  uint32_t *__restrict__ list, uint8_t *__restrict__ owner, uint32_t *__restrict__ cnt) {
    const uint64_t warps = ((uint64_t) gridDim.x * blockDim.x) >> 5;
    const uint64_t w = (blockIdx.x * (uint64_t) blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    for (uint64_t r = w; r < n_rows; r += warps) {
        const uint64_t a = row_off[r], b = row_off[r + 1];
        uint32_t mine = 0;                                  // lane g: hits of this row owned by rank g, g + 32 (G <= 62)
        uint32_t mine_hi = 0;
        for (uint64_t i0 = a; i0 < b; i0 += 32) {
            const uint64_t i = i0 + lane;
            uint32_t o = 0xFFu;
            if (i < b) {
                const uint32_t s = slot[i];
                o = hga_owner_of_slot(s, G);
                list[i] = hga_list_of_slot(s, G);
                owner[i] = (uint8_t) o;
            }
            for (uint32_t g = 0; g < G; g++) {
                const uint32_t c = __popc(__ballot_sync(0xFFFFFFFFu, o == g));
                if ((g & 31) == (uint32_t) lane) { if (g < 32) mine += c; else mine_hi += c; }
            }
        }
        if ((uint32_t) lane < G) cnt[(size_t) lane * n_rows + r] = mine;
        if ((uint32_t) lane + 32 < G) cnt[(size_t) (lane + 32) * n_rows + r] = mine_hi;
    }
}

// send counts of a partitioned array: cnt[g] = number of elements whose (sorted) destination byte is g, g = 0 .. G - 1
__global__ void dest_counts_kernel(const uint8_t *__restrict__ sorted_dest, uint64_t n, int G, unsigned long long *cnt) {
    const int g = threadIdx.x;
    if (g >= G) return;
    uint64_t lo = 0, hi = n;
    while (lo < hi) { const uint64_t mid = (lo + hi) >> 1; if (sorted_dest[mid] < g) lo = mid + 1; else hi = mid; }
    uint64_t lo2 = lo, hi2 = n;
    while (lo2 < hi2) { const uint64_t mid = (lo2 + hi2) >> 1; if (sorted_dest[mid] <= g) lo2 = mid + 1; else hi2 = mid; }
    cnt[g] = lo2 - lo;
}

// partial pair (key = x << 32 | y, score) -> ONE 64-bit record x | y | score (rb bits per row, sb = 64 - 2 rb bits of score) + destination
// owner(x) = x mod G; a score that does not fit raises the flag (every rank then takes the unpacked path together)
__global__ void pack_partials_kernel(const uint64_t *__restrict__ key, const uint32_t *__restrict__ score, uint64_t n, int rb, int sb, uint32_t G,
                                     uint64_t *__restrict__ rec, uint8_t *__restrict__ dest, unsigned long long *flag) {
    bool bad = false;
    for (uint64_t i = blockIdx.x * (uint64_t) blockDim.x + threadIdx.x; i < n; i += (uint64_t) gridDim.x * blockDim.x) {
        const uint64_t k = key[i];
        const uint32_t x = (uint32_t) (k >> 32), y = (uint32_t) k, sc = score[i];
        if (sb < 32 && (sc >> sb)) bad = true;
        rec[i] = ((uint64_t) x << (rb + sb)) | ((uint64_t) y << sb) | sc;
        dest[i] = (uint8_t) (x % G);
    }
    if (bad) atomicExch(flag, 1ull);
}

struct UnpackPairKey {
    int rb, sb;
    __host__ __device__ __forceinline__ uint64_t operator()(const uint64_t &r) const {
        return ((r >> (rb + sb)) << 32) | ((r >> sb) & ((1ull << rb) - 1));
    }
};
struct UnpackPairScore {
    uint64_t mask;
    __host__ __device__ __forceinline__ uint32_t operator()(const uint64_t &r) const { return (uint32_t) (r & mask); }
};

__global__ void pair_dest_kernel(const uint64_t *__restrict__ key, uint64_t n, uint32_t G, uint8_t *__restrict__ dest) {
    for (uint64_t i = blockIdx.x * (uint64_t) blockDim.x + threadIdx.x; i < n; i += (uint64_t) gridDim.x * blockDim.x) dest[i] = (uint8_t) ((uint32_t) (key[i] >> 32) % G);
}

}  // namespace

int hga_comm_rank(const hga_handle *h) { return h->comm ? h->comm->rank : 0; }
int hga_comm_size(const hga_handle *h) { return h->comm ? h->comm->size : 1; }

void hga_comm_destroy(hga_handle *h) {
    if (!h->comm && h->comm_parked) { h->comm = h->comm_parked; h->comm_parked = nullptr; }
    if (!h->comm) return;
    if (h->comm->comm && g_nccl.CommDestroy) g_nccl.CommDestroy(h->comm->comm);
    h->comm->d_small.release();
    h->comm->d_stage.release();
    h->comm->d_rows.release();
    delete h->comm;
    h->comm = nullptr;
}

int hga_comm_allreduce_u64_sum(hga_handle *h, uint64_t *d_buf, size_t n) {
    HGA_NCCL(g_nccl.AllReduce(d_buf, d_buf, n, ncclUint64, ncclSum, h->comm->comm, h->stream));
    return HGA_OK;
}
int hga_comm_allreduce_u32_min(hga_handle *h, uint32_t *d_buf, size_t n) {
    HGA_NCCL(g_nccl.AllReduce(d_buf, d_buf, n, ncclUint32, ncclMin, h->comm->comm, h->stream));
    return HGA_OK;
}
int hga_comm_allreduce_u32_max(hga_handle *h, uint32_t *d_buf, size_t n) {
    HGA_NCCL(g_nccl.AllReduce(d_buf, d_buf, n, ncclUint32, ncclMax, h->comm->comm, h->stream));
    return HGA_OK;
}

// counts[g] for every rank g: cnt_all[g] = value contributed by rank g (host array of size G)
int hga_comm_allgather_u64(hga_handle *h, uint64_t mine, std::vector<uint64_t> &all) {
    const int G = h->comm->size;
    HGA_TRY(h->comm->d_small.ensure((size_t) (G + 1) * 8 * 2));
    uint64_t *d_in = h->comm->d_small.as<uint64_t>(), *d_out = d_in + 1;
    HGA_CUDA(cudaMemcpyAsync(d_in, &mine, 8, cudaMemcpyHostToDevice, h->stream));
    HGA_NCCL(g_nccl.AllGather(d_in, d_out, 1, ncclUint64, h->comm->comm, h->stream));
    all.assign(G, 0);
    HGA_CUDA(cudaMemcpyAsync(all.data(), d_out, (size_t) G * 8, cudaMemcpyDeviceToHost, h->stream));
    HGA_CUDA(cudaStreamSynchronize(h->stream));
    return HGA_OK;
}

// variable-size all-gather: rank g contributes counts[g] elements of elem_bytes (4 or 8) from d_mine; d_all receives the
// concatenation in rank order. Large payloads go through ONE ncclAllGather on segments padded to the largest count
// (the ring / NVLS path that reaches NVLink bandwidth) followed by device-to-device compaction copies; small ones use one
// ncclBroadcast per root inside a group.
int hga_comm_allgatherv(hga_handle *h, const void *d_mine, void *d_all, const std::vector<uint64_t> &counts, int elem_bytes) {
    const int G = h->comm->size, me = h->comm->rank;
    const ncclDataType_t dt = elem_bytes == 8 ? ncclUint64 : ncclUint32;
    uint64_t maxc = 0, total = 0;
    for (uint64_t c : counts) { maxc = std::max(maxc, c); total += c; }
    if (total * elem_bytes >= (8ull << 20)) {
        HGA_TRY(h->comm->d_stage.ensure((size_t) G * maxc * elem_bytes + 256));
        char *stage = h->comm->d_stage.as<char>();
        if (counts[me]) HGA_CUDA(cudaMemcpyAsync(stage + (size_t) me * maxc * elem_bytes, d_mine, counts[me] * elem_bytes, cudaMemcpyDeviceToDevice, h->stream));
        HGA_NCCL(g_nccl.AllGather(stage + (size_t) me * maxc * elem_bytes, stage, maxc, dt, h->comm->comm, h->stream));
        uint64_t base = 0;
        for (int g = 0; g < G; g++) {
            if (counts[g]) HGA_CUDA(cudaMemcpyAsync(reinterpret_cast<char *>(d_all) + base * elem_bytes, stage + (size_t) g * maxc * elem_bytes, counts[g] * elem_bytes,
                                                    cudaMemcpyDeviceToDevice, h->stream));
            base += counts[g];
        }
        return HGA_OK;
    }
    HGA_NCCL(g_nccl.GroupStart());
    uint64_t base = 0;
    for (int g = 0; g < G; g++) {
        char *dst = reinterpret_cast<char *>(d_all) + base * elem_bytes;
        if (counts[g]) HGA_NCCL(g_nccl.Broadcast(g == me ? d_mine : dst, dst, counts[g], dt, g, h->comm->comm, h->stream));
        base += counts[g];
    }
    HGA_NCCL(g_nccl.GroupEnd());
    return HGA_OK;
}

// Count matrix of an exchange: every rank contributes G send counts, two extra values and its STATUS (the return code of the local phase that
// produced the counts); the all-gather of these G + 3 values is the stage's one host synchronisation. A rank whose local phase failed still takes
// part (with zero counts), so that nobody is left waiting in NCCL: every rank sees every status and they all leave the stage together, the failed
// rank with its own error, the others with HGA_E_NCCL. cnt_all[src * HGA_CS(G) + dst], extras at + G and + G + 1.
#define HGA_CS(G) ((size_t) (G) + 3)
static int exchange_counts(hga_handle *h, unsigned long long *d_send_cnt, unsigned long long *d_all, int local_rc, const char *stage, std::vector<unsigned long long> &cnt_all) {
    const int G = h->comm->size, me = h->comm->rank;
    const size_t CS = HGA_CS(G);
    cnt_all.assign((size_t) G * CS, 0);
    const unsigned long long status = (unsigned long long) (local_rc == HGA_OK ? 0 : (unsigned) -local_rc + 1u);
    if (local_rc != HGA_OK) HGA_CUDA(cudaMemsetAsync(d_send_cnt, 0, (CS - 1) * 8, h->stream));
    HGA_CUDA(cudaMemcpyAsync(d_send_cnt + G + 2, &status, 8, cudaMemcpyHostToDevice, h->stream));
    HGA_NCCL(g_nccl.AllGather(d_send_cnt, d_all, CS, ncclUint64, h->comm->comm, h->stream));
    HGA_CUDA(cudaMemcpyAsync(cnt_all.data(), d_all, (size_t) G * CS * 8, cudaMemcpyDeviceToHost, h->stream));
    HGA_CUDA(cudaStreamSynchronize(h->stream));
    if (local_rc != HGA_OK) return local_rc;                         // (the error text of the local phase stands)
    for (int g = 0; g < G; g++)
        if (cnt_all[g * CS + G + 2]) { hga_set_error("%s: rank %d failed before the exchange (rank %d leaves the stage with it)", stage, g, me); return HGA_E_NCCL; }
    return HGA_OK;
}

// test hook: HGA_FAULT="<stage>:<rank>" makes that rank's local phase of the stage fail (tests/multi_gpu_parity.py: nobody may hang)
static bool fault_injected(const hga_handle *h, const char *stage) {
    const char *e = getenv("HGA_FAULT");
    if (!e) return false;
    const size_t n = strlen(stage);
    return strncmp(e, stage, n) == 0 && e[n] == ':' && atoi(e + n + 1) == h->comm->rank;
}

// Steps 1-2 of the header comment. On return h->d_inv_off / h->d_inv_row hold the inverted lists of THIS rank's k-mers (list number
// = kmer_id / G, rows = global row numbers = read id - 1) and h->d_g_row_off / h->d_g_kid the by-row incidence of all rows
// restricted to those k-mers.
int hga_comm_build_owner_index(hga_handle *h) {
    const int G = h->comm->size, me = h->comm->rank;
    const uint64_t E_loc = h->n_hits, R_all = h->n_reads_total;
    const uint32_t n_buckets_all = h->table.n_slots / HGA_BUCKET_SLOTS;                         // n_slots is a multiple of 32
    const uint32_t n_lists = (n_buckets_all + G - 1) / G * HGA_BUCKET_SLOTS;                    // of the fullest owner; a multiple of 32
    const uint32_t row_base = h->read_id_base - 1;
    double comm_ms = 0, part_ms = 0;
    Trace tr(h);

    // 1. list numbers partitioned by owner (ONE stable radix pass: every owner segment keeps row order) + per-row counts per owner.
    // The local phase: whatever goes wrong in it is reported through the count matrix, not by leaving early (exchange_counts).
    const int owner_bits = (int) std::max<uint32_t>(hga_ceil_log2((uint64_t) G), 1);
    const uint64_t R_loc = h->n_reads;
    unsigned long long *d_cnt = h->comm->d_small.as<unsigned long long>(), *d_cnt_all = d_cnt + HGA_CS(G) + 1;     // (sized by hga_comm_init)
    uint32_t *list_out = nullptr, *cnt_send = nullptr, *cnt_recv = nullptr;
    auto local_phase = [&]() -> int {
        if (fault_injected(h, "index")) { hga_set_error("hga_build_index: injected fault (HGA_FAULT)"); return HGA_E_NOMEM; }
        if (E_loc >= (1ull << 32)) { hga_set_error("local incidence of %llu entries exceeds the 32-bit per-GPU limit", (unsigned long long) E_loc); return HGA_E_OVERFLOW; }
        HGA_TRY(h->d_sort_a.ensure((E_loc + 1) * 4));      // list numbers, partitioned
        HGA_TRY(h->d_sort_b.ensure((E_loc + 1) * 4));      // list numbers, stream order
        HGA_TRY(h->d_x_row.ensure((E_loc + 1) * 2));       // owner per hit: in | out
        HGA_TRY(h->comm->d_rows.ensure(((size_t) G * R_loc + R_all + 2) * 4));   // my rows' counts per owner | all rows' counts for my lists
        uint8_t *own_in = h->d_x_row.as<uint8_t>(), *own_out = own_in + (E_loc + 1);
        uint32_t *list_in = h->d_sort_b.as<uint32_t>();
        list_out = h->d_sort_a.as<uint32_t>();
        cnt_send = h->comm->d_rows.as<uint32_t>(); cnt_recv = cnt_send + (size_t) G * R_loc;
        if (R_loc) {
            const int blocks = (int) std::min<uint64_t>((R_loc * 32 + 255) / 256, (uint64_t) h->sm_count * 32);
            pack_lists_kernel<<<blocks, 256, 0, h->stream>>>(h->d_row_off.as<uint64_t>(), R_loc, h->d_hit_slot.as<uint32_t>(), (uint32_t) G, list_in, own_in, cnt_send);
            h->metrics.kernel_launches++;
            HGA_CUDA(cudaGetLastError());
        }
        if (E_loc) {
            size_t tmp = 0;
            HGA_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, tmp, own_in, own_out, list_in, list_out, E_loc, 0, owner_bits, h->stream));
            HGA_TRY(h->d_sort_tmp.ensure(tmp + 16));
            HGA_CUDA(cub::DeviceRadixSort::SortPairs(h->d_sort_tmp.p, tmp, own_in, own_out, list_in, list_out, E_loc, 0, owner_bits, h->stream));
            h->metrics.kernel_launches += 3;
            HGA_CUDA(cudaGetLastError());
        }
        dest_counts_kernel<<<1, 64, 0, h->stream>>>(own_out, E_loc, G, d_cnt);
        const unsigned long long extra[2] = {R_loc, row_base};                          // ride along: the receive layout and the shard-layout check need them from every rank
        HGA_CUDA(cudaMemcpyAsync(d_cnt + G, extra, 16, cudaMemcpyHostToDevice, h->stream));
        h->metrics.kernel_launches++;
        HGA_CUDA(cudaGetLastError());
        return HGA_OK;
    };
    const int local_rc = local_phase();
    tr.mark("pack+partition");
    std::vector<unsigned long long> cnt_all;
    HGA_TRY(exchange_counts(h, d_cnt, d_cnt_all, local_rc, "hga_build_index", cnt_all));   // the only host synchronisation of the stage
    tr.mark("counts");
    const size_t CS = HGA_CS(G);
    std::vector<uint64_t> rows_off(G + 1, 0);
    for (int g = 0; g < G; g++) rows_off[g + 1] = rows_off[g] + cnt_all[g * CS + G];
    // shards must be contiguous read-id ranges in rank order: the row stream of source s must lie in s's range. Every rank checks EVERY rank's layout and share
    // (the matrix holds them all), so they all come to the same verdict.
    for (int g = 0; g < G; g++)
        if (rows_off[g] != cnt_all[g * CS + G + 1]) { hga_set_error("hga_build_index: shards must be contiguous read-id ranges in rank order (rank %d starts at row %llu, expected %llu)", g, (unsigned long long) cnt_all[g * CS + G + 1], (unsigned long long) rows_off[g]); return HGA_E_ARG; }
    if (rows_off[G] != R_all) { hga_set_error("hga_build_index: the ranks scanned %llu reads, hga_comm_init said %llu", (unsigned long long) rows_off[G], (unsigned long long) R_all); return HGA_E_ARG; }
    for (int g = 0; g < G; g++) {
        uint64_t share = 0;
        for (int src = 0; src < G; src++) share += cnt_all[src * CS + g];
        if (share >= (1ull << 32)) { hga_set_error("rank %d's share of the incidence (%llu entries) exceeds the 32-bit per-GPU limit", g, (unsigned long long) share); return HGA_E_OVERFLOW; }
    }

    // 2. all-to-all: the list numbers of my lists from every rank, in rank order = global row order, and the sources' per-row counts
    uint64_t E_own = 0;
    std::vector<uint64_t> recv_off(G + 1, 0), send_off(G + 1, 0);
    for (int src = 0; src < G; src++) { recv_off[src] = E_own; E_own += cnt_all[src * CS + me]; }
    for (int g = 0; g < G; g++) send_off[g + 1] = send_off[g] + cnt_all[me * CS + g];
    HGA_TRY(h->d_g_kid.ensure((E_own + 1) * 4));        // the by-row incidence of all rows restricted to my lists: list number per hit
    HGA_TRY(h->d_g_row_off.ensure((R_all + 2) * 8));
    uint32_t *rx = h->d_g_kid.as<uint32_t>();
    {
        StageTimer xt(h, &part_ms, true);
        HGA_NCCL(g_nccl.GroupStart());
        for (int g = 0; g < G; g++) {
            const uint64_t sc = cnt_all[me * CS + g], rc = cnt_all[g * CS + me];
            const uint64_t rows_g = cnt_all[g * CS + G];
            if (sc) HGA_NCCL(g_nccl.Send(list_out + send_off[g], sc, ncclUint32, g, h->comm->comm, h->stream));
            if (rc) HGA_NCCL(g_nccl.Recv(rx + recv_off[g], rc, ncclUint32, g, h->comm->comm, h->stream));
            if (R_loc) HGA_NCCL(g_nccl.Send(cnt_send + (size_t) g * R_loc, R_loc, ncclUint32, g, h->comm->comm, h->stream));
            if (rows_g) HGA_NCCL(g_nccl.Recv(cnt_recv + rows_off[g], rows_g, ncclUint32, g, h->comm->comm, h->stream));
        }
        HGA_NCCL(g_nccl.GroupEnd());
        xt.stop();
        comm_ms += part_ms;
    }
    tr.mark("alltoall");

    // row offsets of the by-row incidence = exclusive sum of the counts (64-bit accumulator); inverted lists = the single-GPU list builder
    {
        HGA_CUDA(cudaMemsetAsync(cnt_recv + R_all, 0, 4, h->stream));
        size_t tmp = 0;
        HGA_CUDA(cub::DeviceScan::ExclusiveScan(nullptr, tmp, cnt_recv, h->d_g_row_off.as<unsigned long long>(), cub::Sum(), 0ull, R_all + 1, h->stream));
        HGA_TRY(h->d_sort_tmp.ensure(tmp + 16));
        HGA_CUDA(cub::DeviceScan::ExclusiveScan(h->d_sort_tmp.p, tmp, cnt_recv, h->d_g_row_off.as<unsigned long long>(), cub::Sum(), 0ull, R_all + 1, h->stream));
        h->metrics.kernel_launches += 2;
    }
    tr.mark("offsets");
    HGA_TRY(hga_build_lists(h, h->d_g_kid.as<uint32_t>(), h->d_g_row_off.as<uint64_t>(), R_all, E_own, n_lists));
    tr.mark("lists");
    h->inc_rows = R_all;
    h->inc_row_first_id = 1;
    h->inc_entries = E_own;
    h->pair_rows = R_all;
    h->pair_pivot_mul = 1; h->pair_pivot_add = 0;
    h->index_by_kid = true;
    h->index_keys = n_lists;
    h->metrics.exchange_ms = comm_ms;       // NCCL payload calls only (the sorts between them belong to index_ms)
    tr.dump("index", me);
    return HGA_OK;
}

// Step 4 of the header comment: n partial (key = x << 32 | y, score) records of this rank -> owner(x) = x mod G. On return
// *out_n records (unsorted, pairs may repeat: one partial per contributing rank) are in h->d_pair_key2 / h->d_pair_score2.
int hga_comm_exchange_partials(hga_handle *h, uint64_t n, uint64_t *out_n) {
    const int G = h->comm->size, me = h->comm->rank;
    const int owner_bits = (int) std::max<uint32_t>(hga_ceil_log2((uint64_t) G), 1);
    double part_ms = 0;
    Trace tr(h);
    unsigned long long *d_cnt = h->comm->d_small.as<unsigned long long>(), *d_cnt_all = d_cnt + HGA_CS(G) + 1;
    uint64_t *key_part = nullptr;
    uint32_t *score_part = nullptr;
    auto local_phase = [&]() -> int {
        if (fault_injected(h, "partials")) { hga_set_error("hga_pair_count: injected fault (HGA_FAULT)"); return HGA_E_NOMEM; }
        HGA_TRY(h->d_x_row.ensure((n + 1) * 2));
        HGA_TRY(h->d_pair_key2.ensure((n + 1) * 8));
        HGA_TRY(h->d_pair_score2.ensure((n + 1) * 4));
        uint8_t *d_in = h->d_x_row.as<uint8_t>(), *d_out = d_in + (n + 1);
        key_part = h->d_pair_key2.as<uint64_t>();
        score_part = h->d_pair_score2.as<uint32_t>();
        if (n) {
            pair_dest_kernel<<<(int) std::min<uint64_t>((n + 255) / 256, (uint64_t) h->sm_count * 16), 256, 0, h->stream>>>(h->d_pair_key.as<uint64_t>(), n, (uint32_t) G, d_in);
            size_t t1 = 0, t2 = 0;
            HGA_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, t1, d_in, d_out, h->d_pair_key.as<uint64_t>(), key_part, n, 0, owner_bits, h->stream));
            HGA_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, t2, d_in, d_out, h->d_pair_score.as<uint32_t>(), score_part, n, 0, owner_bits, h->stream));
            HGA_TRY(h->d_sort_tmp.ensure(std::max(t1, t2) + 16));
            // two stable passes with the same keys: the same permutation for both value arrays
            HGA_CUDA(cub::DeviceRadixSort::SortPairs(h->d_sort_tmp.p, t1, d_in, d_out, h->d_pair_key.as<uint64_t>(), key_part, n, 0, owner_bits, h->stream));
            HGA_CUDA(cub::DeviceRadixSort::SortPairs(h->d_sort_tmp.p, t2, d_in, d_out, h->d_pair_score.as<uint32_t>(), score_part, n, 0, owner_bits, h->stream));
            h->metrics.kernel_launches += 7;
            HGA_CUDA(cudaGetLastError());
        }
        dest_counts_kernel<<<1, 64, 0, h->stream>>>(d_out, n, G, d_cnt);
        HGA_CUDA(cudaMemsetAsync(d_cnt + G, 0, 16, h->stream));
        h->metrics.kernel_launches++;
        HGA_CUDA(cudaGetLastError());
        return HGA_OK;
    };
    const int local_rc = local_phase();
    tr.mark("partition");
    std::vector<unsigned long long> cnt_all;
    HGA_TRY(exchange_counts(h, d_cnt, d_cnt_all, local_rc, "hga_pair_count", cnt_all));
    tr.mark("counts");
    uint64_t n_recv = 0;
    std::vector<uint64_t> recv_off(G + 1, 0), send_off(G + 1, 0);
    const size_t CS = HGA_CS(G);
    for (int src = 0; src < G; src++) { recv_off[src] = n_recv; n_recv += cnt_all[src * CS + me]; }
    for (int g = 0; g < G; g++) send_off[g + 1] = send_off[g] + cnt_all[me * CS + g];
    // the receive buffers: the (now free) primary pair arrays
    HGA_TRY(h->d_pair_key.ensure((n_recv + 1) * 8));
    HGA_TRY(h->d_pair_score.ensure((n_recv + 1) * 4));
    {
        StageTimer xt(h, &part_ms, true);
        HGA_NCCL(g_nccl.GroupStart());
        for (int g = 0; g < G; g++) {
            const uint64_t sc = cnt_all[me * CS + g], rc = cnt_all[g * CS + me];
            if (sc) {
                HGA_NCCL(g_nccl.Send(key_part + send_off[g], sc, ncclUint64, g, h->comm->comm, h->stream));
                HGA_NCCL(g_nccl.Send(score_part + send_off[g], sc, ncclUint32, g, h->comm->comm, h->stream));
            }
            if (rc) {
                HGA_NCCL(g_nccl.Recv(h->d_pair_key.as<uint64_t>() + recv_off[g], rc, ncclUint64, g, h->comm->comm, h->stream));
                HGA_NCCL(g_nccl.Recv(h->d_pair_score.as<uint32_t>() + recv_off[g], rc, ncclUint32, g, h->comm->comm, h->stream));
            }
        }
        HGA_NCCL(g_nccl.GroupEnd());
        xt.stop();
        h->metrics.exchange_ms += part_ms;
    }
    *out_n = n_recv;
    tr.mark("alltoall");
    if (tr.on) fprintf(stderr, "[hga trace r%d partials] sent=%llu received=%llu\n", me, (unsigned long long) n, (unsigned long long) n_recv);
    tr.dump("partials", me);
    return HGA_OK;
}

// Step 4, the usual way: the n partial records travel PACKED (one u64: x | y | partial score) - one partition pass, 8 instead of 12 bytes
// per record on the wire, one keys-only sort over the 2 x row_bits key bits at the receiver - and are summed per (x, y) there. On return
// *reduced = true and the final pairs (sorted by (x, y), scores summed, *out_n of them) are in h->d_pair_key / h->d_pair_score; when
// the rows or a partial score do not fit 64 bits, *reduced = false and nothing has been exchanged (the caller takes the unpacked path).
int hga_comm_reduce_partials_packed(hga_handle *h, uint64_t n, uint64_t *out_n, bool *reduced) {
    const int G = h->comm->size, me = h->comm->rank;
    *reduced = false;
    const int rb = (int) std::max<uint32_t>(hga_ceil_log2(h->inc_rows + 1), 1), sb = 64 - 2 * rb;
    if (sb < 12) return HGA_OK;                         // (the same on every rank: inc_rows is global)
    const int owner_bits = (int) std::max<uint32_t>(hga_ceil_log2((uint64_t) G), 1);
    double part_ms = 0;
    Trace tr(h);
    unsigned long long *d_cnt = h->comm->d_small.as<unsigned long long>(), *d_cnt_all = d_cnt + HGA_CS(G) + 1;
    uint64_t *rec_part = nullptr;
    auto local_phase = [&]() -> int {
        if (fault_injected(h, "partials")) { hga_set_error("hga_pair_count: injected fault (HGA_FAULT)"); return HGA_E_NOMEM; }
        HGA_TRY(h->d_x_row.ensure((n + 1) * 2));
        HGA_TRY(h->d_pair_key2.ensure((n + 1) * 8));
        HGA_TRY(h->d_x_slot.ensure((n + 1) * 8));
        uint8_t *d_in = h->d_x_row.as<uint8_t>(), *d_out = d_in + (n + 1);
        uint64_t *rec_in = h->d_x_slot.as<uint64_t>();
        rec_part = h->d_pair_key2.as<uint64_t>();
        HGA_CUDA(cudaMemsetAsync(d_cnt, 0, HGA_CS(G) * 8, h->stream));
        if (n) {
            pack_partials_kernel<<<(int) std::min<uint64_t>((n + 255) / 256, (uint64_t) h->sm_count * 16), 256, 0, h->stream>>>(h->d_pair_key.as<uint64_t>(), h->d_pair_score.as<uint32_t>(), n, rb, sb,
                                                                                                                               (uint32_t) G, rec_in, d_in, d_cnt + G);
            size_t t1 = 0;
            HGA_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, t1, d_in, d_out, rec_in, rec_part, n, 0, owner_bits, h->stream));
            HGA_TRY(h->d_sort_tmp.ensure(t1 + 16));
            HGA_CUDA(cub::DeviceRadixSort::SortPairs(h->d_sort_tmp.p, t1, d_in, d_out, rec_in, rec_part, n, 0, owner_bits, h->stream));
            h->metrics.kernel_launches += 4;
            HGA_CUDA(cudaGetLastError());
        }
        dest_counts_kernel<<<1, 64, 0, h->stream>>>(d_out, n, G, d_cnt);
        h->metrics.kernel_launches++;
        HGA_CUDA(cudaGetLastError());
        return HGA_OK;
    };
    const int local_rc = local_phase();
    tr.mark("pack+partition");
    std::vector<unsigned long long> cnt_all;
    HGA_TRY(exchange_counts(h, d_cnt, d_cnt_all, local_rc, "hga_pair_count", cnt_all));
    tr.mark("counts");
    const size_t CS = HGA_CS(G);
    for (int g = 0; g < G; g++) if (cnt_all[g * CS + G]) return HGA_OK;           // a score did not fit somewhere: everybody falls back
    uint64_t n_recv = 0;
    std::vector<uint64_t> recv_off(G + 1, 0), send_off(G + 1, 0);
    for (int src = 0; src < G; src++) { recv_off[src] = n_recv; n_recv += cnt_all[src * CS + me]; }
    for (int g = 0; g < G; g++) send_off[g + 1] = send_off[g] + cnt_all[me * CS + g];
    HGA_TRY(h->d_x_slot.ensure((n_recv + 1) * 8 * 2));                            // received | sorted (rec_in is dead by now)
    uint64_t *rx = h->d_x_slot.as<uint64_t>(), *rx_sorted = rx + (n_recv + 1);
    {
        StageTimer xt(h, &part_ms, true);
        HGA_NCCL(g_nccl.GroupStart());
        for (int g = 0; g < G; g++) {
            const uint64_t sc = cnt_all[me * CS + g], rc = cnt_all[g * CS + me];
            if (sc) HGA_NCCL(g_nccl.Send(rec_part + send_off[g], sc, ncclUint64, g, h->comm->comm, h->stream));
            if (rc) HGA_NCCL(g_nccl.Recv(rx + recv_off[g], rc, ncclUint64, g, h->comm->comm, h->stream));
        }
        HGA_NCCL(g_nccl.GroupEnd());
        xt.stop();
        h->metrics.exchange_ms += part_ms;
    }
    tr.mark("alltoall");
    uint64_t runs_h = 0;
    HGA_TRY(h->d_pair_key.ensure((n_recv + 1) * 8));
    HGA_TRY(h->d_pair_score.ensure((n_recv + 1) * 4));
    if (n_recv) {
        size_t t1 = 0, t2 = 0;
        HGA_CUDA(cub::DeviceRadixSort::SortKeys(nullptr, t1, rx, rx_sorted, n_recv, sb, 64, h->stream));
        cub::TransformInputIterator<uint64_t, UnpackPairKey, const uint64_t *> kit(rx_sorted, UnpackPairKey{rb, sb});
        cub::TransformInputIterator<uint32_t, UnpackPairScore, const uint64_t *> vit(rx_sorted, UnpackPairScore{sb >= 64 ? ~0ull : ((1ull << sb) - 1)});
        unsigned long long *d_runs = d_cnt;                                          // a free scalar
        HGA_CUDA(cub::DeviceReduce::ReduceByKey(nullptr, t2, kit, h->d_pair_key.as<uint64_t>(), vit, h->d_pair_score.as<uint32_t>(), d_runs, cub::Sum(), n_recv, h->stream));
        HGA_TRY(h->d_sort_tmp.ensure(std::max(t1, t2) + 16));
        HGA_CUDA(cub::DeviceRadixSort::SortKeys(h->d_sort_tmp.p, t1, rx, rx_sorted, n_recv, sb, 64, h->stream));
        tr.mark("sort");
        HGA_CUDA(cub::DeviceReduce::ReduceByKey(h->d_sort_tmp.p, t2, kit, h->d_pair_key.as<uint64_t>(), vit, h->d_pair_score.as<uint32_t>(), d_runs, cub::Sum(), n_recv, h->stream));
        unsigned long long runs = 0;
        HGA_CUDA(cudaMemcpyAsync(&runs, d_runs, 8, cudaMemcpyDeviceToHost, h->stream));
        HGA_CUDA(cudaStreamSynchronize(h->stream));
        runs_h = runs;
        h->metrics.kernel_launches += (uint64_t) (2 * rb + 7) / 8 + 5;
        tr.mark("reduce");
    }
    if (tr.on) fprintf(stderr, "[hga trace r%d partials] packed sent=%llu received=%llu final=%llu\n", me, (unsigned long long) n, (unsigned long long) n_recv, (unsigned long long) runs_h);
    tr.dump("partials", me);
    *out_n = runs_h;
    *reduced = true;
    return HGA_OK;
}

namespace {
// row offsets of source s (local, starting at 0) -> global: out[rows_before + i] = local[i] + hits_before, i < n_rows
__global__ void rebase_offsets_kernel(const uint64_t *__restrict__ local, uint64_t n_rows, uint64_t rows_before, uint64_t hits_before, uint64_t *__restrict__ out) {
    for (uint64_t i = blockIdx.x * (uint64_t) blockDim.x + threadIdx.x; i < n_rows; i += (uint64_t) gridDim.x * blockDim.x) out[rows_before + i] = local[i] + hits_before;
}
}  // namespace

// The stages after the scaffold union_find (merge_components, tails, spectral clustering, enrichment: ReadClusteringEngine.cpp:764-794)
// run on ONE GPU: their work is a small fraction of the hot path and their host parts are sequential. This collective turns rank 0's
// handle into a complete single-GPU handle: the hits of all ranks (shards are contiguous id ranges in rank order, slots mean the same
// k-mer on every rank: concatenation IS the single-GPU hit list), the selected edges of all ranks in (x, y) order, the component labels
// (already replicated), and the by-slot inverted index rebuilt from the gathered hits. The communicator is detached from rank 0's
// handle (kept for hga_destroy); the other ranks' handles keep their state and must not enter another collective.
extern "C" int hga_comm_gather_root(hga_handle *h) {
    if (!h) { hga_set_error("NULL handle"); return HGA_E_ARG; }
    if (!h->comm || h->comm->size < 2) return HGA_OK;
    if (!h->have_scan || !h->have_selection || !h->have_components) { hga_set_error("hga_comm_gather_root: needs hga_scan ... hga_components on every rank"); return HGA_E_STATE; }
    HGA_CUDA(cudaSetDevice(h->device));
    const int G = h->comm->size, me = h->comm->rank;
    HGA_TRY(hga_scan_finish_positions(h));
    // (reads, hits, selected edges) of every rank
    HGA_TRY(h->comm->d_small.ensure((size_t) (G + 2) * 8 * (G + 2)));
    unsigned long long *d_mine = h->comm->d_small.as<unsigned long long>(), *d_all = d_mine + 4;
    const unsigned long long mine[3] = {h->n_reads, h->n_hits, h->n_selected};
    HGA_CUDA(cudaMemcpyAsync(d_mine, mine, 24, cudaMemcpyHostToDevice, h->stream));
    HGA_NCCL(g_nccl.AllGather(d_mine, d_all, 3, ncclUint64, h->comm->comm, h->stream));
    std::vector<unsigned long long> all((size_t) 3 * G);
    HGA_CUDA(cudaMemcpyAsync(all.data(), d_all, (size_t) 3 * G * 8, cudaMemcpyDeviceToHost, h->stream));
    HGA_CUDA(cudaStreamSynchronize(h->stream));
    uint64_t R = 0, E = 0, M = 0;
    std::vector<uint64_t> r0(G + 1, 0), e0(G + 1, 0), m0(G + 1, 0);
    for (int g = 0; g < G; g++) { r0[g + 1] = r0[g] + all[3 * g]; e0[g + 1] = e0[g] + all[3 * g + 1]; m0[g + 1] = m0[g] + all[3 * g + 2]; }
    R = r0[G]; E = e0[G]; M = m0[G];
    if (E >= (1ull << 32)) { hga_set_error("hga_comm_gather_root: %llu hits do not fit one GPU's 32-bit incidence", (unsigned long long) E); return HGA_E_OVERFLOW; }

    DevBuf g_off_local, g_off, g_slot, g_pos, g_key, g_score, g_key2, g_score2;
    if (me == 0) {
        HGA_TRY(g_off_local.ensure((R + G + 1) * 8)); HGA_TRY(g_off.ensure((R + 2) * 8));
        HGA_TRY(g_slot.ensure((E + 1) * 4)); HGA_TRY(g_pos.ensure((E + 1) * 4));
        HGA_TRY(g_key.ensure((M + 1) * 8)); HGA_TRY(g_score.ensure((M + 1) * 4));
        HGA_TRY(g_key2.ensure((M + 1) * 8)); HGA_TRY(g_score2.ensure((M + 1) * 4));
    }
    HGA_NCCL(g_nccl.GroupStart());
    if (me != 0) {
        HGA_NCCL(g_nccl.Send(h->d_row_off.p, h->n_reads + 1, ncclUint64, 0, h->comm->comm, h->stream));
        if (h->n_hits) {
            HGA_NCCL(g_nccl.Send(h->d_hit_slot.p, h->n_hits, ncclUint32, 0, h->comm->comm, h->stream));
            HGA_NCCL(g_nccl.Send(h->d_hit_pos.p, h->n_hits, ncclUint32, 0, h->comm->comm, h->stream));
        }
        if (h->n_selected) {
            HGA_NCCL(g_nccl.Send(h->d_sel_key.p, h->n_selected, ncclUint64, 0, h->comm->comm, h->stream));
            HGA_NCCL(g_nccl.Send(h->d_sel_score.p, h->n_selected, ncclUint32, 0, h->comm->comm, h->stream));
        }
    } else {
        for (int g = 1; g < G; g++) {
            const uint64_t nr = all[3 * g], nh = all[3 * g + 1], ns = all[3 * g + 2];
            HGA_NCCL(g_nccl.Recv(g_off_local.as<uint64_t>() + r0[g] + g, nr + 1, ncclUint64, g, h->comm->comm, h->stream));
            if (nh) {
                HGA_NCCL(g_nccl.Recv(g_slot.as<uint32_t>() + e0[g], nh, ncclUint32, g, h->comm->comm, h->stream));
                HGA_NCCL(g_nccl.Recv(g_pos.as<uint32_t>() + e0[g], nh, ncclUint32, g, h->comm->comm, h->stream));
            }
            if (ns) {
                HGA_NCCL(g_nccl.Recv(g_key.as<uint64_t>() + m0[g], ns, ncclUint64, g, h->comm->comm, h->stream));
                HGA_NCCL(g_nccl.Recv(g_score.as<uint32_t>() + m0[g], ns, ncclUint32, g, h->comm->comm, h->stream));
            }
        }
    }
    HGA_NCCL(g_nccl.GroupEnd());
    if (me != 0) { HGA_CUDA(cudaStreamSynchronize(h->stream)); return HGA_OK; }

    // rank 0: its own part, then the global row offsets, the selection in (x, y) order, and the handle's new state
    HGA_CUDA(cudaMemcpyAsync(g_off_local.p, h->d_row_off.p, (h->n_reads + 1) * 8, cudaMemcpyDeviceToDevice, h->stream));
    if (h->n_hits) {
        HGA_CUDA(cudaMemcpyAsync(g_slot.p, h->d_hit_slot.p, h->n_hits * 4, cudaMemcpyDeviceToDevice, h->stream));
        HGA_CUDA(cudaMemcpyAsync(g_pos.p, h->d_hit_pos.p, h->n_hits * 4, cudaMemcpyDeviceToDevice, h->stream));
    }
    if (h->n_selected) {
        HGA_CUDA(cudaMemcpyAsync(g_key.p, h->d_sel_key.p, h->n_selected * 8, cudaMemcpyDeviceToDevice, h->stream));
        HGA_CUDA(cudaMemcpyAsync(g_score.p, h->d_sel_score.p, h->n_selected * 4, cudaMemcpyDeviceToDevice, h->stream));
    }
    for (int g = 0; g < G; g++) {
        const uint64_t nr = all[3 * g];
        if (nr) rebase_offsets_kernel<<<(int) std::min<uint64_t>((nr + 255) / 256, 2048), 256, 0, h->stream>>>(g_off_local.as<uint64_t>() + r0[g] + g, nr, r0[g], e0[g], g_off.as<uint64_t>());
    }
    HGA_CUDA(cudaMemcpyAsync(g_off.as<uint64_t>() + R, &E, 8, cudaMemcpyHostToDevice, h->stream));
    if (M) {
        size_t tmp = 0;
        const int bits = 32 + (int) std::max<uint32_t>(hga_ceil_log2(R + 1), 1);
        HGA_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, tmp, g_key.as<uint64_t>(), g_key2.as<uint64_t>(), g_score.as<uint32_t>(), g_score2.as<uint32_t>(), M, 0, bits, h->stream));
        HGA_TRY(h->d_sort_tmp.ensure(tmp + 16));
        HGA_CUDA(cub::DeviceRadixSort::SortPairs(h->d_sort_tmp.p, tmp, g_key.as<uint64_t>(), g_key2.as<uint64_t>(), g_score.as<uint32_t>(), g_score2.as<uint32_t>(), M, 0, bits, h->stream));
    }
    HGA_CUDA(cudaGetLastError());
    HGA_CUDA(cudaStreamSynchronize(h->stream));
    h->d_row_off.release(); h->d_row_off = g_off;
    h->d_hit_slot.release(); h->d_hit_slot = g_slot;
    h->d_hit_pos.release(); h->d_hit_pos = g_pos;
    h->d_sel_key.release(); h->d_sel_key = g_key2;
    h->d_sel_score.release(); h->d_sel_score = g_score2;
    g_off_local.release(); g_key.release(); g_score.release();
    h->n_reads = R; h->n_hits = E; h->n_selected = M; h->read_id_base = 1;
    h->pos_pending = false; h->scan_tiles = 0;
    h->metrics.n_reads = R; h->metrics.n_hits = E; h->metrics.n_selected = M;
    h->comm_parked = h->comm; h->comm = nullptr;           // from here on a single-GPU handle
    h->have_index = false; h->have_pairs = false;
    const bool had_selection = h->have_selection, had_components = h->have_components;
    HGA_TRY(hga_index_run(h));                               // by-slot index over all reads (clears the later stages' flags)
    h->have_selection = had_selection; h->have_components = had_components;
    return HGA_OK;
}

extern "C" int hga_comm_unique_id(void *id128) {
    if (!id128) { hga_set_error("hga_comm_unique_id: NULL buffer"); return HGA_E_ARG; }
    HGA_TRY(load_nccl());
    static_assert(sizeof(ncclUniqueId) == 128, "ncclUniqueId is expected to be 128 bytes");
    ncclUniqueId id;
    HGA_NCCL(g_nccl.GetUniqueId(&id));
    memcpy(id128, &id, 128);
    return HGA_OK;
}

extern "C" int hga_comm_init(hga_handle *h, const void *id128, int rank, int nranks, uint64_t n_reads_total) {
    if (!h || !id128) { hga_set_error("hga_comm_init: NULL argument"); return HGA_E_ARG; }
    if (nranks < 1 || rank < 0 || rank >= nranks || nranks > 62) { hga_set_error("hga_comm_init: bad rank %d / %d", rank, nranks); return HGA_E_ARG; }
    if (n_reads_total >= (1ull << 32) - 1) { hga_set_error("hga_comm_init: more than 2^32-2 reads"); return HGA_E_ARG; }
    HGA_TRY(load_nccl());
    HGA_CUDA(cudaSetDevice(h->device));
    hga_comm_destroy(h);
    hga_comm *c = new hga_comm();
    c->rank = rank; c->size = nranks;
    ncclUniqueId id;
    memcpy(&id, id128, 128);
    ncclResult_t r = g_nccl.CommInitRank(&c->comm, nranks, id, rank);
    if (r != ncclSuccess) { hga_set_error("ncclCommInitRank failed: %s", g_nccl.GetErrorString(r)); delete c; return HGA_E_NCCL; }
    if (c->d_small.ensure((size_t) (nranks + 4) * 8 * (nranks + 4)) != HGA_OK) { g_nccl.CommDestroy(c->comm); delete c; return HGA_E_NOMEM; }   // count matrices: never allocated inside a stage
    h->comm = c;
    h->n_reads_total = n_reads_total;
    return HGA_OK;
}
