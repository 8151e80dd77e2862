// pair_count: score(x,y) = sum_k mult_x(k) * mult_y(k) for all read pairs sharing a discriminative k-mer.
//
// Replaces ReadClusteringEngine::get_connections / get_all_connections
// (clustering/ReadClusteringEngine.cpp:301-339): per pivot, the reference walks the pivot's k-mer id list
// (duplicates included) and every entry of each k-mer's inverted list (duplicates included) and does
// ++count[candidate] in a tsl::robin_map. This is a sparse integer A * A^T; here it is row-wise Gustavson in
// three tiers:
//   1. pair_count_warp_kernel<512>: one WARP per pivot row, a per-warp shared-memory open-addressing accumulator. Each LANE
//      owns one incidence entry at a time and walks that k-mer's inverted list itself, so a warp has 32 independent list walks
//      (and their random offset look-ups) in flight; a lane that finishes a list picks up the row's next entry without
//      waiting for the others, and the offsets of its next list are prefetched while it walks the current one. Lists are
//      sorted by row, so with all rows as pivots the walk runs from the END of the list and stops at the first row <= pivot:
//      only the half of every list that can produce a (pivot < partner) pair is read, eight entries = one aligned 32 B sector per
//      step, and every unordered pair is produced exactly once. The loop body is ONE predicated path for all 32 lanes (round 1 ran
//      with 10 of 32 lanes per instruction): list switch, the step's eight probes issued together, a predicated shared-memory
//      increment for the partners found at their home slot, and a probe loop the warp steps through together for the misses. Lists
//      longer than PW_LONG are walked by the whole warp with coalesced loads. The first pass runs with 512-entry accumulators
//      (55 registers, 9 CTAs per SM) and the few rows whose partner set does not fit are redone by pair_count_redo_kernel (a CTA
//      per row, four warps on quarter ranges with 1024-entry accumulators that are merged at the end). The pivots take their tickets
//      in min-hash order (row_minhash_kernel); with a communicator the lists are partitioned by whole table buckets, so neighbouring
//      hits still have neighbouring lists and the same kernels run there. What was measured and dropped: DESIGN.md 3.4.
//   2. pair_count_kernel: rows whose partner set overflowed tier 1; one CTA per row, 4096-entry accumulator.
//   3. pair_count_heavy_kernel: rows that overflow tier 2; per-CTA accumulator in HBM.
// Output: (key = min_row << 32 | max_row, score) appended through one atomic cursor bump per row, then one
// radix sort by key puts the pairs in the canonical (x asc, y asc) order that the tie rule of
// hga_select_edges needs.
#include "hga_internal.cuh"

#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_reduce.cuh>
#include <cub/device/device_select.cuh>

#define PC_THREADS 128
#define PC_WARPS (PC_THREADS / 32)
#define PC_CMAX 4096
#define PC_EMPTY 0xFFFFFFFFu
#define HV_THREADS 256
#define PW_THREADS 128
#define PW_WARPS (PW_THREADS / 32)
#define PW_CMAX 1024               // accumulator of the second pass of tier 1
#define PW_CMAX_FIRST 512          // accumulator of the first pass (more resident warps)
#define PW_LONG 96
#define PW_DEFER 32

// which (pivot x, candidate y) combinations a pivot accumulates
#define PAIR_MODE_TAIL 0     // every row is a pivot (on some GPU): y > x (walk list tails only)
#define PAIR_MODE_SUBSET 1   // pivot subset: pair (pivot, non-pivot), or ordered pivot pair

struct PairScalars {
    unsigned long long ticket;
    unsigned long long cursor;        // entries wanted (may exceed capacity)
    unsigned long long heavy_count;
    unsigned long long heavy_ticket;
    unsigned long long increments;
    unsigned long long mid_count;
    unsigned long long mid_ticket;
    unsigned long long redo_count;    // rows whose partner set overflowed the first-pass accumulator of tier 1
    unsigned long long redo_ticket;
    unsigned int overflow;
    unsigned int score_carry;         // a 32-bit score accumulator wrapped (set by the checked kernel variants only)
};

namespace {

struct PairParams {
    const uint64_t *row_off;
    const uint32_t *row_slot;
    uint64_t n_rows;
    uint32_t pivot_mul, pivot_add;  // all-rows mode: pivot t is row t * pivot_mul + pivot_add (multi-GPU: rank, rank + G, ...)
    const uint32_t *inv_off;
    const uint32_t *inv_row;        // global row numbers
    const uint32_t *pivot_rows;     // nullptr: every local row is a pivot
    const uint8_t *pivot_flag;      // SUBSET mode only
    uint64_t n_pivots;
    int mode;
    uint32_t min_score;
    uint64_t *out_key;
    uint32_t *out_score;
    uint64_t capacity;
    uint32_t *redo_list;
    uint32_t *mid_list;
    uint32_t *heavy_list;
    uint32_t *heavy_tab;            // per-CTA tables of heavy_cap (key,val) pairs
    uint32_t heavy_cap;             // power of two
    PairScalars *sc;
};

__device__ __forceinline__ bool keep_candidate(uint32_t x, uint32_t y, int mode, const uint8_t *pivot_flag) {
    if (y == x) return false;                         // :317 erase(pivot)
    if (mode == PAIR_MODE_TAIL) return y > x;         // all rows are pivots: count each unordered pair once
    return !pivot_flag[y] || y > x;
}

__device__ __forceinline__ uint32_t hash_row(uint32_t y) { return y * 2654435761u; }

// score accumulation. A score is at most hits(x) * hits(y), so it cannot exceed 2^32 - 1 while every row holds fewer than 65 536
// hits; hga_pairs_run runs the CHECK = false kernels then (the plain atomic, unchanged). Otherwise the CHECK = true variants look at
// the value the atomic returns: values only grow and every partial sum is a lower bound of a true score, so a carry out of any add
// means a true score above 2^32 - 1, which the host reports as HGA_E_OVERFLOW.
template<bool CHECK>
__device__ __forceinline__ void score_add(uint32_t *v, uint32_t c, unsigned int *carry) {
    if (CHECK) { if (atomicAdd(v, c) > 0xFFFFFFFFu - c) *carry = 1u; }
    else atomicAdd(v, c);
}

template<int THREADS>
__device__ __forceinline__ unsigned long long block_sum(unsigned long long v, unsigned long long *s_red) {
    #pragma unroll
    for (int d = 16; d > 0; d >>= 1) v += __shfl_xor_sync(0xFFFFFFFFu, v, d);
    if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = v;
    __syncthreads();
    unsigned long long t = 0;
    #pragma unroll
    for (int i = 0; i < THREADS / 32; i++) t += s_red[i];
    __syncthreads();
    return t;
}

// exclusive prefix of v over the CTA, total in *total
template<int THREADS>
__device__ __forceinline__ uint32_t block_excl_scan(uint32_t v, uint32_t *s_red, uint32_t *total) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint32_t incl = v;
    #pragma unroll
    for (int d = 1; d < 32; d <<= 1) { uint32_t t = __shfl_up_sync(0xFFFFFFFFu, incl, d); if (lane >= d) incl += t; }
    if (lane == 31) s_red[warp] = incl;
    __syncthreads();
    uint32_t base = 0, tot = 0;
    #pragma unroll
    for (int i = 0; i < THREADS / 32; i++) { if (i < warp) base += s_red[i]; tot += s_red[i]; }
    __syncthreads();
    *total = tot;
    return base + incl - v;
}

// ---- tier 1 ---------------------------------------------------------------------------------------------------
template<int CMAX>
struct WarpAcc {
    uint32_t key[CMAX];
    uint32_t val[CMAX];
    uint2 defer[PW_DEFER];          // long lists: [lo, hi)
    uint32_t distinct, overflow, n_defer, pad;
};

// ++count[y] with shared-memory atomics; most calls find y already present: one plain read, one atomic add
template<int CMAX, bool CHECK = false>
__device__ __forceinline__ void acc_add(WarpAcc<CMAX> &A, uint32_t y, uint32_t c, uint32_t cmask, int cshift, uint32_t limit, unsigned int *carry) {
    uint32_t h = hash_row(y) >> cshift;
    for (;;) {
        uint32_t cur = *reinterpret_cast<volatile uint32_t *>(&A.key[h]);
        if (cur == PC_EMPTY) {
            cur = atomicCAS(&A.key[h], PC_EMPTY, y);
            if (cur == PC_EMPTY) { if (atomicAdd(&A.distinct, 1u) >= limit) A.overflow = 1; cur = y; }
        }
        if (cur == y) { score_add<CHECK>(&A.val[h], c, carry); return; }
        if (*reinterpret_cast<volatile uint32_t *>(&A.overflow)) return;
        h = (h + 1) & cmask;
    }
}

// The walk of one pivot row's incidence entries [a, b) by one warp into its accumulator A.
// TAILONLY: the mode is PAIR_MODE_TAIL at compile time (all rows are pivots: the first-pass kernel of the hot path), so the candidate test is y > x and nothing else
template<int CMAX, int EPS = 4, bool TAILONLY = false, bool CHECK = false>
__device__ __forceinline__ void walk_row(WarpAcc<CMAX> &A, const PairParams &p, uint32_t x, uint64_t a, uint64_t b, bool tail_rt, uint32_t cmask, int cshift,
                                         uint32_t limit, int lane) {
    const bool tail = TAILONLY ? true : tail_rt;
    const int mode = TAILONLY ? PAIR_MODE_TAIL : p.mode;
    // every lane: one list at a time, two lists ahead in flight: the bounds of list j + 64 are being loaded while the
    // last 16 B chunk of list j + 32 (bounds known by now) is prefetched into L2 and list j is walked. (Requesting
    // every chunk one step before it is used - a register double buffer - was measured 14 % SLOWER (r1t). Giving every
    // lane one contiguous block of the row's entries instead of the interleaved lane, lane + 32, ... was 27 % slower (r3v):
    // neighbouring lanes walking neighbouring lists is what coalesces the list loads.)
    uint64_t j = a + lane;
    uint32_t cur_lo = 0, cur_i = 0, n1_lo = 0, n1_hi = 0, n2_lo = 0, n2_hi = 0, slot3 = 0;
    bool have1 = j < b, have2 = j + 32 < b, have3 = j + 64 < b;
    // three lists in flight per lane: list j is walked, the bounds of list j + 32 are known (its last chunk prefetched), and the SLOT of
    // list j + 64 is on its way, so that no load is issued with an address that has to be waited for (r2z: 13 % of the stall samples sat
    // on the slot -> offset chain)
    if (have1) { const uint32_t slot = __ldg(&p.row_slot[j]); n1_lo = __ldg(&p.inv_off[slot]); n1_hi = __ldg(&p.inv_off[slot + 1]); }
    if (have2) { const uint32_t slot = __ldg(&p.row_slot[j + 32]); n2_lo = __ldg(&p.inv_off[slot]); n2_hi = __ldg(&p.inv_off[slot + 1]); }
    if (have3) slot3 = __ldg(&p.row_slot[j + 64]);
    // One loop body for all 32 lanes, predicated rather than branched (r2q: with one branch per list entry - fast path, probe loop, not
    // in range - the warp ran with 10 of 32 lanes per instruction on average): a lane that has finished its list switches to the next
    // one and goes straight on to that list's first chunk; the four entries of a chunk take the fast path together (partner already at
    // its home slot: one predicated shared-memory increment each); the entries that missed are resolved afterwards in a probe loop the
    // whole warp steps through together, one probe per lane and step.
    while (__any_sync(0xFFFFFFFFu, have1 || cur_i > cur_lo)) {
        if (cur_i <= cur_lo && have1) {
            cur_lo = n1_lo; cur_i = n1_hi;
            if (cur_i - cur_lo > PW_LONG) {                           // long list: leave it to the whole warp
                const uint32_t at = atomicAdd(&A.n_defer, 1u);
                if (at < PW_DEFER) { A.defer[at] = make_uint2(cur_lo, cur_i); cur_i = cur_lo; }
            }
            j += 32;
            have1 = have2; n1_lo = n2_lo; n1_hi = n2_hi;
            if (have1 && n1_hi > n1_lo) {
                // (into L1 instead: no change; the sector below the current chunk as well: 53.5 -> 62.3 ms, r3a)
                asm volatile("prefetch.global.L2 [%0];" :: "l"(p.inv_row + (((size_t) n1_hi - 1) & ~(size_t) 3)));
            }
            have2 = have3;
            if (have2) { n2_lo = __ldg(&p.inv_off[slot3]); n2_hi = __ldg(&p.inv_off[slot3 + 1]); }
            have3 = j + 64 < b;
            if (have3) slot3 = __ldg(&p.row_slot[j + 64]);
        }
        // EPS (4 or 8) list entries per step (one aligned 16 / 32 B piece), walked from the end of the list
        const bool act = cur_i > cur_lo;
        uint32_t cb = 0;
        uint32_t ys[EPS];
        #pragma unroll
        for (int e = 0; e < EPS; e++) ys[e] = 0u;
        if (act) {
            const uint32_t q = (cur_i - 1) / EPS;
            cb = q * EPS;
            #pragma unroll
            for (int v = 0; v < EPS / 4; v++) {
                const uint4 c = __ldg(reinterpret_cast<const uint4 *>(p.inv_row) + (size_t) q * (EPS / 4) + v);
                ys[4 * v] = c.x; ys[4 * v + 1] = c.y; ys[4 * v + 2] = c.z; ys[4 * v + 3] = c.w;
            }
        }
        bool ok[EPS], stop = false;
        uint32_t hh[EPS], kk[EPS];
        #pragma unroll
        for (int e = 0; e < EPS; e++) {
            const uint32_t idx = cb + e;
            const bool inr = act && idx < cur_i && idx >= cur_lo;
            stop |= inr && tail && ys[e] <= x;                    // ascending list: nothing further down can be > x
            ok[e] = inr && keep_candidate(x, ys[e], mode, p.pivot_flag);
            hh[e] = hash_row(ys[e]) >> cshift;
        }
        #pragma unroll
        for (int e = 0; e < EPS; e++) kk[e] = ok[e] ? *reinterpret_cast<volatile uint32_t *>(&A.key[hh[e]]) : 0u;
        uint32_t pend = 0;
        #pragma unroll
        for (int e = 0; e < EPS; e++) {
            const bool fast = ok[e] && kk[e] == ys[e];
            if (fast) score_add<CHECK>(&A.val[hh[e]], 1u, &p.sc->score_carry);
            if (ok[e] && !fast) pend |= 1u << e;
        }
        if (__any_sync(0xFFFFFFFFu, pend != 0)) {                  // warp uniform
            uint32_t y = 0, hsl = 0;
            bool busy = false;
            for (;;) {
                if (!busy && pend) {
                    const int e = __ffs(pend) - 1;
                    pend &= pend - 1;
                    #pragma unroll
                    for (int f = 0; f < EPS; f++) if (e == f) { y = ys[f]; hsl = hh[f]; }
                    busy = true;
                }
                if (!__any_sync(0xFFFFFFFFu, busy)) break;
                if (busy) {
                    uint32_t cur = *reinterpret_cast<volatile uint32_t *>(&A.key[hsl]);
                    if (cur == PC_EMPTY) {
                        cur = atomicCAS(&A.key[hsl], PC_EMPTY, y);
                        if (cur == PC_EMPTY) { if (atomicAdd(&A.distinct, 1u) >= limit) A.overflow = 1; cur = y; }
                    }
                    if (cur == y) { score_add<CHECK>(&A.val[hsl], 1u, &p.sc->score_carry); busy = false; }
                    else if (*reinterpret_cast<volatile uint32_t *>(&A.overflow)) { busy = false; pend = 0; }
                    else hsl = (hsl + 1) & cmask;
                }
            }
        }
        if (act) cur_i = stop ? cur_lo : max(cb, cur_lo);
        if (*reinterpret_cast<volatile uint32_t *>(&A.overflow)) { cur_i = cur_lo; have1 = false; }
    }
    __syncwarp();
    const uint32_t nd = min(*reinterpret_cast<volatile uint32_t *>(&A.n_defer), (uint32_t) PW_DEFER);
    for (uint32_t d = 0; d < nd && !*reinterpret_cast<volatile uint32_t *>(&A.overflow); d++) {
        const uint2 r = A.defer[d];
        for (int64_t i = (int64_t) r.y - 1 - lane;; i -= 32) {
            bool go = i >= (int64_t) r.x;
            if (go) {
                const uint32_t y = __ldg(&p.inv_row[i]);
                if (tail && y <= x) go = false;
                else if (keep_candidate(x, y, mode, p.pivot_flag)) acc_add<CMAX, CHECK>(A, y, 1u, cmask, cshift, limit, &p.sc->score_carry);
            }
            if (!__any_sync(0xFFFFFFFFu, go)) break;
        }
    }
    __syncwarp();
}

// entries of A with score >= min_score -> output (one cursor bump per call)
template<int CMAX>
__device__ __forceinline__ void flush_table(WarpAcc<CMAX> &A, const PairParams &p, uint32_t x, uint32_t C, int lane) {
    // flush: entries with score >= min_score
    uint32_t total = 0;
    for (uint32_t i0 = 0; i0 < C; i0 += 32) {
        const bool ok = A.key[i0 + lane] != PC_EMPTY && A.val[i0 + lane] >= p.min_score;
        total += __popc(__ballot_sync(0xFFFFFFFFu, ok));
    }
    if (total) {
        unsigned long long base = 0;
        if (lane == 0) {
            base = atomicAdd(&p.sc->cursor, (unsigned long long) total);
            if (base + total > p.capacity) p.sc->overflow = 1;
        }
        base = __shfl_sync(0xFFFFFFFFu, base, 0);
        if (base + total <= p.capacity) {
            uint32_t off = 0;
            for (uint32_t i0 = 0; i0 < C; i0 += 32) {
                const uint32_t y = A.key[i0 + lane], v = A.val[i0 + lane];
                const bool ok = y != PC_EMPTY && v >= p.min_score;
                const uint32_t bal = __ballot_sync(0xFFFFFFFFu, ok);
                if (ok) {
                    const uint64_t at = base + off + __popc(bal & ((1u << lane) - 1));
                    p.out_key[at] = ((uint64_t) min(x, y) << 32) | max(x, y);
                    p.out_score[at] = v;
                }
                off += __popc(bal);
            }
        }
    }
}

// The kernel is latency bound and its time is inversely proportional to the number of resident warps (r3s: 1 / 2 / 3 / 4 / 6 CTAs
// per SM -> 359 / 186 / 130 / 102 / 75 ms), and the accumulator is what limits them. The first pass therefore runs with a 512-entry
// accumulator (17 KB per CTA), registers limited for 9 CTAs per SM, and eight list entries (one 32 B sector) per step; the rows whose
// partner set does not fit are listed and redone by pair_count_redo_kernel with 1024 entries, and only what overflows that goes on to
// tier 2. (r3p / r3q, config 4, (CTAs per SM the registers are limited for, entries per step): (1, 4) 56 registers 55.5 ms, (1, 8) 75
// registers 53.7, (8, 8) 59 registers 49.8, (9, 8) 48.7, (10, 8) 47 registers 48.7, (8, 16) 60.3, (6, 16) 65.0.)
template<bool TAILONLY, bool CHECK>
__global__ void __launch_bounds__(PW_THREADS, 9) pair_count_warp_kernel(const __grid_constant__ PairParams p) {
    constexpr int CMAX = PW_CMAX_FIRST;
    __shared__ WarpAcc<CMAX> s_acc[PW_WARPS];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    WarpAcc<CMAX> &A = s_acc[warp];
    const bool tail = p.mode == PAIR_MODE_TAIL;
    const unsigned long long n_items = p.n_pivots;

    for (;;) {
        unsigned long long t = 0;
        if (lane == 0) t = atomicAdd(&p.sc->ticket, 1ull);
        t = __shfl_sync(0xFFFFFFFFu, t, 0);
        if (t >= n_items) break;
        // x: global row (what the inverted lists hold); xl: row of the by-read incidence on this GPU
        const uint32_t x = p.pivot_rows ? p.pivot_rows[t] : (uint32_t) t * p.pivot_mul + p.pivot_add;
        const uint32_t xl = p.pivot_rows ? x : (uint32_t) t;
        const uint64_t a = p.row_off[xl], b = p.row_off[xl + 1];
        if (a == b) continue;

        uint32_t C = 64;
        while (C < CMAX && C < 4 * (b - a)) C <<= 1;
        for (bool retry = false;; retry = true) {
            if (retry) C = CMAX;
            const uint32_t cmask = C - 1, limit = (C / 4) * 3;
            const int cshift = 32 - (31 - __clz(C));
            for (uint32_t i = lane; i < C; i += 32) { A.key[i] = PC_EMPTY; A.val[i] = 0; }
            if (lane == 0) { A.distinct = 0; A.overflow = 0; A.n_defer = 0; }
            __syncwarp();

            walk_row<CMAX, 8, TAILONLY, CHECK>(A, p, x, a, b, tail, cmask, cshift, limit, lane);
            if (!*reinterpret_cast<volatile uint32_t *>(&A.overflow)) {
                flush_table<CMAX>(A, p, x, C, lane);
                break;
            }
            if (C == CMAX) {         // more partners than this accumulator holds: second pass, then tier 2
                if (lane == 0) p.redo_list[atomicAdd(&p.sc->redo_count, 1ull)] = xl;
                break;
            }
        }
        __syncwarp();
    }
}

// Second pass of tier 1, for the rows whose partner set overflowed the 512-entry accumulator. They are few (2 732 of 1 M at
// config 4) and they are the longest rows, so one warp per row leaves the GPU waiting for the slowest of them (5.6 ms); here a
// CTA takes a row: every warp walks a quarter of the row's incidence entries into its own 1024-entry accumulator, then warps
// 1 .. 3 pour theirs into warp 0's, which is flushed. A row whose merged partner set still does not fit goes to tier 2.
template<bool CHECK = false>
__global__ void __launch_bounds__(PW_THREADS) pair_count_redo_kernel(const __grid_constant__ PairParams p) {
    __shared__ WarpAcc<PW_CMAX> s_acc[PW_WARPS];
    __shared__ unsigned long long s_ticket;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    WarpAcc<PW_CMAX> &A = s_acc[warp];
    const bool tail = p.mode == PAIR_MODE_TAIL;
    const unsigned long long n_items = p.sc->redo_count;
    const uint32_t C = PW_CMAX, cmask = C - 1, limit = (C / 4) * 3;
    const int cshift = 32 - (31 - __clz(C));

    for (;;) {
        if (threadIdx.x == 0) s_ticket = atomicAdd(&p.sc->redo_ticket, 1ull);
        __syncthreads();
        const unsigned long long t = s_ticket;
        if (t >= n_items) break;
        const uint32_t xl = p.redo_list[t];
        const uint32_t x = p.pivot_rows ? xl : xl * p.pivot_mul + p.pivot_add;
        const uint64_t a0 = p.row_off[xl], b0 = p.row_off[xl + 1];
        // quarters in multiples of 32 entries: inside a warp, neighbouring lanes still walk neighbouring lists
        const uint64_t per = (((b0 - a0 + PW_WARPS - 1) / PW_WARPS) + 31) & ~(uint64_t) 31;
        const uint64_t a = min(b0, a0 + warp * per), b = min(b0, a + per);
        for (uint32_t i = lane; i < C; i += 32) { A.key[i] = PC_EMPTY; A.val[i] = 0; }
        if (lane == 0) { A.distinct = 0; A.overflow = 0; A.n_defer = 0; }
        __syncwarp();
        if (a < b) walk_row<PW_CMAX, 4, false, CHECK>(A, p, x, a, b, tail, cmask, cshift, limit, lane);
        __syncthreads();
        bool over = false;
        #pragma unroll
        for (int w = 0; w < PW_WARPS; w++) over |= *reinterpret_cast<volatile uint32_t *>(&s_acc[w].overflow) != 0;
        if (!over && warp > 0) {
            for (uint32_t i = lane; i < C; i += 32) {
                const uint32_t y = A.key[i];
                if (y != PC_EMPTY) acc_add<PW_CMAX, CHECK>(s_acc[0], y, A.val[i], cmask, cshift, limit, &p.sc->score_carry);
            }
        }
        __syncthreads();
        over |= *reinterpret_cast<volatile uint32_t *>(&s_acc[0].overflow) != 0;
        if (over) {
            if (threadIdx.x == 0) p.mid_list[atomicAdd(&p.sc->mid_count, 1ull)] = xl;
        } else if (warp == 0) {
            flush_table<PW_CMAX>(s_acc[0], p, x, C, lane);
        }
        __syncthreads();
    }
}

// ---- tier 2 ---------------------------------------------------------------------------------------------------
template<bool CHECK = false>
__global__ void __launch_bounds__(PC_THREADS) pair_count_kernel(PairParams p) {
    __shared__ uint32_t s_key[PC_CMAX];
    __shared__ uint32_t s_val[PC_CMAX];
    __shared__ uint32_t s_red[PC_WARPS];
    __shared__ unsigned long long s_red64[PC_WARPS];
    __shared__ unsigned long long s_ticket, s_base;
    __shared__ uint32_t s_distinct;
    __shared__ volatile uint32_t s_overflow;

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint64_t n_mid = p.sc->mid_count;

    for (;;) {
        if (tid == 0) { s_ticket = atomicAdd(&p.sc->mid_ticket, 1ull); s_distinct = 0; s_overflow = 0; }
        __syncthreads();
        const uint64_t t = s_ticket;
        if (t >= n_mid) break;
        const uint32_t xl = p.mid_list[t];
        const uint32_t x = xl * p.pivot_mul + p.pivot_add;
        const uint64_t a = p.row_off[xl], b = p.row_off[xl + 1];
        if (a == b) { __syncthreads(); continue; }

        // pass A: total list length W bounds the number of distinct partners
        unsigned long long w = 0;
        for (uint64_t j = a + tid; j < b; j += PC_THREADS) {
            const uint32_t slot = __ldg(&p.row_slot[j]);
            w += __ldg(&p.inv_off[slot + 1]) - __ldg(&p.inv_off[slot]);
        }
        const unsigned long long W = block_sum<PC_THREADS>(w, s_red64);
        uint32_t C = 64;
        while (C < PC_CMAX && C < 2 * W) C <<= 1;
        const uint32_t limit = (C / 4) * 3;   // never reached unless C was clamped to PC_CMAX (distinct <= W <= C/2)
        const uint32_t cmask = C - 1;
        int cbits = 31 - __clz(C);
        for (uint32_t i = tid; i < C; i += PC_THREADS) { s_key[i] = PC_EMPTY; s_val[i] = 0; }
        __syncthreads();

        // pass B: warp per incidence entry, lanes over the inverted list
        for (uint64_t j = a + warp; j < b && !s_overflow; j += PC_WARPS) {
            const uint32_t slot = __ldg(&p.row_slot[j]);
            const uint32_t lo = __ldg(&p.inv_off[slot]), hi = __ldg(&p.inv_off[slot + 1]);
            for (uint32_t i = lo + lane; i < hi; i += 32) {
                const uint32_t y = __ldg(&p.inv_row[i]);
                if (!keep_candidate(x, y, p.mode, p.pivot_flag)) continue;
                uint32_t hsh = hash_row(y) >> (32 - cbits);
                for (;;) {
                    const uint32_t old = atomicCAS(&s_key[hsh], PC_EMPTY, y);
                    if (old == PC_EMPTY) {
                        if (atomicAdd(&s_distinct, 1u) + 1 > limit) s_overflow = 1;
                    }
                    if (old == PC_EMPTY || old == y) { score_add<CHECK>(&s_val[hsh], 1u, &p.sc->score_carry); break; }
                    if (s_overflow) break;
                    hsh = (hsh + 1) & cmask;
                }
            }
        }
        __syncthreads();
        if (s_overflow) {
            if (tid == 0) {
                const unsigned long long hi = atomicAdd(&p.sc->heavy_count, 1ull);
                p.heavy_list[hi] = xl;
            }
            __syncthreads();
            continue;
        }

        // compaction: entries with score >= min_score
        uint32_t mine = 0;
        for (uint32_t i = tid; i < C; i += PC_THREADS) mine += (s_key[i] != PC_EMPTY && s_val[i] >= p.min_score);
        uint32_t total;
        uint32_t off = block_excl_scan<PC_THREADS>(mine, s_red, &total);
        if (tid == 0) {
            s_base = total ? atomicAdd(&p.sc->cursor, (unsigned long long) total) : 0ull;
            if (total && s_base + total > p.capacity) p.sc->overflow = 1;
        }
        __syncthreads();
        const uint64_t base = s_base;
        if (total && base + total <= p.capacity) {
            for (uint32_t i = tid; i < C; i += PC_THREADS) {
                const uint32_t y = s_key[i], v = s_val[i];
                if (y != PC_EMPTY && v >= p.min_score) {
                    const uint32_t lo = min(x, y), hi = max(x, y);
                    p.out_key[base + off] = ((uint64_t) lo << 32) | hi;
                    p.out_score[base + off] = v;
                    off++;
                }
            }
        }
        __syncthreads();
    }
}

// Rows whose partner set overflowed the shared-memory accumulator: same algorithm, table in HBM.
template<bool CHECK = false>
__global__ void __launch_bounds__(HV_THREADS) pair_count_heavy_kernel(PairParams p) {
    __shared__ uint32_t s_red[HV_THREADS / 32];
    __shared__ unsigned long long s_ticket, s_base;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    uint32_t *tab_key = p.heavy_tab + (size_t) blockIdx.x * 2 * p.heavy_cap;
    uint32_t *tab_val = tab_key + p.heavy_cap;
    const uint32_t cmask = p.heavy_cap - 1;
    const int cbits = 31 - __clz(p.heavy_cap);
    const uint64_t n_heavy = p.sc->heavy_count;

    for (;;) {
        if (tid == 0) s_ticket = atomicAdd(&p.sc->heavy_ticket, 1ull);
        __syncthreads();
        const uint64_t t = s_ticket;
        if (t >= n_heavy) break;
        const uint32_t xl = p.heavy_list[t];
        const uint32_t x = xl * p.pivot_mul + p.pivot_add;
        const uint64_t a = p.row_off[xl], b = p.row_off[xl + 1];
        for (uint32_t i = tid; i < p.heavy_cap; i += HV_THREADS) { tab_key[i] = PC_EMPTY; tab_val[i] = 0; }
        __syncthreads();
        for (uint64_t j = a + warp; j < b; j += HV_THREADS / 32) {
            const uint32_t slot = __ldg(&p.row_slot[j]);
            const uint32_t lo = __ldg(&p.inv_off[slot]), hi = __ldg(&p.inv_off[slot + 1]);
            for (uint32_t i = lo + lane; i < hi; i += 32) {
                const uint32_t y = __ldg(&p.inv_row[i]);
                if (!keep_candidate(x, y, p.mode, p.pivot_flag)) continue;
                uint32_t hsh = hash_row(y) >> (32 - cbits);
                for (;;) {
                    const uint32_t old = atomicCAS(&tab_key[hsh], PC_EMPTY, y);
                    if (old == PC_EMPTY || old == y) { score_add<CHECK>(&tab_val[hsh], 1u, &p.sc->score_carry); break; }
                    hsh = (hsh + 1) & cmask;
                }
            }
        }
        __syncthreads();
        uint32_t mine = 0;
        for (uint32_t i = tid; i < p.heavy_cap; i += HV_THREADS) mine += (tab_key[i] != PC_EMPTY && tab_val[i] >= p.min_score);
        uint32_t total;
        uint32_t off = block_excl_scan<HV_THREADS>(mine, s_red, &total);
        if (tid == 0) {
            s_base = total ? atomicAdd(&p.sc->cursor, (unsigned long long) total) : 0ull;
            if (total && s_base + total > p.capacity) p.sc->overflow = 1;
        }
        __syncthreads();
        const uint64_t base = s_base;
        if (total && base + total <= p.capacity) {
            for (uint32_t i = tid; i < p.heavy_cap; i += HV_THREADS) {
                const uint32_t y = tab_key[i], v = tab_val[i];
                if (y != PC_EMPTY && v >= p.min_score) {
                    const uint32_t lo = min(x, y), hi = max(x, y);
                    p.out_key[base + off] = ((uint64_t) lo << 32) | hi;
                    p.out_score[base + off] = v;
                    off++;
                }
            }
        }
        __syncthreads();
    }
}

// work measure: sum over this GPU's lists of occ*(occ-1)/2
__global__ void increments_kernel(const uint32_t *__restrict__ inv_off, uint32_t n_slots, unsigned long long *out) {
    unsigned long long acc = 0;
    for (uint64_t i = blockIdx.x * (uint64_t) blockDim.x + threadIdx.x; i < n_slots; i += (uint64_t) gridDim.x * blockDim.x) {
        const unsigned long long len = inv_off[i + 1] - inv_off[i];
        acc += len * (len - (len ? 1 : 0)) / 2;
    }
    #pragma unroll
    for (int d = 16; d > 0; d >>= 1) acc += __shfl_xor_sync(0xFFFFFFFFu, acc, d);
    if ((threadIdx.x & 31) == 0 && acc) atomicAdd(out, acc);
}

// Pivot order: min-hash of the row's k-mers (table slots). Reads that overlap on the genome share most of their k-mers, so they
// share their min-hash with a probability equal to their Jaccard similarity: sorting the pivots by it puts groups of overlapping
// reads next to each other in ticket order, and the inverted lists one of them pulls into L2 are found there by the others.
__global__ void row_minhash_kernel(const uint64_t *__restrict__ row_off, const uint32_t *__restrict__ row_slot, uint64_t n_rows, uint32_t *__restrict__ key,
                                   uint32_t *__restrict__ row) {
    const uint64_t warps = ((uint64_t) gridDim.x * blockDim.x) >> 5;
    const uint64_t w = (blockIdx.x * (uint64_t) blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    for (uint64_t r = w; r < n_rows; r += warps) {
        const uint64_t a = row_off[r], b = row_off[r + 1];
        uint32_t m = 0xFFFFFFFFu;
        for (uint64_t i = a + lane; i < b; i += 32) {
            uint32_t h = row_slot[i] * 0x9E3779B1u;
            h ^= h >> 15; h *= 0x85EBCA77u; h ^= h >> 13;
            m = min(m, h);
        }
        #pragma unroll
        for (int d = 16; d > 0; d >>= 1) m = min(m, __shfl_xor_sync(0xFFFFFFFFu, m, d));
        if (lane == 0) { key[r] = m; row[r] = (uint32_t) r; }
    }
}

// largest hit count of a row: bounds every score by its square
__global__ void max_row_hits_kernel(const uint64_t *__restrict__ row_off, uint64_t n_rows, unsigned long long *out) {
    unsigned long long m = 0;
    for (uint64_t i = blockIdx.x * (uint64_t) blockDim.x + threadIdx.x; i < n_rows; i += (uint64_t) gridDim.x * blockDim.x) m = max(m, (unsigned long long) (row_off[i + 1] - row_off[i]));
    #pragma unroll
    for (int d = 16; d > 0; d >>= 1) m = max(m, __shfl_xor_sync(0xFFFFFFFFu, m, d));
    if ((threadIdx.x & 31) == 0 && m) atomicMax(out, m);
}

__global__ void flag_min_score_kernel(const uint32_t *__restrict__ score, uint64_t n, uint32_t min_score, uint8_t *flag) {
    for (uint64_t i = blockIdx.x * (uint64_t) blockDim.x + threadIdx.x; i < n; i += (uint64_t) gridDim.x * blockDim.x) flag[i] = score[i] >= min_score;
}

__global__ void mark_pivots_kernel(const uint32_t *__restrict__ pivot_rows, uint64_t n, uint8_t *flag) {
    for (uint64_t i = blockIdx.x * (uint64_t) blockDim.x + threadIdx.x; i < n; i += (uint64_t) gridDim.x * blockDim.x) flag[pivot_rows[i]] = 1;
}

}  // namespace

int hga_pairs_run(hga_handle *h, uint32_t min_score, const uint32_t *pivots, uint64_t n_pivots) {
    if (!h->have_index) { hga_set_error("hga_pair_count: no index (call hga_build_index)"); return HGA_E_STATE; }
    h->have_pairs = h->have_selection = h->have_components = false;
    const bool multi = h->comm && hga_comm_size(h) > 1;
    const uint64_t n_rows = h->pair_rows;         // rows of the by-read incidence (all reads with a communicator)
    h->pair_min_score = min_score;
    h->pair_subset = pivots != nullptr;
    if (multi && pivots) { hga_set_error("hga_pair_count: pivot subsets are not supported with a communicator"); return HGA_E_ARG; }

    HGA_TRY(h->d_pair_scalars.ensure(sizeof(PairScalars)));
    PairScalars *d_sc = h->d_pair_scalars.as<PairScalars>();
    HGA_TRY(h->d_heavy_list.ensure((n_rows + 1) * 4));
    HGA_TRY(h->d_mid_list.ensure((n_rows + 1) * 4));
    HGA_TRY(h->d_redo_list.ensure((n_rows + 1) * 4));

    // Scores fit 32 bits while every read has fewer than 65 536 hits (score <= hits(x) * hits(y)); above that the checked kernel
    // variants run and a score that does not fit is an error rather than a wrapped value. With a communicator the partial scores
    // are summed in 32 bits by the exchange, which has no such check: such inputs are refused there.
    uint64_t max_hits = 0;
    {
        HGA_CUDA(cudaMemsetAsync(&d_sc->increments, 0, 8, h->stream));
        if (h->n_reads) {
            max_row_hits_kernel<<<(int) std::min<uint64_t>((h->n_reads + 255) / 256, (uint64_t) h->sm_count * 8), 256, 0, h->stream>>>(
                h->d_row_off.as<uint64_t>(), h->n_reads, &d_sc->increments);
            h->metrics.kernel_launches++;
            HGA_CUDA(cudaGetLastError());
        }
        HGA_CUDA(cudaMemcpyAsync(&max_hits, &d_sc->increments, 8, cudaMemcpyDeviceToHost, h->stream));
        HGA_CUDA(cudaStreamSynchronize(h->stream));
        if (multi) {
            std::vector<uint64_t> all;
            HGA_TRY(hga_comm_allgather_u64(h, max_hits, all));
            for (uint64_t v : all) max_hits = std::max(max_hits, v);
        }
    }
    const bool check_scores = max_hits > 65535;
    if (check_scores && multi) {
        hga_set_error("hga_pair_count: a read has %llu hits, so a pair score may exceed 2^32 - 1, which the multi-GPU reduction of partial "
                      "scores cannot detect; run this input on one GPU", (unsigned long long) max_hits);
        return HGA_E_OVERFLOW;
    }

    PairParams p;
    memset(&p, 0, sizeof(p));
    p.n_rows = n_rows;
    // multi-GPU: ALL rows are pivots on every GPU, each row restricted to its hits on this GPU's k-mers (hga_comm.cu): the scores
    // that come out are PARTIAL and are reduced at the owner of x further down
    p.row_off = multi ? h->d_g_row_off.as<uint64_t>() : h->d_row_off.as<uint64_t>();
    p.row_slot = multi ? h->d_g_kid.as<uint32_t>() : h->d_hit_slot.as<uint32_t>();
    p.pivot_mul = h->pair_pivot_mul; p.pivot_add = h->pair_pivot_add;
    p.inv_off = h->d_inv_off.as<uint32_t>(); p.inv_row = h->d_inv_row.as<uint32_t>();
    p.pivot_rows = nullptr; p.pivot_flag = nullptr;
    p.n_pivots = n_rows;
    p.mode = PAIR_MODE_TAIL;
    p.min_score = multi ? 1u : min_score;       // partial scores are filtered after the reduction
    p.mid_list = h->d_mid_list.as<uint32_t>();
    p.redo_list = h->d_redo_list.as<uint32_t>();
    p.heavy_list = h->d_heavy_list.as<uint32_t>();
    p.heavy_tab = nullptr; p.heavy_cap = 0;
    p.sc = d_sc;

    DevBuf &d_pivots = h->d_pivot_rows;      // (a member: released with the handle)
    if (pivots) {
        // caller passes read ids; rows are id - first id
        std::vector<uint32_t> rows(n_pivots);
        for (uint64_t i = 0; i < n_pivots; i++) {
            const uint64_t r = (uint64_t) pivots[i] - h->inc_row_first_id;
            if (pivots[i] < h->inc_row_first_id || r >= n_rows) { hga_set_error("pivot read id %u out of range", pivots[i]); return HGA_E_ARG; }
            rows[i] = (uint32_t) r;
        }
        HGA_TRY(d_pivots.ensure((n_pivots + 1) * 4));
        HGA_TRY(h->d_pivot_flag.ensure(n_rows + 1));
        HGA_CUDA(cudaMemcpyAsync(d_pivots.p, rows.data(), n_pivots * 4, cudaMemcpyHostToDevice, h->stream));
        HGA_CUDA(cudaMemsetAsync(h->d_pivot_flag.p, 0, n_rows + 1, h->stream));
        if (n_pivots) {
            mark_pivots_kernel<<<(int) std::min<uint64_t>((n_pivots + 255) / 256, 1024), 256, 0, h->stream>>>(d_pivots.as<uint32_t>(), n_pivots,
                                                                                                            h->d_pivot_flag.as<uint8_t>());
            h->metrics.kernel_launches++;
        }
        HGA_CUDA(cudaStreamSynchronize(h->stream));   // rows vector goes out of scope below
        p.pivot_rows = d_pivots.as<uint32_t>();
        p.pivot_flag = h->d_pivot_flag.as<uint8_t>();
        p.n_pivots = n_pivots;
        p.mode = PAIR_MODE_SUBSET;
    }

    // pivot order (a performance hint only: the pairs are sorted into canonical order afterwards): the min-hash of the row's k-mers when every
    // row is a pivot, or - HGA_PAIR_ORDER=3 + HGA_PAIR_ORDER_FILE = u32 rows - an order read from a file, loaded before the stage timer
    // (bench.py: the true genome order of its synthetic input, the upper bound of what an order can buy)
    const bool ordered = !pivots && n_rows > 4096;
    const uint32_t *file_order = nullptr;
    if (const char *e = getenv("HGA_PAIR_ORDER")) {
        const char *order_file = getenv("HGA_PAIR_ORDER_FILE");
        if (atoi(e) == 3 && order_file && ordered) {
            std::vector<uint32_t> ord(n_rows);
            FILE *f = fopen(order_file, "rb");
            if (!f || fread(ord.data(), 4, n_rows, f) != n_rows) { if (f) fclose(f); hga_set_error("HGA_PAIR_ORDER_FILE: cannot read %llu rows", (unsigned long long) n_rows); return HGA_E_ARG; }
            fclose(f);
            HGA_TRY(h->d_pivot_order.ensure((n_rows + 1) * 4 * 4));
            HGA_CUDA(cudaMemcpyAsync(h->d_pivot_order.p, ord.data(), n_rows * 4, cudaMemcpyHostToDevice, h->stream));
            HGA_CUDA(cudaStreamSynchronize(h->stream));
            file_order = h->d_pivot_order.as<uint32_t>();
        }
    }

    StageTimer timer(h, &h->metrics.pair_ms);
    Trace tr(h);
    if (file_order) {
        p.pivot_rows = file_order;
    } else if (ordered) {
        HGA_TRY(h->d_pivot_order.ensure((n_rows + 1) * 4 * 4));
        uint32_t *k_in = h->d_pivot_order.as<uint32_t>(), *r_in = k_in + (n_rows + 1), *k_out = r_in + (n_rows + 1), *r_out = k_out + (n_rows + 1);
        row_minhash_kernel<<<(int) std::min<uint64_t>((n_rows * 32 + 255) / 256, (uint64_t) h->sm_count * 32), 256, 0, h->stream>>>(p.row_off, p.row_slot, n_rows, k_in, r_in);
        size_t tmp_bytes = 0;
        HGA_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, tmp_bytes, k_in, k_out, r_in, r_out, n_rows, 0, 32, h->stream));
        HGA_TRY(h->d_sort_tmp.ensure(tmp_bytes + 16));
        HGA_CUDA(cub::DeviceRadixSort::SortPairs(h->d_sort_tmp.p, tmp_bytes, k_in, k_out, r_in, r_out, n_rows, 0, 32, h->stream));
        h->metrics.kernel_launches += 6;
        HGA_CUDA(cudaGetLastError());
        p.pivot_rows = r_out;        // all rows, TAIL mode, in that order
    }
    uint64_t capacity = std::max<uint64_t>(h->pair_capacity, std::max<uint64_t>(64 * n_rows, 1ull << 20));
    int occ_w = 0, occ_c = 0, occ_r = 0;
    typedef void (*pair_kernel_t)(const PairParams);
    pair_kernel_t first_pass = p.mode == PAIR_MODE_TAIL ? pair_count_warp_kernel<true, false> : pair_count_warp_kernel<false, false>;
    pair_kernel_t redo_kernel = pair_count_redo_kernel<false>, mid_kernel = pair_count_kernel<false>, heavy_kernel = pair_count_heavy_kernel<false>;
    if (check_scores) {
        first_pass = p.mode == PAIR_MODE_TAIL ? pair_count_warp_kernel<true, true> : pair_count_warp_kernel<false, true>;
        redo_kernel = pair_count_redo_kernel<true>; mid_kernel = pair_count_kernel<true>; heavy_kernel = pair_count_heavy_kernel<true>;
    }
    HGA_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ_w, first_pass, PW_THREADS, 0));
    HGA_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ_r, redo_kernel, PW_THREADS, 0));
    if (occ_r < 1) occ_r = 1;
    HGA_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ_c, mid_kernel, PC_THREADS, 0));
    if (occ_w < 1) occ_w = 1;
    if (occ_c < 1) occ_c = 1;
    const int grid_w = (int) std::max<uint64_t>(1, std::min<uint64_t>((uint64_t) h->sm_count * occ_w, (p.n_pivots + PW_WARPS - 1) / PW_WARPS));
    PairScalars sc;
    h->metrics.pair_retries = 0;
    for (int attempt = 0;; attempt++) {
        HGA_TRY(h->d_pair_key.ensure((capacity + 1) * 8));
        HGA_TRY(h->d_pair_score.ensure((capacity + 1) * 4));
        p.out_key = h->d_pair_key.as<uint64_t>(); p.out_score = h->d_pair_score.as<uint32_t>(); p.capacity = capacity;
        HGA_CUDA(cudaMemsetAsync(d_sc, 0, sizeof(PairScalars), h->stream));
        if (p.n_pivots) {
            first_pass<<<grid_w, PW_THREADS, 0, h->stream>>>(p);
            h->metrics.kernel_launches++;
            HGA_CUDA(cudaGetLastError());
        }
        HGA_CUDA(cudaMemcpyAsync(&sc, d_sc, sizeof(sc), cudaMemcpyDeviceToHost, h->stream));
        HGA_CUDA(cudaStreamSynchronize(h->stream));
        if (sc.redo_count) {
            const int grid_r = (int) std::max<uint64_t>(1, std::min<uint64_t>((uint64_t) h->sm_count * occ_r, sc.redo_count));
            redo_kernel<<<grid_r, PW_THREADS, 0, h->stream>>>(p);
            h->metrics.kernel_launches++;
            HGA_CUDA(cudaGetLastError());
            HGA_CUDA(cudaMemcpyAsync(&sc, d_sc, sizeof(sc), cudaMemcpyDeviceToHost, h->stream));
            HGA_CUDA(cudaStreamSynchronize(h->stream));
        }
        h->metrics.redo_pivots = sc.redo_count;
        if (sc.mid_count) {
            const int grid_c = (int) std::min<uint64_t>(sc.mid_count, (uint64_t) h->sm_count * occ_c);
            mid_kernel<<<grid_c, PC_THREADS, 0, h->stream>>>(p);
            h->metrics.kernel_launches++;
            HGA_CUDA(cudaGetLastError());
            HGA_CUDA(cudaMemcpyAsync(&sc, d_sc, sizeof(sc), cudaMemcpyDeviceToHost, h->stream));
            HGA_CUDA(cudaStreamSynchronize(h->stream));
        }
        if (sc.heavy_count) {
            uint32_t cap = 1024;
            while (cap < 2 * h->inc_rows && cap < (1u << 30)) cap <<= 1;
            uint64_t budget = 4ull << 30;
            int hgrid = (int) std::min<uint64_t>(sc.heavy_count, (uint64_t) h->sm_count);
            while (hgrid > 1 && (uint64_t) hgrid * cap * 8 > budget) hgrid--;
            HGA_TRY(h->d_heavy_tab.ensure((size_t) hgrid * cap * 8));
            p.heavy_tab = h->d_heavy_tab.as<uint32_t>(); p.heavy_cap = cap;
            heavy_kernel<<<hgrid, HV_THREADS, 0, h->stream>>>(p);
            h->metrics.kernel_launches++;
            HGA_CUDA(cudaGetLastError());
            HGA_CUDA(cudaMemcpyAsync(&sc, d_sc, sizeof(sc), cudaMemcpyDeviceToHost, h->stream));
            HGA_CUDA(cudaStreamSynchronize(h->stream));
        }
        h->metrics.heavy_pivots = sc.heavy_count;
        h->metrics.mid_pivots = sc.mid_count;
        if (sc.score_carry) {
            hga_set_error("hga_pair_count: a pair score exceeds 2^32 - 1 (a read has %llu hits; scores are counted in 32 bits)", (unsigned long long) max_hits);
            return HGA_E_OVERFLOW;
        }
        if (!sc.overflow) break;
        if (attempt >= 1) { hga_set_error("pair_count: output overflow after exact resize (internal error)"); return HGA_E_OVERFLOW; }
        capacity = sc.cursor;
        h->metrics.pair_retries++;
    }
    h->pair_capacity = capacity;
    uint64_t P = sc.cursor;
    tr.mark("kernels");
    // multi-GPU: partial (x, y, score) -> owner(x). Packed records are exchanged, sorted and summed in hga_comm.cu; when they do not fit
    // 64 bits the records travel as (key, score) and the sort / segmented sum below run on them
    bool reduced = false;
    if (multi) HGA_TRY(hga_comm_reduce_partials_packed(h, P, &P, &reduced));
    if (multi && !reduced) HGA_TRY(hga_comm_exchange_partials(h, P, &P));     // received into d_pair_key / d_pair_score
    tr.mark("exchange");

    // canonical physical order: sort by (x_row, y_row)
    HGA_TRY(h->d_pair_key2.ensure((P + 1) * 8));
    HGA_TRY(h->d_pair_score2.ensure((P + 1) * 4));
    unsigned long long *d_runs = &d_sc->heavy_ticket;      // a free scalar
    if (P > 0 && !reduced) {
        // key = x << 32 | y with x, y < 2^row_bits: two stable sorts over the bits that vary (y, then x) instead of one over all 32 + row_bits
        // (config 4: 3 + 3 passes instead of 7); the second one lands in the primary arrays again
        const int row_bits = (int) std::max<uint32_t>(hga_ceil_log2(h->inc_rows + 1), 1);
        size_t t1 = 0, t2 = 0;
        HGA_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, t1, h->d_pair_key.as<uint64_t>(), h->d_pair_key2.as<uint64_t>(),
                                                 h->d_pair_score.as<uint32_t>(), h->d_pair_score2.as<uint32_t>(), P, 0, row_bits, h->stream));
        HGA_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, t2, h->d_pair_key2.as<uint64_t>(), h->d_pair_key.as<uint64_t>(),
                                                 h->d_pair_score2.as<uint32_t>(), h->d_pair_score.as<uint32_t>(), P, 32, 32 + row_bits, h->stream));
        HGA_TRY(h->d_sort_tmp.ensure(std::max(t1, t2) + 16));
        HGA_CUDA(cub::DeviceRadixSort::SortPairs(h->d_sort_tmp.p, t1, h->d_pair_key.as<uint64_t>(), h->d_pair_key2.as<uint64_t>(),
                                                 h->d_pair_score.as<uint32_t>(), h->d_pair_score2.as<uint32_t>(), P, 0, row_bits, h->stream));
        HGA_CUDA(cub::DeviceRadixSort::SortPairs(h->d_sort_tmp.p, t2, h->d_pair_key2.as<uint64_t>(), h->d_pair_key.as<uint64_t>(),
                                                 h->d_pair_score2.as<uint32_t>(), h->d_pair_score.as<uint32_t>(), P, 32, 32 + row_bits, h->stream));
        h->metrics.kernel_launches += 2 * ((uint64_t) (row_bits + 7) / 8 + 2);
    }
    tr.mark("sort");
    if (multi && P > 0 && !reduced) {
        // one record per contributing rank and pair, now adjacent: segmented sum -> final scores (primary -> secondary -> swapped back into the primary arrays)
        size_t tmp_bytes = 0;
        HGA_CUDA(cub::DeviceReduce::ReduceByKey(nullptr, tmp_bytes, h->d_pair_key.as<uint64_t>(), h->d_pair_key2.as<uint64_t>(), h->d_pair_score.as<uint32_t>(),
                                                h->d_pair_score2.as<uint32_t>(), d_runs, cub::Sum(), P, h->stream));
        HGA_TRY(h->d_sort_tmp.ensure(tmp_bytes + 16));
        HGA_CUDA(cub::DeviceReduce::ReduceByKey(h->d_sort_tmp.p, tmp_bytes, h->d_pair_key.as<uint64_t>(), h->d_pair_key2.as<uint64_t>(), h->d_pair_score.as<uint32_t>(),
                                                h->d_pair_score2.as<uint32_t>(), d_runs, cub::Sum(), P, h->stream));
        unsigned long long runs = 0;
        HGA_CUDA(cudaMemcpyAsync(&runs, d_runs, 8, cudaMemcpyDeviceToHost, h->stream));
        HGA_CUDA(cudaStreamSynchronize(h->stream));
        P = runs;
        h->metrics.kernel_launches += 3;
        std::swap(h->d_pair_key, h->d_pair_key2);
        std::swap(h->d_pair_score, h->d_pair_score2);
    }
    if (multi && min_score > 1 && P > 0) {
        // the min_score filter the single-GPU kernels apply when they flush a row
        HGA_TRY(h->d_pair_key2.ensure((P + 1) * 8));
        HGA_TRY(h->d_pair_score2.ensure((P + 1) * 4));
        HGA_TRY(h->d_pivot_flag.ensure(P + 1));
        uint8_t *flag = h->d_pivot_flag.as<uint8_t>();
        flag_min_score_kernel<<<(int) std::min<uint64_t>((P + 255) / 256, (uint64_t) h->sm_count * 16), 256, 0, h->stream>>>(h->d_pair_score.as<uint32_t>(), P, min_score, flag);
        size_t t1 = 0, t2 = 0;
        HGA_CUDA(cub::DeviceSelect::Flagged(nullptr, t1, h->d_pair_key.as<uint64_t>(), flag, h->d_pair_key2.as<uint64_t>(), d_runs, P, h->stream));
        HGA_CUDA(cub::DeviceSelect::Flagged(nullptr, t2, h->d_pair_score.as<uint32_t>(), flag, h->d_pair_score2.as<uint32_t>(), d_runs, P, h->stream));
        HGA_TRY(h->d_sort_tmp.ensure(std::max(t1, t2) + 16));
        HGA_CUDA(cub::DeviceSelect::Flagged(h->d_sort_tmp.p, t1, h->d_pair_key.as<uint64_t>(), flag, h->d_pair_key2.as<uint64_t>(), d_runs, P, h->stream));
        HGA_CUDA(cub::DeviceSelect::Flagged(h->d_sort_tmp.p, t2, h->d_pair_score.as<uint32_t>(), flag, h->d_pair_score2.as<uint32_t>(), d_runs, P, h->stream));
        unsigned long long runs = 0;
        HGA_CUDA(cudaMemcpyAsync(&runs, d_runs, 8, cudaMemcpyDeviceToHost, h->stream));
        HGA_CUDA(cudaStreamSynchronize(h->stream));
        P = runs;
        h->metrics.kernel_launches += 5;
        std::swap(h->d_pair_key, h->d_pair_key2);
        std::swap(h->d_pair_score, h->d_pair_score2);
    }
    h->n_pairs = P;
    tr.mark("reduce");

    {   // work measure
        HGA_CUDA(cudaMemsetAsync(&d_sc->increments, 0, 8, h->stream));
        increments_kernel<<<h->sm_count * 4, 256, 0, h->stream>>>(h->d_inv_off.as<uint32_t>(), h->index_keys, &d_sc->increments);
        h->metrics.kernel_launches++;
        HGA_CUDA(cudaMemcpyAsync(&sc, d_sc, sizeof(sc), cudaMemcpyDeviceToHost, h->stream));
        HGA_CUDA(cudaStreamSynchronize(h->stream));
        h->n_increments = sc.increments;
    }
    tr.mark("increments");
    tr.dump("pairs", hga_comm_rank(h));
    timer.stop();
    h->metrics.n_pairs = h->n_pairs; h->metrics.n_increments = h->n_increments;
    h->have_pairs = true;
    return HGA_OK;
}
