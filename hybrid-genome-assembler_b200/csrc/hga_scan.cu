// scan_probe: fused 2-bit pack + canonical k-mer windows + membership test + hit compaction.
//
// Replaces the per-read half of ReadClusteringEngine::construct_indices
// (clustering/ReadClusteringEngine.cpp:246-277) and KmerIterator (common/KmerIterator.cpp:23-76).
//
// Work decomposition (B200: 148 SMs x 32 resident warps, every WARP is an independent worker, nothing synchronises two warps):
//   * the concatenated base stream is cut into tiles of SCAN_TILE (480) window-end positions; a warp takes tickets of SCAN_TICKETS
//     consecutive tiles (one atomic per ticket, the next one requested while the current is processed);
//   * phase A: every lane loads 16 bytes of ASCII bases (30 lanes hold the tile, lanes 0 and 1 the 32 bases before it) and packs
//     them into one word of forward codes (first base most significant) and one word of complement codes (first base least
//     significant). Bytes outside {A,C,G,T} get code 0 in BOTH streams - the reference's rule (KmerIterator.cpp:56,62:
//     unordered_map::operator[] default-inserts 0 in both tables) - and a bit in an exception bitmap (validity = one PRMT lookup
//     of the expected byte per 4 bases); the two previous lanes' words come over with four shuffles.
//   * phase B, lane-sequential: a lane owns SCAN_LANE (16) CONSECUTIVE window ends. With its 48 bases in registers every piece
//     is a funnel shift with a compile-time register index: the forward and reverse strand's last 16 bases and the 16 before,
//     the two hashed m-mers (one IMAD each: the multiplier shifts out everything above the m-mer), the sliding minimum over the
//     last W symmetric hashes (VIMNMX3, two instructions, no shuffles) and the strand-symmetric bit hash g(F) + g(R). No
//     canonical VALUE and no 64-bit compare is needed (hga_internal.cuh). (minimizer, bit hash) go to shared memory;
//   * phase C, lane-parallel: the 32 lanes take 32 ADJACENT windows from shared memory (a transposition through an 8-byte-
//     entry buffer with an odd row stride, conflict free both ways), so that the ~3.5 consecutive windows that share a
//     minimizer hit the same 32 B filter block and a warp's 32 probes coalesce into ~9 sectors. Windows that pass are queued;
//   * drain, dense, 32 candidates per warp instruction: validity against the read boundaries, the forward k-mer re-extracted
//     from the packed words, its reverse complement, the canonical minimum (KmerIterator.cpp:69), and ONE 256-bit load of the
//     key sector the bit hash points at (a warp-uniform loop goes round the bucket for the few that need more, then the sorted
//     overflow region by bisection);
//   * hits are staged in position order (in the already consumed part of the transposition buffer); a warp reserves the hit
//     buffer in chunks (one atomic per ~64 tiles) and a copy kernel moves the tile segments into stream order (exclusive scan
//     over the tile counts). CSR row offsets are produced per tile and fixed up with the tile's final offset;
//   * windows that contain a non-ACGT byte skip the filter; the drain rebuilds their reverse strand by the reference's rule and
//     takes minimizer and bit hash from the k-mer value; tiles without such bytes never pay for the check.
#include "hga_internal.cuh"

#include <cub/device/device_scan.cuh>

#define SCAN_WARPS 8                             // 5.1 KB of shared memory per warp: 4 CTAs of 8 warps per SM at 64 registers
#define SCAN_THREADS (SCAN_WARPS * 32)
#define SCAN_LANE 16                             // consecutive window ends a lane owns
#define SCAN_TILE (30 * SCAN_LANE)               // window-end positions per warp tile (30 lanes; lanes 0 and 1 hold the 32 bases before it)
#define SCAN_SPAN (32 * SCAN_LANE)               // staged bases per tile: 32 of halo + the tile
#define SCAN_UNROLL 4
#define SCAN_Q 256                               // candidate ring (power of two, >= 31 + 32 * SCAN_UNROLL)
#define SCAN_BND 32                              // read boundaries of a tile staged in shared memory (more: global search)
#define SCAN_TR_STRIDE (SCAN_LANE + 1)            // row stride of the transposition buffer in entries (odd: conflict free)
#define SCAN_CHUNK 2048                          // hit-buffer entries a warp reserves per atomic (a tile holds ~32 hits at config 4); 256 when the scan runs as many launches
#define SCAN_TICKETS 4                           // consecutive tiles per ticket

struct ScanScalars {
    unsigned long long ticket;
    unsigned long long total;        // hits appended so far (= all hits when the kernel ends)
    unsigned long long alloc;        // hit-buffer entries handed out to warps (chunks of SCAN_CHUNK; >= total)
    unsigned long long candidates;   // windows that passed the filter (diagnostic: filter false positives = candidates - hits)
    unsigned int overflow;
    unsigned int pad;
};

namespace {

struct ScanParams {
    const char *frame;                // bases - lead: 16 B aligned
    uint32_t lead;                    // bytes between the aligned frame and the first base
    uint64_t n_bases;
    const uint64_t *read_off;
    uint64_t n_reads;
    KmerTable t;
    uint32_t *out_slot, *out_pos;     // temporary hit arrays (tile segments in completion order)
    uint64_t capacity;
    uint64_t *row_off;
    const uint2 *tile_dir;            // per tile: x = first read starting at/after the tile start, y = read holding the tile start
    unsigned long long *tile_tmp_off; // where the tile's segment starts in the temporary arrays
    uint32_t *tile_cnt;               // hits of the tile
    ScanScalars *scalars;
    uint64_t n_tiles;                 // tickets of this launch
    uint64_t tile_begin;              // first tile of this launch (chunked launches while the bases are still arriving)
    uint64_t tile_stride;             // > 0: sampling mode (count only, tile = tile_begin + ticket * stride)
    uint32_t chunk;                   // hit-buffer entries a warp reserves per atomic
    unsigned long long *warp_chunks;  // chunked launches: every warp's open chunk [pos, end) survives from one launch to the next (nullptr: one launch)
    // packed input (hga_scan_packed*): frame is then 4 B aligned and lead counts bases (0..15)
    const uint64_t *exc_start, *exc_end;  // exception runs, half-open stream positions, sorted and disjoint
    uint64_t n_exc;
    const unsigned long long *exc_dir;    // per tile: the first run that touches its staged span, ~0 = none (nullptr: no runs, never read)
};

// shared memory of one warp
struct WarpTile {
    uint2 tr[SCAN_TR_STRIDE * 32];   // phase B -> C: x = locality hash, y = bit hash; afterwards: staged hits (x = slot, y = window index)
    uint32_t pk[SCAN_SPAN / 16 + 4]; // packed forward codes, 16 bases per word, first base most significant
    uint32_t exc[SCAN_SPAN / 32 + 2];// bit p: staged base p is not one of ACGT (written as u16 halves, one per lane)
    uint16_t q[SCAN_Q];              // candidate windows: staged index | 0x8000 when the window holds a non-ACGT byte
    int32_t bnd[SCAN_BND];           // staged index of the first base of reads r_lo, r_lo + 1, ... (n_bnd of them)
    unsigned long long chunk[2];     // the warp's open chunk of the hit buffer: [pos, end) (lane 0 only; kept out of the registers)
    unsigned long long tk[2];        // the warp's current batch of tile tickets: [next, end)
};

// entry of staged window index i in the transposition buffer
__device__ __forceinline__ int tr_index(int i) { return SCAN_TR_STRIDE * (i / SCAN_LANE) + (i % SCAN_LANE); }

// 4 ASCII bytes (little-endian in w, lowest address = first base) -> forward codes (8 bits, first base most significant) and
// complement codes (8 bits, first base LEAST significant). Codes follow KmerIterator.cpp:7-19 (A0 C1 G2 T3 / complement A3 C2 G1
// T0). diff accumulates w ^ (the byte each code stands for): non-zero exactly when a byte is not one of ACGT (its code bits are
// then garbage; the caller's rare path clears them in both streams).
__device__ __forceinline__ void pack4(uint32_t w, uint32_t &fwd8, uint32_t &rc8, uint32_t &diff) {
    uint32_t x = (w >> 1) & 0x03030303u;          // A0 C1 G3 T2
    x ^= (x >> 1) & 0x01010101u;                  // A0 C1 G2 T3
    const uint32_t sel = __byte_perm(x | (x >> 4), 0u, 0x4420u);      // the four codes as selector nibbles
    diff |= w ^ __byte_perm(0x54474341u, 0u, sel);                    // "ACGT"[code]
    fwd8 = (x * 0x40100401u) >> 24;               // b0<<6 | b1<<4 | b2<<2 | b3
    rc8 = ((x ^ 0x03030303u) * 0x01041040u) >> 24;// c0 | c1<<2 | c2<<4 | c3<<6
}

// last r in [lo, hi] with read_off[r] <= pos (read_off[lo] <= pos is guaranteed by the caller)
__device__ __forceinline__ uint64_t find_read(const uint64_t *__restrict__ read_off, uint64_t lo, uint64_t hi, uint64_t pos) {
    while (lo < hi) {
        uint64_t mid = (lo + hi + 1) >> 1;
        if (__ldg(&read_off[mid]) <= pos) lo = mid; else hi = mid - 1;
    }
    return lo;
}

__device__ __forceinline__ int clamp_local(uint64_t glob, int64_t gbase) {
    const int64_t d = (int64_t) glob - gbase;
    return (int) max((int64_t) -(1 << 30), min((int64_t) (1 << 30), d));
}

// L2 eviction policies: the filter is the one structure every window touches (keep it: evict_last); key sectors are touched
// once per candidate and must not push it out (evict_first); the base stream does not allocate in L1 and leaves L2 first.
__device__ __forceinline__ uint64_t l2_policy_evict_last() {
    uint64_t pol;
    asm("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol));
    return pol;
}
__device__ __forceinline__ uint64_t l2_policy_evict_first() {
    uint64_t pol;
    asm("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
    return pol;
}
__device__ __forceinline__ uint32_t ldg_u32_policy(const uint32_t *a, uint64_t pol) {
    uint32_t v;
    asm("ld.global.nc.L2::cache_hint.u32 %0, [%1], %2;" : "=r"(v) : "l"(a), "l"(pol));
    return v;
}

// one 32 B sector of the key table: one 256-bit load (LDG.E.256), evict-first in L2. Measured (r3i - r3k, ncu, config 4): L1TEX asks for ONE sector
// per probe, but the L2 turns a missing sector into a 64 - 128 B DRAM fetch: 2.5 sectors per probe arrive (4 without the evict-first hint);
// two 128-bit loads, L1::no_allocate and cudaLimitMaxL2FetchGranularity = 32 change nothing. 1.0 G probes x 2.5 x 32 B = the 78 GB that the
// kernel reads from DRAM beyond the 10 GB of bases.
__device__ __forceinline__ void load_sector(const uint64_t *sp, uint64_t pol, unsigned long long &a, unsigned long long &b, unsigned long long &d, unsigned long long &e) {
    asm volatile("ld.global.nc.L2::cache_hint.v4.u64 {%0, %1, %2, %3}, [%4], %5;" : "=l"(a), "=l"(b), "=l"(d), "=l"(e) : "l"(sp), "l"(pol));
}

struct TileCtx {
    const ScanParams *p;
    WarpTile *T;
    int64_t gbase;                   // stream position of staged index 0 (may be negative in the first tile)
    uint64_t r_lo, r_hi;
    uint32_t n_bnd;                  // 0: too many reads in this tile, search read_off in global memory
    int i_end;                       // staged indices >= i_end lie past the end of the stream
};

// staged index of the first base of the read that holds staged base i
__device__ __forceinline__ int read_start_of(const TileCtx &c, int i) {
    if (c.n_bnd) {
        uint32_t lo = 0, hi = c.n_bnd - 1;
        while (lo < hi) { const uint32_t mid = (lo + hi + 1) >> 1; if (c.T->bnd[mid] <= i) lo = mid; else hi = mid - 1; }
        return c.T->bnd[lo];
    }
    const int64_t g = c.gbase + i;
    if (g < 0) return 1 << 30;
    const uint64_t r = find_read(c.p->read_off, c.r_lo, c.r_hi, (uint64_t) g);
    return clamp_local(__ldg(&c.p->read_off[r]), c.gbase);
}

// the 2 x 32 bits of forward codes ending at staged index i (i >= 32): lo = the last 16 bases, hi = the 16 before
__device__ __forceinline__ void extract_window(const uint32_t *pk, int i, uint32_t &lo, uint32_t &hi) {
    const int q = (i - 15) >> 4, sh = ((i + 1) & 15) * 2;
    const uint32_t w0 = pk[q - 1], w1 = pk[q], w2 = pk[q + 1];
    lo = __funnelshift_l(w2, w1, sh);
    hi = __funnelshift_l(w1, w0, sh);
}

// bit b of x -> bits 2b, 2b + 1 (32 -> 64 bits)
__device__ __forceinline__ unsigned long long spread_pairs(uint32_t x) {
    unsigned long long v = x;
    v = (v | (v << 16)) & 0x0000FFFF0000FFFFull;
    v = (v | (v << 8)) & 0x00FF00FF00FF00FFull;
    v = (v | (v << 4)) & 0x0F0F0F0F0F0F0F0Full;
    v = (v | (v << 2)) & 0x3333333333333333ull;
    v = (v | (v << 1)) & 0x5555555555555555ull;
    return v * 3ull;
}

// non-ACGT flags of the k bases ending at staged index i, bit 31 = base i (i >= 32)
__device__ __forceinline__ uint32_t window_exc(const uint32_t *exc, int i, int k) {
    const uint32_t y = __funnelshift_l(exc[(i >> 5) - 1], exc[i >> 5], 31 - (i & 31));
    return k == 32 ? y : (y >> (32 - k)) << (32 - k);
}

#define SCAN_NONE 0xFFFFFFFFu

// one probe step of a lookup: sector `sec` of the bucket at base_slot. Returns true when the lookup is over (slot = the key's slot
// or SCAN_NONE), false when the sector is full of other keys.
__device__ __forceinline__ bool probe_sector(const uint64_t *keys, uint32_t base_slot, uint32_t sec, unsigned long long key, uint64_t pol, uint32_t &slot) {
    const uint32_t s0 = base_slot + (sec & (HGA_BUCKET_SLOTS / HGA_SECTOR_SLOTS - 1)) * HGA_SECTOR_SLOTS;
    unsigned long long a, b, d, e;
    load_sector(keys + s0, pol, a, b, d, e);
    slot = SCAN_NONE;
    if (a == key) slot = s0;
    if (b == key) slot = s0 + 1;
    if (d == key) slot = s0 + 2;
    if (e == key) slot = s0 + 3;
    return slot != SCAN_NONE || a == HGA_EMPTY_KEY || b == HGA_EMPTY_KEY || d == HGA_EMPTY_KEY || e == HGA_EMPTY_KEY;
}

struct QueueState { uint32_t head, tail, st_count; };     // warp uniform

// n (<= 32) queued candidates starting at ring position head: check the window against the read boundaries, rebuild the canonical
// k-mer, probe the key table; hits are appended to the staging area in position order
__device__ __forceinline__ void drain_queue(QueueState &qs, uint32_t n, int lane, const TileCtx &c) {
    const ScanParams &p = *c.p;
    const KmerTable &t = p.t;
    WarpTile &T = *c.T;
    const int k = t.geom.k;
    uint32_t slot = SCAN_NONE, widx = 0, base_slot = 0, sec = 0;
    unsigned long long key = 0;
    bool open = false;
    if ((uint32_t) lane < n) {
        const uint32_t qe = T.q[(qs.head + lane) & (SCAN_Q - 1)];
        widx = qe & 0x7FFFu;
        const int i = (int) widx;
        uint2 en = T.tr[tr_index(i)];     // x = locality hash, y = bit hash (still there: hits are staged below index i - 32)
        const int start = read_start_of(c, i);
        if (i < c.i_end && i - start + 1 >= k) {
            uint32_t lo, hi;
            extract_window(T.pk, i, lo, hi);
            const unsigned long long kmask = k == 32 ? ~0ull : ((1ull << (2 * k)) - 1);
            const unsigned long long F = ((((unsigned long long) hi) << 32) | lo) & kmask;
            unsigned long long Ft = F;                              // the reverse strand reads a non-ACGT byte as code 0 too, i.e. as a T here
            if (qe & 0x8000u) Ft |= spread_pairs(__brev(window_exc(T.exc, i, k)));
            const unsigned long long R = hga_revcomp64(Ft, k);
            key = F < R ? F : R;                                    // KmerIterator.cpp:69
            if (qe & 0x8000u) {                                     // the two strands are not reverse complements: hashes from the VALUE
                en.y = hga_bits_hash(key, t.geom);
                en.x = hga_locality_from_min(hga_minimizer(key, en.y, t.geom));
            }
            base_slot = hga_scale(en.x, t.n_buckets) * HGA_BUCKET_SLOTS;
            sec = hga_start_sector(en.y);
            open = true;
        }
    }
    __syncwarp();
    // go round the bucket, one sector per step, all lanes together: 95 % of the lookups end in the first step
    const uint64_t pol_first = l2_policy_evict_first();
    for (int step = 0; __any_sync(0xFFFFFFFFu, open); step++) {
        if (open) {
            if (probe_sector(t.keys, base_slot, sec + step, key, pol_first, slot)) open = false;
            else if (step == HGA_BUCKET_SLOTS / HGA_SECTOR_SLOTS - 1) {
                open = false;
                if (t.n_over_keys) {      // bucket full: the key, if present, lives in the overflow region (sorted: bisection)
                    uint32_t lo = 0, hi = t.n_over_keys;
                    while (lo < hi) {
                        const uint32_t mid = (lo + hi) >> 1;
                        if (__ldg(t.keys + t.n_main + mid) < key) lo = mid + 1; else hi = mid;
                    }
                    if (lo < t.n_over_keys && __ldg(t.keys + t.n_main + lo) == key) slot = t.n_main + lo;
                }
            }
        }
    }
    const bool hit = slot != SCAN_NONE;
    const uint32_t bal = __ballot_sync(0xFFFFFFFFu, hit);
    if (hit) T.tr[qs.st_count + __popc(bal & ((1u << lane) - 1))] = make_uint2(slot, widx);
    qs.st_count += __popc(bal);
    qs.head += n;
}

// phase B for one lane: P0..P2 / Q0..Q2 = forward / complement codes of the 48 bases ending with the lane's own 16 (P2);
// row = the lane's row of the transposition buffer
template<int W, bool KHI>
__device__ __forceinline__ void phase_b(const uint32_t (&P)[3], const uint32_t (&Q)[3], const KmerGeom &geo, uint2 *row) {
    constexpr int WU = W > 0 ? W - 1 : 0;          // positions before the lane's own that feed its first sliding minima
    uint32_t h[SCAN_LANE + 7], t3[SCAN_LANE + 7];
    const uint32_t cm = geo.cm, mtop = geo.mtop, ca = geo.ca, cb = geo.cb;
    const int k = geo.k;
    const int rsh = KHI ? 64 - 2 * k : 32 - 2 * k; // the reverse strand's pieces are top aligned
    #pragma unroll
    for (int j = -WU; j < SCAN_LANE; j++) {
        const int s0 = j + 17;                     // index (in the 48 bases) of the first of the 16 bases ending at the lane's base j
        const int q = s0 >> 4, off = s0 & 15;
        const uint32_t lo = off ? __funnelshift_l(P[(q + 1) % 3], P[q], 2 * off) : P[q];                 // forward, last 16 bases
        const uint32_t rhi = off ? __funnelshift_r(Q[q], Q[(q + 1) % 3], 2 * off) : Q[q];                // complement of the same, base j on top
        uint32_t mn = 0;
        if (W > 0) {
            h[j + 7] = min(hga_mmer_hash(lo, cm), (rhi & mtop) * HGA_C1 + HGA_C4);
            if (W >= 3 && j >= -WU + 2) t3[j + 7] = __vimin3_u32(h[j + 7], h[j + 6], h[j + 5]);
            if (j >= 0) {
                if (W == 2) mn = min(h[j + 7], h[j + 6]);
                else if (W == 3) mn = t3[j + 7];
                else if (W == 4) mn = min(t3[j + 7], h[j + 4]);
                else if (W == 5) mn = __vimin3_u32(t3[j + 7], h[j + 4], h[j + 3]);
                else if (W == 6) mn = min(t3[j + 7], t3[j + 4]);
                else if (W == 7) mn = __vimin3_u32(t3[j + 7], t3[j + 4], h[j + 1]);
                else mn = __vimin3_u32(t3[j + 7], t3[j + 4], t3[j + 2]);
            }
        }
        if (j >= 0) {
            uint32_t hb;
            if (KHI) {
                const uint32_t hi = off ? __funnelshift_l(P[q], P[(q + 2) % 3], 2 * off) : P[(q + 2) % 3];   // ca discards what lies above the k-mer
                const uint32_t rlo = off ? __funnelshift_r(Q[(q + 2) % 3], Q[q], 2 * off) : Q[(q + 2) % 3];
                const uint32_t Rlo = __funnelshift_r(rlo, rhi, rsh), Rhi = rhi >> rsh;
                hb = (hi * ca + lo) * cb + (Rhi * ca + Rlo) * cb;
            } else {
                hb = lo * cb + (rhi >> rsh) * cb;                                                           // cb discards what lies above the k-mer
            }
            if (W == 0) mn = hga_mix_bits(hb);
            row[j] = make_uint2(hga_locality_from_min(mn), hb);
        }
    }
}

template<bool KHI>
__device__ __forceinline__ void phase_b_dispatch(const uint32_t (&P)[3], const uint32_t (&Q)[3], const KmerGeom &geo, uint2 *row) {
    switch (geo.use_min ? geo.W : 0) {
        case 2: phase_b<2, KHI>(P, Q, geo, row); break;
        case 3: phase_b<3, KHI>(P, Q, geo, row); break;
        case 4: phase_b<4, KHI>(P, Q, geo, row); break;
        case 5: phase_b<5, KHI>(P, Q, geo, row); break;
        case 6: phase_b<6, KHI>(P, Q, geo, row); break;
        case 7: phase_b<7, KHI>(P, Q, geo, row); break;
        case 8: phase_b<8, KHI>(P, Q, geo, row); break;
        default: phase_b<0, KHI>(P, Q, geo, row); break;
    }
}

// phase C + drains: returns the number of staged hits. Step s = the 32 adjacent staged windows 32 s .. 32 s + 31 (two lanes' rows); step 0
// is the halo. One loop, one drain call site (the unrolled code of phases B and C already fills the instruction cache).
template<bool EXC>
__device__ __forceinline__ uint32_t phase_c(const TileCtx &c, int lane, uint32_t &n_cand) {
    const ScanParams &p = *c.p;
    WarpTile &T = *c.T;
    const uint64_t pol_last = l2_policy_evict_last();
    const uint32_t n_blocks = p.t.n_blocks, lane_lt = (1u << lane) - 1;
    const uint32_t *filter = p.t.filter;
    QueueState qs = {0, 0, 0};
    #pragma unroll 1
    for (int s0 = 0; s0 <= SCAN_SPAN / 32; s0 += SCAN_UNROLL) {
        const bool last = s0 >= SCAN_SPAN / 32;                     // one more round that only empties the queue
        if (!last) {
            uint2 en[SCAN_UNROLL];
            uint32_t fw[SCAN_UNROLL];
            #pragma unroll
            for (int u = 0; u < SCAN_UNROLL; u++) {
                en[u] = T.tr[tr_index(32 * (s0 + u) + lane)];       // x = locality hash, y = bit hash
                fw[u] = ldg_u32_policy(filter + (__umulhi(en[u].x, n_blocks) * 8 + hga_bits_word(en[u].y)), pol_last);
            }
            #pragma unroll
            for (int u = 0; u < SCAN_UNROLL; u++) {
                if (u == 0 && s0 == 0) continue;                    // the halo's windows belong to the previous tile
                const int i = 32 * (s0 + u) + lane;
                bool pass = hga_bits_test(fw[u], en[u].y);
                bool exc = false;
                if (EXC) { exc = window_exc(T.exc, i, p.t.geom.k) != 0; pass |= exc; }
                const uint32_t bal = __ballot_sync(0xFFFFFFFFu, pass);
                if (bal) {                                           // warp uniform
                    if (pass) T.q[(qs.tail + __popc(bal & lane_lt)) & (SCAN_Q - 1)] = (uint16_t) ((uint32_t) i | (exc ? 0x8000u : 0u));
                    qs.tail += __popc(bal);
                }
            }
        }
        const uint32_t need = last ? 1u : 32u;
        if (qs.tail - qs.head >= need) {
            __syncwarp();
            do drain_queue(qs, min(32u, qs.tail - qs.head), lane, c); while (qs.tail - qs.head >= need);
            __syncwarp();
        }
    }
    n_cand += qs.tail;
    return qs.st_count;
}

// 32 independent warps per SM (4 CTAs of 8 at 64 registers; 5.2 KB of shared memory per warp). The parameters are __grid_constant__ and
// every helper is inlined so that nothing lives in local memory.
// PACKED: the bases arrive 2-bit packed (4 per byte, first base most significant): a lane loads one 4-byte word = its 16 bases, the
// exception runs of the tile come from the run directory. Phases B and C, the drain and the hit staging are the same code.
template<bool PACKED>
__global__ void __launch_bounds__(SCAN_THREADS, 4) scan_probe_kernel(const __grid_constant__ ScanParams p) {
    extern __shared__ __align__(16) unsigned char s_raw[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    WarpTile &T = reinterpret_cast<WarpTile *>(s_raw)[warp];
    uint32_t n_cand = 0;
    const int kk = p.t.geom.k;

    if (lane < 4) T.pk[SCAN_SPAN / 16 + lane] = 0;
    if (lane < 2) T.exc[SCAN_SPAN / 32 + lane] = 0;
    __syncwarp();

    const uint64_t pol_stream = l2_policy_evict_first();               // the base stream passes through L2 once
    // a ticket = SCAN_TICKETS consecutive tiles (one atomic per batch, the next one requested while this batch is processed); the
    // hit buffer is handed out in chunks of SCAN_CHUNK entries, so a tile's segment costs no atomic round trip of its own (r2r: the
    // two per-tile atomics were 9 % of the stall samples). scan_reorder_kernel closes the gaps the chunks leave.
    unsigned long long next_batch = 0;
    if (lane == 0) {
        const size_t warp_id = (size_t) blockIdx.x * SCAN_WARPS + warp;
        T.chunk[0] = p.warp_chunks ? p.warp_chunks[2 * warp_id] : 0ull;
        T.chunk[1] = p.warp_chunks ? p.warp_chunks[2 * warp_id + 1] : 0ull;
        T.tk[0] = T.tk[1] = 0;
        next_batch = atomicAdd(&p.scalars->ticket, 1ull);
    }
    // lane 0: the next tile ticket of this warp (>= n_tiles: none left)
    auto take_ticket = [&]() -> unsigned long long {
        unsigned long long t = T.tk[0];
        if (t == T.tk[1]) {                                        // batch used up: on to the one requested a batch ago, request the next
            t = next_batch * SCAN_TICKETS;
            if (t < p.n_tiles) next_batch = atomicAdd(&p.scalars->ticket, 1ull);
            T.tk[1] = min((unsigned long long) p.n_tiles, t + SCAN_TICKETS);
        }
        T.tk[0] = t + 1;
        return t;
    };
    unsigned long long cur = 0;
    if (lane == 0) cur = take_ticket();
    for (;;) {
        const unsigned long long ticket = __shfl_sync(0xFFFFFFFFu, cur, 0);
        if (ticket >= p.n_tiles) break;
        if (lane == 0) cur = take_ticket();                            // the tile after this one
        const uint64_t tile = p.tile_begin + (p.tile_stride ? ticket * p.tile_stride : ticket);
        // frame coordinate u = stream position + lead; the tile's window ends are u in [480 tile, 480 tile + 480); staged index 0 is u = 480 tile - 32
        const int64_t ubase = (int64_t) (tile * SCAN_TILE) - 32;
        const int64_t gbase = ubase - (int64_t) p.lead;
        const int64_t u_end = (int64_t) p.lead + (int64_t) p.n_bases;                 // first frame position past the stream

        // ---- phase A: 16 bases per lane, packed to one word per strand -----------------------------------------------
        uint32_t P[3], Q[3], bad = 0;
        if (PACKED) {
            const int64_t u = ubase + SCAN_LANE * lane;
            uint32_t w = 0;                                                            // outside the stream: code 0 (never inside a valid window)
            if (u >= 0 && u < u_end)
                asm volatile("ld.global.L1::no_allocate.L2::cache_hint.u32 %0, [%1], %2;" : "=r"(w) : "l"(p.frame + u / 4), "l"(pol_stream));
            P[2] = __byte_perm(w, 0u, 0x0123u);                                        // byte 0 holds the first 4 bases: to the top
            uint32_t x = __brev(P[2]);                                                 // base j's pair at bits 2j, 2j + 1, its two bits swapped
            x = ((x >> 1) & 0x55555555u) | ((x & 0x55555555u) << 1);
            Q[2] = ~x;                                                                 // complement codes (3 - c), first base least significant
            if (p.exc_dir != nullptr) {
                const unsigned long long r0 = __ldg(&p.exc_dir[tile]);
                if (r0 != ~0ull) {                                                     // rare: the runs that touch the tile, warp uniform
                    const int64_t g0 = gbase + SCAN_LANE * lane, g_end = gbase + SCAN_SPAN;
                    for (uint64_t r = r0; r < p.n_exc; r++) {
                        const int64_t s = (int64_t) __ldg(&p.exc_start[r]);
                        if (s >= g_end) break;
                        const int64_t e = (int64_t) __ldg(&p.exc_end[r]);
                        const int64_t lo = max(s - g0, (int64_t) 0), hi = min(e - g0, (int64_t) SCAN_LANE);
                        if (lo < hi) bad |= (0xFFFFu >> (SCAN_LANE - (int) (hi - lo))) << (int) lo;
                    }
                    uint32_t m = bad;                                                  // bit j -> bits 2j, 2j + 1: clear those codes on both strands
                    m = (m | (m << 8)) & 0x00FF00FFu; m = (m | (m << 4)) & 0x0F0F0F0Fu;
                    m = (m | (m << 2)) & 0x33333333u; m = (m | (m << 1)) & 0x55555555u;
                    m *= 3u;
                    Q[2] &= ~m; P[2] &= ~__brev(m);
                }
            }
        } else {
            const int64_t u = ubase + SCAN_LANE * lane;
            uint32_t v[4];
            if (u >= 0 && u < u_end) {
                asm volatile("ld.global.L1::no_allocate.L2::cache_hint.v4.u32 {%0, %1, %2, %3}, [%4], %5;"
                             : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]) : "l"(p.frame + u), "l"(pol_stream));
            } else {
                #pragma unroll
                for (int i = 0; i < 4; i++) v[i] = 0x41414141u;                        // outside the stream: 'A' (never inside a valid window)
            }
            uint32_t diff = 0, f[4], r[4];
            #pragma unroll
            for (int i = 0; i < 4; i++) pack4(v[i], f[i], r[i], diff);
            P[2] = (f[0] << 24) | (f[1] << 16) | (f[2] << 8) | f[3];
            Q[2] = r[0] | (r[1] << 8) | (r[2] << 16) | (r[3] << 24);
            if (diff) {                                                                // rare: clear the codes of the non-ACGT bytes, note them
                #pragma unroll
                for (int i = 0; i < 4; i++) {
                    uint32_t d = 0, f0, r0;
                    pack4(v[i], f0, r0, d);
                    #pragma unroll
                    for (int b = 0; b < 4; b++) {
                        if ((d >> (8 * b)) & 0xFFu) {
                            const int pos = 4 * i + b;
                            bad |= 1u << pos;
                            P[2] &= ~(3u << (30 - 2 * pos)); Q[2] &= ~(3u << (2 * pos));
                        }
                    }
                }
            }
        }
        T.pk[lane] = P[2];
        reinterpret_cast<uint16_t *>(T.exc)[lane] = (uint16_t) bad;
        P[0] = __shfl_up_sync(0xFFFFFFFFu, P[2], 2); P[1] = __shfl_up_sync(0xFFFFFFFFu, P[2], 1);   // lanes 0 and 1 are the halo: their own windows are never used
        Q[0] = __shfl_up_sync(0xFFFFFFFFu, Q[2], 2); Q[1] = __shfl_up_sync(0xFFFFFFFFu, Q[2], 1);
        const bool exc_any = __any_sync(0xFFFFFFFFu, bad != 0);

        // read boundaries of the tile (reads r_lo .. r_hi start at or before the tile's last base)
        const uint2 d0 = __ldg(&p.tile_dir[tile]), d1 = __ldg(&p.tile_dir[tile + 1]);
        TileCtx ctx;
        ctx.p = &p; ctx.T = &T; ctx.gbase = gbase;
        ctx.i_end = (int) min((int64_t) SCAN_SPAN, u_end - ubase);
        ctx.r_lo = d0.y; ctx.r_hi = min((uint64_t) d1.y, p.n_reads - 1);
        const uint64_t nb = ctx.r_hi - ctx.r_lo + 1;
        ctx.n_bnd = nb <= SCAN_BND ? (uint32_t) nb : 0u;
        if (nb <= SCAN_BND) for (uint32_t i = lane; i < nb; i += 32) T.bnd[i] = clamp_local(__ldg(&p.read_off[ctx.r_lo + i]), gbase);

        // ---- phase B: lane-sequential hashing of the lane's 32 windows -------------------------------------------------
        if (kk > 16) phase_b_dispatch<true>(P, Q, p.t.geom, T.tr + SCAN_TR_STRIDE * lane);
        else phase_b_dispatch<false>(P, Q, p.t.geom, T.tr + SCAN_TR_STRIDE * lane);
        __syncwarp();

        // ---- phase C: lane-parallel filter probes, drains ------------------------------------------------------------
        uint32_t total;
        if (exc_any) total = phase_c<true>(ctx, lane, n_cand);
        else total = phase_c<false>(ctx, lane, n_cand);
        __syncwarp();

        // ---- append the tile's hits (one atomic), tile directory, tile-local CSR row offsets ---------------------
        if (p.tile_stride) {
            if (lane == 0 && total) atomicAdd(&p.scalars->total, (unsigned long long) total);
            continue;
        }
        unsigned long long tile_off = 0;
        if (lane == 0) {
            unsigned long long chunk_pos = T.chunk[0], chunk_end = T.chunk[1];
            if (chunk_end - chunk_pos < total) {                       // new chunk (what is left of the old one stays unused)
                const unsigned long long want = max((unsigned long long) p.chunk, (unsigned long long) total);
                chunk_pos = atomicAdd(&p.scalars->alloc, want);
                chunk_end = chunk_pos + want;
                if (chunk_end > p.capacity) { p.scalars->overflow = 1; chunk_end = chunk_pos; }     // nothing fits any more
                T.chunk[1] = chunk_end;
            }
            tile_off = chunk_pos;
            const bool fits = chunk_end - chunk_pos >= total;
            if (fits) chunk_pos += total; else tile_off = ~0ull;
            T.chunk[0] = chunk_pos;
            if (total) atomicAdd(&p.scalars->total, (unsigned long long) total);                   // no return value: a reduction, nobody waits for it
            p.tile_tmp_off[tile] = tile_off; p.tile_cnt[tile] = total;
        }
        tile_off = __shfl_sync(0xFFFFFFFFu, tile_off, 0);
        // rows starting in this tile: number of tile hits whose window ends before the read's first base
        for (uint64_t rr = (uint64_t) d0.x + lane; rr <= ctx.r_hi; rr += 32) {
            const uint64_t ro = __ldg(&p.read_off[rr]);
            if (ro < p.n_bases && (ro + p.lead) / SCAN_TILE == tile) {
                const uint32_t q = (uint32_t) ((int64_t) ro - gbase);
                uint32_t lo = 0, hi = total;
                while (lo < hi) { const uint32_t mid = (lo + hi) >> 1; if (T.tr[mid].y < q) lo = mid + 1; else hi = mid; }
                p.row_off[rr] = lo;       // tile-local; scan_fix_rows_kernel adds the tile's final offset
            }
        }
        if (tile_off != ~0ull) {
            for (uint32_t i = lane; i < total; i += 32) {
                const uint2 hit = T.tr[i];
                const int e = (int) hit.y;
                __stcs(&p.out_slot[tile_off + i], hit.x);
                __stcs(&p.out_pos[tile_off + i], (uint32_t) (e - read_start_of(ctx, e) + 1));   // KmerIterator::position_in_sequence
            }
        }
        __syncwarp();
    }
    if (lane == 0 && p.warp_chunks) {
        const size_t warp_id = (size_t) blockIdx.x * SCAN_WARPS + warp;
        p.warp_chunks[2 * warp_id] = T.chunk[0]; p.warp_chunks[2 * warp_id + 1] = T.chunk[1];
    }
    if (lane == 0 && n_cand) atomicAdd(&p.scalars->candidates, (unsigned long long) n_cand);
}

// per tile: x = first r in [0, n_reads] with read_off[r] >= tile start, y = last r in [0, n_reads) with read_off[r] <= tile start
// (tile start = stream position of the tile's first window end, 992 t - lead, clamped at 0)
__global__ void scan_tile_dir_kernel(const uint64_t *__restrict__ read_off, uint64_t n_reads, uint64_t n_tiles, uint32_t lead, uint2 *dir) {
    for (uint64_t t = blockIdx.x * (uint64_t) blockDim.x + threadIdx.x; t <= n_tiles; t += (uint64_t) gridDim.x * blockDim.x) {
        const uint64_t pos = t * SCAN_TILE > lead ? t * SCAN_TILE - lead : 0;
        uint64_t lo = 0, hi = n_reads;        // lower bound over read_off[0 .. n_reads]
        while (lo < hi) { const uint64_t mid = (lo + hi) >> 1; if (read_off[mid] < pos) lo = mid + 1; else hi = mid; }
        const uint64_t first = lo;
        // the read holding pos: the one before `first`, unless a read starts exactly at pos (then the LAST read that starts there: empty reads
        // share their offset with their successor)
        if (first < n_reads && read_off[first] == pos) {
            lo = first; hi = n_reads - 1;
            while (lo < hi) { const uint64_t mid = (lo + hi + 1) >> 1; if (read_off[mid] <= pos) lo = mid; else hi = mid - 1; }
        } else {
            lo = first > 0 ? std::min<uint64_t>(first, n_reads) - 1 : 0;
        }
        dir[t] = make_uint2((uint32_t) first, (uint32_t) lo);
    }
}

// packed scans: per tile, the first exception run that touches the tile's staged span (stream positions [480 t - 32 - lead, + 512)), ~0
// when none does, so that a tile without exceptions pays one directory load
__global__ void scan_exc_dir_kernel(const uint64_t *__restrict__ exc_start, const uint64_t *__restrict__ exc_end, uint64_t n_exc, uint64_t n_tiles, uint32_t lead,
                                    unsigned long long *dir) {
    for (uint64_t t = blockIdx.x * (uint64_t) blockDim.x + threadIdx.x; t < n_tiles; t += (uint64_t) gridDim.x * blockDim.x) {
        const int64_t s0 = (int64_t) (t * SCAN_TILE) - 32 - (int64_t) lead;
        uint64_t lo = 0, hi = n_exc;          // first run ending after s0
        while (lo < hi) { const uint64_t mid = (lo + hi) >> 1; if ((int64_t) exc_end[mid] <= s0) lo = mid + 1; else hi = mid; }
        dir[t] = (lo < n_exc && (int64_t) exc_start[lo] < s0 + SCAN_SPAN) ? lo : ~0ull;
    }
}

// input of a device entry. Every read is shorter than 2^30 bases (a tile sees its reads' starts through clamp_local, 31 bits): flag[0] = the
// first read that is not (flag[0] starts at ~0). Packed input: read_off[0] must be 0 and the runs non-empty, sorted, disjoint and inside
// [0, n_bases); a violation sets flag[1]. The last read ends at n_bases.
__global__ void scan_input_check_kernel(const uint64_t *__restrict__ read_off, uint64_t n_reads, const uint64_t *__restrict__ exc_start,
                                        const uint64_t *__restrict__ exc_end, uint64_t n_exc, uint64_t n_bases, bool packed, unsigned long long *flag) {
    if (blockIdx.x == 0 && threadIdx.x == 0 && packed && read_off[0] != 0) flag[1] = 1;
    for (uint64_t i = blockIdx.x * (uint64_t) blockDim.x + threadIdx.x; i < n_reads || i < n_exc; i += (uint64_t) gridDim.x * blockDim.x) {
        if (i < n_reads) {
            const uint64_t a = read_off[i], b = i + 1 < n_reads ? read_off[i + 1] : n_bases;
            if (b > a && b - a >= (1ull << 30)) atomicMin(&flag[0], (unsigned long long) i);
        }
        if (i < n_exc) {
            const uint64_t s = exc_start[i], e = exc_end[i];
            if (s >= e || e > n_bases || (i + 1 < n_exc && exc_start[i + 1] < e)) flag[1] = 1;
        }
    }
}

// tile segments (completion order, with the gaps the chunked allocation leaves) -> stream order. A warp takes 32 consecutive tiles: their
// directory entries arrive in three coalesced loads (one tile per lane) and are handed round with shuffles; the 32 destinations are
// one contiguous range. (One warp per tile with three dependent scalar loads each: 3.1 ms at config 4, r2q.)
// (one array per launch: the slots are needed by the very next stage, the positions only by hga_get_hits, which moves them on demand)
__global__ void scan_reorder_kernel(const uint32_t *__restrict__ tmp, const unsigned long long *__restrict__ tile_tmp_off, const uint32_t *__restrict__ tile_cnt,
                                    const unsigned long long *__restrict__ tile_off, uint64_t n_tiles, uint32_t *out) {
    const uint64_t warps = ((uint64_t) gridDim.x * blockDim.x) >> 5;
    const uint64_t w = (blockIdx.x * (uint64_t) blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    for (uint64_t t0 = w * 32; t0 < n_tiles; t0 += warps * 32) {
        const uint64_t t = t0 + lane;
        unsigned long long src = 0, dst = 0;
        uint32_t n = 0;
        if (t < n_tiles) { src = tile_tmp_off[t]; dst = tile_off[t]; n = tile_cnt[t]; }
        #pragma unroll 4
        for (int j = 0; j < 32; j++) {
            const unsigned long long s = __shfl_sync(0xFFFFFFFFu, src, j), d = __shfl_sync(0xFFFFFFFFu, dst, j);
            const uint32_t m = __shfl_sync(0xFFFFFFFFu, n, j);
            for (uint32_t i = lane; i < m; i += 32) __stcs(&out[d + i], __ldcs(&tmp[s + i]));
        }
    }
}

// row_off[r] (tile-local count) += final offset of the tile holding the read's first base; rows at or past the end
// of the stream (trailing empty reads, terminal entry) get E
__global__ void scan_fix_rows_kernel(const uint64_t *__restrict__ read_off, uint64_t n_reads, uint64_t n_bases, uint32_t lead,
                                     const unsigned long long *__restrict__ tile_off, uint64_t n_tiles, uint64_t *row_off) {
    const unsigned long long E = tile_off[n_tiles];
    uint64_t i = blockIdx.x * (uint64_t) blockDim.x + threadIdx.x;
    const uint64_t stride = (uint64_t) gridDim.x * blockDim.x;
    for (; i <= n_reads; i += stride) {
        const uint64_t ro = (i == n_reads) ? n_bases : read_off[i];
        row_off[i] = (ro >= n_bases) ? E : row_off[i] + tile_off[(ro + lead) / SCAN_TILE];
    }
}

// what a scan reads back at its synchronisation: the scalars and, for a device entry, the flags of scan_input_check_kernel
struct ScanReadback {
    ScanScalars sc;
    unsigned long long bad_read;     // first read of 2^30 bases or more, ~0 = none
    unsigned long long bad_runs;     // packed: read_off[0] != 0 or a bad exception run
};

typedef void (*scan_kernel_t)(const ScanParams);
scan_kernel_t scan_kernel(bool packed) { return packed ? scan_probe_kernel<true> : scan_probe_kernel<false>; }
constexpr size_t SCAN_SMEM_BYTES = SCAN_WARPS * sizeof(WarpTile);

int launch_scan(hga_handle *h, const ScanParams &p, int grid, bool packed) {
    scan_kernel(packed)<<<grid, SCAN_THREADS, SCAN_SMEM_BYTES, h->stream>>>(p);
    HGA_CUDA(cudaGetLastError());
    h->metrics.kernel_launches++;
    return HGA_OK;
}

}  // namespace

int hga_scan_run(hga_handle *h, const char *d_bases, const uint64_t *d_read_off, uint64_t n_reads, uint64_t n_bases, const char *h_bases,
                 const ScanPackedInput *packed, const char *check) {
    h->have_scan = h->have_index = h->have_pairs = h->have_selection = h->have_components = h->have_enrichment = false;
    h->n_reads = n_reads; h->n_bases = n_bases; h->n_hits = 0;
    if (n_reads >= (1ull << 32) - 1) { hga_set_error("hga_scan: more than 2^32-2 reads per GPU"); return HGA_E_ARG; }
    HGA_TRY(h->d_row_off.ensure((n_reads + 1) * 8));
    // the scalars, then the two words of the input check (read back with them), then the warps' open chunks (chunked launches)
    HGA_TRY(h->d_scan_scalars.ensure(sizeof(ScanReadback) + (size_t) h->sm_count * 8 * SCAN_WARPS * 16));
    ScanScalars *d_sc = h->d_scan_scalars.as<ScanScalars>();
    unsigned long long *d_check = reinterpret_cast<unsigned long long *>(h->d_scan_scalars.as<char>() + offsetof(ScanReadback, bad_read));
    unsigned long long *d_warp_chunks = reinterpret_cast<unsigned long long *>(h->d_scan_scalars.as<char>() + sizeof(ScanReadback));
    // the kernel loads aligned 16 B pieces (packed: 4 B words): frame = the bases aligned down; lead = bases between frame and the first base
    const bool pk = packed != nullptr;
    const uint32_t frame_bytes = (uint32_t) (reinterpret_cast<uintptr_t>(d_bases) & (pk ? 3 : 15));
    const uint32_t lead = pk ? 4 * frame_bytes + packed->sub : frame_bytes;
    const uint64_t per_byte = pk ? 4 : 1;                                          // bases per byte
    const uint64_t src_bytes = n_bases == 0 ? 0 : pk ? (packed->sub + n_bases + 3) / 4 : n_bases;   // bytes from d_bases / h_bases on
    const uint64_t n_exc = pk ? packed->n_exc : 0;
    const uint64_t n_tiles = (n_reads == 0 || n_bases == 0) ? 0 : (lead + n_bases + SCAN_TILE - 1) / SCAN_TILE;
    HGA_TRY(h->d_tile_state.ensure((n_tiles + 2) * (8 + 8 + 4)));   // tile directory: tmp offset | final offset | count
    unsigned long long *tile_tmp_off = h->d_tile_state.as<unsigned long long>();
    unsigned long long *tile_off = tile_tmp_off + (n_tiles + 2);
    uint32_t *tile_cnt = reinterpret_cast<uint32_t *>(tile_off + (n_tiles + 2));
    HGA_TRY(h->d_tile_dir.ensure((n_tiles + 2) * sizeof(uint2)));

    ScanParams p;
    memset(&p, 0, sizeof(p));
    p.frame = d_bases - frame_bytes; p.lead = lead; p.n_bases = n_bases; p.read_off = d_read_off; p.n_reads = n_reads;
    p.t = h->table;
    p.row_off = h->d_row_off.as<uint64_t>();
    p.tile_dir = h->d_tile_dir.as<uint2>();
    p.tile_tmp_off = tile_tmp_off; p.tile_cnt = tile_cnt;
    p.scalars = d_sc;
    unsigned long long *exc_dir = nullptr;
    if (n_exc) {                                                                   // run directory: n_tiles entries
        HGA_TRY(h->d_exc_dir.ensure((n_tiles + 1) * 8));
        exc_dir = h->d_exc_dir.as<unsigned long long>();
        p.exc_start = packed->d_exc_start; p.exc_end = packed->d_exc_end; p.n_exc = n_exc; p.exc_dir = exc_dir;
    }

    int occ = 0;
    HGA_CUDA(cudaFuncSetAttribute(scan_kernel(pk), cudaFuncAttributeMaxDynamicSharedMemorySize, (int) SCAN_SMEM_BYTES));
    HGA_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, scan_kernel(pk), SCAN_THREADS, SCAN_SMEM_BYTES));
    if (occ < 1) occ = 1;
    const int grid_full = (int) std::min<uint64_t>((uint64_t) h->sm_count * occ, std::max<uint64_t>((n_tiles + SCAN_WARPS - 1) / SCAN_WARPS, 1));

    auto launch_scan_pk = [&](const ScanParams &lp, int grid) { return launch_scan(h, lp, grid, pk); };
    StageTimer timer(h, &h->metrics.scan_ms);
    ScanReadback rb;
    memset(&rb, 0, sizeof(rb));
    ScanScalars &sc = rb.sc;
    uint64_t capacity = 0, E = 0;
    h->metrics.scan_retries = 0;
    // Hit-buffer sizes. Warps reserve chunks, so the buffer holds gaps: what is left of a chunk when the next tile does not fit (less
    // than one tile's hits, <= SCAN_TILE) and every warp's last chunk. `expected` sizes the first attempt from an estimate of the hit
    // count (an overflow is detected and the scan reruns), `certain` is the bound that cannot overflow for an exact count.
    const uint64_t warps_full = (uint64_t) grid_full * SCAN_WARPS;
    auto expected = [&](double hits, double margin, uint64_t launches, uint32_t chunk) {
        return (uint64_t) (hits * (margin + 0.05)) + launches * warps_full * chunk + (1ull << 20);
    };
    auto certain = [&](uint64_t hits, uint64_t launches, uint32_t chunk) {
        return hits + hits * SCAN_TILE / (chunk - SCAN_TILE + 1) + launches * warps_full * chunk + 1024;
    };
    // Host source (hga_scan): the bases travel in chunks on a second stream and every chunk is scanned as soon as it has
    // landed (a tile only needs bases at or before its own end, so chunk c can run while chunk c + 1 is in flight).
    uint64_t chunk_mb = 256;                                                      // bases per chunk; HGA_SCAN_CHUNK_MB lets the tests reach this path with small inputs
    if (const char *e = getenv("HGA_SCAN_CHUNK_MB")) chunk_mb = std::max(1, atoi(e));
    const uint64_t chunk_tiles = (chunk_mb << 20) / SCAN_TILE;
    const bool pipelined = h_bases != nullptr && n_tiles > 2 * chunk_tiles && h->copy_stream != nullptr;
    // the host entry of a packed scan copies its runs with the bases (pipelined: with the first chunk)
    auto copy_runs = [&](cudaStream_t st) -> int {
        if (!pk || !packed->h_exc_start || !n_exc) return HGA_OK;
        HGA_CUDA(cudaMemcpyAsync(const_cast<uint64_t *>(packed->d_exc_start), packed->h_exc_start, n_exc * 8, cudaMemcpyHostToDevice, st));
        HGA_CUDA(cudaMemcpyAsync(const_cast<uint64_t *>(packed->d_exc_end), packed->h_exc_end, n_exc * 8, cudaMemcpyHostToDevice, st));
        return HGA_OK;
    };
    auto launch_exc_dir = [&]() -> int {
        if (check) {                                                               // device entry: its flags come back with the scalars of the scan
            HGA_CUDA(cudaMemsetAsync(d_check, 0xFF, 8, h->stream));
            HGA_CUDA(cudaMemsetAsync(d_check + 1, 0, 8, h->stream));
            scan_input_check_kernel<<<(int) std::min<uint64_t>((std::max(n_reads, n_exc) + 256) / 256, (uint64_t) h->sm_count * 8), 256, 0, h->stream>>>(
                d_read_off, n_reads, p.exc_start, p.exc_end, n_exc, n_bases, pk, d_check);
            h->metrics.kernel_launches++;
        }
        if (n_exc && n_tiles > 0) {
            scan_exc_dir_kernel<<<(int) std::min<uint64_t>((n_tiles + 255) / 256, (uint64_t) h->sm_count * 8), 256, 0, h->stream>>>(p.exc_start, p.exc_end, n_exc, n_tiles, lead,
                                                                                                                                    exc_dir);
            h->metrics.kernel_launches++;
        }
        HGA_CUDA(cudaGetLastError());
        return HGA_OK;
    };
    if (h_bases != nullptr && !pipelined && n_bases) {
        StageTimer t(h, &h->metrics.h2d_ms, true);
        HGA_CUDA(cudaMemcpyAsync(const_cast<char *>(d_bases), h_bases, src_bytes, cudaMemcpyHostToDevice, h->stream));
        HGA_TRY(copy_runs(h->stream));
        t.stop();
    }
    if (n_tiles > 0) {
        scan_tile_dir_kernel<<<(int) std::min<uint64_t>((n_tiles + 256) / 256, (uint64_t) h->sm_count * 8), 256, 0, h->stream>>>(d_read_off, n_reads, n_tiles, lead,
                                                                                                                               h->d_tile_dir.as<uint2>());
        h->metrics.kernel_launches++;
        HGA_CUDA(cudaGetLastError());
    }
    if (!pipelined) HGA_TRY(launch_exc_dir());
    bool done = false;
    if (pipelined) {
        const uint64_t n_chunks = (n_tiles + chunk_tiles - 1) / chunk_tiles;
        std::vector<cudaEvent_t> landed(n_chunks, nullptr);
        // chunk c = the bytes of tiles [c * chunk_tiles, (c + 1) * chunk_tiles): a tile reads no base past its own end (the host entries' device buffers
        // start aligned, so frame and d_bases coincide)
        auto chunk_bytes = [&](uint64_t c, uint64_t &lo, uint64_t &hi) {
            lo = c * chunk_tiles * SCAN_TILE / per_byte; hi = std::min<uint64_t>(src_bytes, (c + 1) * chunk_tiles * SCAN_TILE / per_byte);
        };
        cudaEvent_t ev_begin = nullptr, ev_end = nullptr;
        HGA_CUDA(cudaEventCreate(&ev_begin)); HGA_CUDA(cudaEventCreate(&ev_end));
        HGA_CUDA(cudaEventRecord(ev_begin, h->stream));
        HGA_CUDA(cudaStreamWaitEvent(h->copy_stream, ev_begin, 0));               // the destination buffer was (re)allocated on h->stream
        for (uint64_t c = 0; c < n_chunks; c++) {
            uint64_t lo, hi;
            chunk_bytes(c, lo, hi);
            HGA_CUDA(cudaMemcpyAsync(const_cast<char *>(d_bases) + lo, h_bases + lo, hi - lo, cudaMemcpyHostToDevice, h->copy_stream));
            if (c == 0) HGA_TRY(copy_runs(h->copy_stream));
            HGA_CUDA(cudaEventCreateWithFlags(&landed[c], cudaEventDisableTiming));
            HGA_CUDA(cudaEventRecord(landed[c], h->copy_stream));
        }
        HGA_CUDA(cudaEventRecord(ev_end, h->copy_stream));
        // capacity from a count-only sample of the first chunk (1 tile in 16)
        HGA_CUDA(cudaStreamWaitEvent(h->stream, landed[0], 0));
        HGA_TRY(launch_exc_dir());
        {
            const uint64_t stride = 16, n_sample = (chunk_tiles + stride - 1) / stride;
            HGA_CUDA(cudaMemsetAsync(d_sc, 0, sizeof(ScanScalars), h->stream));
            ScanParams ps = p;
            ps.tile_stride = stride; ps.n_tiles = n_sample; ps.tile_begin = 0; ps.capacity = 0;
            HGA_TRY(launch_scan_pk(ps, (int) std::min<uint64_t>((uint64_t) h->sm_count * occ, (n_sample + SCAN_WARPS - 1) / SCAN_WARPS)));
            HGA_CUDA(cudaMemcpyAsync(&sc, d_sc, sizeof(sc), cudaMemcpyDeviceToHost, h->stream));
            HGA_CUDA(cudaStreamSynchronize(h->stream));
            const double est = (double) sc.total * (double) n_tiles / (double) n_sample;
            capacity = std::min<uint64_t>(certain(n_bases, 1, SCAN_CHUNK), expected(est, 1.15, 1, SCAN_CHUNK));
        }
        HGA_TRY(h->d_sort_a.ensure((capacity + 1) * 4));
        HGA_TRY(h->d_pos_tmp.ensure((capacity + 1) * 4));
        p.out_slot = h->d_sort_a.as<uint32_t>(); p.out_pos = h->d_pos_tmp.as<uint32_t>();
        p.capacity = capacity; p.tile_stride = 0; p.chunk = SCAN_CHUNK;
        p.warp_chunks = d_warp_chunks;
        HGA_CUDA(cudaMemsetAsync(d_sc, 0, sizeof(ScanScalars), h->stream));
        HGA_CUDA(cudaMemsetAsync(d_warp_chunks, 0, warps_full * 16, h->stream));
        for (uint64_t c = 0; c < n_chunks; c++) {
            HGA_CUDA(cudaStreamWaitEvent(h->stream, landed[c], 0));
            p.tile_begin = c * chunk_tiles; p.n_tiles = std::min<uint64_t>(chunk_tiles, n_tiles - p.tile_begin);
            HGA_CUDA(cudaMemsetAsync(&d_sc->ticket, 0, 8, h->stream));
            HGA_TRY(launch_scan_pk(p, (int) std::min<uint64_t>((uint64_t) h->sm_count * occ, (p.n_tiles + SCAN_WARPS - 1) / SCAN_WARPS)));
        }
        HGA_CUDA(cudaMemcpyAsync(&sc, d_sc, sizeof(sc), cudaMemcpyDeviceToHost, h->stream));
        HGA_CUDA(cudaStreamSynchronize(h->stream));
        HGA_CUDA(cudaStreamSynchronize(h->copy_stream));
        float ms = 0.f;
        cudaEventElapsedTime(&ms, ev_begin, ev_end);
        h->metrics.h2d_ms = ms;
        for (cudaEvent_t e : landed) cudaEventDestroy(e);
        cudaEventDestroy(ev_begin); cudaEventDestroy(ev_end);
        E = sc.total;
        p.tile_begin = 0; p.warp_chunks = nullptr;
        if (!sc.overflow) done = true;
        else { capacity = certain(E, 1, SCAN_CHUNK); h->metrics.scan_retries++; }     // the bases are resident now: one plain rerun with the exact count
    } else if (n_tiles > 0) {
        // capacity of the hit arrays: exact upper bound for small inputs, otherwise estimated from a strided
        // count-only sample (1 tile in 64)
        const uint64_t small_limit = 32ull << 20;
        if (n_bases <= small_limit) {
            capacity = certain(n_bases, 1, SCAN_CHUNK);
        } else if (h->scan_density > 0) {
            // this handle has scanned before: size from the hit density it saw (a denser input overflows and reruns with the exact count below)
            capacity = std::min<uint64_t>(certain(n_bases, 1, SCAN_CHUNK), expected((double) n_bases * h->scan_density, 1.25, 1, SCAN_CHUNK));
        } else {
            const uint64_t stride = 64;
            const uint64_t n_sample = (n_tiles + stride - 1) / stride;
            HGA_CUDA(cudaMemsetAsync(d_sc, 0, sizeof(ScanScalars), h->stream));
            ScanParams ps = p;
            ps.tile_stride = stride; ps.n_tiles = n_sample; ps.capacity = 0;
            const int grid_s = (int) std::min<uint64_t>((uint64_t) h->sm_count * occ, (n_sample + SCAN_WARPS - 1) / SCAN_WARPS);
            HGA_TRY(launch_scan_pk(ps, grid_s));
            HGA_CUDA(cudaMemcpyAsync(&sc, d_sc, sizeof(sc), cudaMemcpyDeviceToHost, h->stream));
            HGA_CUDA(cudaStreamSynchronize(h->stream));
            const double est = (double) sc.total * (double) n_tiles / (double) n_sample;
            capacity = std::min<uint64_t>(certain(n_bases, 1, SCAN_CHUNK), expected(est, 1.10, 1, SCAN_CHUNK));
        }
    }

    for (int attempt = 0; attempt < 2 && n_tiles > 0 && !done; attempt++) {
        HGA_TRY(h->d_sort_a.ensure((capacity + 1) * 4));      // temporary slots (reused by the index sort later)
        HGA_TRY(h->d_pos_tmp.ensure((capacity + 1) * 4));     // temporary positions (kept until hga_get_hits asks for them)
        p.out_slot = h->d_sort_a.as<uint32_t>(); p.out_pos = h->d_pos_tmp.as<uint32_t>();
        p.capacity = capacity; p.n_tiles = n_tiles; p.tile_begin = 0; p.tile_stride = 0; p.chunk = SCAN_CHUNK;
        HGA_CUDA(cudaMemsetAsync(d_sc, 0, sizeof(ScanScalars), h->stream));
        HGA_TRY(launch_scan_pk(p, grid_full));
        HGA_CUDA(cudaMemcpyAsync(&rb, d_sc, check ? sizeof(rb) : sizeof(sc), cudaMemcpyDeviceToHost, h->stream));   // with the check's flags
        HGA_CUDA(cudaStreamSynchronize(h->stream));
        E = sc.total;
        if (!sc.overflow) break;
        if (attempt == 1) { hga_set_error("scan: hit buffer overflow after exact resize (internal error)"); return HGA_E_OVERFLOW; }
        capacity = certain(E, 1, SCAN_CHUNK);   // cannot overflow; rerun once
        h->metrics.scan_retries++;
    }

    if (check) {                                                                   // the check ran before the scan; its flags came back with the scalars
        if (n_tiles == 0) {                                                        // no scan ran: read them on their own
            HGA_CUDA(cudaMemcpyAsync(&rb, d_sc, sizeof(rb), cudaMemcpyDeviceToHost, h->stream));
            HGA_CUDA(cudaStreamSynchronize(h->stream));
        }
        if (rb.bad_runs) {
            hga_set_error("%s: read_off[0] must be 0 and the exception runs non-empty, sorted, non-overlapping and inside [0, %llu)", check,
                          (unsigned long long) n_bases);
            return HGA_E_ARG;
        }
        if (rb.bad_read != ~0ull) {
            hga_set_error("%s: read %llu has 2^30 bases or more (reads must be shorter than 2^30 bases)", check, rb.bad_read);
            return HGA_E_ARG;
        }
    }
    HGA_TRY(h->d_hit_slot.ensure((E + 1) * 4));
    if (n_tiles > 0) {
        size_t tmp_bytes = 0;
        HGA_CUDA(cudaMemsetAsync(tile_cnt + n_tiles, 0, 4, h->stream));
        HGA_CUDA(cub::DeviceScan::ExclusiveScan(nullptr, tmp_bytes, tile_cnt, tile_off, cub::Sum(), 0ull, n_tiles + 1, h->stream));   // 64-bit accumulator
        HGA_TRY(h->d_sort_tmp.ensure(tmp_bytes + 16));
        HGA_CUDA(cub::DeviceScan::ExclusiveScan(h->d_sort_tmp.p, tmp_bytes, tile_cnt, tile_off, cub::Sum(), 0ull, n_tiles + 1, h->stream));
        const int blocks = (int) std::max<uint64_t>(1, std::min<uint64_t>((n_tiles + 255) / 256, (uint64_t) h->sm_count * 16));
        scan_reorder_kernel<<<blocks, 256, 0, h->stream>>>(h->d_sort_a.as<uint32_t>(), tile_tmp_off, tile_cnt, tile_off, n_tiles, h->d_hit_slot.as<uint32_t>());
        const int rblocks = (int) std::min<uint64_t>((n_reads + 256) / 256, 2048);
        scan_fix_rows_kernel<<<rblocks, 256, 0, h->stream>>>(d_read_off, n_reads, n_bases, lead, tile_off, n_tiles, p.row_off);
        h->metrics.kernel_launches += 4;
        HGA_CUDA(cudaGetLastError());
    } else {
        HGA_CUDA(cudaMemsetAsync(p.row_off, 0, (n_reads + 1) * 8, h->stream));
    }
    timer.stop();
    h->n_hits = E;
    h->scan_tiles = n_tiles; h->pos_pending = n_tiles > 0;
    if (n_bases) h->scan_density = (double) E / (double) n_bases;
    h->metrics.n_bases = n_bases; h->metrics.n_reads = n_reads; h->metrics.n_hits = E; h->metrics.n_candidates = sc.candidates;
    h->have_scan = true;
    return HGA_OK;
}

// the hit positions, still in tile-completion order after the scan, into stream order (hga_get_hits is their only reader)
int hga_scan_finish_positions(hga_handle *h) {
    if (!h->pos_pending) return HGA_OK;
    const uint64_t n_tiles = h->scan_tiles;
    HGA_TRY(h->d_hit_pos.ensure((h->n_hits + 1) * 4));
    unsigned long long *tile_tmp_off = h->d_tile_state.as<unsigned long long>();
    unsigned long long *tile_off = tile_tmp_off + (n_tiles + 2);
    uint32_t *tile_cnt = reinterpret_cast<uint32_t *>(tile_off + (n_tiles + 2));
    const int blocks = (int) std::max<uint64_t>(1, std::min<uint64_t>((n_tiles + 255) / 256, (uint64_t) h->sm_count * 16));
    scan_reorder_kernel<<<blocks, 256, 0, h->stream>>>(h->d_pos_tmp.as<uint32_t>(), tile_tmp_off, tile_cnt, tile_off, n_tiles, h->d_hit_pos.as<uint32_t>());
    HGA_CUDA(cudaGetLastError());
    h->metrics.kernel_launches++;
    h->pos_pending = false;
    return HGA_OK;
}
