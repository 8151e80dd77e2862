// count: exact canonical k-mer counts of a set of reads (SURVEY.md §8f-4, the GPU half of the SDK selection).
//
// Replaces what occurrences/run_jellyfish.sh asks jellyfish for, per read file (occurrences/JellyfishOccurrenceReader.cpp:16-38):
//   jellyfish bc -C -m k ...; jellyfish count -C -m k --bc ...; jellyfish dump -c; LC_ALL=C sort
// i.e. the canonical k-mers (-C: the smaller of a k-mer and its reverse complement; with A < C < G < T that is the smaller 2-bit
// value, the same canonical form as KmerIterator.cpp:69) that occur at least twice (the two-pass Bloom-counter filter, here without
// its false positives), with their exact counts, in ascending order (string order = value order for equal-length ACGT strings).
// jellyfish itself is not in this image and is not vendored by the reference: the counting is pinned with the reference's own KmerIterator +
// std::map on ACGT-only reads (oracle/_ref/occ_driver count) and checked against exact counting in numpy elsewhere (DESIGN.md §3.10).
// Windows containing a byte other than A C G T a c g t are skipped, as jellyfish does (NOT the code-0 rule of KmerIterator).
//
// Small inputs (at most one budget of windows, 2^29): count_emit_kernel (one thread per window start: binary search of the read, k byte
// loads, canonical value or a sentinel), CUB radix sort + run-length encode, count_flag_kernel + CUB select for count >= min_count.
// Large inputs run in KEY-RANGE passes, so that the scratch is one budget of keys whatever the input size: a strided sample of the
// windows gives the quantiles of the key distribution; pass r emits only the k-mers of range [q_r, q_r+1) (count_emit_range_kernel: the
// same per-window code, matches compacted with one atomic per warp), sorts, run-length encodes, filters and appends its (k-mer, count)
// runs to the host result; ranges ascend, so the result is sorted without a merge and every k-mer is counted in exactly one pass. A
// range that overflows the budget is split at its midpoint and redone. HBM-bound by the sort passes of the emitted keys plus one read
// of the bases per pass.
// Packed input (hga_count_kmers_packed: the case-folded 2-bit codes, exception runs for the bytes outside ACGTacgt): the same two modes
// with count_emit_packed_kernel in place of the two emit kernels. A thread owns a span of consecutive window starts; it searches once for
// its read and once for the first exception run that can touch the span, then rolls the forward and reverse-complement values over the
// span plus k - 1 bases, reading one 32-bit word per 16 bases and stepping over read ends and runs. Every later step (sort, run-length
// encode, filter, quantiles, range splitting) is shared with the ASCII input, so the results are the same values in the same order.
// Spectrum mode (hga_count_spectrum[_packed]): the same emits, passes and sorts; count_spectrum_kernel then adds each pass's runs to a
// device histogram and totals in place of the run-length encode, filter and D2H, so no k-mer leaves the device.
// SDK mode (hga_sdk_count_packed: the read set cut into files): the same sample, key ranges, passes and splits over the whole stream.
// A pass emits file by file, so file f's keys fill one contiguous segment (one pass: the segment of its bases; key-range passes: one
// emit launch per file on its own rebased read_off and runs, the shared cursor snapshotted after each launch). Each segment is sorted,
// run-length encoded and filtered (count >= min_count) on its own; the survivors, tagged (count, file), are sorted by k-mer together
// and sdk_merge_kernel writes one (k-mer, total, max, files) entry per distinct k-mer into a device chunk of exactly that many entries.
// A range split down to one k-mer gets its entry from the per-file cursor snapshots. hga_sdk_specificity (sdk_spec_kernel: dense
// [threshold][total] bins for small totals, a sorted (threshold, total) list for the rest) and hga_sdk_range (count, then an exactly
// sized select) run over the chunks; only the rows and the range come back to the host.
#include "hga_internal.cuh"

#include <algorithm>
#include <cstdio>
#include <cstdlib>

#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_reduce.cuh>
#include <cub/device/device_run_length_encode.cuh>
#include <cub/device/device_scan.cuh>
#include <cub/device/device_select.cuh>

namespace {

constexpr unsigned long long COUNT_SENTINEL = ~0ull;      // no canonical k-mer has this value (the reverse complement of T...T is 0)

__device__ __forceinline__ int count_base_code(unsigned char c) {
    switch (c) {
        case 'A': case 'a': return 0;
        case 'C': case 'c': return 1;
        case 'G': case 'g': return 2;
        case 'T': case 't': return 3;
        default: return -1;
    }
}

// canonical k-mer of the window starting at position p, or COUNT_SENTINEL (window crosses a read end / holds a byte other than ACGTacgt)
__device__ __forceinline__ unsigned long long count_window_key(const char *__restrict__ bases, const uint64_t *__restrict__ read_off, uint64_t n_reads, int k, uint64_t p) {
    // the read that holds position p: the last r with read_off[r] <= p
    uint64_t lo = 0, hi = n_reads;
    while (lo < hi) { const uint64_t mid = (lo + hi + 1) >> 1; if (read_off[mid] <= p) lo = mid; else hi = mid - 1; }
    if (p + (uint64_t) k > read_off[lo + 1]) return COUNT_SENTINEL;
    unsigned long long fwd = 0, rc = 0;
    for (int j = 0; j < k; j++) {
        const int c = count_base_code((unsigned char) bases[p + j]);
        if (c < 0) return COUNT_SENTINEL;
        fwd = (fwd << 2) | (unsigned long long) c;
        rc = (rc >> 2) | ((unsigned long long) (3 - c) << (2 * (k - 1)));
    }
    if (k < 32) fwd &= (1ull << (2 * k)) - 1;
    return fwd < rc ? fwd : rc;
}

__global__ void count_emit_kernel(const char *__restrict__ bases, const uint64_t *__restrict__ read_off, uint64_t n_reads, int k, uint64_t p0, uint64_t p1,
                                  unsigned long long *__restrict__ out) {
    for (uint64_t p = p0 + blockIdx.x * (uint64_t) blockDim.x + threadIdx.x; p < p1; p += (uint64_t) gridDim.x * blockDim.x)
        out[p - p0] = count_window_key(bases, read_off, n_reads, k, p);
}

// Key-range pass: the canonical k-mers in [key_lo, key_hi) of the windows of every span_stride-th span of COUNT_SPAN positions, compacted into out
// (unordered). cursor counts every match, stored or not (capacity overflow is detected from it); one atomic per warp on the device.
#define COUNT_SPAN 8
__global__ void count_emit_range_kernel(const char *__restrict__ bases, const uint64_t *__restrict__ read_off, uint64_t n_reads, int k, uint64_t n_bases,
                                        unsigned long long key_lo, unsigned long long key_hi, uint64_t span_stride, unsigned long long *__restrict__ out,
                                        uint64_t capacity, unsigned long long *cursor) {
    const uint64_t n_spans = (n_bases + COUNT_SPAN - 1) / COUNT_SPAN, n_sel = (n_spans + span_stride - 1) / span_stride;
    const uint64_t threads = (uint64_t) gridDim.x * blockDim.x, rounds = (n_sel + threads - 1) / threads;
    for (uint64_t round = 0; round < rounds; round++) {                      // the same trip count for every thread: the warp stays together
        const uint64_t t = round * threads + blockIdx.x * (uint64_t) blockDim.x + threadIdx.x;
        unsigned long long keys[COUNT_SPAN];
        uint32_t cnt = 0;
        if (t < n_sel) {
            const uint64_t p0 = t * span_stride * COUNT_SPAN;
            #pragma unroll
            for (int j = 0; j < COUNT_SPAN; j++) {
                unsigned long long key = COUNT_SENTINEL;
                if (p0 + j < n_bases) key = count_window_key(bases, read_off, n_reads, k, p0 + j);
                if (key != COUNT_SENTINEL && key >= key_lo && key < key_hi) keys[cnt++] = key;
            }
        }
        unsigned long long at;
#ifdef __CUDA_ARCH__
        const int lane = threadIdx.x & 31;
        uint32_t incl = cnt;
        #pragma unroll
        for (int d = 1; d < 32; d <<= 1) { const uint32_t v = __shfl_up_sync(0xFFFFFFFFu, incl, d); if (lane >= d) incl += v; }
        unsigned long long base = 0;
        if (lane == 31 && incl) base = atomicAdd(cursor, (unsigned long long) incl);
        base = __shfl_sync(0xFFFFFFFFu, base, 31);
        at = base + incl - cnt;
#else
        at = atomicAdd(cursor, (unsigned long long) cnt);
#endif
        for (uint32_t j = 0; j < cnt; j++) if (at + j < capacity) out[at + j] = keys[j];
    }
}

// ---- packed input ----------------------------------------------------------------------------------------------------------------
// Base i of a slice sits at position g = sub + i of the device buffer (which starts at the byte holding the slice's first base): bits
// 30 - 2 * (g & 15) of 32-bit word g >> 4 once its bytes are swapped (the first base of a byte is in its most significant bits).
#define COUNT_PACKED_SPAN 32            // window starts per thread where every window is emitted (one pass, key-range passes)
__device__ __forceinline__ uint32_t count_packed_word(const uint32_t *__restrict__ words, uint64_t w) {
#ifdef __CUDA_ARCH__
    return __byte_perm(__ldg(words + w), 0, 0x0123);
#else
    return __builtin_bswap32(words[w]);
#endif
}

// The rolling state of one thread: push() takes base q and says whether the k bases ending at q form a window to count (all in one
// read, none under an exception run). rend = the end of read r (the read holding q); [xs, xe) = run x, the first run that ends after q.
struct CountRoll {
    const uint32_t *words;
    const uint64_t *read_off, *exc_start, *exc_end;
    uint64_t n_exc, q, g, r, rend, x, xs, xe;
    unsigned long long fwd, rc, mask;
    uint32_t word;
    int k, vlen;

    __device__ __forceinline__ void start(const uint32_t *w, uint32_t sub, const uint64_t *ro, uint64_t n_reads, const uint64_t *es, const uint64_t *ee, uint64_t ne, int kk,
                                          uint64_t p0) {
        words = w; read_off = ro; exc_start = es; exc_end = ee; n_exc = ne; k = kk; vlen = 0; fwd = rc = 0;
        mask = k < 32 ? (1ull << (2 * k)) - 1 : ~0ull;
        uint64_t lo = 0, hi = n_reads;                      // the read that holds p0: the last r with read_off[r] <= p0
        while (lo < hi) { const uint64_t mid = (lo + hi + 1) >> 1; if (read_off[mid] <= p0) lo = mid; else hi = mid - 1; }
        r = lo; rend = read_off[r + 1];
        lo = 0; hi = n_exc;                                 // the first run that ends after p0 (the ends ascend)
        while (lo < hi) { const uint64_t mid = (lo + hi) >> 1; if (exc_end[mid] <= p0) lo = mid + 1; else hi = mid; }
        x = lo;
        xs = x < n_exc ? exc_start[x] : ~0ull; xe = x < n_exc ? exc_end[x] : ~0ull;
        q = p0; g = sub + p0;
        word = count_packed_word(words, g >> 4);
    }
    // q < read_off[n_reads]
    __device__ __forceinline__ bool push() {
        if ((g & 15) == 0) word = count_packed_word(words, g >> 4);
        const uint32_t c = (word >> (30 - 2 * (uint32_t) (g & 15))) & 3u;
        if (q == rend) { do rend = read_off[++r + 1]; while (rend == q); vlen = 0; }       // a new read (empty ones skipped)
        if (q == xe) { x++; xs = x < n_exc ? exc_start[x] : ~0ull; xe = x < n_exc ? exc_end[x] : ~0ull; }   // the next run starts at xe or later
        fwd = ((fwd << 2) | c) & mask;
        rc = (rc >> 2) | ((unsigned long long) (3u - c) << (2 * (k - 1)));
        vlen = q >= xs ? 0 : vlen + 1;
        q++; g++;
        return vlen >= k;
    }
};

// Window starts [p0, p0 + span) of every span_stride-th span (span: a multiple of COUNT_SPAN), in chunks of COUNT_SPAN windows.
// RANGE == false (one pass; span_stride 1): out[p] = the key of window p or COUNT_SENTINEL, the layout of count_emit_kernel.
// RANGE == true: the keys in [key_lo, key_hi), compacted into out as count_emit_range_kernel does (span COUNT_SPAN: the same sample).
template<bool RANGE>
__global__ void count_emit_packed_kernel(const uint32_t *__restrict__ words, uint32_t sub, const uint64_t *__restrict__ read_off, uint64_t n_reads,
                                         const uint64_t *__restrict__ exc_start, const uint64_t *__restrict__ exc_end, uint64_t n_exc, int k, uint64_t n_bases,
                                         uint32_t span, uint64_t span_stride, unsigned long long key_lo, unsigned long long key_hi,
                                         unsigned long long *__restrict__ out, uint64_t capacity, unsigned long long *cursor) {
    const uint64_t n_units = (n_bases + span - 1) / span, n_sel = (n_units + span_stride - 1) / span_stride;
    const uint64_t threads = (uint64_t) gridDim.x * blockDim.x, rounds = (n_sel + threads - 1) / threads;
    for (uint64_t round = 0; round < rounds; round++) {                      // the same trip counts for every thread: the warp stays together
        const uint64_t t = round * threads + blockIdx.x * (uint64_t) blockDim.x + threadIdx.x;
        const bool live = t < n_sel;
        const uint64_t p0 = t * span_stride * span;
        CountRoll roll;
        if (live) {
            roll.start(words, sub, read_off, n_reads, exc_start, exc_end, n_exc, k, p0);
            for (int j = 0; j < k - 1 && roll.q < n_bases; j++) roll.push();      // the first k - 1 bases end no window of the span
        }
        for (uint32_t c0 = 0; c0 < span; c0 += COUNT_SPAN) {
            unsigned long long keys[COUNT_SPAN];
            #pragma unroll
            for (int j = 0; j < COUNT_SPAN; j++) {                             // window p0 + c0 + j ends at base roll.q
                keys[j] = COUNT_SENTINEL;
                if (live && roll.q < n_bases && roll.push()) keys[j] = roll.fwd < roll.rc ? roll.fwd : roll.rc;
            }
            if (!RANGE) {
                if (live) {
                    #pragma unroll
                    for (int j = 0; j < COUNT_SPAN; j++) if (p0 + c0 + j < n_bases) out[p0 + c0 + j] = keys[j];
                }
                continue;
            }
            uint32_t m = 0;
            #pragma unroll
            for (int j = 0; j < COUNT_SPAN; j++) if (keys[j] != COUNT_SENTINEL && keys[j] >= key_lo && keys[j] < key_hi) m |= 1u << j;
            unsigned long long at;
#ifdef __CUDA_ARCH__
            const uint32_t cnt = (uint32_t) __popc(m);
            const int lane = threadIdx.x & 31;
            uint32_t incl = cnt;
            #pragma unroll
            for (int d = 1; d < 32; d <<= 1) { const uint32_t v = __shfl_up_sync(0xFFFFFFFFu, incl, d); if (lane >= d) incl += v; }
            unsigned long long base = 0;
            if (lane == 31 && incl) base = atomicAdd(cursor, (unsigned long long) incl);
            base = __shfl_sync(0xFFFFFFFFu, base, 31);
            at = base + incl - cnt;
#else
            at = atomicAdd(cursor, (unsigned long long) __builtin_popcount(m));
#endif
            #pragma unroll
            for (int j = 0; j < COUNT_SPAN; j++) if ((m >> j) & 1u) { if (at < capacity) out[at] = keys[j]; at++; }
        }
    }
}

__global__ void count_flag_kernel(const unsigned long long *__restrict__ keys, const uint32_t *__restrict__ cnt, uint64_t n, uint32_t min_count, uint8_t *__restrict__ flag) {
    for (uint64_t i = blockIdx.x * (uint64_t) blockDim.x + threadIdx.x; i < n; i += (uint64_t) gridDim.x * blockDim.x)
        flag[i] = keys[i] != COUNT_SENTINEL && cnt[i] >= min_count;
}

// ---- spectrum ----------------------------------------------------------------------------------------------------------------------
#define COUNT_SPECTRUM_CHUNK 16          // sorted positions a thread owns per round
#define COUNT_SPECTRUM_REG_BINS 4        // bins counted in registers (runs of 1..4 for error-rich reads) and reduced per warp
#define COUNT_SPECTRUM_SHARED_BINS 4096  // bins privatised per CTA as u32 in shared memory (16 KB: 8 CTAs of 256 threads per SM)

// the first index >= j whose key is not `key`, given s[j - 1] == key: doubling steps, then bisection (O(log(run length)) loads)
__device__ __forceinline__ uint64_t count_run_end(const unsigned long long *__restrict__ s, uint64_t m, uint64_t j, unsigned long long key) {
    uint64_t lo = j - 1, hi, step = 1;                                       // s[lo] == key
    for (;; step <<= 1) { hi = lo + step; if (hi >= m) { hi = m; break; } if (s[hi] != key) break; lo = hi; }
    while (hi - lo > 1) { const uint64_t mid = lo + (hi - lo) / 2; if (s[mid] == key) lo = mid; else hi = mid; }
    return hi;
}

// The runs of s[0 .. m) (one pass's keys, ascending; the sentinels of one-pass mode sort last and are skipped) added to acc:
// acc[0] distinct keys, acc[1] windows (the sum of the run lengths), acc[2] the longest run, acc[3 + b] for b < n_bins the runs of
// length b + 1 (the last bin: n_bins or more). A thread owns chunks of COUNT_SPECTRUM_CHUNK positions and counts the runs that start in
// them; a run that reaches the end of its chunk finds its end with count_run_end. The counters a thread or a CTA keeps privately stay
// below 2^32: a pass holds at most the keys of one device allocation, far fewer than 2^32 per CTA of the persistent grid.
__global__ void count_spectrum_kernel(const unsigned long long *__restrict__ s, uint64_t m, uint32_t n_bins, unsigned long long *__restrict__ acc) {
    unsigned long long *bins = acc + 3;
    unsigned long long windows = 0, longest = 0;
    uint32_t distinct = 0, reg[COUNT_SPECTRUM_REG_BINS] = {};
#ifdef __CUDA_ARCH__
    __shared__ uint32_t sh[COUNT_SPECTRUM_SHARED_BINS];
    const uint32_t n_sh = n_bins < COUNT_SPECTRUM_SHARED_BINS ? n_bins : COUNT_SPECTRUM_SHARED_BINS;
    for (uint32_t b = threadIdx.x; b < n_sh; b += blockDim.x) sh[b] = 0;
    __syncthreads();
#endif
    auto add = [&](unsigned long long c) {
        distinct++; windows += c; longest = c > longest ? c : longest;
        if (n_bins == 0) return;
        const uint32_t bin = (uint32_t) ((c < n_bins ? c : n_bins) - 1);
        if (bin < COUNT_SPECTRUM_REG_BINS) {
            #pragma unroll
            for (uint32_t r = 0; r < COUNT_SPECTRUM_REG_BINS; r++) reg[r] += bin == r;
        } else {
#ifdef __CUDA_ARCH__
            if (bin < COUNT_SPECTRUM_SHARED_BINS) atomicAdd(&sh[bin], 1u);
            else atomicAdd(&bins[bin], 1ull);
#else
            bins[bin]++;
#endif
        }
    };
    const uint64_t n_chunks = (m + COUNT_SPECTRUM_CHUNK - 1) / COUNT_SPECTRUM_CHUNK;
    for (uint64_t t = blockIdx.x * (uint64_t) blockDim.x + threadIdx.x; t < n_chunks; t += (uint64_t) gridDim.x * blockDim.x) {
        const uint64_t a = t * COUNT_SPECTRUM_CHUNK, e = a + COUNT_SPECTRUM_CHUNK < m ? a + COUNT_SPECTRUM_CHUNK : m;
        uint64_t i = a;
        if (a) { const unsigned long long before = s[a - 1]; while (i < e && s[i] == before) i++; }     // the run of the previous chunk
        while (i < e) {
            const unsigned long long key = s[i];
            if (key == COUNT_SENTINEL) break;
            uint64_t j = i + 1;
            while (j < e && s[j] == key) j++;
            if (j == e) j = count_run_end(s, m, j, key);
            add(j - i);
            i = j;
        }
    }
#ifdef __CUDA_ARCH__
    distinct = __reduce_add_sync(0xFFFFFFFFu, distinct);
    #pragma unroll
    for (int r = 0; r < COUNT_SPECTRUM_REG_BINS; r++) reg[r] = __reduce_add_sync(0xFFFFFFFFu, reg[r]);
    #pragma unroll
    for (int d = 16; d; d >>= 1) {
        windows += __shfl_xor_sync(0xFFFFFFFFu, windows, d);
        const unsigned long long o = __shfl_xor_sync(0xFFFFFFFFu, longest, d);
        longest = o > longest ? o : longest;
    }
    if ((threadIdx.x & 31) == 0 && distinct) {
        atomicAdd(&acc[0], (unsigned long long) distinct); atomicAdd(&acc[1], windows); atomicMax(&acc[2], longest);
        #pragma unroll
        for (uint32_t r = 0; r < COUNT_SPECTRUM_REG_BINS; r++) if (reg[r]) atomicAdd(&sh[r], reg[r]);       // reg[r] != 0: r < n_bins
    }
    __syncthreads();
    for (uint32_t b = threadIdx.x; b < n_sh; b += blockDim.x) if (sh[b]) atomicAdd(&bins[b], (unsigned long long) sh[b]);
#else
    acc[0] += distinct; acc[1] += windows; acc[2] = longest > acc[2] ? longest : acc[2];
    for (uint32_t r = 0; r < COUNT_SPECTRUM_REG_BINS; r++) if (reg[r]) bins[r] += reg[r];
#endif
}

// ---- SDK selection (hga_sdk_*) ---------------------------------------------------------------------------------------------------
// One file's runs of a pass (k-mer, count), n of them: flag[i] = the run is a k-mer (not the sentinel) seen at least min_count times,
// tag[i] = its count in the high 32 bits and the file in the low 32 bits (what the merge needs once the files' runs are mixed).
__global__ void sdk_tag_kernel(const unsigned long long *__restrict__ keys, const uint32_t *__restrict__ cnt, uint64_t n, uint32_t min_count, uint32_t file,
                               uint8_t *__restrict__ flag, unsigned long long *__restrict__ tag) {
    for (uint64_t i = blockIdx.x * (uint64_t) blockDim.x + threadIdx.x; i < n; i += (uint64_t) gridDim.x * blockDim.x) {
        flag[i] = keys[i] != COUNT_SENTINEL && cnt[i] >= min_count;
        tag[i] = ((unsigned long long) cnt[i] << 32) | file;
    }
}

// The merge of one pass: distinct k-mer j = ukey[j] holds the tags [start[j], start[j] + len[j]) of the pass's tags sorted by k-mer, one
// per file that keeps it, so at most n_files of them. Writes (k-mer, total, largest count, files) to entry j (j < capacity) and sets
// *overflow when a total does not fit 32 bits.
__global__ void sdk_merge_kernel(const unsigned long long *__restrict__ ukey, const uint32_t *__restrict__ len, const unsigned long long *__restrict__ start,
                                 const unsigned long long *__restrict__ tag, uint64_t n_uniq, uint64_t n_tag, uint32_t n_files, unsigned long long *__restrict__ out_kmer,
                                 uint32_t *__restrict__ out_total, uint32_t *__restrict__ out_max, uint32_t *__restrict__ out_files, uint64_t capacity,
                                 unsigned long long *__restrict__ overflow) {
    const uint64_t n = n_uniq < capacity ? n_uniq : capacity;
    for (uint64_t j = blockIdx.x * (uint64_t) blockDim.x + threadIdx.x; j < n; j += (uint64_t) gridDim.x * blockDim.x) {
        const uint64_t s = start[j], l = len[j] < n_files ? len[j] : n_files, e = s + l < n_tag ? s + l : n_tag;
        unsigned long long total = 0;
        uint32_t mx = 0, files = 0;
        for (uint64_t i = s; i < e; i++) {
            const uint32_t c = (uint32_t) (tag[i] >> 32);
            total += c; mx = c > mx ? c : mx; files += c > 0;
        }
        if (total > 0xFFFFFFFFull) *overflow = 1;
        out_kmer[j] = ukey[j]; out_total[j] = (uint32_t) total; out_max[j] = mx; out_files[j] = files;
    }
}

// Specificity of n merged k-mers (entries base .. base + n of the table): bin = the first of the n_thr ascending thresholds strictly
// greater than ((double) max / (double) total) * 100. COUNT pass: totals below dense_lim are added to dense[bin * dense_lim + total],
// the others are counted in *cursor, and the smallest entry without a bin goes to *bad. FILL pass: the others are written as
// bin << 32 | total to tail (below capacity).
template<bool FILL>
__global__ void sdk_spec_kernel(const uint32_t *__restrict__ total, const uint32_t *__restrict__ max, uint64_t n, const double *__restrict__ thr, uint32_t n_thr,
                                uint32_t dense_lim, unsigned long long *__restrict__ dense, unsigned long long *__restrict__ tail, uint64_t capacity,
                                unsigned long long *cursor, unsigned long long *bad, uint64_t base) {
    for (uint64_t i = blockIdx.x * (uint64_t) blockDim.x + threadIdx.x; i < n; i += (uint64_t) gridDim.x * blockDim.x) {
        const double v = ((double) max[i] / (double) total[i]) * 100;
        uint32_t lo = 0, hi = n_thr;
        while (lo < hi) { const uint32_t mid = (lo + hi) >> 1; if (thr[mid] > v) hi = mid; else lo = mid + 1; }
        if (lo == n_thr) {
            if (!FILL) {
#ifdef __CUDA_ARCH__
                atomicMin(bad, (unsigned long long) (base + i));
#else
                if (base + i < *bad) *bad = base + i;
#endif
            }
            continue;
        }
        if (total[i] < dense_lim) {
            if (!FILL) atomicAdd(&dense[(uint64_t) lo * dense_lim + total[i]], 1ull);
            continue;
        }
        const unsigned long long at = atomicAdd(cursor, 1ull);
        if (FILL && at < capacity) tail[at] = ((unsigned long long) lo << 32) | total[i];
    }
}

// lower <= total[i] <= upper: flag[i] (when flag is not NULL), and the number of such entries added to *count
__global__ void sdk_range_kernel(const uint32_t *__restrict__ total, uint64_t n, uint32_t lower, uint32_t upper, uint8_t *__restrict__ flag, unsigned long long *count) {
    unsigned long long c = 0;
    for (uint64_t i = blockIdx.x * (uint64_t) blockDim.x + threadIdx.x; i < n; i += (uint64_t) gridDim.x * blockDim.x) {
        const bool in = lower <= total[i] && total[i] <= upper;
        if (flag) flag[i] = in;
        c += in;
    }
    if (c) atomicAdd(count, c);
}

struct Bufs {
    DevBuf bases, off, exc, keys, sorted, run_key, run_len, acc_key2, acc_cnt2, tmp, scalars, flag, spectrum, f_off, f_exc, f_cnt, tag, sel_tag, m_key, m_tag, m_start;
    ~Bufs() {
        for (DevBuf *b : {&bases, &off, &exc, &keys, &sorted, &run_key, &run_len, &acc_key2, &acc_cnt2, &tmp, &scalars, &flag, &spectrum, &f_off, &f_exc, &f_cnt, &tag,
                          &sel_tag, &m_key, &m_tag, &m_start})
            b->release();
    }
};

// the message of a k-mer whose count does not fit the 32-bit counts
void count_too_many(const char *who, int k, unsigned long long kmer, unsigned long long m) {
    char s[33];
    for (int i = 0; i < k; i++) s[i] = "ACGT"[(kmer >> (2 * (k - 1 - i))) & 3];
    s[k] = '\0';
    hga_set_error("%s: k-mer %s occurs %llu times, more than a 32-bit count holds (2^32 - 1); hga_count_spectrum gives its exact count", who, s, m);
}

}  // namespace

// The merged table of hga_sdk_count_packed: chunks in ascending k-mer order, each one device block of exactly its entries (one chunk
// per key-range pass, plus one per range split down to a single k-mer). A chunk is never grown or copied once written.
struct hga_sdk {
    struct Chunk {
        void *p;
        uint64_t n;
        unsigned long long *kmer() const { return (unsigned long long *) p; }
        uint32_t *total() const { return (uint32_t *) (kmer() + n); }
        uint32_t *max() const { return total() + n; }
        uint32_t *files() const { return max() + n; }
    };
    int device = 0;
    uint64_t n = 0;
    std::vector<Chunk> chunks;
    int add(uint64_t n_entries, Chunk *c) {            // a new chunk of n_entries entries, owned by the handle from here on
        void *p = nullptr;
        const cudaError_t e = cudaMalloc(&p, n_entries * 20);
        if (e != cudaSuccess) { hga_set_error("cudaMalloc(%llu) failed: %s", (unsigned long long) n_entries * 20, cudaGetErrorString(e)); cudaGetLastError(); return HGA_E_NOMEM; }
        chunks.push_back({p, n_entries});
        n += n_entries;
        *c = chunks.back();
        return HGA_OK;
    }
};

// the files of hga_sdk_count_packed: file f = reads [first[f], first[f + 1])
struct SdkFiles {
    int n;
    const uint64_t *first;
};

static int count_run(const char *who, int device, int k, const char *bases, const uint8_t *packed, uint64_t first_base, const uint64_t *read_off,
                     uint64_t n_reads, const uint64_t *exc_start, const uint64_t *exc_end, uint64_t n_exc, uint32_t min_count, hga_kmer_counts_t *out,
                     hga_kmer_spectrum_t *spec, uint32_t n_bins, uint64_t *hist, const SdkFiles *files, hga_sdk *sdk);

int hga_count_run(const char *who, int device, int k, const char *bases, const uint8_t *packed, uint64_t first_base, const uint64_t *read_off,
                  uint64_t n_reads, const uint64_t *exc_start, const uint64_t *exc_end, uint64_t n_exc, uint32_t min_count, hga_kmer_counts_t *out,
                  hga_kmer_spectrum_t *spec, uint32_t n_bins, uint64_t *hist) {
    return count_run(who, device, k, bases, packed, first_base, read_off, n_reads, exc_start, exc_end, n_exc, min_count, out, spec, n_bins, hist, nullptr, nullptr);
}

// SDK mode (files != NULL, packed input): every pass's keys are emitted file by file into one contiguous segment per file, each
// segment is counted on its own (sort, run-length encode, count >= min_count), and the files' runs are merged by k-mer on the device
// into a new chunk of sdk; nothing per k-mer comes back to the host.
static int count_run(const char *who, int device, int k, const char *bases, const uint8_t *packed, uint64_t first_base, const uint64_t *read_off,
                     uint64_t n_reads, const uint64_t *exc_start, const uint64_t *exc_end, uint64_t n_exc, uint32_t min_count, hga_kmer_counts_t *out,
                     hga_kmer_spectrum_t *spec, uint32_t n_bins, uint64_t *hist, const SdkFiles *files, hga_sdk *sdk) {
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) { cudaGetLastError(); hga_set_error("%s: no usable CUDA device (this library has no CPU path)", who); return HGA_E_CUDA; }
    HGA_CUDA(cudaSetDevice(device));
    if (n_reads == 0) return HGA_OK;
    const uint64_t base0 = read_off[0], n_bases = read_off[n_reads] - base0;
    if (n_bases == 0) return HGA_OK;
    cudaStream_t st = nullptr;      // legacy default stream: every call below is ordered on it
    Bufs b;
    // only the bytes that hold the read set travel; packed, they start at an aligned buffer, first_base % 4 bases into its first byte
    const uint32_t sub = (uint32_t) (first_base & 3);
    const uint64_t in_bytes = packed ? (sub + n_bases + 3) / 4 : n_bases;
    HGA_TRY(b.bases.ensure(in_bytes + 64));
    HGA_TRY(b.off.ensure((n_reads + 1) * 8));
    HGA_TRY(b.scalars.ensure(64));
    std::vector<uint64_t> off(n_reads + 1);
    for (uint64_t i = 0; i <= n_reads; i++) off[i] = read_off[i] - base0;
    HGA_CUDA(cudaMemcpyAsync(b.bases.p, packed ? (const void *) (packed + first_base / 4) : (const void *) (bases + base0), in_bytes, cudaMemcpyHostToDevice, st));
    HGA_CUDA(cudaMemcpyAsync(b.off.p, off.data(), (n_reads + 1) * 8, cudaMemcpyHostToDevice, st));
    if (packed) {
        HGA_TRY(b.exc.ensure(n_exc * 16 + 16));
        if (n_exc) {
            HGA_CUDA(cudaMemcpyAsync(b.exc.p, exc_start, n_exc * 8, cudaMemcpyHostToDevice, st));
            HGA_CUDA(cudaMemcpyAsync(b.exc.as<uint64_t>() + n_exc, exc_end, n_exc * 8, cudaMemcpyHostToDevice, st));
        }
    }
    const uint32_t *d_words = b.bases.as<uint32_t>();
    const uint64_t *d_off = b.off.as<uint64_t>(), *d_xs = b.exc.as<uint64_t>(), *d_xe = d_xs + n_exc;
    unsigned long long *d_scal = b.scalars.as<unsigned long long>();
    // keys per pass (the scratch is ~6 arrays of this many entries); HGA_COUNT_CHUNK overrides it (tests force the multi-pass path on small inputs with it)
    const char *ch_env = getenv("HGA_COUNT_CHUNK");
    const uint64_t B = ch_env && std::strtoull(ch_env, nullptr, 10) >= 256 ? std::strtoull(ch_env, nullptr, 10) : (1ull << 29);
    // 2k key bits are enough: no canonical k-mer has all of them set (T...T is not canonical), so the sentinels still sort behind
    // every k-mer and stay together
    const int end_bit = 2 * k;
    int sm = 148;
    cudaDeviceGetAttribute(&sm, cudaDevAttrMultiProcessorCount, device);
    auto grid = [&](uint64_t n) { return (int) std::max<uint64_t>(1, std::min<uint64_t>((n + 255) / 256, (uint64_t) sm * 16)); };
    std::vector<uint64_t> res_k;
    std::vector<uint32_t> res_c;
    // spectrum mode: device accumulators of count_spectrum_kernel across the passes. No count exceeds n_bases, so bins past it stay
    // empty and the device keeps min(n_bins, n_bases) of them
    const uint32_t spec_bins = (uint32_t) std::min<uint64_t>(n_bins, n_bases);
    if (spec) {
        HGA_TRY(b.spectrum.ensure((spec_bins + 3ull) * 8));
        HGA_CUDA(cudaMemsetAsync(b.spectrum.p, 0, (spec_bins + 3ull) * 8, st));
    }
    // SDK mode: fb[f] = the first base of file f (relative to the read set); its keys of a one-pass run are keys[fb[f] .. fb[f + 1])
    const uint32_t n_files = files ? (uint32_t) files->n : 0;
    std::vector<uint64_t> fb(n_files + 1);
    if (files) {
        for (uint32_t f = 0; f <= n_files; f++) fb[f] = off[files->first[f]];
        HGA_TRY(b.f_cnt.ensure(n_files * 8ull + 8));
    }

    // SDK mode: the keys of one pass, file f's in keys[seg[f] .. seg[f + 1]) -> the merged entries of the pass as a new chunk of sdk
    auto merge_pass = [&](const std::vector<uint64_t> &seg) -> int {
        const uint64_t m = seg[n_files];
        if (m == 0) return HGA_OK;
        HGA_TRY(b.sorted.ensure(m * 8)); HGA_TRY(b.run_key.ensure(m * 8)); HGA_TRY(b.run_len.ensure(m * 4));
        HGA_TRY(b.flag.ensure(m + 16)); HGA_TRY(b.tag.ensure(m * 8));
        unsigned long long *d_keys = b.keys.as<unsigned long long>(), *d_sorted = b.sorted.as<unsigned long long>(), *d_rk = b.run_key.as<unsigned long long>();
        unsigned long long *d_fcnt = b.f_cnt.as<unsigned long long>(), *d_tag = b.tag.as<unsigned long long>();
        uint32_t *d_rl = b.run_len.as<uint32_t>();
        uint8_t *d_flag = b.flag.as<uint8_t>();
        // each file on its own: its segment sorted and run-length encoded into the same positions of the run arrays (a segment of n keys
        // has at most n runs), the number of runs to d_fcnt[f]
        HGA_CUDA(cudaMemsetAsync(d_fcnt, 0, n_files * 8ull, st));
        for (uint32_t f = 0; f < n_files; f++) {
            const uint64_t s0 = seg[f], n = seg[f + 1] - seg[f];
            if (n == 0) continue;
            size_t t1 = 0, t2 = 0;
            HGA_CUDA(cub::DeviceRadixSort::SortKeys(nullptr, t1, d_keys + s0, d_sorted + s0, n, 0, end_bit, st));
            HGA_CUDA(cub::DeviceRunLengthEncode::Encode(nullptr, t2, d_sorted + s0, d_rk + s0, d_rl + s0, d_fcnt + f, n, st));
            HGA_TRY(b.tmp.ensure(std::max(t1, t2) + 16));
            HGA_CUDA(cub::DeviceRadixSort::SortKeys(b.tmp.p, t1, d_keys + s0, d_sorted + s0, n, 0, end_bit, st));
            HGA_CUDA(cub::DeviceRunLengthEncode::Encode(b.tmp.p, t2, d_sorted + s0, d_rk + s0, d_rl + s0, d_fcnt + f, n, st));
        }
        HGA_CUDA(cudaGetLastError());
        std::vector<unsigned long long> runs(n_files);
        HGA_CUDA(cudaMemcpyAsync(runs.data(), d_fcnt, n_files * 8ull, cudaMemcpyDeviceToHost, st));
        HGA_CUDA(cudaStreamSynchronize(st));
        // the runs that reach min_count, tagged with count and file; the positions past a file's runs stay unflagged
        HGA_CUDA(cudaMemsetAsync(d_flag, 0, m, st));
        for (uint32_t f = 0; f < n_files; f++) {
            const uint64_t r = std::min<uint64_t>(runs[f], seg[f + 1] - seg[f]);
            if (r) sdk_tag_kernel<<<grid(r), 256, 0, st>>>(d_rk + seg[f], d_rl + seg[f], r, min_count, f, d_flag + seg[f], d_tag + seg[f]);
        }
        HGA_CUDA(cudaGetLastError());
        HGA_TRY(b.acc_key2.ensure(m * 8)); HGA_TRY(b.sel_tag.ensure(m * 8));
        unsigned long long *d_sk = b.acc_key2.as<unsigned long long>(), *d_st = b.sel_tag.as<unsigned long long>();
        size_t t1 = 0, t2 = 0;
        HGA_CUDA(cub::DeviceSelect::Flagged(nullptr, t1, d_rk, d_flag, d_sk, d_scal, m, st));
        HGA_CUDA(cub::DeviceSelect::Flagged(nullptr, t2, d_tag, d_flag, d_st, d_scal + 3, m, st));
        HGA_TRY(b.tmp.ensure(std::max(t1, t2) + 16));
        HGA_CUDA(cub::DeviceSelect::Flagged(b.tmp.p, t1, d_rk, d_flag, d_sk, d_scal, m, st));
        HGA_CUDA(cub::DeviceSelect::Flagged(b.tmp.p, t2, d_tag, d_flag, d_st, d_scal + 3, m, st));
        HGA_CUDA(cudaGetLastError());
        unsigned long long ns = 0;
        HGA_CUDA(cudaMemcpyAsync(&ns, d_scal, 8, cudaMemcpyDeviceToHost, st));
        HGA_CUDA(cudaStreamSynchronize(st));
        if (ns == 0) return HGA_OK;
        // the files' runs mixed and sorted by k-mer (a k-mer has one run per file that keeps it), then one entry per distinct k-mer
        HGA_TRY(b.m_key.ensure(ns * 8)); HGA_TRY(b.m_tag.ensure(ns * 8));
        unsigned long long *d_mk = b.m_key.as<unsigned long long>(), *d_mt = b.m_tag.as<unsigned long long>();
        HGA_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, t1, d_sk, d_mk, d_st, d_mt, ns, 0, end_bit, st));
        HGA_CUDA(cub::DeviceRunLengthEncode::Encode(nullptr, t2, d_mk, d_rk, d_rl, d_scal, ns, st));
        HGA_TRY(b.tmp.ensure(std::max(t1, t2) + 16));
        HGA_CUDA(cub::DeviceRadixSort::SortPairs(b.tmp.p, t1, d_sk, d_mk, d_st, d_mt, ns, 0, end_bit, st));
        HGA_CUDA(cub::DeviceRunLengthEncode::Encode(b.tmp.p, t2, d_mk, d_rk, d_rl, d_scal, ns, st));
        HGA_CUDA(cudaGetLastError());
        unsigned long long nu = 0;
        HGA_CUDA(cudaMemcpyAsync(&nu, d_scal, 8, cudaMemcpyDeviceToHost, st));
        HGA_CUDA(cudaStreamSynchronize(st));
        HGA_TRY(b.m_start.ensure(nu * 8));
        unsigned long long *d_ms = b.m_start.as<unsigned long long>();
        HGA_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, t1, d_rl, d_ms, nu, st));
        HGA_TRY(b.tmp.ensure(t1 + 16));
        HGA_CUDA(cub::DeviceScan::ExclusiveSum(b.tmp.p, t1, d_rl, d_ms, nu, st));
        hga_sdk::Chunk c;
        HGA_TRY(sdk->add(nu, &c));
        HGA_CUDA(cudaMemsetAsync(d_scal + 2, 0, 8, st));
        sdk_merge_kernel<<<grid(nu), 256, 0, st>>>(d_rk, d_rl, d_ms, d_mt, nu, ns, n_files, c.kmer(), c.total(), c.max(), c.files(), c.n, d_scal + 2);
        HGA_CUDA(cudaGetLastError());
        unsigned long long overflow = 0;
        HGA_CUDA(cudaMemcpyAsync(&overflow, d_scal + 2, 8, cudaMemcpyDeviceToHost, st));
        HGA_CUDA(cudaStreamSynchronize(st));
        if (overflow) { hga_set_error("%s: total count overflows 32 bits", who); return HGA_E_OVERFLOW; }
        return HGA_OK;
    };

    // m unsorted keys in b.keys -> sorted runs -> (k-mer, count >= min_count, sentinel dropped) appended to the host result, or in
    // spectrum mode the runs added to the device spectrum
    auto finish_pass = [&](uint64_t m) -> int {
        if (m == 0) return HGA_OK;
        if (spec) {
            HGA_TRY(b.sorted.ensure(m * 8));
            unsigned long long *d_keys = b.keys.as<unsigned long long>(), *d_sorted = b.sorted.as<unsigned long long>();
            size_t t1 = 0;
            HGA_CUDA(cub::DeviceRadixSort::SortKeys(nullptr, t1, d_keys, d_sorted, m, 0, end_bit, st));
            HGA_TRY(b.tmp.ensure(t1 + 16));
            HGA_CUDA(cub::DeviceRadixSort::SortKeys(b.tmp.p, t1, d_keys, d_sorted, m, 0, end_bit, st));
            count_spectrum_kernel<<<grid((m + COUNT_SPECTRUM_CHUNK - 1) / COUNT_SPECTRUM_CHUNK), 256, 0, st>>>(d_sorted, m, spec_bins, b.spectrum.as<unsigned long long>());
            HGA_CUDA(cudaGetLastError());
            return HGA_OK;
        }
        HGA_TRY(b.sorted.ensure(m * 8)); HGA_TRY(b.run_key.ensure(m * 8)); HGA_TRY(b.run_len.ensure(m * 4));
        unsigned long long *d_keys = b.keys.as<unsigned long long>(), *d_sorted = b.sorted.as<unsigned long long>(), *d_rk = b.run_key.as<unsigned long long>();
        uint32_t *d_rl = b.run_len.as<uint32_t>();
        size_t t1 = 0, t2 = 0;
        HGA_CUDA(cub::DeviceRadixSort::SortKeys(nullptr, t1, d_keys, d_sorted, m, 0, end_bit, st));
        HGA_CUDA(cub::DeviceRunLengthEncode::Encode(nullptr, t2, d_sorted, d_rk, d_rl, d_scal, m, st));
        HGA_TRY(b.tmp.ensure(std::max(t1, t2) + 16));
        HGA_CUDA(cub::DeviceRadixSort::SortKeys(b.tmp.p, t1, d_keys, d_sorted, m, 0, end_bit, st));
        HGA_CUDA(cub::DeviceRunLengthEncode::Encode(b.tmp.p, t2, d_sorted, d_rk, d_rl, d_scal, m, st));
        HGA_CUDA(cudaGetLastError());
        unsigned long long runs = 0;
        HGA_CUDA(cudaMemcpyAsync(&runs, d_scal, 8, cudaMemcpyDeviceToHost, st));
        HGA_CUDA(cudaStreamSynchronize(st));
        if (runs == 0) return HGA_OK;
        HGA_TRY(b.flag.ensure(runs + 16));
        HGA_TRY(b.acc_key2.ensure(runs * 8)); HGA_TRY(b.acc_cnt2.ensure(runs * 4));
        uint8_t *d_flag = b.flag.as<uint8_t>();
        count_flag_kernel<<<grid(runs), 256, 0, st>>>(d_rk, d_rl, runs, min_count, d_flag);
        HGA_CUDA(cub::DeviceSelect::Flagged(nullptr, t1, d_rk, d_flag, b.acc_key2.as<unsigned long long>(), d_scal, runs, st));
        HGA_CUDA(cub::DeviceSelect::Flagged(nullptr, t2, d_rl, d_flag, b.acc_cnt2.as<uint32_t>(), d_scal, runs, st));
        HGA_TRY(b.tmp.ensure(std::max(t1, t2) + 16));
        HGA_CUDA(cub::DeviceSelect::Flagged(b.tmp.p, t1, d_rk, d_flag, b.acc_key2.as<unsigned long long>(), d_scal, runs, st));
        HGA_CUDA(cub::DeviceSelect::Flagged(b.tmp.p, t2, d_rl, d_flag, b.acc_cnt2.as<uint32_t>(), d_scal, runs, st));
        HGA_CUDA(cudaGetLastError());
        unsigned long long ns = 0;
        HGA_CUDA(cudaMemcpyAsync(&ns, d_scal, 8, cudaMemcpyDeviceToHost, st));
        HGA_CUDA(cudaStreamSynchronize(st));
        if (ns) {
            const size_t at = res_k.size();
            res_k.resize(at + ns); res_c.resize(at + ns);
            HGA_CUDA(cudaMemcpy(res_k.data() + at, b.acc_key2.p, ns * 8, cudaMemcpyDeviceToHost));
            HGA_CUDA(cudaMemcpy(res_c.data() + at, b.acc_cnt2.p, ns * 4, cudaMemcpyDeviceToHost));
        }
        return HGA_OK;
    };

    if (n_bases <= B) {
        // one pass: a key (or the sentinel) per window start
        HGA_TRY(b.keys.ensure(n_bases * 8));
        if (packed)
            count_emit_packed_kernel<false><<<grid((n_bases + COUNT_PACKED_SPAN - 1) / COUNT_PACKED_SPAN), 256, 0, st>>>(d_words, sub, d_off, n_reads, d_xs, d_xe, n_exc, k, n_bases,
                                                                                                                    COUNT_PACKED_SPAN, 1, 0ull, COUNT_SENTINEL, b.keys.as<unsigned long long>(),
                                                                                                                    n_bases, nullptr);
        else
            count_emit_kernel<<<grid(n_bases), 256, 0, st>>>(b.bases.as<char>(), b.off.as<uint64_t>(), n_reads, k, 0, n_bases, b.keys.as<unsigned long long>());
        if (files) HGA_TRY(merge_pass(fb));       // the reads of a file are contiguous, so are the keys (and sentinels) of its windows
        else HGA_TRY(finish_pass(n_bases));
    } else {
        // key-range passes. Quantiles of the key distribution from a strided sample of the windows (about 2^24 of them, all of them when the input is small)
        HGA_TRY(b.keys.ensure(B * 8));
        const uint64_t n_spans = (n_bases + COUNT_SPAN - 1) / COUNT_SPAN;
        const uint64_t sample_stride = std::max<uint64_t>(1, n_bases / std::min<uint64_t>(B, 1ull << 24));
        const uint64_t sample_cap = std::min<uint64_t>(B, (n_spans + sample_stride - 1) / sample_stride * COUNT_SPAN);
        HGA_CUDA(cudaMemsetAsync(d_scal + 1, 0, 8, st));
        if (packed)
            count_emit_packed_kernel<true><<<grid((n_spans + sample_stride - 1) / sample_stride), 256, 0, st>>>(d_words, sub, d_off, n_reads, d_xs, d_xe, n_exc, k, n_bases, COUNT_SPAN,
                                                                                                           sample_stride, 0ull, COUNT_SENTINEL, b.keys.as<unsigned long long>(),
                                                                                                           sample_cap, d_scal + 1);
        else
            count_emit_range_kernel<<<grid((n_spans + sample_stride - 1) / sample_stride), 256, 0, st>>>(b.bases.as<char>(), b.off.as<uint64_t>(), n_reads, k, n_bases, 0ull, COUNT_SENTINEL,
                                                                                                        sample_stride, b.keys.as<unsigned long long>(), sample_cap, d_scal + 1);
        unsigned long long n_sample = 0;
        HGA_CUDA(cudaMemcpyAsync(&n_sample, d_scal + 1, 8, cudaMemcpyDeviceToHost, st));
        HGA_CUDA(cudaStreamSynchronize(st));
        n_sample = std::min<unsigned long long>(n_sample, sample_cap);
        // ranges that are expected to hold ~0.6 B keys each
        const double est_keys = (double) n_sample * (double) sample_stride;
        const uint64_t n_ranges = std::max<uint64_t>(1, (uint64_t) (est_keys / (0.6 * (double) B)) + 1);
        std::vector<unsigned long long> cut(n_ranges + 1, 0ull);
        cut[n_ranges] = COUNT_SENTINEL;                                     // exclusive: no canonical k-mer has this value
        if (n_sample && n_ranges > 1) {
            HGA_TRY(b.sorted.ensure(n_sample * 8));
            size_t t1 = 0;
            HGA_CUDA(cub::DeviceRadixSort::SortKeys(nullptr, t1, b.keys.as<unsigned long long>(), b.sorted.as<unsigned long long>(), n_sample, 0, end_bit, st));
            HGA_TRY(b.tmp.ensure(t1 + 16));
            HGA_CUDA(cub::DeviceRadixSort::SortKeys(b.tmp.p, t1, b.keys.as<unsigned long long>(), b.sorted.as<unsigned long long>(), n_sample, 0, end_bit, st));
            for (uint64_t r = 1; r < n_ranges; r++)
                HGA_CUDA(cudaMemcpy(&cut[r], b.sorted.as<unsigned long long>() + (size_t) ((double) n_sample * (double) r / (double) n_ranges), 8, cudaMemcpyDeviceToHost));
        }
        // the ranges, ascending; one that overflows the budget is split at its midpoint and redone (a single value that overflows IS its own count)
        std::vector<std::pair<unsigned long long, unsigned long long>> todo;
        uint64_t passes = 0, splits = 0;
        for (uint64_t r = n_ranges; r-- > 0;) if (cut[r] < cut[r + 1]) todo.push_back({cut[r], cut[r + 1]});
        // SDK mode: every file as a read set of its own (read_off rebased to its first base, its runs clipped to it and rebased),
        // uploaded once; after file f's emit the cursor is copied to d_snap[f], so file f's keys of a pass are keys[snap[f - 1] .. snap[f])
        std::vector<uint64_t> f_off_at(n_files + 1, 0), f_exc_at(n_files + 1, 0), snap(n_files + 1, 0);
        unsigned long long *d_snap = b.f_cnt.as<unsigned long long>();
        const uint64_t *d_foff = nullptr, *d_fxs = nullptr, *d_fxe = nullptr;
        if (files) {
            std::vector<uint64_t> f_off, f_es, f_ee;
            f_off.reserve(n_reads + n_files);
            for (uint32_t f = 0; f < n_files; f++) {
                f_off_at[f] = f_off.size();
                for (uint64_t i = files->first[f]; i <= files->first[f + 1]; i++) f_off.push_back(off[i] - fb[f]);
                f_exc_at[f] = f_es.size();
                for (uint64_t j = (uint64_t) (std::upper_bound(exc_end, exc_end + n_exc, fb[f]) - exc_end); j < n_exc && exc_start[j] < fb[f + 1]; j++) {
                    f_es.push_back(std::max(exc_start[j], fb[f]) - fb[f]);
                    f_ee.push_back(std::min(exc_end[j], fb[f + 1]) - fb[f]);
                }
            }
            f_off_at[n_files] = f_off.size(); f_exc_at[n_files] = f_es.size();
            HGA_TRY(b.f_off.ensure(f_off.size() * 8 + 8)); HGA_TRY(b.f_exc.ensure(f_es.size() * 16 + 16));
            HGA_CUDA(cudaMemcpy(b.f_off.p, f_off.data(), f_off.size() * 8, cudaMemcpyHostToDevice));
            if (!f_es.empty()) {
                HGA_CUDA(cudaMemcpy(b.f_exc.p, f_es.data(), f_es.size() * 8, cudaMemcpyHostToDevice));
                HGA_CUDA(cudaMemcpy(b.f_exc.as<uint64_t>() + f_es.size(), f_ee.data(), f_ee.size() * 8, cudaMemcpyHostToDevice));
            }
            d_foff = b.f_off.as<uint64_t>(); d_fxs = b.f_exc.as<uint64_t>(); d_fxe = d_fxs + f_es.size();
        }
        while (!todo.empty()) {
            const unsigned long long lo = todo.back().first, hi = todo.back().second;
            todo.pop_back();
            passes++;
            HGA_CUDA(cudaMemsetAsync(d_scal + 1, 0, 8, st));
            if (files) {
                for (uint32_t f = 0; f < n_files; f++) {
                    const uint64_t nb = fb[f + 1] - fb[f], g0 = sub + fb[f];
                    if (nb)
                        count_emit_packed_kernel<true><<<grid((nb + COUNT_PACKED_SPAN - 1) / COUNT_PACKED_SPAN), 256, 0, st>>>(d_words + (g0 >> 4), (uint32_t) (g0 & 15), d_foff + f_off_at[f],
                                                                                                                        files->first[f + 1] - files->first[f], d_fxs + f_exc_at[f],
                                                                                                                        d_fxe + f_exc_at[f], f_exc_at[f + 1] - f_exc_at[f], k, nb,
                                                                                                                        COUNT_PACKED_SPAN, 1, lo, hi, b.keys.as<unsigned long long>(), B,
                                                                                                                        d_scal + 1);
                    HGA_CUDA(cudaMemcpyAsync(d_snap + f, d_scal + 1, 8, cudaMemcpyDeviceToDevice, st));
                }
                HGA_CUDA(cudaGetLastError());
                HGA_CUDA(cudaMemcpyAsync(snap.data() + 1, d_snap, n_files * 8ull, cudaMemcpyDeviceToHost, st));
                HGA_CUDA(cudaStreamSynchronize(st));
                const unsigned long long m = snap[n_files];
                if (m <= B) { HGA_TRY(merge_pass(snap)); continue; }
                if (hi - lo > 1) {
                    splits++;
                    const unsigned long long mid = lo + (hi - lo) / 2;
                    todo.push_back({mid, hi});
                    todo.push_back({lo, mid});
                    continue;
                }
                // one k-mer, seen snap[f + 1] - snap[f] times in file f: its merged entry is built here, a chunk of its own
                unsigned long long total = 0;
                uint32_t mx = 0, nf = 0;
                for (uint32_t f = 0; f < n_files; f++) {
                    const unsigned long long c = snap[f + 1] - snap[f];
                    if (c > 0xFFFFFFFFull) { count_too_many(who, k, lo, c); return HGA_E_OVERFLOW; }
                    if (c == 0 || c < min_count) continue;
                    total += c; mx = std::max<uint32_t>(mx, (uint32_t) c); nf++;
                }
                if (nf == 0) continue;
                if (total > 0xFFFFFFFFull) { hga_set_error("%s: total count overflows 32 bits", who); return HGA_E_OVERFLOW; }
                hga_sdk::Chunk c;
                HGA_TRY(sdk->add(1, &c));
                const unsigned long long key = lo;
                const uint32_t tot = (uint32_t) total;
                HGA_CUDA(cudaMemcpy(c.kmer(), &key, 8, cudaMemcpyHostToDevice));
                HGA_CUDA(cudaMemcpy(c.total(), &tot, 4, cudaMemcpyHostToDevice));
                HGA_CUDA(cudaMemcpy(c.max(), &mx, 4, cudaMemcpyHostToDevice));
                HGA_CUDA(cudaMemcpy(c.files(), &nf, 4, cudaMemcpyHostToDevice));
                continue;
            }
            if (packed)
                count_emit_packed_kernel<true><<<grid((n_bases + COUNT_PACKED_SPAN - 1) / COUNT_PACKED_SPAN), 256, 0, st>>>(d_words, sub, d_off, n_reads, d_xs, d_xe, n_exc, k, n_bases,
                                                                                                                       COUNT_PACKED_SPAN, 1, lo, hi, b.keys.as<unsigned long long>(), B,
                                                                                                                       d_scal + 1);
            else
                count_emit_range_kernel<<<grid(n_spans), 256, 0, st>>>(b.bases.as<char>(), b.off.as<uint64_t>(), n_reads, k, n_bases, lo, hi, 1, b.keys.as<unsigned long long>(), B, d_scal + 1);
            HGA_CUDA(cudaGetLastError());
            unsigned long long m = 0;
            HGA_CUDA(cudaMemcpyAsync(&m, d_scal + 1, 8, cudaMemcpyDeviceToHost, st));
            HGA_CUDA(cudaStreamSynchronize(st));
            if (m > B) {
                if (hi - lo == 1) {                                          // one k-mer, seen m times
                    if (spec) {
                        spec->n_distinct++; spec->n_windows += m; spec->max_count = std::max<uint64_t>(spec->max_count, m);
                        if (n_bins) hist[std::min<uint64_t>(m, n_bins) - 1]++;
                        continue;
                    }
                    if (m > 0xFFFFFFFFull) { count_too_many(who, k, lo, m); return HGA_E_OVERFLOW; }      // the counts are 32-bit: refuse rather than clip
                    if (m >= min_count) { res_k.push_back(lo); res_c.push_back((uint32_t) m); }
                    continue;
                }
                splits++;
                const unsigned long long mid = lo + (hi - lo) / 2;
                todo.push_back({mid, hi});
                todo.push_back({lo, mid});
                continue;
            }
            HGA_TRY(finish_pass(m));
        }
        // HGA_COUNT_STATS=1: how the key range was cut (a split range counts its pass and the passes of its halves)
        if (getenv("HGA_COUNT_STATS")) fprintf(stderr, "%s: %llu key-range passes (%llu ranges split)\n", who, (unsigned long long) passes, (unsigned long long) splits);
    }
    if (spec) {
        std::vector<unsigned long long> h(spec_bins + 3ull);
        HGA_CUDA(cudaMemcpy(h.data(), b.spectrum.p, h.size() * 8, cudaMemcpyDeviceToHost));
        spec->n_distinct += h[0]; spec->n_windows += h[1]; spec->max_count = std::max<uint64_t>(spec->max_count, h[2]);
        for (uint32_t i = 0; i < spec_bins; i++) hist[i] += h[3 + i];
        return HGA_OK;
    }
    if (files) return HGA_OK;
    const uint64_t n_out = res_k.size();
    uint64_t *hk = (uint64_t *) std::malloc((n_out + 1) * 8);
    uint32_t *hc = (uint32_t *) std::malloc((n_out + 1) * 4);
    if (!hk || !hc) { std::free(hk); std::free(hc); hga_set_error("%s: out of host memory", who); return HGA_E_NOMEM; }
    if (n_out) { std::memcpy(hk, res_k.data(), n_out * 8); std::memcpy(hc, res_c.data(), n_out * 4); }
    out->n = n_out; out->kmer = hk; out->count = hc;
    return HGA_OK;
}

extern "C" int hga_count_kmers(int device, int k, const char *bases, const uint64_t *read_off, uint64_t n_reads, uint32_t min_count, hga_kmer_counts_t *out) {
    if (!out) { hga_set_error("hga_count_kmers: NULL argument"); return HGA_E_ARG; }
    out->n = 0; out->kmer = nullptr; out->count = nullptr;
    if (k < 1 || k > 32) { hga_set_error("Kmer size is too big or too small (k = %d)", k); return HGA_E_ARG; }
    if (n_reads && (!bases || !read_off)) { hga_set_error("hga_count_kmers: NULL argument"); return HGA_E_ARG; }
    return hga_count_run("hga_count_kmers", device, k, bases, nullptr, 0, read_off, n_reads, nullptr, nullptr, 0, min_count, out, nullptr, 0, nullptr);
}

extern "C" int hga_count_spectrum(int device, int k, const char *bases, const uint64_t *read_off, uint64_t n_reads, uint32_t n_bins, uint64_t *hist,
                                  hga_kmer_spectrum_t *out) {
    if (out) std::memset(out, 0, sizeof *out);
    if (hist && n_bins) std::memset(hist, 0, (size_t) n_bins * 8);
    if (!out || (n_bins && !hist)) { hga_set_error("hga_count_spectrum: NULL argument"); return HGA_E_ARG; }
    if (k < 1 || k > 32) { hga_set_error("Kmer size is too big or too small (k = %d)", k); return HGA_E_ARG; }
    if (n_reads && (!bases || !read_off)) { hga_set_error("hga_count_spectrum: NULL argument"); return HGA_E_ARG; }
    return hga_count_run("hga_count_spectrum", device, k, bases, nullptr, 0, read_off, n_reads, nullptr, nullptr, 0, 0, nullptr, out, n_bins, hist);
}

extern "C" void hga_free_kmer_counts(hga_kmer_counts_t *c) {
    if (!c) return;
    std::free((void *) c->kmer); std::free((void *) c->count);
    c->kmer = nullptr; c->count = nullptr; c->n = 0;
}

// ---- SDK selection handle -----------------------------------------------------------------------------------------------------------
extern "C" void hga_sdk_free(hga_sdk *s) {
    if (!s) return;
    if (!s->chunks.empty()) cudaSetDevice(s->device);
    for (const hga_sdk::Chunk &c : s->chunks) cudaFree(c.p);
    delete s;
}

// the device half of hga_sdk_count_packed (hga_capi.cu checks the arguments): on failure nothing is left on the device
int hga_sdk_run(const char *who, int device, int k, const uint8_t *packed, uint64_t first_base, const uint64_t *read_off, uint64_t n_reads,
                const uint64_t *exc_start, const uint64_t *exc_end, uint64_t n_exc, int n_files, const uint64_t *file_first, uint32_t min_count, hga_sdk **out) {
    hga_sdk *s = new hga_sdk;
    s->device = device;
    const SdkFiles files{n_files, file_first};
    const int rc = count_run(who, device, k, nullptr, packed, first_base, read_off, n_reads, exc_start, exc_end, n_exc, min_count, nullptr, nullptr, 0, nullptr, &files, s);
    if (rc != HGA_OK) { hga_sdk_free(s); return rc; }
    *out = s;
    return HGA_OK;
}

extern "C" int hga_sdk_size(const hga_sdk *s, uint64_t *n_kmers) {
    if (!s || !n_kmers) { hga_set_error("hga_sdk_size: NULL argument"); return HGA_E_ARG; }
    *n_kmers = s->n;
    return HGA_OK;
}

// Bins of hga_host_sdk_specificity on the device: totals below dense_lim in a dense [bin][total] table, larger totals as a sorted list
// of (bin, total) keys run-length encoded; rows in (threshold, total) order, as the reference's nested std::map gives them.
extern "C" int hga_sdk_specificity(const hga_sdk *s, const double *thresholds, int n_thresholds, double *out_threshold, uint32_t *out_occurrences,
                                   uint64_t *out_unique, uint64_t capacity, uint64_t *out_n) {
    if (!s || !out_n || n_thresholds < 1 || !thresholds) { hga_set_error("hga_sdk_specificity: bad argument"); return HGA_E_ARG; }
    for (int i = 0; i < n_thresholds; i++)
        if (thresholds[i] != thresholds[i]) { hga_set_error("hga_sdk_specificity: threshold %d is NaN", i); return HGA_E_ARG; }
    std::vector<double> thr(thresholds, thresholds + n_thresholds);         // ascending, without repeats: the bins of the table
    std::sort(thr.begin(), thr.end());
    thr.erase(std::unique(thr.begin(), thr.end()), thr.end());
    *out_n = 0;
    if (s->n == 0) return HGA_OK;
    HGA_CUDA(cudaSetDevice(s->device));
    cudaStream_t st = nullptr;
    const uint32_t n_thr = (uint32_t) thr.size(), dense_lim = n_thr <= 64 ? 65536u : 256u;
    int sm = 148;
    cudaDeviceGetAttribute(&sm, cudaDevAttrMultiProcessorCount, s->device);
    auto grid = [&](uint64_t n) { return (int) std::max<uint64_t>(1, std::min<uint64_t>((n + 255) / 256, (uint64_t) sm * 16)); };
    Bufs b;
    HGA_TRY(b.acc_key2.ensure(n_thr * 8ull)); HGA_TRY(b.spectrum.ensure((uint64_t) n_thr * dense_lim * 8)); HGA_TRY(b.scalars.ensure(64));
    const double *d_thr = b.acc_key2.as<double>();
    unsigned long long *d_dense = b.spectrum.as<unsigned long long>(), *d_scal = b.scalars.as<unsigned long long>();
    HGA_CUDA(cudaMemcpy(b.acc_key2.p, thr.data(), n_thr * 8ull, cudaMemcpyHostToDevice));
    HGA_CUDA(cudaMemsetAsync(d_dense, 0, (uint64_t) n_thr * dense_lim * 8, st));
    HGA_CUDA(cudaMemsetAsync(d_scal, 0, 8, st));
    HGA_CUDA(cudaMemsetAsync(d_scal + 1, 0xFF, 8, st));
    uint64_t base = 0;
    for (const hga_sdk::Chunk &c : s->chunks) {
        sdk_spec_kernel<false><<<grid(c.n), 256, 0, st>>>(c.total(), c.max(), c.n, d_thr, n_thr, dense_lim, d_dense, nullptr, 0, d_scal, d_scal + 1, base);
        base += c.n;
    }
    HGA_CUDA(cudaGetLastError());
    unsigned long long h[2] = {0, 0};
    HGA_CUDA(cudaMemcpyAsync(h, d_scal, 16, cudaMemcpyDeviceToHost, st));
    HGA_CUDA(cudaStreamSynchronize(st));
    if (h[1] != ~0ull) {                                                     // the first k-mer without a bin, as the host loop meets it
        uint64_t i = h[1];
        for (const hga_sdk::Chunk &c : s->chunks) {
            if (i >= c.n) { i -= c.n; continue; }
            uint32_t t = 0, m = 0;
            HGA_CUDA(cudaMemcpy(&t, c.total() + i, 4, cudaMemcpyDeviceToHost));
            HGA_CUDA(cudaMemcpy(&m, c.max() + i, 4, cudaMemcpyDeviceToHost));
            const double v = ((double) m / (double) t) * 100;
            hga_set_error("hga_sdk_specificity: no threshold above %.4f (the reference dereferences end() here)", v);
            return HGA_E_ARG;
        }
    }
    // the totals of dense_lim and more: (bin, total) keys, exactly as many as counted, sorted and run-length encoded
    const unsigned long long n_tail = h[0];
    std::vector<unsigned long long> t_key, t_len;
    if (n_tail) {
        HGA_TRY(b.keys.ensure(n_tail * 8)); HGA_TRY(b.sorted.ensure(n_tail * 8)); HGA_TRY(b.run_key.ensure(n_tail * 8)); HGA_TRY(b.run_len.ensure(n_tail * 4));
        unsigned long long *d_keys = b.keys.as<unsigned long long>(), *d_sorted = b.sorted.as<unsigned long long>(), *d_rk = b.run_key.as<unsigned long long>();
        uint32_t *d_rl = b.run_len.as<uint32_t>();
        HGA_CUDA(cudaMemsetAsync(d_scal, 0, 8, st));
        for (const hga_sdk::Chunk &c : s->chunks)
            sdk_spec_kernel<true><<<grid(c.n), 256, 0, st>>>(c.total(), c.max(), c.n, d_thr, n_thr, dense_lim, d_dense, d_keys, n_tail, d_scal, d_scal + 1, 0);
        HGA_CUDA(cudaGetLastError());
        size_t t1 = 0, t2 = 0;
        HGA_CUDA(cub::DeviceRadixSort::SortKeys(nullptr, t1, d_keys, d_sorted, n_tail, 0, 64, st));
        HGA_CUDA(cub::DeviceRunLengthEncode::Encode(nullptr, t2, d_sorted, d_rk, d_rl, d_scal + 2, n_tail, st));
        HGA_TRY(b.tmp.ensure(std::max(t1, t2) + 16));
        HGA_CUDA(cub::DeviceRadixSort::SortKeys(b.tmp.p, t1, d_keys, d_sorted, n_tail, 0, 64, st));
        HGA_CUDA(cub::DeviceRunLengthEncode::Encode(b.tmp.p, t2, d_sorted, d_rk, d_rl, d_scal + 2, n_tail, st));
        HGA_CUDA(cudaGetLastError());
        unsigned long long nr = 0;
        HGA_CUDA(cudaMemcpyAsync(&nr, d_scal + 2, 8, cudaMemcpyDeviceToHost, st));
        HGA_CUDA(cudaStreamSynchronize(st));
        t_key.resize(nr);
        std::vector<uint32_t> l32(nr);
        if (nr) {
            HGA_CUDA(cudaMemcpy(t_key.data(), d_rk, nr * 8, cudaMemcpyDeviceToHost));
            HGA_CUDA(cudaMemcpy(l32.data(), d_rl, nr * 4, cudaMemcpyDeviceToHost));
        }
        t_len.assign(l32.begin(), l32.end());     // a (bin, total) run holds k-mers seen dense_lim times or more: far fewer than 2^32 of them
    }
    std::vector<unsigned long long> dense((uint64_t) n_thr * dense_lim);
    HGA_CUDA(cudaMemcpy(dense.data(), d_dense, dense.size() * 8, cudaMemcpyDeviceToHost));
    uint64_t m = 0, j = 0;
    auto row = [&](double t, uint32_t occ, uint64_t cnt) {
        if (m < capacity && out_threshold && out_occurrences && out_unique) { out_threshold[m] = t; out_occurrences[m] = occ; out_unique[m] = cnt; }
        m++;
    };
    for (uint32_t bin = 0; bin < n_thr; bin++) {
        for (uint32_t t = 0; t < dense_lim; t++)
            if (dense[(uint64_t) bin * dense_lim + t]) row(thr[bin], t, dense[(uint64_t) bin * dense_lim + t]);
        for (; j < t_key.size() && (t_key[j] >> 32) == bin; j++) row(thr[bin], (uint32_t) t_key[j], t_len[j]);
    }
    *out_n = m;                                                              // > capacity: call again with more room
    return HGA_OK;
}

extern "C" int hga_sdk_range(const hga_sdk *s, uint32_t lower, uint32_t upper, hga_sdk_range_t *out) {
    if (!out) { hga_set_error("hga_sdk_range: NULL argument"); return HGA_E_ARG; }
    std::memset(out, 0, sizeof *out);
    if (!s) { hga_set_error("hga_sdk_range: NULL argument"); return HGA_E_ARG; }
    std::vector<unsigned long long> cnt(s->chunks.size() + 1, 0);
    Bufs b;
    cudaStream_t st = nullptr;
    int sm = 148;
    auto grid = [&](uint64_t n) { return (int) std::max<uint64_t>(1, std::min<uint64_t>((n + 255) / 256, (uint64_t) sm * 16)); };
    unsigned long long n_out = 0;
    if (lower <= upper && s->n) {
        HGA_CUDA(cudaSetDevice(s->device));
        cudaDeviceGetAttribute(&sm, cudaDevAttrMultiProcessorCount, s->device);
        // count per chunk, then fill arrays of exactly that size
        HGA_TRY(b.scalars.ensure(cnt.size() * 8 + 8));
        unsigned long long *d_cnt = b.scalars.as<unsigned long long>();
        HGA_CUDA(cudaMemsetAsync(d_cnt, 0, cnt.size() * 8, st));
        uint64_t largest = 0;
        for (size_t i = 0; i < s->chunks.size(); i++) {
            const hga_sdk::Chunk &c = s->chunks[i];
            sdk_range_kernel<<<grid(c.n), 256, 0, st>>>(c.total(), c.n, lower, upper, nullptr, d_cnt + i);
            largest = std::max<uint64_t>(largest, c.n);
        }
        HGA_CUDA(cudaGetLastError());
        HGA_CUDA(cudaMemcpyAsync(cnt.data(), d_cnt, s->chunks.size() * 8, cudaMemcpyDeviceToHost, st));
        HGA_CUDA(cudaStreamSynchronize(st));
        for (size_t i = 0; i < s->chunks.size(); i++) n_out += cnt[i];
        if (n_out) {
            HGA_TRY(b.flag.ensure(largest + 16)); HGA_TRY(b.keys.ensure(n_out * 8)); HGA_TRY(b.run_len.ensure(n_out * 12));
            unsigned long long *d_k = b.keys.as<unsigned long long>();
            uint32_t *d_t = b.run_len.as<uint32_t>(), *d_m = d_t + n_out, *d_f = d_m + n_out;
            uint8_t *d_flag = b.flag.as<uint8_t>();
            unsigned long long *d_ns = d_cnt + s->chunks.size();
            uint64_t at = 0;
            for (size_t i = 0; i < s->chunks.size(); i++) {
                const hga_sdk::Chunk &c = s->chunks[i];
                if (!cnt[i]) continue;
                sdk_range_kernel<<<grid(c.n), 256, 0, st>>>(c.total(), c.n, lower, upper, d_flag, d_ns);
                size_t t1 = 0, t2 = 0;
                HGA_CUDA(cub::DeviceSelect::Flagged(nullptr, t1, c.kmer(), d_flag, d_k + at, d_ns, c.n, st));
                HGA_CUDA(cub::DeviceSelect::Flagged(nullptr, t2, c.total(), d_flag, d_t + at, d_ns, c.n, st));
                HGA_TRY(b.tmp.ensure(std::max(t1, t2) + 16));
                HGA_CUDA(cub::DeviceSelect::Flagged(b.tmp.p, t1, c.kmer(), d_flag, d_k + at, d_ns, c.n, st));
                HGA_CUDA(cub::DeviceSelect::Flagged(b.tmp.p, t2, c.total(), d_flag, d_t + at, d_ns, c.n, st));
                HGA_CUDA(cub::DeviceSelect::Flagged(b.tmp.p, t2, c.max(), d_flag, d_m + at, d_ns, c.n, st));
                HGA_CUDA(cub::DeviceSelect::Flagged(b.tmp.p, t2, c.files(), d_flag, d_f + at, d_ns, c.n, st));
                HGA_CUDA(cudaGetLastError());
                at += cnt[i];
            }
        }
    }
    uint64_t *hk = (uint64_t *) std::malloc((n_out + 1) * 8);
    uint32_t *ht = (uint32_t *) std::malloc((n_out + 1) * 12);
    if (!hk || !ht) { std::free(hk); std::free(ht); hga_set_error("hga_sdk_range: out of host memory"); return HGA_E_NOMEM; }
    if (n_out) {
        cudaError_t e = cudaMemcpy(hk, b.keys.p, n_out * 8, cudaMemcpyDeviceToHost);
        for (int a = 0; a < 3 && e == cudaSuccess; a++) e = cudaMemcpy(ht + a * (n_out + 1), b.run_len.as<uint32_t>() + a * n_out, n_out * 4, cudaMemcpyDeviceToHost);
        if (e != cudaSuccess) { std::free(hk); std::free(ht); hga_set_error("hga_sdk_range: copy to the host failed: %s", cudaGetErrorString(e)); return HGA_E_CUDA; }
    }
    out->n = n_out; out->kmer = hk; out->total = ht; out->max = ht + n_out + 1; out->files = ht + 2 * (n_out + 1);
    return HGA_OK;
}

extern "C" void hga_free_sdk_range(hga_sdk_range_t *r) {
    if (!r) return;
    std::free((void *) r->kmer); std::free((void *) r->total);      // total, max and files share one block
    std::memset(r, 0, sizeof *r);
}
