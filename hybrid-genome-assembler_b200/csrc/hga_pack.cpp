// hga_host_pack_bases[_folded]: ASCII bases -> the 2-bit packed format of hga_scan_packed, or its case-folded form that
// hga_count_kmers_packed takes (host arithmetic, no GPU). The stream is cut into one range per thread at multiples of 4 bases (a thread
// owns whole bytes); every range collects its exception runs, and the runs of neighbouring ranges are joined where one ends at the seam
// and the next starts there.
#include "hga_b200.h"
#include "hga_pack.h"

#include <algorithm>
#include <cstdio>
#include <thread>
#include <vector>

void hga_set_error(const char *fmt, ...);

static int pack_bases(const char *who, bool fold, const char *bases, uint64_t n_bases, uint8_t *packed, uint64_t *exc_start, uint64_t *exc_end,
                      uint64_t exc_capacity, uint64_t *n_exc, int threads) {
    if (!n_exc) { hga_set_error("%s: n_exc is NULL", who); return HGA_E_ARG; }
    *n_exc = 0;
    if (n_bases && (!bases || !packed)) { hga_set_error("%s: NULL buffer", who); return HGA_E_ARG; }
    if (exc_capacity && (!exc_start || !exc_end)) { hga_set_error("%s: NULL run arrays with a non-zero capacity", who); return HGA_E_ARG; }
    int T = threads > 0 ? threads : (n_bases < ((uint64_t) 8 << 20) ? 1 : (int) std::min(16u, std::max(1u, std::thread::hardware_concurrency())));
    const uint64_t n_bytes = (n_bases + 3) / 4;
    T = (int) std::max<uint64_t>(1, std::min<uint64_t>((uint64_t) T, n_bytes));
    const uint64_t per = (n_bytes + T - 1) / T * 4;                         // bases per thread, a multiple of 4
    std::vector<hga_pack::Packer> part;
    part.reserve(T);
    for (int t = 0; t < T; t++) part.emplace_back(packed, std::min(n_bases, per * t), fold);
    auto work = [&](int t) {
        const uint64_t a = std::min(n_bases, per * t), b = std::min(n_bases, per * (t + 1));
        if (a < b) part[t].put(bases + a, b - a);
    };
    if (T == 1) work(0);
    else {
        std::vector<std::thread> pool;
        for (int t = 0; t < T; t++) pool.emplace_back(work, t);
        for (auto &th : pool) th.join();
    }
    hga_pack::Runs all;
    all.start.swap(part[0].runs.start); all.end.swap(part[0].runs.end);
    for (int t = 1; t < T; t++) all.append(part[t].runs);
    *n_exc = all.size();
    if (all.size() > exc_capacity) {
        hga_set_error("%s: %llu exception runs, capacity %llu", who, (unsigned long long) all.size(), (unsigned long long) exc_capacity);
        return HGA_E_ARG;
    }
    std::copy(all.start.begin(), all.start.end(), exc_start);
    std::copy(all.end.begin(), all.end.end(), exc_end);
    return HGA_OK;
}

extern "C" int hga_host_pack_bases(const char *bases, uint64_t n_bases, uint8_t *packed, uint64_t *exc_start, uint64_t *exc_end, uint64_t exc_capacity,
                                   uint64_t *n_exc, int threads) {
    return pack_bases("hga_host_pack_bases", false, bases, n_bases, packed, exc_start, exc_end, exc_capacity, n_exc, threads);
}

extern "C" int hga_host_pack_bases_folded(const char *bases, uint64_t n_bases, uint8_t *packed, uint64_t *exc_start, uint64_t *exc_end, uint64_t exc_capacity,
                                          uint64_t *n_exc, int threads) {
    return pack_bases("hga_host_pack_bases_folded", true, bases, n_bases, packed, exc_start, exc_end, exc_capacity, n_exc, threads);
}
