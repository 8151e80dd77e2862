// Host-side 2-bit packing of ASCII bases (no CUDA): the formats hga_scan_packed and hga_count_kmers_packed take (include/hga_b200.h).
// Header only, shared by hga_host_pack_bases[_folded] (hga_pack.cpp) and the packing loader of the CLIs (cli/hga_host.h).
//   codes  : A0 C1 G2 T3 (KmerIterator.cpp:7-19), four bases per byte, the first base in the most significant bits
//   exceptions: every byte other than uppercase A C G T gets code 0 and is covered by a maximal half-open run [start, end)
//   fold   : (the count's case-folded packing, jellyfish's rule) lowercase a c g t are packed as their bases; only bytes outside
//            A C G T a c g t are exceptions. Clearing bit 5 maps exactly a c g t (and A C G T themselves) onto A C G T.
#pragma once

#include <cstdint>
#include <cstring>
#include <vector>

namespace hga_pack {

// maximal, sorted exception runs; a run that continues one that ends where it starts extends it
struct Runs {
    std::vector<uint64_t> start, end;
    void add(uint64_t s, uint64_t e) {
        if (!end.empty() && end.back() == s) end.back() = e;
        else { start.push_back(s); end.push_back(e); }
    }
    // appends the runs of the next piece of the stream (a run across the seam becomes one)
    void append(const Runs &o) {
        for (size_t i = 0; i < o.start.size(); i++) add(o.start[i], o.end[i]);
    }
    size_t size() const { return start.size(); }
};

constexpr uint64_t FOLD8 = ~0x2020202020202020ull;      // clears bit 5 of 8 bytes at once

// 8 ASCII bytes (little-endian in w): true when all are one of A C G T; then b0 / b1 = the two packed bytes (bases 0-3 / 4-7)
inline bool pack8(uint64_t w, uint8_t &b0, uint8_t &b1) {
    auto zero_bytes = [](uint64_t z) { return ~(((z & 0x7F7F7F7F7F7F7F7Full) + 0x7F7F7F7F7F7F7F7Full) | z) & 0x8080808080808080ull; };
    const uint64_t ok = zero_bytes(w ^ 0x4141414141414141ull) | zero_bytes(w ^ 0x4343434343434343ull) | zero_bytes(w ^ 0x4747474747474747ull) |
                        zero_bytes(w ^ 0x5454545454545454ull);
    if (ok != 0x8080808080808080ull) return false;
    uint64_t x = (w >> 1) & 0x0303030303030303ull;    // A0 C1 G3 T2
    x ^= (x >> 1) & 0x0101010101010101ull;             // A0 C1 G2 T3
    b0 = (uint8_t) (((uint32_t) x * 0x40100401u) >> 24);
    b1 = (uint8_t) (((uint32_t) (x >> 32) * 0x40100401u) >> 24);
    return true;
}

inline int code_of(unsigned char c) {
    switch (c) {
        case 'A': return 0;
        case 'C': return 1;
        case 'G': return 2;
        case 'T': return 3;
        default: return -1;
    }
}

// Packs a stream piece by piece. A packer owns the bytes from base `pos` (a multiple of 4) on: it writes the first base of a byte with
// '=', the others with '|', so the output needs no clearing. fold: the case-folded packing.
struct Packer {
    uint8_t *out;
    uint64_t pos;
    Runs runs;
    bool fold;
    Packer(uint8_t *o, uint64_t first, bool fold_case = false) : out(o), pos(first), fold(fold_case) {}

    void put1(unsigned char c) {
        int v = code_of(fold ? (unsigned char) (c & 0xDF) : c);
        if (v < 0) { runs.add(pos, pos + 1); v = 0; }
        const unsigned sh = 6 - 2 * (unsigned) (pos & 3);
        if ((pos & 3) == 0) out[pos >> 2] = (uint8_t) (v << sh);
        else out[pos >> 2] |= (uint8_t) (v << sh);
        pos++;
    }
    void put(const char *s, uint64_t n) {
        const unsigned char *u = reinterpret_cast<const unsigned char *>(s);
        while (n && (pos & 3)) { put1(*u++); n--; }
        while (n >= 8) {
            uint64_t w;
            memcpy(&w, u, 8);
            if (fold) w &= FOLD8;
            uint8_t b0, b1;
            if (pack8(w, b0, b1)) { out[pos >> 2] = b0; out[(pos >> 2) + 1] = b1; pos += 8; }
            else for (int i = 0; i < 8; i++) put1(u[i]);
            u += 8; n -= 8;
        }
        while (n) { put1(*u++); n--; }
    }
};

}  // namespace hga_pack
