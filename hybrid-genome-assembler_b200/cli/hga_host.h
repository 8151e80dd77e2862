// Host side of the drop-in `categorization` executable: the k-mer file loader and the FASTA/FASTQ record loader,
// with the reference's rules (paths relative to /root/reference/src):
//   load_text_file_kmers   read_clustering.cpp:18-33      one KmerIterator per line, first window only, k = last line
//   KmerIterator tables    common/KmerIterator.cpp:6-21   A0 C1 G2 T3 / complement A3 C2 G1 T0, any other byte 0 in BOTH
//   SequenceRecords        common/SequenceRecordIterator.cpp:73-173   format sniffed per file from its first record,
//                          FASTQ = 4 lines / record, FASTA = 2 lines / record, the record reader runs on across file
//                          boundaries, header = line minus its first character, ReadID = 1, 2, ... over all files,
//                          per-file and aggregate MetaData (the aggregate max_read_length is never updated: prints 0)
// Nothing here touches the GPU; the arithmetic on reads happens behind include/hga_b200.h.
#pragma once

#include <algorithm>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <exception>
#include <fstream>
#include <iterator>
#include <sstream>
#include <stdexcept>
#include <string>
#include <string_view>
#include <thread>
#include <vector>

#include "../csrc/hga_pack.h"

#include <fcntl.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <unistd.h>

namespace hga_host {

inline uint64_t canonical_first_window(const std::string &s, int k) {
    if (k > 32) throw std::invalid_argument("Kmer size is too big");     // KmerIterator.cpp:24-26
    if (k == 0 || (int) s.size() < k) return 0;                          // no window: current_kmer stays 0
    uint64_t fwd = 0, rev = 0;
    for (int i = 0; i < k; i++) {
        uint64_t c = 0, cc = 0;
        switch (s[i]) {
            case 'A': c = 0; cc = 3; break;
            case 'C': c = 1; cc = 2; break;
            case 'G': c = 2; cc = 1; break;
            case 'T': c = 3; cc = 0; break;
            default: c = 0; cc = 0; break;                                // operator[] default-inserts 0 in both tables
        }
        fwd |= c << (2 * (k - 1 - i));
        rev |= cc << (2 * i);
    }
    return std::min(fwd, rev);
}

// A read-only view of one input file (mmap; kept mapped so that export_components can re-emit headers and qualities
// without a second copy in memory).
struct MappedFile {
    const char *data = nullptr;
    size_t size = 0;
    int fd = -1;
    MappedFile() = default;
    MappedFile(const MappedFile &) = delete;
    MappedFile &operator=(const MappedFile &) = delete;
    MappedFile(MappedFile &&o) noexcept : data(o.data), size(o.size), fd(o.fd), owned(o.owned) { o.data = nullptr; o.size = 0; o.fd = -1; o.owned = nullptr; }
    bool open(const std::string &path) {
        fd = ::open(path.c_str(), O_RDONLY);
        if (fd < 0) return false;
        struct stat st;
        if (fstat(fd, &st) != 0) { ::close(fd); fd = -1; return false; }
        size = (size_t) st.st_size;
        if (size) {
            void *p = mmap(nullptr, size, PROT_READ, MAP_PRIVATE | MAP_POPULATE, fd, 0);   // populate: one bulk fault-in instead of one fault per page
            if (p == MAP_FAILED) {                      // not mappable (pipe, special file): read it
                std::ifstream f(path, std::ios::binary);
                std::string *buf = new std::string((std::istreambuf_iterator<char>(f)), std::istreambuf_iterator<char>());
                owned = buf; data = buf->data(); size = buf->size();
            } else {
                data = (const char *) p;
                madvise(p, size, MADV_SEQUENTIAL);
            }
        }
        return true;
    }
    ~MappedFile() {
        if (owned) delete owned;
        else if (data && size) munmap((void *) data, size);
        if (fd >= 0) ::close(fd);
    }
private:
    std::string *owned = nullptr;
};

struct KmerSet {
    std::vector<uint64_t> kmers;   // sorted, unique canonical values
    int k = 0;
};

inline uint64_t canonical_first_window(const char *s, size_t len) {
    const int k = (int) len;
    if (len > 32) throw std::invalid_argument("Kmer size is too big");    // KmerIterator.cpp:24-26
    uint64_t fwd = 0, rev = 0;
    for (int i = 0; i < k; i++) {
        uint64_t c = 0, cc = 0;
        switch (s[i]) {
            case 'A': c = 0; cc = 3; break;
            case 'C': c = 1; cc = 2; break;
            case 'G': c = 2; cc = 1; break;
            case 'T': c = 3; cc = 0; break;
            default: break;                                               // operator[] default-inserts 0 in both tables
        }
        fwd |= c << (2 * (k - 1 - i));
        rev |= cc << (2 * i);
    }
    return std::min(fwd, rev);
}

// read_clustering.cpp:18-33: one KmerIterator per line (k = the length of THAT line), first window only; the k that the run
// uses is the length of the LAST line; duplicates collapse. The file is mapped and cut at line ends into one piece per thread;
// every piece is canonicalised and sorted on its own, then the pieces are merged pairwise.
inline KmerSet load_text_file_kmers(const std::string &path, int threads = 0) {
    KmerSet out;
    MappedFile f;
    if (!f.open(path) || f.size == 0) return out;                         // a missing file yields an empty set, as in the reference
    const char *d = f.data, *e = d + f.size;
    int T = threads > 0 ? threads : (int) std::min(16u, std::max(1u, std::thread::hardware_concurrency()));
    if (f.size < ((size_t) 4 << 20)) T = 1;
    std::vector<const char *> cut(T + 1, e);
    cut[0] = d;
    for (int t = 1; t < T; t++) {
        const char *q = d + f.size / T * t;
        const char *nl = (const char *) memchr(q, '\n', (size_t) (e - q));
        cut[t] = nl ? nl + 1 : e;
    }
    for (int t = 1; t <= T; t++) cut[t] = std::max(cut[t], cut[t - 1]);
    std::vector<std::vector<uint64_t>> part(T);
    std::vector<int> last_k(T, -1);
    std::vector<std::exception_ptr> err(T);
    auto work = [&](int t) {
        try {
            const char *p = cut[t], *pe = cut[t + 1];
            part[t].reserve((size_t) (pe - p) / 16 + 16);
            while (p < pe) {                                              // std::getline: a last line without '\n' counts
                const char *nl = (const char *) memchr(p, '\n', (size_t) (pe - p));
                const size_t len = nl ? (size_t) (nl - p) : (size_t) (pe - p);
                last_k[t] = (int) len;
                part[t].push_back(canonical_first_window(p, len));
                p = nl ? nl + 1 : pe;
            }
            std::sort(part[t].begin(), part[t].end());
        } catch (...) { err[t] = std::current_exception(); }
    };
    if (T == 1) work(0);
    else {
        std::vector<std::thread> pool;
        for (int t = 0; t < T; t++) pool.emplace_back(work, t);
        for (auto &th : pool) th.join();
    }
    for (int t = 0; t < T; t++) if (err[t]) std::rethrow_exception(err[t]);
    for (int t = 0; t < T; t++) if (last_k[t] >= 0) out.k = last_k[t];
    for (int step = 1; step < T; step *= 2) {                             // pairwise merges, each round in parallel
        std::vector<std::thread> pool;
        for (int a = 0; a + step < T; a += 2 * step)
            pool.emplace_back([&, a, step] {
                std::vector<uint64_t> m(part[a].size() + part[a + step].size());
                std::merge(part[a].begin(), part[a].end(), part[a + step].begin(), part[a + step].end(), m.begin());
                part[a].swap(m);
                std::vector<uint64_t>().swap(part[a + step]);
            });
        for (auto &th : pool) th.join();
    }
    out.kmers.swap(part[0]);
    out.kmers.erase(std::unique(out.kmers.begin(), out.kmers.end()), out.kmers.end());
    return out;
}

struct MetaData {
    std::string filename;
    uint64_t records = 0, min_read_length = UINT64_MAX, max_read_length = 0, avg_read_length = 0, total_bases = 0;
    std::string repr() const {                                            // SequenceRecordIterator.h:60-63
        std::ostringstream o;
        o << filename << ":\n- " << records << " reads\n- " << total_bases << " total bases\n- " << avg_read_length << " average read length\n- "
          << max_read_length << " max read length\n- " << min_read_length << " min read length\n\n";
        return o.str();
    }
};

// All records of the input files, loaded in ONE pass over the mapped files (the reference reads every file twice: once for
// load_meta_data, SequenceRecordIterator.cpp:31-71, once for the records). Phase 1 (sequential, memchr) finds the lines and
// applies the record rules; phase 2 writes the sequences into one contiguous buffer with several threads: the ASCII bytes (what
// hga_scan and hga_count_kmers take) or, with `packed`, the 2-bit codes and exception runs of hga_scan_packed, a quarter of the
// bytes, written straight from the mappings; `packed` with `fold_case`: the case-folded packing of hga_count_kmers_packed. The buffer is 2 MB aligned and advised MADV_HUGEPAGE: first-touch page faults, not
// memcpy, are what bounds the copy (measured on 1.2 GB: 1.17 s single thread with 4 KB pages, 0.29 s with huge pages and 8 threads).
// Headers, sequences and qualities stay views into the mappings.
struct SequenceRecords {
    struct View { uint32_t file; uint32_t len; uint64_t off; };
    std::vector<std::string> paths;
    std::vector<MappedFile> files;
    std::vector<MetaData> file_meta;
    MetaData meta;
    char *bases_data = nullptr;          // ASCII mode: sequences back to back
    uint8_t *packed_data = nullptr;      // packed mode: the same stream, 2-bit codes, (bases_size + 3) / 4 bytes
    std::vector<uint64_t> exc_start, exc_end;   // packed mode: maximal runs of bytes other than A C G T (folded: A C G T a c g t), stream positions
    uint64_t bases_size = 0;
    std::vector<uint64_t> seq_off;       // n_reads + 1
    std::vector<View> header_v, quality_v, seq_v;
    std::vector<uint8_t> is_fastq;       // per record: 4-line record (re-emitted with '+' and qualities)
    std::vector<int> file_index;
    bool fastq_last = true;

    size_t n_reads() const { return header_v.size(); }
    std::string_view header(size_t i) const { return {files[header_v[i].file].data + header_v[i].off, header_v[i].len}; }
    std::string_view quality(size_t i) const { return is_fastq[i] ? std::string_view{files[quality_v[i].file].data + quality_v[i].off, quality_v[i].len} : std::string_view{}; }
    std::string_view sequence(size_t i) const { return {files[seq_v[i].file].data + seq_v[i].off, seq_v[i].len}; }
    ~SequenceRecords() { free(bases_data); free(packed_data); }
    SequenceRecords(const SequenceRecords &) = delete;
    SequenceRecords &operator=(const SequenceRecords &) = delete;

    // GenomeReadData::fastX_string (SequenceRecordIterator.h:36-48): FASTQ iff the record has qualities
    void write_fastx(std::ostream &o, size_t i) const {
        const std::string_view q = quality(i), hd = header(i), sq = sequence(i);
        if (!q.empty()) { o.put('@'); o.write(hd.data(), hd.size()); o.put('\n'); o.write(sq.data(), sq.size()); o.write("\n+\n", 3); o.write(q.data(), q.size()); }
        else { o.put('>'); o.write(hd.data(), hd.size()); o.put('\n'); o.write(sq.data(), sq.size()); }
    }
    std::string fastx_string(size_t i) const {
        std::ostringstream o;
        write_fastx(o, i);
        return o.str();
    }

    // threads <= 0: automatic (one thread below 8 MB of bases)
    explicit SequenceRecords(const std::vector<std::string> &read_paths, int threads = 0, bool packed = false, bool fold_case = false)
        : paths(read_paths), file_meta(read_paths.size()) {
        files.reserve(paths.size());
        int cur = -1, method = 4;
        const char *p = nullptr, *end = nullptr;       // cursor in the current file
        uint64_t total_size = 0;
        // std::getline semantics: lines end at '\n' (dropped); a last line without '\n' counts; no empty line after a final '\n'
        auto peek_line = [](const char *&q, const char *e, const char *&ls, size_t &ln) -> bool {
            if (q >= e) return false;
            const char *nl = (const char *) memchr(q, '\n', (size_t) (e - q));
            ls = q; ln = nl ? (size_t) (nl - q) : (size_t) (e - q);
            q = nl ? nl + 1 : e;
            return true;
        };
        auto open_file = [&](int pos) {
            files.emplace_back();
            if (!files.back().open(paths[pos])) throw std::invalid_argument("File with path \"" + paths[pos] + "\" does not exist");
            p = files.back().data; end = p + files.back().size;
            total_size += files.back().size;
            // sniff (load_file_at_position :85-99): first and third line of the file
            const char *q = p, *l0 = nullptr, *l1 = nullptr, *l2 = nullptr;
            size_t n0 = 0, n1 = 0, n2 = 0;
            const bool h0 = peek_line(q, end, l0, n0), h1 = h0 && peek_line(q, end, l1, n1), h2 = h1 && peek_line(q, end, l2, n2);
            (void) l1; (void) n1;
            if (!h1) throw std::logic_error("File is empty");
            const char c0 = n0 ? l0[0] : '\0';
            if (c0 == '@') {
                if (!h2) throw std::logic_error("File is empty");
                if (n2 && l2[0] == '+') method = 4;
            } else if (c0 == '>') {
                method = 2;
            } else {
                throw std::logic_error("Unrecognized file format");
            }
        };
        // the line stream runs on across file boundaries (a record may start in one file and end in the next)
        auto next_line = [&](const char *&ls, size_t &ln, int &file) -> bool {
            while (p >= end) {
                if (cur + 1 >= (int) paths.size()) return false;
                cur++;
                open_file(cur);
            }
            file = cur;
            return peek_line(p, end, ls, ln);
        };
        cur = 0;
        open_file(0);
        int prev_file = -1;
        std::vector<std::string> names;
        seq_off.push_back(0);
        for (;;) {
            const int n = method;
            const char *ls[4] = {nullptr, nullptr, nullptr, nullptr};
            size_t ln[4] = {0, 0, 0, 0};
            int lf[4] = {0, 0, 0, 0};
            int got = 0;
            for (; got < n; got++) if (!next_line(ls[got], ln[got], lf[got])) break;
            if (got < n) break;
            if (ln[0] == 0) throw std::out_of_range("basic_string::substr");    // header.substr(1) on an empty header
            header_v.push_back({(uint32_t) lf[0], (uint32_t) (ln[0] - 1), (uint64_t) (ls[0] + 1 - files[lf[0]].data)});
            seq_v.push_back({(uint32_t) lf[1], (uint32_t) ln[1], (uint64_t) (ls[1] - files[lf[1]].data)});
            seq_off.push_back(seq_off.back() + ln[1]);
            if (n == 4 && ln[3]) { quality_v.push_back({(uint32_t) lf[3], (uint32_t) ln[3], (uint64_t) (ls[3] - files[lf[3]].data)}); is_fastq.push_back(1); }
            else { quality_v.push_back({0, 0, 0}); is_fastq.push_back(0); }
            file_index.push_back(cur);
            if (cur != prev_file) {
                file_meta[cur] = MetaData();
                const size_t slash = paths[cur].find_last_of('/');
                file_meta[cur].filename = slash == std::string::npos ? paths[cur] : paths[cur].substr(slash + 1);
                names.push_back(file_meta[cur].filename);
                prev_file = cur;
            }
            MetaData &fm = file_meta[cur];
            const uint64_t L = ln[1];
            fm.total_bases += L; fm.min_read_length = std::min(fm.min_read_length, L); fm.max_read_length = std::max(fm.max_read_length, L);
            fm.records++; fm.avg_read_length += L;
            meta.total_bases += L; meta.min_read_length = std::min(meta.min_read_length, L); meta.records++; meta.avg_read_length += L;
        }
        fastq_last = method == 4;
        if (meta.records == 0) throw std::logic_error("File is empty");
        meta.avg_read_length /= meta.records;          // aggregate max_read_length stays 0 (never updated, :59-62)
        for (size_t i = 0; i < names.size(); i++) meta.filename += (i ? "__" : "") + names[i];
        // data.avg_read_length /= data.records for EVERY file (:69-71): a file to which no record was attributed (its lines were
        // swallowed by a record that began in the previous file and ended in the next one) is a division by zero there, and the
        // reference dies with SIGFPE; the drop-in refuses the input as well
        for (auto &fm : file_meta) {
            if (!fm.records) throw std::runtime_error("Floating point exception: a read file contributed no record (division by zero in load_meta_data)");
            fm.avg_read_length /= fm.records;
        }

        // phase 2: the sequence bytes, in parallel
        bases_size = seq_off.back();
        const size_t huge = (size_t) 1 << 21;
        const size_t cap = ((size_t) (packed ? (bases_size + 3) / 4 : bases_size) + 64 + huge - 1) & ~(huge - 1);
        void *buf = aligned_alloc(huge, cap);
        if (!buf) throw std::bad_alloc();
        madvise(buf, cap, MADV_HUGEPAGE);
        if (packed) { packed_data = (uint8_t *) buf; pack_from_mappings(threads, fold_case); return; }
        bases_data = (char *) buf;
        int T = threads > 0 ? threads : (int) std::min(16u, std::max(1u, std::thread::hardware_concurrency()));
        if (bases_size < ((uint64_t) 8 << 20)) T = 1;
        const size_t n = seq_v.size();
        auto copy_range = [&](size_t a, size_t b) {
            for (size_t i = a; i < b; i++) memcpy(bases_data + seq_off[i], files[seq_v[i].file].data + seq_v[i].off, seq_v[i].len);
        };
        if (T == 1) copy_range(0, n);
        else {
            // ranges balanced by bytes
            std::vector<std::thread> pool;
            size_t a = 0;
            for (int t = 0; t < T; t++) {
                const uint64_t want = bases_size / T * (t + 1);
                size_t b = t == T - 1 ? n : (size_t) (std::upper_bound(seq_off.begin(), seq_off.end(), want) - seq_off.begin());
                b = std::min(std::max(b, a), n);
                pool.emplace_back(copy_range, a, b);
                a = b;
            }
            for (auto &th : pool) th.join();
        }
    }

private:
    // packed mode of phase 2: thread t packs stream positions [per * t, per * (t + 1)) (per: a multiple of 4, so a thread owns whole
    // bytes) piece by piece from the mappings; the runs of neighbouring threads are joined at the seams
    void pack_from_mappings(int threads, bool fold_case) {
        const uint64_t n_bytes = (bases_size + 3) / 4;
        int T = threads > 0 ? threads : (bases_size < ((uint64_t) 8 << 20) ? 1 : (int) std::min(16u, std::max(1u, std::thread::hardware_concurrency())));
        T = (int) std::max<uint64_t>(1, std::min<uint64_t>((uint64_t) T, n_bytes));
        const uint64_t per = (n_bytes + T - 1) / T * 4;
        std::vector<hga_pack::Packer> part;
        part.reserve(T);
        for (int t = 0; t < T; t++) part.emplace_back(packed_data, std::min(bases_size, per * t), fold_case);
        auto work = [&](int t) {
            const uint64_t a = std::min(bases_size, per * t), b = std::min(bases_size, per * (t + 1));
            if (a >= b) return;
            size_t i = (size_t) (std::upper_bound(seq_off.begin(), seq_off.end(), a) - seq_off.begin()) - 1;     // the read holding a
            for (; i < seq_v.size() && seq_off[i] < b; i++) {
                const uint64_t lo = std::max(a, seq_off[i]), hi = std::min(b, seq_off[i + 1]);
                if (lo < hi) part[t].put(files[seq_v[i].file].data + seq_v[i].off + (lo - seq_off[i]), hi - lo);
            }
        };
        if (T == 1) work(0);
        else {
            std::vector<std::thread> pool;
            for (int t = 0; t < T; t++) pool.emplace_back(work, t);
            for (auto &th : pool) th.join();
        }
        hga_pack::Runs all;
        for (int t = 0; t < T; t++) all.append(part[t].runs);
        exc_start.swap(all.start); exc_end.swap(all.end);
    }
};

// export_components (clustering/ReadClusteringEngine.cpp:804-826): <dir>/#<component id>.fa per component, the records of its
// reads in input order, each followed by a newline (operator<< std::endl, :820). The bytes are the reference's; the writing is
// parallel: every record's size is known, so every record has a fixed offset in its file and `threads` workers pwrite
// disjoint read ranges into the pre-sized files.
inline void export_components(const SequenceRecords &reads, const std::vector<uint32_t> &component_ids, const uint32_t *component_of_read /* 0 = none */,
                              const std::string &dir, int threads = 0) {
    const size_t n = reads.n_reads();
    std::vector<uint32_t> ids(component_ids);
    std::sort(ids.begin(), ids.end());
    auto file_of = [&](uint32_t c) -> int {
        auto it = std::lower_bound(ids.begin(), ids.end(), c);
        return (it != ids.end() && *it == c) ? (int) (it - ids.begin()) : -1;
    };
    auto rec_size = [&](size_t r) -> uint64_t {
        const uint64_t q = reads.quality(r).size();
        return 1 + reads.header(r).size() + 1 + reads.sequence(r).size() + (q ? 3 + q : 0) + 1;
    };
    std::vector<uint64_t> file_size(ids.size(), 0), rec_off(n, 0);
    std::vector<int> rec_file(n, -1);
    for (size_t r = 0; r < n; r++) {
        const int f = component_of_read[r] ? file_of(component_of_read[r]) : -1;
        rec_file[r] = f;
        if (f >= 0) { rec_off[r] = file_size[f]; file_size[f] += rec_size(r); }
    }
    std::vector<int> fds(ids.size(), -1);
    for (size_t f = 0; f < ids.size(); f++) {
        const std::string path = dir + "/#" + std::to_string(ids[f]) + ".fa";
        fds[f] = ::open(path.c_str(), O_CREAT | O_TRUNC | O_WRONLY, 0644);
        if (fds[f] < 0) throw std::runtime_error("cannot create " + path);
        if (file_size[f] && ftruncate(fds[f], (off_t) file_size[f]) != 0) throw std::runtime_error("cannot size " + path);
    }
    int T = threads > 0 ? threads : (reads.bases_size < ((uint64_t) 8 << 20) ? 1 : (int) std::min(16u, std::max(1u, std::thread::hardware_concurrency())));
    std::vector<std::string> errors(T);
    auto work = [&](int t) {
        const size_t a = n * (size_t) t / T, b = n * (size_t) (t + 1) / T;
        std::string buf;
        buf.reserve(1 << 20);
        int cur = -1;
        uint64_t cur_off = 0;
        auto flush = [&]() {
            size_t done = 0;
            while (cur >= 0 && done < buf.size()) {
                const ssize_t w = pwrite(fds[cur], buf.data() + done, buf.size() - done, (off_t) (cur_off + done));
                if (w <= 0) { errors[t] = "write failed"; break; }
                done += (size_t) w;
            }
            buf.clear();
        };
        for (size_t r = a; r < b; r++) {
            const int f = rec_file[r];
            if (f < 0) continue;
            if (f != cur || cur_off + buf.size() != rec_off[r] || buf.size() > (1u << 20)) { flush(); cur = f; cur_off = rec_off[r]; }
            const std::string_view q = reads.quality(r), hd = reads.header(r), sq = reads.sequence(r);
            buf.push_back(q.empty() ? '>' : '@');
            buf.append(hd.data(), hd.size());
            buf.push_back('\n');
            buf.append(sq.data(), sq.size());
            if (!q.empty()) { buf.append("\n+\n", 3); buf.append(q.data(), q.size()); }
            buf.push_back('\n');
        }
        flush();
    };
    if (T == 1) work(0);
    else {
        std::vector<std::thread> pool;
        for (int t = 0; t < T; t++) pool.emplace_back(work, t);
        for (auto &th : pool) th.join();
    }
    for (int fd : fds) if (fd >= 0) ::close(fd);
    for (const auto &e : errors) if (!e.empty()) throw std::runtime_error("export_components: " + e);
}

}  // namespace hga_host
