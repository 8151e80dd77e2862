// jf_occurrences - the reference's SDK-selection front end (jellyfish_occurrences.cpp) on top of libhga_b200.so: it produces the
// --kmers file `categorization` takes (SURVEY.md §8f-4).
//
//   jf_occurrences <read files...> [-k K] [-o OUT]           then, on stdin:  <lower> <upper> <percent>
//
// Same options as jellyfish_occurrences.cpp:22-30 (read_paths, --k-size / -k, --output / -o, --help). Where the reference shells out
// to jellyfish once per read file (occurrences/run_jellyfish.sh) this program counts the canonical k-mers of every file on the GPU
// (hga_count_kmers_packed: exact counts, k-mers seen at least twice). The reads are packed while they load, in the case-folded 2-bit
// form (lowercase a c g t are bases, as for jellyfish; other bytes travel as exception runs), so a quarter of the bytes crosses to the
// GPU; a file is counted in place as a slice of that stream, with its runs clipped to the slice and rebased. The counts equal
// hga_count_kmers on the ASCII bytes, so every output is unchanged. The merge of the per-file lists, the specificity table and the
// export of a count range are the reader's host arithmetic (hga_host_sdk_*; JellyfishOccurrenceReader.cpp:63-134). Differences,
// on purpose: the specificity table is printed as text (the reference pipes it into a Python plot, Plotting.cpp); without -k the k
// sweep of get_unique_k_length (occurrences/KmerAnalysis.cpp:41-56: k = 11, 13, ... until the number of distinct k-mers changes by
// less than 10 %) uses EXACT distinct counts instead of a HyperLogLog estimate (hga_count_spectrum_packed: the distinct count of every
// k of the sweep is computed on the GPU, so host memory does not grow with the number of distinct k-mers); the `percent` sampling draws from a generator
// seeded with --seed (default 0) instead of std::random_device. No GPU, no result: there is no CPU path.
#include <algorithm>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <fstream>
#include <iostream>
#include <stdexcept>
#include <string>
#include <vector>

#include "hga_b200.h"
#include "hga_host.h"

namespace {

void check(int rc, const char *what) {
    if (rc != HGA_OK) {
        std::cerr << "jf_occurrences: " << what << " failed (" << rc << "): " << hga_last_error() << "\n";
        std::exit(2);
    }
}

std::string number_to_sequence(uint64_t v, int k) {            // KmerIterator::number_to_sequence
    std::string s((size_t) k, 'A');
    for (int i = k - 1; i >= 0; i--) { s[(size_t) i] = "ACGT"[v & 3]; v >>= 2; }
    return s;
}

}  // namespace

int main(int argc, char **argv) {
    std::vector<std::string> read_paths;
    std::string output_path;
    int k = 0, device = 0, threads = 0;
    uint64_t seed = 0;
    for (int i = 1; i < argc; i++) {
        const std::string a = argv[i];
        auto need = [&]() -> const char * { if (i + 1 >= argc) throw std::invalid_argument("the required argument for option '" + a + "' is missing"); return argv[++i]; };
        if (a == "-h" || a == "--help") {
            std::cout << "Options:\n  -h [ --help ]         Help screen\n  --read_paths arg      Path to file with reads (FASTA or FASTQ)\n"
                         "  -k [ --k-size ] arg   Size of kmer to analyze & select\n  -o [ --output ] arg   Output path for the exported kmers\n";
            return 0;
        } else if (a == "-k" || a == "--k-size") k = std::atoi(need());
        else if (a == "-o" || a == "--output") output_path = need();
        else if (a == "--read_paths") read_paths.push_back(need());
        else if (a == "--device") device = std::atoi(need());
        else if (a == "--threads" || a == "-t") threads = std::atoi(need());
        else if (a == "--seed") seed = std::strtoull(need(), nullptr, 10);
        else if (a.size() > 1 && a[0] == '-') throw std::invalid_argument("unrecognised option '" + a + "'");
        else read_paths.push_back(a);
    }
    if (read_paths.empty()) throw std::invalid_argument("You need to specify paths to read files");      // jellyfish_occurrences.cpp:38

    hga_host::SequenceRecords reads(read_paths, threads, /*packed=*/true, /*fold_case=*/true);
    std::vector<uint64_t> file_first{0};                       // first read of every file
    for (const auto &m : reads.file_meta) file_first.push_back(file_first.back() + m.records);
    // reads [lo, hi) in place: bases seq_off[lo] .. seq_off[hi] of the packed stream, their runs clipped to them and rebased
    struct Slice { uint64_t b0; std::vector<uint64_t> off, es, ee; };
    auto slice = [&](size_t lo, size_t hi) {
        Slice s;
        s.b0 = reads.seq_off[lo];
        const uint64_t b1 = reads.seq_off[hi];
        for (size_t i = lo; i <= hi; i++) s.off.push_back(reads.seq_off[i] - s.b0);
        for (size_t j = (size_t) (std::upper_bound(reads.exc_end.begin(), reads.exc_end.end(), s.b0) - reads.exc_end.begin());
             j < reads.exc_start.size() && reads.exc_start[j] < b1; j++) {
            s.es.push_back(std::max(reads.exc_start[j], s.b0) - s.b0);
            s.ee.push_back(std::min(reads.exc_end[j], b1) - s.b0);
        }
        return s;
    };
    auto count = [&](int kk, size_t lo, size_t hi, uint32_t min_count, hga_kmer_counts_t *c) {
        const Slice s = slice(lo, hi);
        check(hga_count_kmers_packed(device, kk, reads.packed_data, s.b0, s.off.data(), hi - lo, s.es.data(), s.ee.data(), s.es.size(), min_count, c),
              "hga_count_kmers_packed");
    };

    if (k == 0) {
        // get_unique_k_length (KmerAnalysis.cpp:41-56) with exact distinct counts: the spectrum's totals, no k-mer leaves the GPU
        const Slice all = slice(0, reads.n_reads());
        auto distinct = [&](int kk) {
            hga_kmer_spectrum_t sp;
            check(hga_count_spectrum_packed(device, kk, reads.packed_data, all.b0, all.off.data(), reads.n_reads(), all.es.data(), all.ee.data(), all.es.size(), 0,
                                            nullptr, &sp),
                  "hga_count_spectrum_packed");
            return (long long) sp.n_distinct;
        };
        k = 11;
        long long previous = distinct(k);
        std::cout << "k=11 : " << previous << " kmers" << std::endl;
        while (k < 33 && k + 2 <= 32) {
            const long long count = distinct(k + 2);
            std::cout << "k=" << (k + 2) << " : " << count << " kmers" << std::endl;
            if (((double) std::llabs(count - previous) / ((double) (count + previous) / 2.0)) < 0.1) break;
            k += 2;
            previous = count;
        }
    }

    // per file: exact canonical counts, k-mers seen at least twice (run_jellyfish.sh: bc + count --bc + dump + sort)
    std::vector<uint64_t> file_off{0}, kmers;
    std::vector<uint32_t> counts;
    for (size_t f = 0; f + 1 < file_first.size(); f++) {
        hga_kmer_counts_t c;
        count(k, file_first[f], file_first[f + 1], 2, &c);
        kmers.insert(kmers.end(), c.kmer, c.kmer + c.n);
        counts.insert(counts.end(), c.count, c.count + c.n);
        file_off.push_back(kmers.size());
        hga_free_kmer_counts(&c);
    }
    const uint64_t cap = kmers.size() + 1;
    std::vector<uint64_t> m_kmer(cap);
    std::vector<uint32_t> m_total(cap), m_max(cap), m_files(cap);
    uint64_t n = 0;
    check(hga_host_sdk_merge((int) (file_off.size() - 1), file_off.data(), kmers.data(), counts.data(), m_kmer.data(), m_total.data(), m_max.data(), m_files.data(), &n),
          "hga_host_sdk_merge");

    const double thresholds[] = {70, 85, 90, 95, 99, 100, 100.01};      // jellyfish_occurrences.cpp:47
    uint64_t rows = 0;
    check(hga_host_sdk_specificity(n, m_total.data(), m_max.data(), thresholds, 7, nullptr, nullptr, nullptr, 0, &rows), "hga_host_sdk_specificity");
    std::vector<double> s_thr(rows + 1);
    std::vector<uint32_t> s_occ(rows + 1);
    std::vector<uint64_t> s_cnt(rows + 1);
    check(hga_host_sdk_specificity(n, m_total.data(), m_max.data(), thresholds, 7, s_thr.data(), s_occ.data(), s_cnt.data(), rows, &rows), "hga_host_sdk_specificity");
    std::cout << "# k = " << k << ": upper specificity, occurrences, unique k-mers\n";
    for (uint64_t i = 0; i < rows; i++) std::printf("%.2f %u %llu\n", s_thr[i], s_occ[i], (unsigned long long) s_cnt[i]);
    std::fflush(stdout);

    int lower = 0, upper = 0;
    double percent = 0;
    std::cout << "Enter lower and upper bounds for exported kmers as well as percentage\n";      // :52
    if (!(std::cin >> lower >> upper >> percent)) { std::cerr << "jf_occurrences: expected <lower> <upper> <percent> on stdin\n"; return 2; }
    if (output_path.empty()) {
        char buf[128];
        std::snprintf(buf, sizeof buf, "%d-mers_%d_%d_%g%%.txt", k, lower, upper, percent * 100);      // :57
        output_path = buf;
    }
    std::vector<uint8_t> sel(n + 1);
    uint64_t n_sel = 0, n_disc = 0;
    check(hga_host_sdk_select(n, m_total.data(), m_files.data(), (uint32_t) std::max(lower, 0), (uint32_t) std::max(upper, 0), percent, seed, sel.data(), &n_sel, &n_disc),
          "hga_host_sdk_select");
    std::ofstream out(output_path);
    for (uint64_t i = 0; i < n; i++) if (sel[i]) out << number_to_sequence(m_kmer[i], k) << "\n";
    out.close();
    std::cout << n_disc << " out of " << n_sel << " exported kmers are discriminative\n";      // :132
    return 0;
}
