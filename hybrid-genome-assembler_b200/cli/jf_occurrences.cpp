// jf_occurrences - the reference's SDK-selection front end (jellyfish_occurrences.cpp) on top of libhga_b200.so: it produces the
// --kmers file `categorization` takes (SURVEY.md §8f-4).
//
//   jf_occurrences <read files...> [-k K] [-o OUT]           then, on stdin:  <lower> <upper> <percent>
//
// Same options as jellyfish_occurrences.cpp:22-30 (read_paths, --k-size / -k, --output / -o, --help). Where the reference shells out
// to jellyfish once per read file (occurrences/run_jellyfish.sh) this program counts the canonical k-mers of every file on the GPU
// (exact counts, k-mers seen at least twice in the file). The reads are packed while they load, in the case-folded 2-bit form
// (lowercase a c g t are bases, as for jellyfish; other bytes travel as exception runs), so a quarter of the bytes crosses to the GPU.
// One call (hga_sdk_count_packed) counts every file and merges the files' counts on the GPU; the merged table stays there, the
// specificity table is computed there (hga_sdk_specificity) and only the k-mers of the chosen count range come back (hga_sdk_range).
// The results are those of the reader's host arithmetic on the per-file hga_count_kmers_packed lists (hga_host_sdk_merge /
// _specificity; JellyfishOccurrenceReader.cpp:63-134), and the sampling stays on the host (hga_host_sdk_select on the range). Differences,
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

    // per file: exact canonical counts, k-mers seen at least twice (run_jellyfish.sh: bc + count --bc + dump + sort), merged over
    // the files; the merged table stays on the GPU
    hga_sdk *sdk = nullptr;
    {
        const Slice all = slice(0, reads.n_reads());
        check(hga_sdk_count_packed(device, k, reads.packed_data, all.b0, all.off.data(), reads.n_reads(), all.es.data(), all.ee.data(), all.es.size(),
                                   (int) (file_first.size() - 1), file_first.data(), 2, &sdk),
              "hga_sdk_count_packed");
    }

    const double thresholds[] = {70, 85, 90, 95, 99, 100, 100.01};      // jellyfish_occurrences.cpp:47
    uint64_t rows = 0;
    check(hga_sdk_specificity(sdk, thresholds, 7, nullptr, nullptr, nullptr, 0, &rows), "hga_sdk_specificity");
    std::vector<double> s_thr(rows + 1);
    std::vector<uint32_t> s_occ(rows + 1);
    std::vector<uint64_t> s_cnt(rows + 1);
    check(hga_sdk_specificity(sdk, thresholds, 7, s_thr.data(), s_occ.data(), s_cnt.data(), rows, &rows), "hga_sdk_specificity");
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
    // only the k-mers of the count range come back; the sampler draws for in-range k-mers only, in ascending order, so it keeps the
    // same ones as on the whole merged table
    const uint32_t lo = (uint32_t) std::max(lower, 0), hi = (uint32_t) std::max(upper, 0);
    hga_sdk_range_t r;
    check(hga_sdk_range(sdk, lo, hi, &r), "hga_sdk_range");
    hga_sdk_free(sdk);
    std::vector<uint8_t> sel(r.n + 1);
    uint64_t n_sel = 0, n_disc = 0;
    check(hga_host_sdk_select(r.n, r.total, r.files, lo, hi, percent, seed, sel.data(), &n_sel, &n_disc), "hga_host_sdk_select");
    std::ofstream out(output_path);
    for (uint64_t i = 0; i < r.n; i++) if (sel[i]) out << number_to_sequence(r.kmer[i], k) << "\n";
    out.close();
    hga_free_sdk_range(&r);
    std::cout << n_disc << " out of " << n_sel << " exported kmers are discriminative\n";      // :132
    return 0;
}
