// `categorization` — drop-in command line for the hot path of the reference executable of the same name
// (/root/reference/src/read_clustering.cpp:35-85): same positional read files, same option names and defaults
// (:41-58, ReadClusteringEngine.h:138-148), same per-file meta blocks, "<stage> took <ms>ms" lines (common/Utils.h:17-35)
// and the same output layout: <dir>/#<component id>.fa, records re-emitted in input order (export_components,
// clustering/ReadClusteringEngine.cpp:804-826).
//
// The arithmetic (scan -> membership -> incidence -> pair counting -> edge selection -> components) runs on the GPU
// behind include/hga_b200.h; there is no CPU path. After the scaffold components (union_find at :763) the run continues
// with the merge of the scaffold components and the core enrichment (hga_enrich; run_clustering :764, :785-794) and exports
// the final components under the surviving component ids, like the reference. The tail / spectral block in between
// (:768-777, SURVEY.md §8f-2: spanning-tree tails, tail amplification, spectral clustering of the scaffold components, merge of
// the clusters) is part of the run, as in the reference (hga_enrich_full); --no-tail-block leaves it out: with more than two
// scaffold components the run then says so on stderr and goes on the way the reference does when it finds no strong tail
// connection (:771), i.e. every scaffold component becomes a core. --spectral (:739-746) takes get_all_connections(5) from
// the GPU and runs the reference's host-side spectral clustering of the whole data set (hga_spectral_clustering).
//
// Extra switches: --no-tail-block (above; --tail-block is accepted and is the default), --scaffolds-only (stop after union_find and export the scaffold components), --load-only (load the k-mers and
// the reads, print the meta data and the load time, no GPU), --export-test (writer self-test, no GPU), --parse-only (print the
// record stream and meta data, no GPU), --dump-kmers (print the canonical k-mer values of the --kmers file, no GPU), --device N.
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <filesystem>
#include <iostream>
#include <map>
#include <condition_variable>
#include <mutex>
#include <thread>

#include "hga_b200.h"
#include "hga_host.h"

namespace {

struct Config {                                     // ReadClusteringConfig, ReadClusteringEngine.h:138-148
    int scaffold_component_min_size = 30;
    int scaffold_component_max_size = -1;
    double scaffold_forming_fraction = 0.15;
    uint64_t scaffold_forming_score = 0;
    uint64_t enrichment_connections_min_score = 20;
    uint64_t tail_amplification_min_score = 40;
    int threads = 1;
    int spectral_dims = 16;
    bool force_spectral = false;
};

void usage() {
    std::cout << "Options:\n"
                 "  -h [ --help ]             Help screen\n"
                 "  --read_paths arg          Path to file with reads (FASTA or FASTQ)\n"
                 "  -k [ --kmers ] arg        Path to text file with kmers\n"
                 "  -o [ --output ] arg       Path to folder with exported clusters\n"
                 "  --sc_max_size arg         Maximum size for a scaffold component\n"
                 "  --sc_min_size arg         Minimum size for a scaffold component\n"
                 "  --sc_fraction arg         Minimum score for a scaffold component forming connection\n"
                 "  --sc_score arg            Minimum score for a scaffold component forming connection\n"
                 "  --tail_amplification arg  Minimal score for tail amplifying connections\n"
                 "  --core_enrichment arg     Minimal score for connections enriching core components\n"
                 "  --spectral_dims arg       Number of dimensions for spectral embedding\n"
                 "  -s [ --spectral ]         Forces the usage of spectral clustering on the entire dataset\n"
                 "  -d [ --debug ]            Debug flag. Treat read files as separate haplotype reads.\n"
                 "  -t [ --threads ] arg      Number of threads to use\n"
                 "  --gpus arg (=1)           hga_b200: GPUs for the hot path (devices --device .. --device + N - 1, NCCL)\n";
}

struct Timer {
    const char *label;
    std::chrono::steady_clock::time_point t0 = std::chrono::steady_clock::now();
    explicit Timer(const char *l) : label(l) {}
    void done() {
        const auto ms = std::chrono::duration_cast<std::chrono::milliseconds>(std::chrono::steady_clock::now() - t0).count();
        std::cout << label << " took " << ms << "ms\n";               // Utils.h:17-35
    }
};

void check(int rc, const char *what) {
    if (rc != HGA_OK) {
        std::cerr << "categorization: " << what << " failed (" << rc << "): " << hga_last_error() << "\n";
        std::exit(2);
    }
}

// --gpus N: the hot path (scan -> index -> pair count -> edge selection -> union-find) on N GPUs, one rank thread per GPU: reads shard by
// contiguous id ranges balanced by bases, the inverted index is partitioned by k-mer owner, partial pair scores are reduced at the owner of
// x (hga_comm.cu). hga_comm_gather_root then leaves a complete single-GPU handle on the first GPU, and the rest of run_clustering
// (ReadClusteringEngine.cpp:764-794) goes on there as with one GPU. Returns rank 0's handle; the stage lines are printed from rank 0's clock.
hga_handle *run_hot_path_multi(const hga_host::KmerSet &ks, const hga_host::SequenceRecords &reads, const Config &config, int device, int gpus) {
    const uint64_t n_reads = reads.n_reads();
    const uint64_t total = reads.seq_off[n_reads];
    std::vector<uint64_t> bound(gpus + 1, n_reads);
    bound[0] = 0;
    for (int r = 1; r < gpus; r++)
        bound[r] = (uint64_t) (std::lower_bound(reads.seq_off.begin(), reads.seq_off.begin() + (ptrdiff_t) n_reads, total / gpus * r) - reads.seq_off.begin());
    unsigned char id[128];
    check(hga_comm_unique_id(id), "hga_comm_unique_id");
    std::vector<hga_handle *> hs(gpus, nullptr);
    std::vector<std::string> errors(gpus);
    std::vector<double> stamp(6, 0.0);                        // rank 0: create, scan, index, pairs + select, components, gather
    std::vector<std::thread> workers;
    // the rank threads meet after every stage: a rank that failed in a purely local stage (hga_create, hga_scan) must not leave the others waiting in the
    // next stage's collective
    std::mutex mu;
    std::condition_variable cv;
    int arrived = 0, generation = 0;
    bool any_failed = false;
    auto meet = [&](bool ok) {
        std::unique_lock<std::mutex> lk(mu);
        if (!ok) any_failed = true;
        const int gen = generation;
        if (++arrived == gpus) { arrived = 0; generation++; cv.notify_all(); }
        else cv.wait(lk, [&] { return generation != gen; });
        return !any_failed;
    };
    for (int r = 0; r < gpus; r++) {
        workers.emplace_back([&, r] {
            bool alive = true;
            auto fail = [&](int rc, const char *what) {
                if (!alive) return true;
                if (rc == HGA_OK) return false;
                errors[r] = std::string(what) + " failed (" + std::to_string(rc) + "): " + hga_last_error();
                alive = false;
                return true;
            };
            auto now = [] { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
            const uint64_t lo = bound[r], hi = bound[r + 1];
            std::vector<uint64_t> off(hi - lo + 1);
            for (uint64_t i = lo; i <= hi; i++) off[i - lo] = reads.seq_off[i] - reads.seq_off[lo];
            // the rank's slice of the packed stream is scanned in place: its exception runs, clipped to the slice and rebased
            const uint64_t b0 = reads.seq_off[lo], b1 = reads.seq_off[hi];
            std::vector<uint64_t> es, ee;
            for (size_t j = (size_t) (std::upper_bound(reads.exc_end.begin(), reads.exc_end.end(), b0) - reads.exc_end.begin());
                 j < reads.exc_start.size() && reads.exc_start[j] < b1; j++) {
                es.push_back(std::max(reads.exc_start[j], b0) - b0);
                ee.push_back(std::min(reads.exc_end[j], b1) - b0);
            }
            double t = now();
            auto lap = [&](int i) { const double n2 = now(); if (r == 0) stamp[i] = n2 - t; t = n2; };
            // every stage is entered by all ranks or by none
            alive = !fail(hga_create(device + r, ks.k, ks.kmers.data(), ks.kmers.size(), &hs[r]), "hga_create");
            if (!meet(alive)) return;
            alive = !fail(hga_comm_init(hs[r], id, r, gpus, n_reads), "hga_comm_init");
            if (!meet(alive)) return;
            lap(0);
            alive = !fail(hga_scan_packed(hs[r], reads.packed_data, b0, off.data(), hi - lo, es.data(), ee.data(), es.size(), (uint32_t) (lo + 1)), "hga_scan_packed");
            if (!meet(alive)) return;
            lap(1);
            alive = !fail(hga_build_index(hs[r]), "hga_build_index");
            if (!meet(alive)) return;
            lap(2);
            alive = !fail(hga_pair_count(hs[r], 1, nullptr, 0), "hga_pair_count");
            if (!meet(alive)) return;
            alive = !fail(hga_select_edges(hs[r], config.scaffold_forming_fraction, 0), "hga_select_edges");
            if (!meet(alive)) return;
            lap(3);
            alive = !fail(hga_components(hs[r], config.scaffold_component_min_size), "hga_components");
            if (!meet(alive)) return;
            lap(4);
            alive = !fail(hga_comm_gather_root(hs[r]), "hga_comm_gather_root");
            if (!meet(alive)) return;
            lap(5);
        });
    }
    for (auto &w : workers) w.join();
    bool failed = false;
    for (int r = 0; r < gpus; r++)
        if (!errors[r].empty()) { std::cerr << "categorization: rank " << r << ": " << errors[r] << "\n"; failed = true; }
    if (failed) std::exit(2);
    std::cout << "Index construction took " << (long long) (stamp[0] + stamp[1] + stamp[2]) << "ms\n";
    std::cout << "Calculation of connections between reads took " << (long long) stamp[3] << "ms\n";
    std::cout << "Union-find took " << (long long) stamp[4] << "ms\n";
    std::fprintf(stderr, "hga_b200: %d GPUs, wall ms on rank 0: create (CUDA context + table + NCCL) %.0f, scan (H2D inside) %.0f, index %.0f, pairs + select %.0f, "
                         "components %.0f, gather to GPU %d %.0f\n", gpus, stamp[0], stamp[1], stamp[2], stamp[3], stamp[4], device, stamp[5]);
    for (int r = 1; r < gpus; r++) hga_destroy(hs[r]);
    return hs[0];
}

}  // namespace

int main(int argc, char **argv) {
    std::vector<std::string> read_paths;
    std::string kmer_path, output_folder_path;
    Config config;
    bool debug = false, parse_only = false, dump_kmers = false, scaffolds_only = false, load_only = false, export_test = false, tail_block = true;
    int device = 0, gpus = 1;

    // boost::program_options' default style (read_clustering.cpp:60-66): --name=value and --name value, -k value and -kvalue,
    // and unambiguous prefixes of long names (--kmer for --kmers)
    static const char *long_names[] = {"--help", "--read_paths", "--kmers", "--output", "--sc_max_size", "--sc_min_size", "--sc_fraction", "--sc_score",
                                       "--tail_amplification", "--core_enrichment", "--spectral_dims", "--spectral", "--debug", "--threads",
                                       "--parse-only", "--dump-kmers", "--scaffolds-only", "--load-only", "--export-test", "--device", "--tail-block", "--no-tail-block", "--gpus"};
    std::vector<std::string> args;
    for (int i = 1; i < argc; i++) {
        std::string a = argv[i];
        std::string value;
        bool has_value = false;
        if (a.rfind("--", 0) == 0 && a.size() > 2) {
            const size_t eq = a.find('=');
            if (eq != std::string::npos) { value = a.substr(eq + 1); a = a.substr(0, eq); has_value = true; }
            std::vector<std::string> matches;
            bool exact = false;
            for (const char *n : long_names) {
                if (a == n) { exact = true; break; }
                if (std::string(n).rfind(a, 0) == 0) matches.push_back(n);
            }
            if (!exact) {
                if (matches.size() == 1) a = matches[0];
                else if (matches.size() > 1) throw std::invalid_argument("option '" + a + "' is ambiguous");
            }
        } else if (a.size() > 2 && a[0] == '-' && a[1] != '-' && std::string("kot").find(a[1]) != std::string::npos) {
            value = a.substr(2); a = a.substr(0, 2); has_value = true;      // -kFILE
        }
        args.push_back(a);
        if (has_value) args.push_back(value);
    }
    const int nargs = (int) args.size();
    auto need = [&](int &i) -> const char * {
        if (i + 1 >= nargs) throw std::invalid_argument("the required argument for option '" + args[i] + "' is missing");
        return args[++i].c_str();
    };
    for (int i = 0; i < nargs; i++) {
        const std::string a = args[i];
        if (a == "-h" || a == "--help") { usage(); return 0; }
        else if (a == "-k" || a == "--kmers") kmer_path = need(i);
        else if (a == "-o" || a == "--output") output_folder_path = need(i);
        else if (a == "--read_paths") read_paths.push_back(need(i));
        else if (a == "--sc_max_size") config.scaffold_component_max_size = std::atoi(need(i));
        else if (a == "--sc_min_size") config.scaffold_component_min_size = std::atoi(need(i));
        else if (a == "--sc_fraction") config.scaffold_forming_fraction = std::atof(need(i));
        else if (a == "--sc_score") config.scaffold_forming_score = std::strtoull(need(i), nullptr, 10);
        else if (a == "--tail_amplification") config.tail_amplification_min_score = std::strtoull(need(i), nullptr, 10);
        else if (a == "--core_enrichment") config.enrichment_connections_min_score = std::strtoull(need(i), nullptr, 10);
        else if (a == "--spectral_dims") config.spectral_dims = std::atoi(need(i));
        else if (a == "-s" || a == "--spectral") config.force_spectral = true;
        else if (a == "-d" || a == "--debug") debug = true;
        else if (a == "-t" || a == "--threads") config.threads = std::atoi(need(i));
        else if (a == "--parse-only") parse_only = true;
        else if (a == "--dump-kmers") dump_kmers = true;
        else if (a == "--scaffolds-only") scaffolds_only = true;
        else if (a == "--load-only") load_only = true;
        else if (a == "--export-test") export_test = true;
        else if (a == "--device") device = std::atoi(need(i));
        else if (a == "--gpus") gpus = std::max(1, std::atoi(need(i)));
        else if (a == "--tail-block") tail_block = true;
        else if (a == "--no-tail-block") tail_block = false;
        else if (a.size() > 1 && a[0] == '-') throw std::invalid_argument("unrecognised option '" + a + "'");
        else read_paths.push_back(a);
    }
    (void) debug;   // haplotype annotation / plots are debug output of the reference, not part of the hot path

    if (kmer_path.empty() && !parse_only && !load_only && !export_test) throw std::invalid_argument("You need to specify path to kmers");
    if (dump_kmers) {
        const hga_host::KmerSet ks = hga_host::load_text_file_kmers(kmer_path);
        std::cout << "#K " << ks.k << " " << ks.kmers.size() << "\n";
        for (uint64_t v : ks.kmers) std::cout << v << "\n";
        return 0;
    }
    if (read_paths.empty()) throw std::invalid_argument("You need to specify paths to read files");

    // the CUDA context is created on a second thread while the files are read (seconds on a cold machine)
    std::thread cuda_start;
    if (!parse_only && !load_only && !export_test) cuda_start = std::thread([device] { (void) hga_init(device); });
    struct Joiner { std::thread &t; ~Joiner() { if (t.joinable()) t.join(); } } joiner{cuda_start};
    hga_host::KmerSet ks;
    Timer t_load("Loading of k-mers and reads");
    if (!parse_only && !kmer_path.empty()) ks = hga_host::load_text_file_kmers(kmer_path, config.threads > 1 ? config.threads : 0);
    // the reads are packed while they load (2-bit codes + exception runs: a quarter of the bytes to copy to the GPU)
    hga_host::SequenceRecords reads(read_paths, config.threads > 1 ? config.threads : 0, /*packed=*/true);
    if (!parse_only) t_load.done();
    if (export_test) {   // writer self-test (no GPU): read r (1-based) goes to component 1 + r % 3, every 7th read to none
        std::vector<uint32_t> of_read(reads.n_reads());
        for (size_t r = 0; r < reads.n_reads(); r++) of_read[r] = ((r + 1) % 7 == 0) ? 0u : (uint32_t) (1 + (r + 1) % 3);
        std::filesystem::remove_all(output_folder_path);
        std::filesystem::create_directories(output_folder_path);
        hga_host::export_components(reads, {1, 2, 3}, of_read.data(), output_folder_path, config.threads);
        return 0;
    }
    if (load_only) {
        for (const auto &m : reads.file_meta) std::cout << m.repr();
        std::cout << ks.kmers.size() << " k-mers, k = " << ks.k << "\n";
        return 0;
    }
    if (parse_only) {
        for (const auto &m : reads.file_meta)
            std::cout << "#META " << m.filename << " " << m.records << " " << m.total_bases << " " << m.avg_read_length << " " << m.max_read_length << " "
                      << m.min_read_length << "\n";
        const auto &m = reads.meta;
        std::cout << "#AGG " << m.filename << " " << m.records << " " << m.total_bases << " " << m.avg_read_length << " " << m.max_read_length << " "
                  << m.min_read_length << "\n";
        for (size_t i = 0; i < reads.n_reads(); i++)
            std::cout << (i + 1) << "\t" << reads.header(i) << "\t" << reads.sequence(i) << "\t" << reads.quality(i) << "\n";
        return 0;
    }
    for (const auto &m : reads.file_meta) std::cout << m.repr();
    if (output_folder_path.empty()) output_folder_path = "./" + reads.meta.filename + "_clusters/";
    if (config.scaffold_component_max_size != -1 && scaffolds_only) {
        std::cerr << "categorization: --sc_max_size makes the scaffold components depend on the edge order (sequential union_find); they are computed "
                     "inside the merge + enrichment stage, not by the GPU components stage --scaffolds-only exports\n";
        return 3;
    }

    if (gpus > 1 && (config.force_spectral || config.scaffold_forming_score > 0 || reads.n_reads() < (size_t) gpus)) {
        std::cerr << "categorization: --gpus " << gpus << " applies to the default path (all reads as pivots, --sc_fraction); --spectral / --sc_score and inputs with "
                     "fewer reads than GPUs run on one GPU\n";
        gpus = 1;
    }
    hga_handle *h = nullptr;
    if (gpus > 1) {
        if (cuda_start.joinable()) cuda_start.join();
        int n_dev = 0;
        check(hga_device_count(&n_dev), "hga_device_count");
        if (device < 0 || device + gpus > n_dev) {            // checked here: a rank thread that cannot create its handle would leave the others waiting in ncclCommInitRank
            std::cerr << "categorization: --gpus " << gpus << " from --device " << device << " needs devices " << device << " .. " << device + gpus - 1 << ", this machine has " << n_dev << "\n";
            return 2;
        }
        h = run_hot_path_multi(ks, reads, config, device, gpus);
    } else {
        Timer t("Index construction");               // table build + scan + inverted index = construct_indices (:234-299)
        if (cuda_start.joinable()) cuda_start.join();
        const auto w0 = std::chrono::steady_clock::now();
        check(hga_create(device, ks.k, ks.kmers.data(), ks.kmers.size(), &h), "hga_create");
        const auto w1 = std::chrono::steady_clock::now();
        check(hga_scan_packed(h, reads.packed_data, 0, reads.seq_off.data(), reads.n_reads(), reads.exc_start.data(), reads.exc_end.data(), reads.exc_start.size(), 1),
              "hga_scan_packed");
        const auto w2 = std::chrono::steady_clock::now();
        check(hga_build_index(h), "hga_build_index");
        const auto w3 = std::chrono::steady_clock::now();
        t.done();
        std::fprintf(stderr, "hga_b200: wall ms: create (CUDA context + table) %.0f, scan (H2D inside) %.0f, index %.0f\n",
                     std::chrono::duration<double, std::milli>(w1 - w0).count(), std::chrono::duration<double, std::milli>(w2 - w1).count(),
                     std::chrono::duration<double, std::milli>(w3 - w2).count());
    }
    if (config.force_spectral) {
        // run_clustering :739-746: get_all_connections(5) on the GPU; spectral clustering of the WHOLE data set on the host (an S x S
        // eigen-problem over all connected reads, lib/clustering: small inputs only, in the reference as well); merge_components
        // (element [0] of a cluster survives); components with >= sc_min_size reads are exported. The connection list goes to the
        // spectral stage in the canonical order (score desc, min id asc, max id asc, x asc), both directions as the reference emits them.
        hga_pairs pr;
        {
            Timer t("Calculation of connections between reads");
            check(hga_pair_count(h, 5, nullptr, 0), "hga_pair_count");
            check(hga_get_pairs(h, &pr), "hga_get_pairs");
            t.done();
        }
        std::vector<uint32_t> final_ids, of_read(reads.n_reads(), 0);
        {
            Timer t("Forced spectral clustering");
            std::vector<uint64_t> order(pr.n_pairs);
            for (uint64_t i = 0; i < pr.n_pairs; i++) order[i] = i;
            std::stable_sort(order.begin(), order.end(), [&](uint64_t a, uint64_t b) { return pr.score[a] > pr.score[b]; });   // pairs arrive in (x, y) order
            std::vector<uint32_t> cx(2 * pr.n_pairs + 1), cy(2 * pr.n_pairs + 1), member(4 * pr.n_pairs + 1);
            std::vector<uint64_t> cs(2 * pr.n_pairs + 1), coff((size_t) config.spectral_dims + 2, 0);
            for (uint64_t i = 0; i < pr.n_pairs; i++) {
                const uint64_t j = order[i];
                cx[2 * i] = pr.x[j]; cy[2 * i] = pr.y[j]; cs[2 * i] = pr.score[j];
                cx[2 * i + 1] = pr.y[j]; cy[2 * i + 1] = pr.x[j]; cs[2 * i + 1] = pr.score[j];
            }
            uint64_t n_nodes = 0, n_clusters = 0;
            check(hga_spectral_clustering(cx.data(), cy.data(), cs.data(), 2 * pr.n_pairs, config.spectral_dims, member.data(), coff.data(), &n_nodes, &n_clusters),
                  "hga_spectral_clustering");
            std::vector<std::pair<uint32_t, uint64_t>> by_first;          // (smallest member, cluster) of the clusters that are large enough
            for (uint64_t c = 0; c < n_clusters; c++) {
                const uint64_t a = coff[c], b = coff[c + 1];
                if (b == a || b - a < (uint64_t) std::max(config.scaffold_component_min_size, 1)) continue;
                by_first.push_back({*std::min_element(member.begin() + (ptrdiff_t) a, member.begin() + (ptrdiff_t) b), c});
            }
            std::sort(by_first.begin(), by_first.end());
            for (const auto &bc : by_first) {
                const uint32_t id = member[coff[bc.second]];
                final_ids.push_back(id);
                for (uint64_t i = coff[bc.second]; i < coff[bc.second + 1]; i++) of_read[member[i] - 1] = id;
            }
            t.done();
        }
        std::filesystem::remove_all(output_folder_path);
        std::filesystem::create_directories(output_folder_path);
        hga_host::export_components(reads, final_ids, of_read.data(), output_folder_path, config.threads > 1 ? config.threads : 0);
        std::cout << "Exported " << final_ids.size() << " components\n";
        hga_destroy(h);
        return 0;
    }
    if (gpus == 1) {
        Timer t("Calculation of connections between reads");
        if (config.scaffold_forming_score > 0) {
            // pivots = components with at least sc_score discriminative k-mers (:750-752)
            hga_hits hits;
            check(hga_get_hits(h, 0, &hits), "hga_get_hits");
            std::vector<uint32_t> pivots;
            for (uint64_t r = 0; r < hits.n_reads; r++)
                if (hits.row_off[r + 1] - hits.row_off[r] >= config.scaffold_forming_score) pivots.push_back((uint32_t) (r + 1));
            const uint32_t none = 0;       // no read reaches the threshold: the EMPTY subset (a NULL pointer would mean "all reads")
            check(hga_pair_count(h, (uint32_t) config.scaffold_forming_score, pivots.empty() ? &none : pivots.data(), pivots.size()), "hga_pair_count");
            check(hga_select_edges(h, 0.0, (uint32_t) config.scaffold_forming_score), "hga_select_edges");
        } else {
            check(hga_pair_count(h, 1, nullptr, 0), "hga_pair_count");
            check(hga_select_edges(h, config.scaffold_forming_fraction, 0), "hga_select_edges");
        }
        t.done();
    }
    hga_components_t comp;
    if (gpus == 1) {
        Timer t("Union-find");
        check(hga_components(h, config.scaffold_component_min_size), "hga_components");
        check(hga_get_components(h, &comp), "hga_get_components");
        t.done();
    } else {
        check(hga_get_components(h, &comp), "hga_get_components");
    }

    // export_components (:804-826): one file per component, records in input order; reads of no component are dropped
    std::filesystem::remove_all(output_folder_path);
    std::filesystem::create_directories(output_folder_path);
    const int io_threads = config.threads > 1 ? config.threads : 0;
    if (scaffolds_only) {
        std::vector<uint32_t> of_read(comp.n_reads, 0), ids(comp.comp_label, comp.comp_label + comp.n_components);
        std::sort(ids.begin(), ids.end());
        for (uint64_t r = 0; r < comp.n_reads; r++)
            if (std::binary_search(ids.begin(), ids.end(), comp.label[r])) of_read[r] = comp.label[r];
        hga_host::export_components(reads, ids, of_read.data(), output_folder_path, io_threads);
        std::cout << "Exported " << comp.n_components << " components\n";
    } else {
        if (!tail_block && (comp.n_components > 2 || config.scaffold_component_max_size != -1))
            std::cerr << "categorization: " << comp.n_components << " scaffold components; the tail / spectral merge of scaffold components "
                         "(ReadClusteringEngine.cpp:768-777) is left out (--no-tail-block): every scaffold component becomes a core, as in the reference "
                         "when it finds no strong tail connection\n";
        hga_enrichment_t fin;
        {
            if (tail_block)
                check(hga_enrich_full(h, config.scaffold_component_min_size, config.scaffold_component_max_size, (uint32_t) config.enrichment_connections_min_score,
                                      (uint32_t) config.tail_amplification_min_score, config.spectral_dims, reads.seq_off.data()), "hga_enrich_full");
            else
                check(hga_enrich_ex(h, config.scaffold_component_min_size, config.scaffold_component_max_size, (uint32_t) config.enrichment_connections_min_score),
                      "hga_enrich");
            check(hga_get_enrichment(h, &fin), "hga_get_enrichment");
            // one library call, reported under the reference's own timer labels (ReadClusteringEngine.cpp:765-791)
            hga_metrics_t pm;
            hga_tail_block_t tb;
            check(hga_metrics(h, &pm), "hga_metrics");
            const bool block_ran = tail_block && hga_get_tail_block(h, &tb) == HGA_OK && tb.ran;
            const char *labels[6] = {"Merging of initial components", "Calculation of tail connections", "Spectral clustering", "Merging of scaffold components",
                                     "Calculation of enrichment connections", "Merging into core components"};
            for (int i = 0; i < 6; i++) {
                if (i >= 1 && i <= 3 && !(block_ran && (i == 1 || pm.enrich_phase_ms[i] > 0))) continue;   // :768-775: only with more than two scaffold components / strong tail connections
                std::cout << labels[i] << " took " << (long long) pm.enrich_phase_ms[i] << "ms\n";
            }
        }
        Timer t_exp("Export of components");
        hga_host::export_components(reads, std::vector<uint32_t>(fin.final_id, fin.final_id + fin.n_final), fin.assignment, output_folder_path, io_threads);
        t_exp.done();
        std::cout << "Exported " << fin.n_final << " components\n";
    }

    hga_metrics_t m;
    if (hga_metrics(h, &m) == HGA_OK) {
        std::fprintf(stderr,
                     "hga_b200: %llu reads, %llu bases, %llu hits, %llu pairs, %llu selected edges, %llu components | GPU ms: table %.2f h2d %.2f scan %.2f "
                     "index %.2f pairs %.2f select %.2f components %.2f enrich %.2f (%llu cores, %llu enrichment connections, %llu final components)\n",
                     (unsigned long long) m.n_reads, (unsigned long long) m.n_bases, (unsigned long long) m.n_hits, (unsigned long long) m.n_pairs,
                     (unsigned long long) m.n_selected, (unsigned long long) m.n_components, m.table_build_ms, m.h2d_ms, m.scan_ms, m.index_ms, m.pair_ms,
                     m.select_ms, m.components_ms, m.enrich_ms, (unsigned long long) m.n_cores, (unsigned long long) m.n_enrich_connections,
                     (unsigned long long) m.n_final_components);
    }
    hga_destroy(h);
    return 0;
}
