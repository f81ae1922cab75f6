// kmer_count -- reads -> the reference's k-mer file, or straight to contigs, on the B200 library.
//
//   kmer_count K reads_file [--histo HISTO_FILE] kmer_file_out   [min_count [min_ext]]
//   kmer_count K reads_file [--histo HISTO_FILE] --contigs PREFIX [min_count [min_ext]]
//   kmer_count K reads_file --histo HISTO_FILE
//
// The first form writes what the reference's read_kmers parses (read_kmers.hpp:64-76: K bases, a blank, backward and
// forward extension, '\n' per unique k-mer) -- the output of "the first preprocessing stage" the assignment assumes done
// (README.md:19-21) -- so `kmer_hash_<K> kmer_file_out test` (ours or the reference's) can follow.  The second form keeps
// the records on the GPU (kh_count_extract_device -> kh_insert_pairs_device -> kh_assemble) and writes PREFIX_0.dat, one
// contig per line, the file scripts/check_it.sh:47-48 sorts and diffs: no k-mer text in between.
//
// reads_file: one read per line, FASTA or FASTQ (detected from the first byte; header / quality lines are blanked on
// the host).  Bases are upper-case ACGT; anything else (N, ...) splits a read.  Defaults: min_count = min_ext = 2.
//
// --histo HISTO_FILE writes the k-mer spectrum (kh_count_histogram) in the two-column format of `jellyfish histo`, which
// GenomeScope reads: "c n" per line for every count c in 1..255 with n > 0 distinct k-mers, ascending; 255 stands for
// 255 or more.  With --histo alone nothing else is written.  min_count may be the word `auto`: the valley of the
// spectrum (kh_count_auto_min_count).  Whenever the spectrum is computed, one more stdout line reports it.
// Environment: KH_DEVICE, KH_LOAD_FACTOR (0.5), KH_COUNT_DISTINCT = distinct k-mers to size the table for, erroneous
// ones included (default: half the input bytes).
//
// KH_RANKS=P (2..8): the analysis on P ranks (GPU r % visible GPUs, KH_DEVICE is not used), kh_sharded::CountCluster:
// the pieces of the file are dealt to the ranks in turn, every rank counts its pieces, and reduce() merges all counts at
// the k-mers' owner ranks -- whenever a rank has counted KH_COUNT_BATCH_BYTES since the last reduce (then pieces are
// that size too; default: no intermediate reduce) and once at the end.  The k-mer file is the ranks' k-mers in rank
// order; with --contigs, every rank's records go on its GPU into kh_sharded::Cluster (17 <= K <= 54) and rank r writes
// PREFIX_r.dat.  Same k-mers, counters and contigs as P = 1, in another order.
#include <algorithm>
#include <array>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <stdexcept>
#include <string>
#include <vector>

#include "kh/kmer_counter.hpp"
#include "kh/sharded_counter.hpp"
#include "kh/sharded_host.hpp"

namespace {

void must(int status, kh_table* t, const char* what) {
    if (status == KH_OK) return;
    const char* detail = t ? kh_last_error(t) : "";
    throw std::runtime_error(std::string(detail && *detail ? detail : kh_status_string(status)) + " [" + what + "]");
}

int usage() {
    fprintf(stderr, "Usage: kmer_count K reads_file [--histo HISTO_FILE] [kmer_file_out | --contigs PREFIX] [min_count|auto [min_ext]]\n"
                    "       (the output may be left out only with --histo)\n");
    return 1;
}

// The spectrum once counting is done: written to `histo` (if named), min_count resolved when it is `auto`, one line on
// stdout.
void spectrum(const std::array<uint64_t, 256>& hist, int k, const std::string& histo, bool auto_min_count, uint32_t& min_count) {
    if (!histo.empty()) {
        FILE* o = fopen(histo.c_str(), "wb");
        if (o == nullptr) throw std::runtime_error("kmer_count: could not open " + histo);
        for (size_t c = 1; c < hist.size(); ++c)
            if (hist[c] && fprintf(o, "%zu %llu\n", c, (unsigned long long)hist[c]) < 0) throw std::runtime_error("kmer_count: short write to " + histo);
        if (fclose(o) != 0) throw std::runtime_error("kmer_count: short write to " + histo);
    }
    uint64_t distinct = 0;
    for (uint64_t n : hist) distinct += n;
    const uint32_t valley = kh_count_auto_min_count(hist.data());
    if (auto_min_count) min_count = valley;
    printf("Spectrum of %llu distinct %d-mers%s%s: min_count %u, auto min_count %u\n", (unsigned long long)distinct, k,
           histo.empty() ? "" : " written to ", histo.c_str(), min_count, valley);
}

// The file goes through in pieces of about `buffer` bytes that end on a line boundary (FASTA: before a header); each
// piece's sequence lines (kh::sequence_lines) go to sink(text, n).
template <class Sink> void read_pieces(FILE* f, size_t buffer, Sink sink) {
    std::vector<char> buf(buffer);
    size_t carry = 0;
    char format = 0;
    unsigned state = 0;
    for (;;) {
        if (carry == buf.size()) buf.resize(buf.size() * 2);                  // a single line longer than the buffer
        const size_t got = fread(buf.data() + carry, 1, buf.size() - carry, f);
        const size_t have = carry + got;
        if (have == 0) break;
        if (format == 0) format = buf[0] == '>' ? 'a' : (buf[0] == '@' ? 'q' : 'p');
        size_t cut = have;
        if (got != 0) {                                                       // not at the end of the file: stop where a new read starts
            cut = kh::sequence_cut(buf.data(), have, format);
            if (cut == 0) { carry = have; continue; }
        }
        size_t len = cut;
        kh::sequence_lines(buf.data(), len, format, state);
        sink(buf.data(), len);
        carry = have - cut;
        memmove(buf.data(), buf.data() + cut, carry);
        if (got == 0) break;
    }
}

int count_sharded(FILE* f, int k, int ranks, uint64_t distinct, double lf, bool contigs, const std::string& out_name,
                  const std::string& histo, bool auto_min_count, uint32_t min_count, uint32_t min_ext) {
    using clock = std::chrono::high_resolution_clock;
    const uint64_t batch = getenv("KH_COUNT_BATCH_BYTES") ? strtoull(getenv("KH_COUNT_BATCH_BYTES"), nullptr, 10) : 0;
    const size_t buffer = batch ? (size_t)std::min<uint64_t>(128u << 20, std::max<uint64_t>(batch, 4096)) : (128u << 20) + (1u << 20);
    const auto t0 = clock::now();
    kh_sharded::CountCluster cluster(k, ranks, distinct, lf);
    int next = 0;
    read_pieces(f, buffer, [&](const char* p, size_t n) {
        const int r = next;
        next = (next + 1) % ranks;
        cluster.count(r, p, n);
        if (batch && cluster.batch_bytes(r) >= batch) cluster.reduce();
    });
    fclose(f);
    cluster.reduce();
    const auto t1 = clock::now();
    printf("Counted %llu k-mer occurrences, %llu distinct %d-mers, from %llu bytes of reads in %lf s\n",
           (unsigned long long)cluster.n_occurrences(), (unsigned long long)cluster.n_distinct(), k,
           (unsigned long long)cluster.n_bytes(), std::chrono::duration<double>(t1 - t0).count());
    if (!histo.empty() || auto_min_count) spectrum(cluster.histogram(), k, histo, auto_min_count, min_count);
    if (out_name.empty()) return 0;

    if (!contigs) {
        FILE* o = fopen(out_name.c_str(), "wb");
        if (o == nullptr) throw std::runtime_error("kmer_count: could not open " + out_name);
        uint64_t lines = 0;
        for (int r = 0; r < ranks; ++r) {
            const std::string text = cluster.extract_lines(r, min_count, min_ext);
            if (fwrite(text.data(), 1, text.size(), o) != text.size()) throw std::runtime_error("kmer_count: short write to " + out_name);
            lines += text.size() / (size_t)(k + 4);
        }
        fclose(o);
        printf("Wrote %llu k-mers (count >= %u, extensions seen >= %u times) to %s\n", (unsigned long long)lines, min_count,
               min_ext, out_name.c_str());
        return 0;
    }
    std::vector<const void*> recs(ranks);
    std::vector<uint64_t> n(ranks);
    for (int r = 0; r < ranks; ++r) recs[r] = cluster.extract_device(r, min_count, min_ext, n[r]);
    uint64_t n_local_max = 1, n_total = 0;
    for (uint64_t x : n) { n_local_max = std::max(n_local_max, x); n_total += x; }
    const auto t2 = clock::now();
    kh_sharded::Cluster tables(k, ranks, n_local_max, std::max<uint64_t>(n_total, 1), lf);
    tables.begin();
    tables.insert(recs, n);
    const std::vector<kh_sharded::RankOutput> outs = tables.assemble();
    const auto t3 = clock::now();
    uint64_t nc = 0, nodes = 0;
    for (int r = 0; r < ranks; ++r) {
        const std::string dat = out_name + "_" + std::to_string(r) + ".dat";
        FILE* o = fopen(dat.c_str(), "wb");
        if (o == nullptr) throw std::runtime_error("kmer_count: could not open " + dat);
        const std::vector<char>& text = outs[r].text;
        if (!text.empty() && fwrite(text.data(), 1, text.size(), o) != text.size()) throw std::runtime_error("kmer_count: short write to " + dat);
        fclose(o);
        nc += outs[r].n_contigs;
        nodes += outs[r].n_nodes;
    }
    printf("Assembled %llu k-mers into %llu contigs with %llu nodes in %lf s; wrote %s_0.dat .. %s_%d.dat\n",
           (unsigned long long)n_total, (unsigned long long)nc, (unsigned long long)nodes,
           std::chrono::duration<double>(t3 - t2).count(), out_name.c_str(), out_name.c_str(), ranks - 1);
    return 0;
}

}  // namespace

int main(int argc, char** argv) {
    if (argc < 4) return usage();
    const int k = atoi(argv[1]);
    const std::string reads_file = argv[2];
    int a = 3;
    std::string histo;
    if (std::string(argv[a]) == "--histo") {
        if (++a >= argc) return usage();
        histo = argv[a++];
    }
    if (histo.empty() && a >= argc) return usage();
    const bool contigs = a < argc && std::string(argv[a]) == "--contigs";
    if (contigs && ++a >= argc) return usage();
    const std::string out_name = a < argc ? argv[a++] : "";              // empty: --histo alone
    const bool auto_min_count = a < argc && std::string(argv[a]) == "auto";
    uint32_t min_count = a < argc ? (auto_min_count ? 0u : (uint32_t)atoi(argv[a])) : 2u;
    if (a < argc) ++a;
    const uint32_t min_ext = a < argc ? (uint32_t)atoi(argv[a++]) : 2u;
    if (k < 2 || k > 61) { fprintf(stderr, "kmer_count: K must be 2..61\n"); return 1; }
    const int device = getenv("KH_DEVICE") ? atoi(getenv("KH_DEVICE")) : 0;
    const double lf = getenv("KH_LOAD_FACTOR") ? atof(getenv("KH_LOAD_FACTOR")) : 0.5;

    FILE* f = fopen(reads_file.c_str(), "rb");
    if (f == nullptr) throw std::runtime_error("kmer_count: could not open " + reads_file);
    fseek(f, 0, SEEK_END);
    const uint64_t file_bytes = (uint64_t)ftell(f);
    fseek(f, 0, SEEK_SET);
    const uint64_t distinct = getenv("KH_COUNT_DISTINCT") ? strtoull(getenv("KH_COUNT_DISTINCT"), nullptr, 10)
                                                          : (file_bytes / 2 > 1024 ? file_bytes / 2 : 1024);
    const int ranks = getenv("KH_RANKS") ? atoi(getenv("KH_RANKS")) : 1;
    if (ranks < 1 || ranks > 8) { fprintf(stderr, "kmer_count: KH_RANKS must be 1..8\n"); return 1; }
    if (ranks > 1 && contigs && (k < 17 || k > 54)) { fprintf(stderr, "kmer_count: --contigs with KH_RANKS > 1 needs 17 <= K <= 54\n"); return 1; }
    if (ranks > 1) return count_sharded(f, k, ranks, distinct, lf, contigs, out_name, histo, auto_min_count, min_count, min_ext);
    const auto t0 = std::chrono::high_resolution_clock::now();
    kh::KmerCounter counter(k, distinct, lf, device);

    read_pieces(f, (128u << 20) + (1u << 20), [&](const char* p, size_t n) { counter.count_reads(p, n); });
    fclose(f);
    const auto t1 = std::chrono::high_resolution_clock::now();
    kh_count_stats st = counter.stats();
    printf("Counted %llu k-mer occurrences, %llu distinct %d-mers, from %llu bytes of reads in %lf s\n",
           (unsigned long long)st.n_occurrences, (unsigned long long)st.n_distinct, k, (unsigned long long)st.n_bytes,
           std::chrono::duration<double>(t1 - t0).count());
    if (!histo.empty() || auto_min_count) spectrum(counter.histogram(), k, histo, auto_min_count, min_count);
    if (out_name.empty()) return 0;

    if (!contigs) {
        const std::string lines = counter.extract_lines(min_count, min_ext);
        FILE* o = fopen(out_name.c_str(), "wb");
        if (o == nullptr) throw std::runtime_error("kmer_count: could not open " + out_name);
        if (fwrite(lines.data(), 1, lines.size(), o) != lines.size()) throw std::runtime_error("kmer_count: short write to " + out_name);
        fclose(o);
        printf("Wrote %llu k-mers (count >= %u, extensions seen >= %u times) to %s\n",
               (unsigned long long)(lines.size() / (size_t)(k + 4)), min_count, min_ext, out_name.c_str());
        return 0;
    }
    uint64_t n = 0;
    const void* recs = counter.extract_device(min_count, min_ext, n);
    kh_table* t = nullptr;
    must(kh_create(k, n ? n : 1, lf, device, &t), nullptr, "kh_create");
    const auto t2 = std::chrono::high_resolution_clock::now();
    must(kh_insert_pairs_device(t, recs, n), t, "insert");
    const char* text = nullptr;
    const uint64_t* offs = nullptr;
    uint64_t nc = 0, bytes = 0, nodes = 0;
    must(kh_assemble(t, &text, &offs, &nc, &bytes, &nodes), t, "assemble");
    const auto t3 = std::chrono::high_resolution_clock::now();
    const std::string dat = out_name + "_0.dat";
    FILE* o = fopen(dat.c_str(), "wb");
    if (o == nullptr) throw std::runtime_error("kmer_count: could not open " + dat);
    if (bytes && fwrite(text, 1, bytes, o) != bytes) throw std::runtime_error("kmer_count: short write to " + dat);
    fclose(o);
    printf("Assembled %llu k-mers into %llu contigs with %llu nodes in %lf s; wrote %s\n", (unsigned long long)n,
           (unsigned long long)nc, (unsigned long long)nodes, std::chrono::duration<double>(t3 - t2).count(), dat.c_str());
    kh_destroy(t);
    return 0;
}
