// kmer_counter.hpp -- the k-mer analysis stage (kh_count_* in kh_capi.h) for C++ callers: reads in, the reference's
// kmer_pair records (or its k-mer file) out.  This is the stage README.md:19-21 assumes done before the homework starts;
// its output is what read_kmers (read_kmers.hpp:54-79) returns, so `kh::KmerCounter::extract()` can stand in for
// `read_kmers(file)` in kmer_hash.cpp:122 when the input is reads instead of a k-mer file.
//
// Also here: `kh::sequence_lines`, which blanks everything but the sequence lines of FASTA / FASTQ text (header and
// quality lines contain letters that would read as bases).
#pragma once

#include <array>
#include <cstdint>
#include <stdexcept>
#include <string>
#include <vector>

#include "../kh_capi.h"
#include "record_line.hpp"

namespace kh {

// n kmer_pair records -> the reference's k-mer file text (K + 4 bytes per record, kc_record_to_line)
inline std::string pair_lines(const unsigned char* recs, uint64_t n, int k) {
    const uint64_t pb = kh_pair_bytes(k), ll = (uint64_t)k + 4;
    std::string out(n * ll, '\0');
    for (uint64_t i = 0; i < n; ++i) kc_record_to_line(recs + i * pb, k, reinterpret_cast<unsigned char*>(&out[i * ll]));
    return out;
}

// Contig depth partials of disjoint window sets (one per owner of a sharded counter) -> the record over all of them
inline void combine_depth(kh_contig_depth& into, const kh_contig_depth& part) {
    into.n_kmers += part.n_kmers;
    into.sum += part.sum;
    into.min = part.min < into.min ? part.min : into.min;
    into.max = part.max > into.max ? part.max : into.max;
}

class KmerCounter {
    kh_counter* c_ = nullptr;
    int k_;

    void check(int status, const char* what) const {
        if (status == KH_OK) return;
        const char* detail = c_ ? kh_count_last_error(c_) : "";
        throw std::runtime_error(std::string(detail && *detail ? detail : kh_status_string(status)) + " [" + what + "]");
    }

  public:
    // n_distinct_expected counts every distinct k-mer of the reads (erroneous ones too).  count_reads doubles the table
    // when it runs short (kh_count_create), so a good estimate only saves the rehashes.
    KmerCounter(int k, uint64_t n_distinct_expected, double load_factor = 0.5, int device = 0) : k_(k) {
        if (kh_device_count() <= 0) throw std::runtime_error("KmerCounter: no CUDA device (libkh_b200 has no CPU fallback)");
        check(kh_count_create(k, n_distinct_expected, load_factor, device, &c_), "kh_count_create");
    }
    ~KmerCounter() { kh_count_destroy(c_); }
    KmerCounter(const KmerCounter&) = delete;
    KmerCounter& operator=(const KmerCounter&) = delete;

    int k() const { return k_; }
    void clear() { check(kh_count_clear(c_), "clear"); }
    // any byte outside ACGT separates reads; the buffer begins and ends at a read boundary; may be called repeatedly
    void count_reads(const char* reads, uint64_t n_bytes) { check(kh_count_reads(c_, reads, n_bytes), "count_reads"); }
    void count_reads(const std::string& reads) { count_reads(reads.data(), reads.size()); }

    // the reported k-mers as kmer_pair bytes (kh_pair_bytes(k) each), in table order
    std::vector<unsigned char> extract(uint32_t min_count = 2, uint32_t min_ext = 2) {
        uint64_t n = 0;
        check(kh_count_extract(c_, min_count, min_ext, nullptr, 0, &n), "extract");
        std::vector<unsigned char> out(n * kh_pair_bytes(k_));
        check(kh_count_extract(c_, min_count, min_ext, out.data(), n, &n), "extract");
        return out;
    }
    // the same as lines of the reference's k-mer file (K + 4 bytes each)
    std::string extract_lines(uint32_t min_count = 2, uint32_t min_ext = 2) {
        uint64_t n = 0;
        check(kh_count_extract_lines(c_, min_count, min_ext, nullptr, 0, &n), "extract_lines");
        std::string out(n * (uint64_t)(k_ + 4), '\0');
        check(kh_count_extract_lines(c_, min_count, min_ext, &out[0], n, &n), "extract_lines");
        return out;
    }
    // records stay in device memory (owned by the counter): hand the pointer to kh_insert_pairs_device
    const void* extract_device(uint32_t min_count, uint32_t min_ext, uint64_t& n) {
        const void* p = nullptr;
        check(kh_count_extract_device(c_, min_count, min_ext, &p, &n), "extract_device");
        return p;
    }
    // the k-mer spectrum: [c] = distinct k-mers seen exactly c times, [255] = 255 times or more (kh_count_histogram);
    // kh_count_auto_min_count(h.data()) picks min_count at its valley
    std::array<uint64_t, 256> histogram() {
        std::array<uint64_t, 256> h{};
        check(kh_count_histogram(c_, h.data()), "histogram");
        return h;
    }
    // per contig [offsets[i], offsets[i+1]) of text: its k-mers' occurrence counts, kh_count_contig_depth (world 1)
    std::vector<kh_contig_depth> contig_depth(const char* text, const uint64_t* offsets, uint64_t n) {
        std::vector<kh_contig_depth> out(n);
        check(kh_count_contig_depth(c_, text, offsets, n, 1, 0, out.data()), "contig_depth");
        return out;
    }
    // unitig extensions (kh_count_link_check*): extensions whose neighbour does not name the k-mer back become 'F';
    // returns the sides cut.  Host records in place, or device records (any device; out may be in).
    uint64_t link_check(std::vector<unsigned char>& pairs, uint32_t min_count = 2, uint32_t min_ext = 2, uint32_t world = 1, uint32_t rank = 0) {
        uint64_t n_cut = 0;
        check(kh_count_link_check(c_, pairs.data(), pairs.size() / kh_pair_bytes(k_), min_count, min_ext, world, rank, &n_cut), "link_check");
        return n_cut;
    }
    uint64_t link_check_device(const void* in, void* out, uint64_t n, uint32_t min_count = 2, uint32_t min_ext = 2, uint32_t world = 1,
                               uint32_t rank = 0) {
        uint64_t n_cut = 0;
        check(kh_count_link_check_device(c_, in, out, n, min_count, min_ext, world, rank, &n_cut), "link_check_device");
        return n_cut;
    }
    kh_count_stats stats() {
        kh_count_stats s{};
        check(kh_count_get_stats(c_, &s), "stats");
        return s;
    }
    kh_counter* handle() { return c_; }
};

// FASTA ('>' headers, sequences possibly wrapped over several lines) / FASTQ ('@' header, sequence, '+', quality) /
// plain (one read per line) text, in place: what is not sequence must not reach the counter (header and quality lines
// contain letters that would read as bases), and the lines of one FASTA record are joined (a line break would cut the
// k-mers that span it).  n is updated to the new length (FASTA text shrinks).  A piece must end on a line boundary --
// for FASTA before a header line, see sequence_cut -- and `state` carries the FASTQ line phase from piece to piece
// (start with 0).  format 0 = detect from the first byte.  Returns the format: 'a', 'q' or 'p'.
inline char sequence_lines(char* text, size_t& n, char format, unsigned& state) {
    if (format == 0) format = n && text[0] == '>' ? 'a' : (n && text[0] == '@' ? 'q' : 'p');
    if (format == 'p') return format;
    size_t i = 0, w = 0;
    while (i < n) {
        size_t e = i;
        while (e < n && text[e] != '\n') ++e;
        if (format == 'a') {
            if (text[i] == '>' || text[i] == ';') text[w++] = '\n';          // the record before this header ends here
            else for (size_t j = i; j < e; ++j) text[w++] = text[j];          // joined to the previous sequence line
        } else {
            const bool keep = (state & 3u) == 1u;                             // FASTQ: line 1 of every 4 (0-based) is the sequence
            ++state;
            if (!keep) for (size_t j = i; j < e; ++j) text[j] = '\n';
        }
        i = e + 1;
    }
    if (format == 'a') { if (w < n) text[w++] = '\n'; n = w; }
    return format;
}
// Where a piece of `have` bytes may end so that the next piece starts a new read: after the last line break -- for
// FASTA ('a') after the last line break that is followed by a header.  0 = no such place in this piece (read more).
inline size_t sequence_cut(const char* text, size_t have, char format) {
    size_t cut = have;
    if (format == 'a') {
        while (cut > 1 && !(text[cut - 1] == '\n' && cut < have && text[cut] == '>')) --cut;
        return cut > 1 ? cut : 0;
    }
    while (cut > 0 && text[cut - 1] != '\n') --cut;
    return cut;
}

}  // namespace kh
