// kh/sharded_counter.hpp -- k-mer analysis (kh_count_*) over several ranks (GPUs) in ONE host process, over the C ABI.
//
// Counting the reads on P GPUs and extracting on each alone is wrong: a k-mer seen once on each of two GPUs has count 2,
// and min_count / min_ext only mean something for the global counts.  So every rank keeps two counters:
//   batch  -- counts this rank's reads (kh_count_reads*, unchanged);
//   owned  -- holds the k-mers this rank OWNS (kh_count_partition's owner rank), merged from every rank's batch.
// reduce() partitions every batch by owner, every owner merges the group addressed to it from every rank (records cross
// between GPUs with one peer copy each), and the batches are cleared.  Count / reduce may alternate: batches bound the
// batch tables' memory, the owned tables hold ~1/P of the distinct k-mers each.  Saturating counters add exactly
// (kh_capi.h), so the union of the owned extracts is, record for record, what one counter over all reads reports --
// provided each rank's reads begin and end at a non-base byte (split_reads) and nothing is dropped before the reduce.
//
// Every step is host-synchronous (no in-stream barriers), so ranks that share a device simply run in turn; ranks with
// a device of their own run on one host thread each.  Rank r lives on device r % (visible devices), as in Cluster
// (sharded_host.hpp), so the owned records can go straight into a kh_sharded::Cluster of the same world.
#pragma once

#include <algorithm>
#include <array>
#include <cstdint>
#include <exception>
#include <memory>
#include <mutex>
#include <stdexcept>
#include <string>
#include <thread>
#include <vector>

#include "../kh_capi.h"
#include "kmer_counter.hpp"

namespace kh_sharded {

inline void count_must(int status, kh_counter* c, const char* what) {
    if (status == KH_OK) return;
    const char* detail = c ? kh_count_last_error(c) : "";
    throw std::runtime_error(std::string(detail && *detail ? detail : kh_status_string(status)) + " [" + what + "]");
}

// world + 1 cut points that split text[0, n) into world pieces of about n / world bytes each.  A cut lies at 0, at n or
// right behind a byte that is not a base, so no k-mer and no extension observation spans two pieces.
inline std::vector<size_t> split_reads(const char* text, size_t n, int world) {
    auto is_base = [](char ch) { return ch == 'A' || ch == 'C' || ch == 'G' || ch == 'T'; };
    std::vector<size_t> cut(world + 1, n);
    cut[0] = 0;
    for (int r = 1; r < world; ++r) {
        size_t c = std::max(cut[r - 1], (size_t)((unsigned __int128)n * r / world));
        while (c < n && c > 0 && is_base(text[c - 1])) ++c;
        cut[r] = c;
    }
    return cut;
}

class CountCluster {
    int k_, world_;
    bool in_turn_ = false;
    std::vector<kh_counter*> batch_, owned_;
    std::vector<int> dev_;
    std::vector<uint64_t> occ_, bytes_;           // per rank: what earlier batches counted (before their clear)
    std::vector<void*> unitigs_;                   // per rank: extract_unitigs_device's records, on device(rank)
    std::vector<uint64_t> unitigs_cap_;
    std::unique_ptr<std::mutex[]> owner_lock_;     // extract_unitigs*: one call at a time on each owned counter

    template <class F> void each_rank(F fn) {
        if (in_turn_ || world_ == 1) {
            for (int r = 0; r < world_; ++r) fn(r);
            return;
        }
        std::vector<std::exception_ptr> err(world_);
        std::vector<std::thread> th;
        for (int r = 0; r < world_; ++r)
            th.emplace_back([&, r] { try { fn(r); } catch (...) { err[r] = std::current_exception(); } });
        for (auto& x : th) x.join();
        for (auto& e : err) if (e) std::rethrow_exception(e);
    }
    kh_count_stats stats_of(kh_counter* c) {
        kh_count_stats s{};
        count_must(kh_count_get_stats(c, &s), c, "stats");
        return s;
    }

  public:
    // n_distinct_expected_total: distinct k-mers of all reads (erroneous ones included); both tables grow when short.
    // A batch table is sized for all of them (one rank's reads may hold nearly every k-mer), an owned table for its share.
    CountCluster(int k, int world, uint64_t n_distinct_expected_total, double load_factor = 0.5)
        : k_(k), world_(world), batch_(world, nullptr), owned_(world, nullptr), dev_(world, 0), occ_(world, 0), bytes_(world, 0),
          unitigs_(world, nullptr), unitigs_cap_(world, 0), owner_lock_(new std::mutex[world]) {
        const int ndev = kh_device_count();
        if (ndev <= 0) throw std::runtime_error("CountCluster: no CUDA device (libkh_b200 has no CPU fallback)");
        if (world < 1 || world > 64) throw std::runtime_error("CountCluster: world must be between 1 and 64");
        in_turn_ = world > ndev;
        const uint64_t share = n_distinct_expected_total / world + n_distinct_expected_total / (8 * (uint64_t)world) + 4096;
        try {
            for (int r = 0; r < world; ++r) {
                dev_[r] = r % ndev;
                count_must(kh_count_create(k, n_distinct_expected_total, load_factor, dev_[r], &batch_[r]), nullptr, "kh_count_create");
                count_must(kh_count_create(k, share, load_factor, dev_[r], &owned_[r]), nullptr, "kh_count_create");
            }
        } catch (...) {
            for (int r = 0; r < world; ++r) { kh_count_destroy(batch_[r]); kh_count_destroy(owned_[r]); }
            throw;
        }
    }
    ~CountCluster() {
        for (int r = 0; r < world_; ++r) { kh_count_destroy(batch_[r]); kh_count_destroy(owned_[r]); kh_device_free(unitigs_[r]); }
    }
    CountCluster(const CountCluster&) = delete;
    CountCluster& operator=(const CountCluster&) = delete;

    int world() const { return world_; }
    int device(int rank) const { return dev_[rank]; }
    kh_counter* owned(int rank) { return owned_[rank]; }

    // rank's reads (begin and end at a non-base byte): host memory, or device memory on device(rank) (only enqueued;
    // must stay valid until the next reduce)
    void count(int rank, const char* reads_host, uint64_t n) { count_must(kh_count_reads(batch_[rank], reads_host, n), batch_[rank], "count"); }
    void count_device(int rank, const char* reads_dev, uint64_t n) {
        count_must(kh_count_reads_device(batch_[rank], reads_dev, n), batch_[rank], "count_device");
    }
    // read bytes counted on this rank since the last reduce
    uint64_t batch_bytes(int rank) { return stats_of(batch_[rank]).n_bytes; }

    // every rank's batch into the owners' tables, then the batches are cleared
    void reduce() {
        std::vector<const unsigned char*> recs(world_, nullptr);
        std::vector<std::vector<uint64_t>> offs(world_, std::vector<uint64_t>(world_ + 1, 0));
        const uint64_t rb = kh_count_record_bytes(k_);
        each_rank([&](int r) {
            const void* p = nullptr;
            count_must(kh_count_partition(batch_[r], world_, &p, offs[r].data()), batch_[r], "partition");
            recs[r] = static_cast<const unsigned char*>(p);
        });
        each_rank([&](int o) {
            for (int i = 0; i < world_; ++i) {
                const int r = (o + i) % world_;                // owners start at different sources
                const uint64_t n = offs[r][o + 1] - offs[r][o];
                if (n) count_must(kh_count_merge_device(owned_[o], recs[r] + offs[r][o] * rb, n), owned_[o], "merge");
            }
        });
        each_rank([&](int r) {
            const kh_count_stats s = stats_of(batch_[r]);
            occ_[r] += s.n_occurrences;
            bytes_[r] += s.n_bytes;
            count_must(kh_count_clear(batch_[r]), batch_[r], "clear");
        });
    }

    // After reduce(): the k-mers rank `rank` owns, as with kh::KmerCounter (records stay on device(rank), owned by the
    // counter until its next extract)
    const void* extract_device(int rank, uint32_t min_count, uint32_t min_ext, uint64_t& n) {
        const void* p = nullptr;
        count_must(kh_count_extract_device(owned_[rank], min_count, min_ext, &p, &n), owned_[rank], "extract_device");
        return p;
    }
    std::string extract_lines(int rank, uint32_t min_count = 2, uint32_t min_ext = 2) {
        uint64_t n = 0;
        count_must(kh_count_extract_lines(owned_[rank], min_count, min_ext, nullptr, 0, &n), owned_[rank], "extract_lines");
        std::string out(n * (uint64_t)(k_ + 4), '\0');
        count_must(kh_count_extract_lines(owned_[rank], min_count, min_ext, &out[0], n, &n), owned_[rank], "extract_lines");
        return out;
    }

    // After reduce(): rank's records with unitig extensions (kh_count_link_check*) -- rank's extract, checked by every
    // owner for the sides whose neighbour it owns; the partials apply in any order and give the one-counter records.
    // The device form leaves them in a buffer the cluster owns on device(rank), valid until the next call for this rank;
    // the owners start at `rank` and go round, and the records cross devices 2 (P - 1) times (in and back for every other
    // owner).  Calls for different ranks may run concurrently (each owner checks one rank's records at a time, and rotated
    // starts keep them apart); calls for the same rank must not overlap.  n_cut: the sides turned to 'F'.
    const void* extract_unitigs_device(int rank, uint32_t min_count, uint32_t min_ext, uint64_t& n, uint64_t& n_cut) {
        n_cut = 0;
        const void* p = nullptr;
        {
            std::lock_guard<std::mutex> g(owner_lock_[rank]);
            count_must(kh_count_extract_device(owned_[rank], min_count, min_ext, &p, &n), owned_[rank], "extract_unitigs");
            const uint64_t bytes = n * kh_pair_bytes(k_);
            if (bytes > unitigs_cap_[rank]) {
                kh_device_free(unitigs_[rank]);
                unitigs_[rank] = nullptr;
                unitigs_cap_[rank] = 0;
                count_must(kh_device_alloc_on(dev_[rank], &unitigs_[rank], bytes), nullptr, "extract_unitigs: device buffer");
                unitigs_cap_[rank] = bytes;
            }
            // the owner on rank's device checks first and moves the records out of its extract buffer as it goes
            uint64_t cut = 0;
            count_must(kh_count_link_check_device(owned_[rank], p, unitigs_[rank], n, min_count, min_ext, (uint32_t)world_, (uint32_t)rank, &cut),
                       owned_[rank], "extract_unitigs");
            n_cut += cut;
        }
        for (int i = 1; i < world_; ++i) {
            const int o = (rank + i) % world_;
            std::lock_guard<std::mutex> g(owner_lock_[o]);
            uint64_t cut = 0;
            count_must(kh_count_link_check_device(owned_[o], unitigs_[rank], unitigs_[rank], n, min_count, min_ext, (uint32_t)world_, (uint32_t)o, &cut),
                       owned_[o], "extract_unitigs");
            n_cut += cut;
        }
        return unitigs_[rank];
    }
    // the same records in host memory (kh_count_link_check per owner)
    std::vector<unsigned char> extract_unitigs(int rank, uint32_t min_count, uint32_t min_ext, uint64_t& n_cut) {
        n_cut = 0;
        std::vector<unsigned char> recs;
        uint64_t n = 0;
        {
            std::lock_guard<std::mutex> g(owner_lock_[rank]);
            count_must(kh_count_extract(owned_[rank], min_count, min_ext, nullptr, 0, &n), owned_[rank], "extract_unitigs");
            recs.resize(n * kh_pair_bytes(k_));
            count_must(kh_count_extract(owned_[rank], min_count, min_ext, recs.data(), n, &n), owned_[rank], "extract_unitigs");
        }
        for (int i = 0; i < world_; ++i) {
            const int o = (rank + i) % world_;
            std::lock_guard<std::mutex> g(owner_lock_[o]);
            uint64_t cut = 0;
            count_must(kh_count_link_check(owned_[o], recs.data(), n, min_count, min_ext, (uint32_t)world_, (uint32_t)o, &cut), owned_[o],
                       "extract_unitigs");
            n_cut += cut;
        }
        return recs;
    }

    // After reduce(): the k-mer spectrum of everything reduced so far (kh_count_histogram).  Every k-mer has exactly one
    // owner and the owned counters are bit-identical to one counter's, so the bin-by-bin sum of the owners' spectra is
    // exact.  Reads counted since the last reduce are not in it.
    std::array<uint64_t, 256> histogram() {
        std::array<uint64_t, 256> sum{};
        for (int r = 0; r < world_; ++r) {
            std::array<uint64_t, 256> h{};
            count_must(kh_count_histogram(owned_[r], h.data()), owned_[r], "histogram");
            for (size_t c = 0; c < h.size(); ++c) sum[c] += h[c];
        }
        return sum;
    }

    // After reduce(): the depth of contigs [offsets[i], offsets[i+1]) of host text against everything reduced so far.
    // Every owner looks up the windows whose k-mer it owns (kh_count_contig_depth with world, rank = owner); every
    // k-mer has exactly one owner, so the partials combine into exactly one counter's records.
    std::vector<kh_contig_depth> contig_depth(const char* text, const uint64_t* offsets, uint64_t n) {
        std::vector<std::vector<kh_contig_depth>> part(world_, std::vector<kh_contig_depth>(n));
        each_rank([&](int o) {
            count_must(kh_count_contig_depth(owned_[o], text, offsets, n, (uint32_t)world_, (uint32_t)o, part[o].data()), owned_[o],
                       "contig_depth");
        });
        std::vector<kh_contig_depth> out(n, kh_contig_depth{0, 0, UINT32_MAX, 0});
        for (int o = 0; o < world_; ++o)
            for (uint64_t i = 0; i < n; ++i) kh::combine_depth(out[i], part[o][i]);
        return out;
    }

    // totals over all ranks: occurrences and read bytes counted (reduced or not), distinct k-mers reduced so far
    uint64_t n_occurrences() {
        uint64_t s = 0;
        for (int r = 0; r < world_; ++r) s += occ_[r] + stats_of(batch_[r]).n_occurrences;
        return s;
    }
    uint64_t n_bytes() {
        uint64_t s = 0;
        for (int r = 0; r < world_; ++r) s += bytes_[r] + stats_of(batch_[r]).n_bytes;
        return s;
    }
    uint64_t n_distinct() {
        uint64_t s = 0;
        for (int r = 0; r < world_; ++r) s += stats_of(owned_[r]).n_distinct;
        return s;
    }
};

}  // namespace kh_sharded
