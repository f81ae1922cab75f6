// Host-only run of the sharded-counting functions in cs267_hw3_b200/csrc/count_core.cuh (built with nvcc, runs without a
// GPU): kc_count_kernel's loops count every rank's piece of the reads into its own table, the table is partitioned by
// owner rank (kc_slot_owner, kc_partition_kernel's grouping, serially) and every group merged into its owner's table with
// kc_merge_slot -- batch after batch into the same owner tables.  tests/test_count_sharded.py compares with the oracle.
//
//   count_merge_host_check merge K world batches n_slots min_count min_ext reads_file
//     the reads are cut into `batches` parts and every part into `world` pieces with kh_sharded::split_reads; prints
//     "n_occurrences sum_owned_distinct n_reported errors max_local_occurrences max_local_observation", then per reported
//     k-mer: rank record(hex) occurrences backA..T fwdA..T
//   count_merge_host_check spread world n_slots n_keys
//     the home slots (kc_home over n_slots) of the random keys rank 0 owns, counted in `world` equal ranges of the table
//   count_merge_host_check add a b
//     kc_add(a, b)
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "../../cs267_hw3_b200/csrc/count_core.cuh"
#include "../../include/kh/sharded_counter.hpp"

using namespace kh;

template <int W>
static void count_piece(const unsigned char* buf, u64 n, u64* table, u64 n_slots, int k, KcCounters& ctr) {
    std::vector<u32> s_code(kKcWords), s_inv(kKcWords);
    for (u64 t0 = 0; t0 < n; t0 += kKcTile) {
        for (u32 i = 0; i < kKcWords; ++i) kc_pack_word(buf, n, (long long)t0 - 16 + 16ll * (long long)i, s_code[i], s_inv[i]);
        for (u32 local = 0; local < kKcTile && t0 + local < n; ++local) {
            if (!kc_kmer_valid(s_inv.data(), local, k)) continue;
            const KcOcc o = kc_position(s_code.data(), s_inv.data(), local, k);
            bool f;
            if (!kc_upsert<W>(table, n_slots, o, kc_home(o.key_hi, o.key_lo, n_slots), f)) { ctr.errors |= kKcErrFull; continue; }
            ++ctr.n_occurrences;
            ctr.n_distinct += f ? 1 : 0;
        }
    }
}

template <int W>
static int merge(int k, u32 world, int batches, u64 n_slots, u32 min_count, u32 min_ext, const std::vector<char>& reads) {
    constexpr int S = KcSlot<W>::kWords;
    std::vector<std::vector<u64>> owned(world, std::vector<u64>(n_slots * S, 0ull));
    std::vector<KcCounters> octr(world, KcCounters{});
    u64 n_occ = 0;
    u32 errors = 0, max_total = 0, max_obs = 0;
    const std::vector<size_t> bcut = kh_sharded::split_reads(reads.data(), reads.size(), batches);
    for (int b = 0; b < batches; ++b) {
        const char* part = reads.data() + bcut[b];
        const size_t part_n = bcut[b + 1] - bcut[b];
        const std::vector<size_t> cut = kh_sharded::split_reads(part, part_n, (int)world);
        // count: one batch table per rank
        std::vector<std::vector<u64>> batch(world, std::vector<u64>(n_slots * S, 0ull));
        for (u32 r = 0; r < world; ++r) {
            KcCounters c = {};
            count_piece<W>(reinterpret_cast<const unsigned char*>(part + cut[r]), cut[r + 1] - cut[r], batch[r].data(), n_slots, k, c);
            n_occ += c.n_occurrences;
            errors |= c.errors;
            for (u64 i = 0; i < n_slots; ++i) {
                const u64* p = batch[r].data() + i * S;
                const u64 q[4] = {p[0], p[1], 0ull, 0ull};
                if (kc_slot_empty<W>(q)) continue;
                const u64 w = p[W == 1 ? 1 : 2];
                max_total = std::max(max_total, kc_total(w));
                for (u32 x = 0; x < 4; ++x) max_obs = std::max(max_obs, std::max(kc_back_count(w, x), kc_fwd_count(w, x)));
            }
        }
        // partition: every rank's slots grouped by owner; then every owner merges its group from every rank
        for (u32 r = 0; r < world; ++r) {
            std::vector<std::vector<u64>> outbox(world);
            for (u64 i = 0; i < n_slots; ++i) {
                const u32 o = kc_slot_owner<W>(batch[r].data(), i, world);
                if (o < world) outbox[o].insert(outbox[o].end(), batch[r].data() + i * S, batch[r].data() + (i + 1) * S);
            }
            for (u32 o = 0; o < world; ++o) {
                for (size_t j = 0; j < outbox[o].size(); j += S) {
                    bool f;
                    if (!kc_merge_slot<W>(owned[o].data(), n_slots, outbox[o].data() + j, f)) { errors |= kKcErrFull; continue; }
                    octr[o].n_distinct += f ? 1 : 0;
                }
            }
        }
    }
    u64 n_distinct = 0, n_rep = 0;
    std::string body;
    const int pb = (k + 3) / 4 + 2;
    char tmp[64];
    for (u32 o = 0; o < world; ++o) {
        n_distinct += octr[o].n_distinct;
        for (u64 i = 0; i < n_slots; ++i) {
            if (!kc_slot_reported<W>(owned[o].data(), i, min_count)) continue;
            unsigned char rec[18];
            kc_slot_record<W>(owned[o].data(), i, k, min_ext, rec);
            ++n_rep;
            snprintf(tmp, sizeof tmp, "%u ", o);
            body += tmp;
            for (int j = 0; j < pb; ++j) { snprintf(tmp, sizeof tmp, "%02x", rec[j]); body += tmp; }
            const u64 c = owned[o][i * S + (W == 1 ? 1 : 2)];
            snprintf(tmp, sizeof tmp, " %u", kc_total(c));
            body += tmp;
            for (u32 x = 0; x < 4; ++x) { snprintf(tmp, sizeof tmp, " %u", kc_back_count(c, x)); body += tmp; }
            for (u32 x = 0; x < 4; ++x) { snprintf(tmp, sizeof tmp, " %u", kc_fwd_count(c, x)); body += tmp; }
            body += '\n';
        }
    }
    printf("%llu %llu %llu %u %u %u\n", n_occ, n_distinct, n_rep, errors, max_total, max_obs);
    fwrite(body.data(), 1, body.size(), stdout);
    return 0;
}

static u64 splitmix(u64& s) {
    u64 z = (s += 0x9E3779B97F4A7C15ull);
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}

int main(int argc, char** argv) {
    const std::string mode = argc > 1 ? argv[1] : "";
    if (mode == "add" && argc == 4) {
        printf("%llu\n", kc_add(strtoull(argv[2], nullptr, 10), strtoull(argv[3], nullptr, 10)));
        return 0;
    }
    if (mode == "spread" && argc == 5) {
        const u32 world = (u32)atoi(argv[2]);
        const u64 n_slots = strtoull(argv[3], nullptr, 10), n_keys = strtoull(argv[4], nullptr, 10);
        std::vector<u64> hist(world, 0);
        u64 s = 267;
        for (u64 i = 0; i < n_keys; ++i) {
            const u64 lo = splitmix(s) >> 2, hi = (i & 1) ? splitmix(s) >> 10 : 0ull;     // 31-mers and 59-mers
            if (kc_owner(hi, lo, world) != 0) continue;
            ++hist[kc_home(hi, lo, n_slots) * world / n_slots];
        }
        for (u32 o = 0; o < world; ++o) printf("%llu%c", hist[o], o + 1 == world ? '\n' : ' ');
        return 0;
    }
    if (mode == "merge" && argc == 9) {
        const int k = atoi(argv[2]);
        const u32 world = (u32)atoi(argv[3]);
        const int batches = atoi(argv[4]);
        const u64 n_slots = strtoull(argv[5], nullptr, 10);
        const u32 min_count = (u32)atoi(argv[6]), min_ext = (u32)atoi(argv[7]);
        FILE* f = fopen(argv[8], "rb");
        if (!f) return 2;
        fseek(f, 0, SEEK_END);
        const long n = ftell(f);
        fseek(f, 0, SEEK_SET);
        std::vector<char> reads((size_t)n);
        if (fread(reads.data(), 1, (size_t)n, f) != (size_t)n) return 2;
        fclose(f);
        return kc_slot_words(k) == 1 ? merge<1>(k, world, batches, n_slots, min_count, min_ext, reads)
                                     : merge<2>(k, world, batches, n_slots, min_count, min_ext, reads);
    }
    fprintf(stderr, "usage: count_merge_host_check (merge K world batches n_slots min_count min_ext reads_file | spread world n_slots n_keys | add a b)\n");
    return 2;
}
