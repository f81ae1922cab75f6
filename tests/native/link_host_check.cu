// Host-only run of kc_link_kernel's per-record logic (cs267_hw3_b200/csrc/count.cu) built from the functions of
// count_core.cuh (nvcc, runs without a GPU): the reads are counted serially as kc_count_kernel counts them, the reported
// records are taken from the table as kc_extract_kernel takes them, and every record then goes through kc_link_plan,
// kc_find_pair and kc_link_apply -- once with world = 1, and as the partials of owners 0..world-1 applied one after
// another in forward and in reverse owner order.  tests/test_unitigs.py compares the output with a numpy restatement.
//
//   link_host_check K n_slots min_count min_ext world reads_file
// prints the world = 1 records as k-mer file lines, then one line
//   n_cut n_cut_forward n_cut_reverse same_forward same_reverse
// (same_*: 1 when the partials applied in that order gave the world = 1 records byte for byte).
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "../../cs267_hw3_b200/csrc/count_core.cuh"

using namespace kh;

template <int W>
static void count_reads(const unsigned char* buf, u64 n, u64* table, u64 n_slots, int k) {
    std::vector<u32> s_code(kKcWords), s_inv(kKcWords);
    for (u64 t0 = 0; t0 < n; t0 += kKcTile) {
        for (u32 i = 0; i < kKcWords; ++i) kc_pack_word(buf, n, (long long)t0 - 16 + 16ll * (long long)i, s_code[i], s_inv[i]);
        for (u32 local = 0; local < kKcTile; ++local) {
            if (t0 + local >= n || !kc_kmer_valid(s_inv.data(), local, k)) continue;
            const KcOcc o = kc_position(s_code.data(), s_inv.data(), local, k);
            bool f;
            if (!kc_upsert<W>(table, n_slots, o, kc_home(o.key_hi, o.key_lo, n_slots), f)) { fprintf(stderr, "table full\n"); exit(3); }
        }
    }
}

// the per-record logic of kc_link_kernel over all records; returns the sides cut
template <int W>
static u64 link(std::vector<unsigned char>& recs, int k, const u64* table, u64 n_slots, u32 min_count, u32 min_ext, u32 world, u32 rank) {
    const int pb = ((k + 3) >> 2) + 2;
    u64 cut = 0;
    for (size_t i = 0; i + pb <= recs.size(); i += pb) {
        const KcLinkPlan p = kc_link_plan(&recs[i], k, world, rank);
        if (p.bad) { fprintf(stderr, "bad record\n"); exit(3); }
        u64 c[2];
        kc_find_pair<W>(table, n_slots, p, c);
        cut += kc_link_apply(p, c, k, min_count, min_ext, &recs[i]);
    }
    return cut;
}

static std::vector<unsigned char> slurp(const char* path) {
    FILE* f = fopen(path, "rb");
    if (!f) exit(2);
    fseek(f, 0, SEEK_END);
    const long n = ftell(f);
    fseek(f, 0, SEEK_SET);
    std::vector<unsigned char> b((size_t)n);
    if (n && fread(b.data(), 1, (size_t)n, f) != (size_t)n) exit(2);
    fclose(f);
    return b;
}

template <int W>
static int run(int k, u64 n_slots, u32 min_count, u32 min_ext, u32 world, const char* reads_file) {
    const std::vector<unsigned char> reads = slurp(reads_file);
    std::vector<u64> table(n_slots * KcSlot<W>::kWords, 0ull);
    count_reads<W>(reads.data(), reads.size(), table.data(), n_slots, k);
    const int pb = ((k + 3) >> 2) + 2;
    std::vector<unsigned char> recs;
    for (u64 i = 0; i < n_slots; ++i) {
        if (!kc_slot_reported<W>(table.data(), i, min_count)) continue;
        unsigned char rec[18];
        kc_slot_record<W>(table.data(), i, k, min_ext, rec);
        recs.insert(recs.end(), rec, rec + pb);
    }
    std::vector<unsigned char> one = recs, fwd = recs, rev = recs;
    const u64 cut = link<W>(one, k, table.data(), n_slots, min_count, min_ext, 1, 0);
    u64 cut_f = 0, cut_r = 0;
    for (u32 r = 0; r < world; ++r) {
        cut_f += link<W>(fwd, k, table.data(), n_slots, min_count, min_ext, world, r);
        cut_r += link<W>(rev, k, table.data(), n_slots, min_count, min_ext, world, world - 1 - r);
    }
    std::vector<unsigned char> line((size_t)k + 4);
    for (size_t i = 0; i < one.size(); i += pb) {
        kc_record_to_line(&one[i], k, line.data());
        fwrite(line.data(), 1, line.size(), stdout);
    }
    printf("%llu %llu %llu %d %d\n", (unsigned long long)cut, (unsigned long long)cut_f, (unsigned long long)cut_r, (int)(fwd == one),
           (int)(rev == one));
    return 0;
}

int main(int argc, char** argv) {
    if (argc != 7) { fprintf(stderr, "usage: link_host_check K n_slots min_count min_ext world reads_file\n"); return 2; }
    const int k = atoi(argv[1]);
    const u64 n_slots = strtoull(argv[2], nullptr, 10);
    const u32 min_count = (u32)atoi(argv[3]), min_ext = (u32)atoi(argv[4]), world = (u32)atoi(argv[5]);
    if (k < 2 || k > 61 || world < 1 || world > kKcMaxWorld) return 2;
    return kc_slot_words(k) == 1 ? run<1>(k, n_slots, min_count, min_ext, world, argv[6]) : run<2>(k, n_slots, min_count, min_ext, world, argv[6]);
}
