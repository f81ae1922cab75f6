// Host-only run of kc_depth_kernel (cs267_hw3_b200/csrc/count.cu) built from the functions of count_core.cuh (nvcc, runs
// without a GPU): the reads are counted serially as kc_count_kernel counts them, then the depth kernel's loops run block
// by block -- the tile pack and list, the block's contig range and each position's search inside it, the window's end
// check, the owner filter, the read-only lookup -- and its warp reduction lane group by lane group (the lanes of a warp
// grouped by contig, one update per group).  tests/test_contig_depth.py compares the records with a numpy restatement.
//
//   depth_host_check K n_slots world reads_file text_file offsets_file
// (offsets_file: n_contigs + 1 little-endian uint64 offsets into the text) prints one line per contig:
//   n_kmers sum min max  n_kmers sum min max
// first the world = 1 record, then the partials of ranks 0..world-1 combined with kh::combine_depth.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "../../cs267_hw3_b200/csrc/count_core.cuh"
#include "../../include/kh/kmer_counter.hpp"

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

// kc_depth_kernel, serially: seg = the text at p_begin, span bytes of it
template <int W>
static void depth(const unsigned char* seg, u64 span, u64 p_begin, const u64* offsets, u64 n, const u64* table, u64 n_slots, int k,
                  u32 world, u32 rank, kh_contig_depth* out) {
    for (u64 i = 0; i < n; ++i) out[i] = kh_contig_depth{0, 0, kKcDepthNoMin, 0};
    std::vector<u32> s_code(kKcWords), s_inv(kKcWords);
    const u64 blocks = (span + kKcTile - 1) / kKcTile;
    for (u64 block = 0; block < blocks; ++block) {
        const u64 t0 = block * kKcTile;
        const u64 lo = kc_contig_of(offsets, 0, n, p_begin + t0);
        const u64 last = p_begin + (t0 + kKcTile < span ? t0 + kKcTile : span) - 1;
        u64 hi = kc_contig_of(offsets, 0, n, last) + 1;
        if (hi <= lo) hi = lo + 1;
        for (u32 i = 0; i < kKcWords; ++i) kc_pack_word(seg, span, (long long)t0 - 16 + 16ll * (long long)i, s_code[i], s_inv[i]);
        std::vector<unsigned short> list;
        for (int r = 0; r < kKcPer; ++r)
            for (u32 thread = 0; thread < (u32)kKcThreads; ++thread) {
                const u32 local = thread + (u32)r * kKcThreads;
                if (t0 + local < span && kc_kmer_valid(s_inv.data(), local, k)) list.push_back((unsigned short)local);
            }
        const u32 cnt = (u32)list.size();
        for (u32 warp = 0; warp < (u32)kKcThreads / 32; ++warp) {
            for (u32 i0 = 32 * warp; i0 < cnt; i0 += kKcThreads) {
                u64 c[32];
                u32 v[32];
                for (u32 lane = 0; lane < 32; ++lane) {
                    const u32 i = i0 + lane;
                    c[lane] = kKcNoContig;
                    v[lane] = 0;
                    if (i >= cnt) continue;
                    const u32 local = list[i];
                    const u64 p = p_begin + t0 + local;
                    const u64 cc = kc_contig_of(offsets, lo, hi, p);
                    if (!kc_window_in_contig(offsets, cc, p, k)) continue;
                    const KcOcc o = kc_position(s_code.data(), s_inv.data(), local, k);
                    if (world != 1 && kc_owner(o.key_hi, o.key_lo, world) != rank) continue;
                    c[lane] = cc;
                    v[lane] = kc_depth_value<W>(table, n_slots, o.key_hi, o.key_lo);
                }
                // __match_any_sync groups; the group's first lane applies the group's reduction
                for (u32 lead = 0; lead < 32; ++lead) {
                    if (c[lead] == kKcNoContig) continue;
                    bool first = true;
                    for (u32 l = 0; l < lead; ++l) first = first && c[l] != c[lead];
                    if (!first) continue;
                    u64 m = 0, s = 0;
                    u32 mn = kKcDepthNoMin, mx = 0;
                    for (u32 l = lead; l < 32; ++l) {
                        if (c[l] != c[lead]) continue;
                        ++m; s += v[l];
                        mn = v[l] < mn ? v[l] : mn;
                        mx = v[l] > mx ? v[l] : mx;
                    }
                    kh_contig_depth& rec = out[c[lead]];
                    rec.n_kmers += m; rec.sum += s;
                    rec.min = mn < rec.min ? mn : rec.min;
                    rec.max = mx > rec.max ? mx : rec.max;
                }
            }
        }
    }
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
static int run(int k, u64 n_slots, u32 world, const char* reads_file, const char* text_file, const char* offsets_file) {
    const std::vector<unsigned char> reads = slurp(reads_file), text = slurp(text_file), ob = slurp(offsets_file);
    std::vector<u64> offsets(ob.size() / 8);
    if (offsets.empty()) return 2;
    memcpy(offsets.data(), ob.data(), offsets.size() * 8);
    const u64 n = offsets.size() - 1;
    if (offsets[n] > text.size()) return 2;
    std::vector<u64> table(n_slots * KcSlot<W>::kWords, 0ull);
    count_reads<W>(reads.data(), reads.size(), table.data(), n_slots, k);
    // the text range alone, at an address that is not 16-byte aligned unless offsets[0] is: both tile loaders run
    const u64 p_begin = offsets[0], span = offsets[n] > p_begin ? offsets[n] - p_begin : 0;
    std::vector<kh_contig_depth> one(n), all(n, kh_contig_depth{0, 0, kKcDepthNoMin, 0}), part(n);
    depth<W>(text.data() + p_begin, span, p_begin, offsets.data(), n, table.data(), n_slots, k, 1, 0, one.data());
    for (u32 r = 0; r < world; ++r) {
        depth<W>(text.data() + p_begin, span, p_begin, offsets.data(), n, table.data(), n_slots, k, world, r, part.data());
        for (u64 i = 0; i < n; ++i) combine_depth(all[i], part[i]);
    }
    for (u64 i = 0; i < n; ++i)
        printf("%llu %llu %u %u %llu %llu %u %u\n", (unsigned long long)one[i].n_kmers, (unsigned long long)one[i].sum, one[i].min,
               one[i].max, (unsigned long long)all[i].n_kmers, (unsigned long long)all[i].sum, all[i].min, all[i].max);
    return 0;
}

int main(int argc, char** argv) {
    if (argc != 7) { fprintf(stderr, "usage: depth_host_check K n_slots world reads_file text_file offsets_file\n"); return 2; }
    const int k = atoi(argv[1]);
    const u64 n_slots = strtoull(argv[2], nullptr, 10);
    const u32 world = (u32)atoi(argv[3]);
    if (k < 2 || k > 61 || world < 1 || world > kKcMaxWorld) return 2;
    return kc_slot_words(k) == 1 ? run<1>(k, n_slots, world, argv[4], argv[5], argv[6]) : run<2>(k, n_slots, world, argv[4], argv[5], argv[6]);
}
