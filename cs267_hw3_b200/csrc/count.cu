// count.cu -- k-mer analysis on the GPU (kh_count_* of include/kh_capi.h): reads -> unique k-mers with their
// backward / forward extensions, as kmer_pair records in device memory.  The algorithm and the table format are in
// count_core.cuh; this file holds the three kernels and the host runtime.
//
//   kc_count_kernel    a block packs a tile of 2048 read characters (+ halo) to 2 bits each in shared memory, lists the
//                      positions that hold a k-mer, and its threads cut the k-mers with their two neighbour characters
//                      out of the packed stream (five LDS + funnel shifts each, whatever K is) and count them: one
//                      sector read + one CAS on the counter word
//   kc_extract_kernel  table scan -> kmer_pair records of the k-mers with enough occurrences (block-wise compaction)
//   kc_lookup_kernel   counters of given k-mers
//   kc_histogram_kernel  table scan -> the k-mer spectrum (distinct k-mers per occurrence count)
//   kc_depth_kernel    contig text -> per contig: windows, sum / min / max of their k-mers' occurrences (read-only)
//   kc_link_kernel     kmer_pair records -> the same records with every extension whose neighbour does not name the k-mer
//                      back turned to 'F' (unitig extensions; read-only on the table)
//
// HBM-bound integer work like the rest of the library: what an occurrence costs is one random 32-byte sector (the slot)
// read and written back.  Algorithmic bytes per occurrence = 1 (the character) + 64.
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>

#include "../../include/kh_capi.h"
#include "count_core.cuh"

using namespace kh;

namespace {
constexpr u32 kFull = 0xFFFFFFFFu;
constexpr u64 kKcChunk = 64ull << 20;                       // positions per host chunk (multiple of the tile and of 16)
constexpr u64 kKcHalo = 16 + 64;                            // bytes around a chunk: 16 before (keeps the alignment), 64 behind
constexpr double kKcMaxLoad = 0.9;                          // a launch never takes the table past this load
constexpr u64 kKcMinLaunch = 4ull << 20;                    // grow rather than count in launches smaller than this
}  // namespace

// Pass 1 compacts the tile's positions that hold a k-mer into a list (reads end every ~150 characters and K - 1
// positions before every end hold none: a third of the lanes would idle through the table code otherwise); pass 2 runs
// over the list with full warps (2.22 -> 1.69 ms for 52.7 M occurrences of 51-mers).  A software prefetch of a thread's
// next occurrence one iteration ahead, and 6 instead of 8 blocks per SM for 128-bit keys, were measured with no gain:
// the kernel is issue-bound.
template <int W>
__global__ void __launch_bounds__(kKcThreads, 8)
kc_count_kernel(const unsigned char* __restrict__ buf, u64 n, u64 p_begin, u64 p_end, u64* __restrict__ table, u64 n_slots, int k,
                KcCounters* ctr) {
    __shared__ u32 s_code[kKcWords], s_inv[kKcWords];
    __shared__ unsigned short s_list[kKcTile];
    __shared__ u32 s_n, s_fresh, s_fail;
    const u64 t0 = (p_begin & ~15ull) + (u64)blockIdx.x * kKcTile;
    if (threadIdx.x == 0) { s_n = 0; s_fresh = 0; s_fail = 0; }
    for (u32 i = threadIdx.x; i < kKcWords; i += kKcThreads)
        kc_pack_word(buf, n, (long long)t0 - 16 + 16ll * (long long)i, s_code[i], s_inv[i]);
    __syncthreads();
    const u32 lane = threadIdx.x & 31u;
#pragma unroll
    for (int r = 0; r < kKcPer; ++r) {
        const u32 local = threadIdx.x + (u32)r * kKcThreads;
        const u64 p = t0 + local;
        const bool ok = p >= p_begin && p < p_end && kc_kmer_valid(s_inv, local, k);
        const u32 bal = __ballot_sync(kFull, ok);
        u32 base = 0;
        if (lane == 0 && bal) base = atomicAdd(&s_n, (u32)__popc(bal));
        base = __shfl_sync(kFull, base, 0);
        if (ok) s_list[base + (u32)__popc(bal & ((1u << lane) - 1u))] = (unsigned short)local;
    }
    __syncthreads();
    // a table that has overflowed stays wrong whatever follows: later blocks do not probe it slot by slot any more
    const u32 cnt = *reinterpret_cast<volatile u32*>(&ctr->errors) ? 0u : s_n;
    u32 fresh = 0, fail = 0;
#pragma unroll 1
    for (u32 i = threadIdx.x; i < cnt; i += kKcThreads) {
        const KcOcc o = kc_position(s_code, s_inv, s_list[i], k);
        bool f;
        if (kc_upsert<W>(table, n_slots, o, kc_home(o.key_hi, o.key_lo, n_slots), f)) fresh += f ? 1u : 0u;
        else ++fail;
    }
    __syncwarp();
    fresh = __reduce_add_sync(kFull, fresh);
    fail = __reduce_add_sync(kFull, fail);
    if (lane == 0) {
        if (fresh) atomicAdd(&s_fresh, fresh);
        if (fail) atomicAdd(&s_fail, fail);
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        if (cnt > s_fail) atomicAdd(&ctr->n_occurrences, (u64)(cnt - s_fail));
        if (s_fresh) atomicAdd(&ctr->n_distinct, (u64)s_fresh);
        if (s_fail) atomicOr(&ctr->errors, kKcErrFull);
    }
}

// table growth: every occupied slot of the old table moves to its place in the new one
template <int W>
__global__ void __launch_bounds__(256)
kc_rehash_kernel(const u64* __restrict__ old_table, u64 old_slots, u64* __restrict__ table, u64 n_slots, KcCounters* ctr) {
    const u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < old_slots && !kc_move_slot<W>(old_table, i, table, n_slots)) atomicOr(&ctr->errors, kKcErrFull);
}

constexpr int kKcExtThreads = 256;
constexpr int kKcExtPer = 4;

template <int W>
__global__ void __launch_bounds__(kKcExtThreads)
kc_extract_kernel(const u64* __restrict__ table, u64 n_slots, int k, u32 min_count, u32 min_ext, unsigned char* __restrict__ out, u64 cap,
                  KcCounters* ctr) {
    __shared__ u32 s_warp[kKcExtThreads / 32];
    __shared__ u64 s_base;
    const u64 first = (u64)blockIdx.x * (kKcExtThreads * kKcExtPer);
    const int pb = ((k + 3) >> 2) + 2;
    u32 flags = 0, mine = 0;
#pragma unroll
    for (int r = 0; r < kKcExtPer; ++r) {
        const u64 i = first + (u64)r * kKcExtThreads + threadIdx.x;
        const bool rep = i < n_slots && kc_slot_reported<W>(table, i, min_count);
        flags |= rep ? (1u << r) : 0u;
        mine += rep ? 1u : 0u;
    }
    // exclusive scan of `mine` over the block
    const u32 lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
    u32 incl = mine;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const u32 up = __shfl_up_sync(kFull, incl, d);
        if ((int)lane >= d) incl += up;
    }
    if (lane == 31u) s_warp[warp] = incl;
    __syncthreads();
    if (threadIdx.x == 0) {
        u32 run = 0;
        for (int w = 0; w < kKcExtThreads / 32; ++w) { const u32 c = s_warp[w]; s_warp[w] = run; run += c; }
        s_base = run ? atomicAdd(&ctr->n_reported, (u64)run) : 0ull;
    }
    __syncthreads();
    u64 at = s_base + s_warp[warp] + (incl - mine);
#pragma unroll
    for (int r = 0; r < kKcExtPer; ++r) {
        if (!((flags >> r) & 1u)) continue;
        const u64 i = first + (u64)r * kKcExtThreads + threadIdx.x;
        if (at < cap) {
            unsigned char rec[18];
            kc_slot_record<W>(table, i, k, min_ext, rec);
            unsigned char* dst = out + at * (u64)pb;
            for (int j = 0; j < pb; ++j) dst[j] = rec[j];
        }
        ++at;
    }
}

// Sharded counting, step 1: the occupied slots grouped by owner rank (kc_owner).  Two launches over the table, the same
// block-wise pattern as kc_extract_kernel: a warp aggregates the slots of one owner with __match_any_sync, the block
// collects per-owner counts in shared memory and reserves its run in each owner's segment with ONE global atomicAdd per
// owner.  scatter = false: cursor[o] ends as owner o's slot count (the histogram); scatter = true: cursor[o] starts at
// owner o's segment offset and the slots are copied there verbatim (order within a segment is arbitrary).
template <int W>
__global__ void __launch_bounds__(kKcExtThreads)
kc_partition_kernel(const u64* __restrict__ table, u64 n_slots, u32 world, bool scatter, u64* __restrict__ cursor, u64* __restrict__ out) {
    __shared__ u32 s_cnt[kKcMaxWorld];
    __shared__ u64 s_base[kKcMaxWorld];
    for (u32 o = threadIdx.x; o < world; o += kKcExtThreads) s_cnt[o] = 0;
    __syncthreads();
    const u64 first = (u64)blockIdx.x * (kKcExtThreads * kKcExtPer);
    const u32 lane = threadIdx.x & 31u;
    u32 own[kKcExtPer], at[kKcExtPer];
#pragma unroll
    for (int r = 0; r < kKcExtPer; ++r) {
        const u64 i = first + (u64)r * kKcExtThreads + threadIdx.x;
        own[r] = i < n_slots ? kc_slot_owner<W>(table, i, world) : world;
        const u32 peers = __match_any_sync(kFull, own[r]);
        const u32 leader = (u32)__ffs(peers) - 1u;
        u32 base = 0;
        if (lane == leader && own[r] < world) base = atomicAdd(&s_cnt[own[r]], (u32)__popc(peers));
        at[r] = __shfl_sync(kFull, base, leader) + (u32)__popc(peers & ((1u << lane) - 1u));
    }
    __syncthreads();
    for (u32 o = threadIdx.x; o < world; o += kKcExtThreads)
        if (s_cnt[o]) s_base[o] = atomicAdd(&cursor[o], (u64)s_cnt[o]);
    if (!scatter) return;
    __syncthreads();
#pragma unroll
    for (int r = 0; r < kKcExtPer; ++r) {
        if (own[r] >= world) continue;
        const u64 i = first + (u64)r * kKcExtThreads + threadIdx.x;
        const u64* src = table + i * (u64)KcSlot<W>::kWords;
        u64* dst = out + (s_base[own[r]] + at[r]) * (u64)KcSlot<W>::kWords;
#pragma unroll
        for (int j = 0; j < KcSlot<W>::kWords; ++j) dst[j] = src[j];
    }
}

// Sharded counting, step 2: records (slots of other tables of the same K) merged into this table, one per thread
template <int W>
__global__ void __launch_bounds__(256)
kc_merge_kernel(const u64* __restrict__ recs, u64 n, u64* __restrict__ table, u64 n_slots, KcCounters* ctr) {
    __shared__ u32 s_fresh, s_fail;
    if (threadIdx.x == 0) { s_fresh = 0; s_fail = 0; }
    __syncthreads();
    const u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    u32 fresh = 0, fail = 0;
    if (i < n) {
        bool f = false;
        if (kc_merge_slot<W>(table, n_slots, recs + i * (u64)KcSlot<W>::kWords, f)) fresh = f ? 1u : 0u;
        else fail = 1u;
    }
    fresh = __reduce_add_sync(kFull, fresh);
    fail = __reduce_add_sync(kFull, fail);
    if ((threadIdx.x & 31u) == 0) {
        if (fresh) atomicAdd(&s_fresh, fresh);
        if (fail) atomicAdd(&s_fail, fail);
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        if (s_fresh) atomicAdd(&ctr->n_distinct, (u64)s_fresh);
        if (s_fail) atomicOr(&ctr->errors, kKcErrFull);
    }
}

// The k-mer spectrum (kc_slot_total per slot, binned): one read of the table, grid-stride with a few blocks per SM so the
// global flush stays at about blocks x 256 atomics.  The bins are very skewed -- half the slots are empty at load 0.5 and
// most k-mers of error-rich reads sit in bin 1 -- so a warp aggregates its equal values with __match_any_sync before
// the shared atomic, as kc_partition_kernel does.  Empty slots (value 0) are not binned.
constexpr int kKcHistThreads = 256;
constexpr int kKcHistBlocksPerSm = 4;

template <int W>
__global__ void __launch_bounds__(kKcHistThreads)
kc_histogram_kernel(const u64* __restrict__ table, u64 n_slots, u64* __restrict__ hist) {
    __shared__ u32 s_bin[kKcHistBins];
    for (u32 b = threadIdx.x; b < kKcHistBins; b += kKcHistThreads) s_bin[b] = 0;
    __syncthreads();
    const u32 lane = threadIdx.x & 31u;
    const u64 stride = (u64)gridDim.x * kKcHistThreads;
    // the bound is block-uniform: every lane reaches __match_any_sync
    for (u64 first = (u64)blockIdx.x * kKcHistThreads; first < n_slots; first += stride) {
        const u64 i = first + threadIdx.x;
        const u32 v = i < n_slots ? kc_slot_total<W>(table, i) : 0u;
        const u32 peers = __match_any_sync(kFull, v);
        if (v && lane == (u32)__ffs(peers) - 1u) atomicAdd(&s_bin[v], (u32)__popc(peers));
    }
    __syncthreads();
    for (u32 b = threadIdx.x; b < kKcHistBins; b += kKcHistThreads)
        if (s_bin[b]) atomicAdd(&hist[b], (u64)s_bin[b]);
}

// Contig depth (kh_count_contig_depth*): one block per 2048-byte tile of the contig text [offsets[0], offsets[n]), seen
// through `seg` = the text at offsets[0], so nothing outside that range is read.  The tile is packed and its windows
// listed as in kc_count_kernel (positions past the range read as separators).  A block first finds the contigs its
// tile touches (two binary searches over offsets), then every listed position searches only that range; windows that
// run past their contig's end, or whose k-mer another rank owns, are dropped.  The lookup is read-only (kc_find).  The
// loop bound is warp-uniform: lanes without a window carry kKcNoContig, the lanes of one contig are grouped with
// __match_any_sync and reduced with __reduce_*_sync, and the group's first lane adds the group into the record with
// integer atomics -- the records do not depend on the schedule.  Tiles cost the same whatever the contig lengths: a
// 10^6-k-mer contig is spread over ~500 blocks, and a tile of hundreds of short contigs costs one more search level.
template <int W>
__global__ void __launch_bounds__(kKcThreads, 8)
kc_depth_kernel(const unsigned char* __restrict__ seg, u64 span, u64 p_begin, const u64* __restrict__ offsets, u64 n_contigs,
                const u64* __restrict__ table, u64 n_slots, int k, u32 world, u32 rank, KcDepth* __restrict__ out) {
    __shared__ u32 s_code[kKcWords], s_inv[kKcWords];
    __shared__ unsigned short s_list[kKcTile];
    __shared__ u32 s_n;
    __shared__ u64 s_lo, s_hi;
    const u64 t0 = (u64)blockIdx.x * kKcTile;
    if (threadIdx.x == 0) {
        s_n = 0;
        s_lo = kc_contig_of(offsets, 0, n_contigs, p_begin + t0);
    } else if (threadIdx.x == 32) {
        const u64 last = p_begin + (t0 + kKcTile < span ? t0 + kKcTile : span) - 1;
        s_hi = kc_contig_of(offsets, 0, n_contigs, last) + 1;
    }
    for (u32 i = threadIdx.x; i < kKcWords; i += kKcThreads)
        kc_pack_word(seg, span, (long long)t0 - 16 + 16ll * (long long)i, s_code[i], s_inv[i]);
    __syncthreads();
    const u32 lane = threadIdx.x & 31u;
#pragma unroll
    for (int r = 0; r < kKcPer; ++r) {
        const u32 local = threadIdx.x + (u32)r * kKcThreads;
        const bool ok = t0 + local < span && kc_kmer_valid(s_inv, local, k);
        const u32 bal = __ballot_sync(kFull, ok);
        u32 base = 0;
        if (lane == 0 && bal) base = atomicAdd(&s_n, (u32)__popc(bal));
        base = __shfl_sync(kFull, base, 0);
        if (ok) s_list[base + (u32)__popc(bal & ((1u << lane) - 1u))] = (unsigned short)local;
    }
    __syncthreads();
    // offsets that decrease somewhere could give hi <= lo: the range stays non-empty and inside [0, n_contigs)
    const u64 lo = s_lo, hi = s_hi > lo ? s_hi : lo + 1;
    const u32 cnt = s_n;
#pragma unroll 1
    for (u32 i0 = threadIdx.x & ~31u; i0 < cnt; i0 += kKcThreads) {
        const u32 i = i0 + lane;
        u64 c = kKcNoContig;
        u32 v = 0;
        if (i < cnt) {
            const u32 local = s_list[i];
            const u64 p = p_begin + t0 + local;
            const u64 cc = kc_contig_of(offsets, lo, hi, p);
            if (kc_window_in_contig(offsets, cc, p, k)) {
                const KcOcc o = kc_position(s_code, s_inv, local, k);
                if (world == 1 || kc_owner(o.key_hi, o.key_lo, world) == rank) {
                    c = cc;
                    v = kc_depth_value<W>(table, n_slots, o.key_hi, o.key_lo);
                }
            }
        }
        const u32 peers = __match_any_sync(kFull, c);
        if (c != kKcNoContig) {
            const u32 sum = __reduce_add_sync(peers, v), mn = __reduce_min_sync(peers, v), mx = __reduce_max_sync(peers, v);
            if (lane == (u32)__ffs(peers) - 1u) {
                KcDepth* rec = out + c;
                atomicAdd(&rec->n_kmers, (u64)__popc(peers));
                atomicAdd(&rec->sum, (u64)sum);
                atomicMin(&rec->min, mn);
                atomicMax(&rec->max, mx);
            }
        }
    }
}

__global__ void __launch_bounds__(256) kc_depth_init_kernel(KcDepth* __restrict__ out, u64 n) {
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x)
        out[i] = KcDepth{0ull, 0ull, kKcDepthNoMin, 0u};
}

// Unitig extensions (kh_count_link_check*): one block per kKcLinkRecs records.  Records are K/4 + 2 = 3..18 bytes at
// any alignment, so the block stages its byte range through shared memory -- aligned 32-bit loads in, one byte per
// thread out, both coalesced -- and every thread checks kKcLinkPer records there (kc_link_plan, kc_find_pair with the
// successor and predecessor lookups in flight together, kc_link_apply).  The table is only read.  `out` may be `in`: a
// block reads its whole range before it writes any of it, and ranges of blocks are disjoint.  Cuts and malformed
// records are summed per warp, one atomic each.
struct KcLink {
    u64 n_cut;
    u32 bad, pad;
};
constexpr int kKcLinkThreads = 256;
constexpr int kKcLinkPer = 4;
constexpr u32 kKcLinkRecs = kKcLinkThreads * kKcLinkPer;
constexpr u32 kKcLinkWords = (kKcLinkRecs * 18 + 3 + 3) / 4;          // the longest record (K = 61) + the first word's head

template <int W>
__global__ void __launch_bounds__(kKcLinkThreads)
kc_link_kernel(const unsigned char* in, unsigned char* out, u64 n, const u64* __restrict__ table, u64 n_slots, int k, u32 min_count,
               u32 min_ext, u32 world, u32 rank, KcLink* __restrict__ acc) {
    __shared__ u32 s_w[kKcLinkWords];
    const u64 pb = (u64)((k + 3) >> 2) + 2, first = (u64)blockIdx.x * kKcLinkRecs;
    const u32 cnt = n - first < kKcLinkRecs ? (u32)(n - first) : kKcLinkRecs;
    const u32 bytes = cnt * (u32)pb;
    const unsigned char* src = in + first * pb;
    const u32 head = (u32)(reinterpret_cast<uintptr_t>(src) & 3u);
    const u32* words = reinterpret_cast<const u32*>(src - head);     // aligned words that hold a byte of the range
    for (u32 i = threadIdx.x; i < (head + bytes + 3u) / 4u; i += kKcLinkThreads) s_w[i] = words[i];
    __syncthreads();
    unsigned char* s_b = reinterpret_cast<unsigned char*>(s_w) + head;
    u32 cut = 0, bad = 0;
#pragma unroll 1
    for (u32 i = threadIdx.x; i < cnt; i += kKcLinkThreads) {
        unsigned char* rec = s_b + i * (u32)pb;
        const KcLinkPlan p = kc_link_plan(rec, k, world, rank);
        u64 c[2];
        kc_find_pair<W>(table, n_slots, p, c);
        bad |= p.bad ? 1u : 0u;
        cut += kc_link_apply(p, c, k, min_count, min_ext, rec);
    }
    __syncthreads();
    unsigned char* dst = out + first * pb;
    for (u32 j = threadIdx.x; j < bytes; j += kKcLinkThreads) dst[j] = s_b[j];
    cut = __reduce_add_sync(kFull, cut);
    bad = __reduce_or_sync(kFull, bad);
    if ((threadIdx.x & 31u) == 0u) {
        if (cut) atomicAdd(&acc->n_cut, (u64)cut);
        if (bad) atomicOr(&acc->bad, 1u);
    }
}

template <int W>
__global__ void __launch_bounds__(256)
kc_lookup_kernel(const u64* __restrict__ table, u64 n_slots, int k, const unsigned char* __restrict__ pkmers, u64 n, u32* __restrict__ counts_out) {
    const u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int pl = (k + 3) >> 2;
    unsigned char key[16];
    for (int j = 0; j < pl; ++j) key[j] = pkmers[i * pl + j];
    u64 kh_, kl_;
    kc_packed_to_key(key, k, kh_, kl_);
    const u64 c = kc_find<W>(table, n_slots, kh_, kl_);
    u32* o = counts_out + 9 * i;
    o[0] = kc_total(c);
    for (u32 b = 0; b < 4u; ++b) { o[1 + b] = kc_back_count(c, b); o[5 + b] = kc_fwd_count(c, b); }
}

// records -> lines of the reference's k-mer file; a warp writes 32 consecutive lines (one contiguous run of bytes)
__global__ void __launch_bounds__(256)
kc_lines_kernel(const unsigned char* __restrict__ recs, u64 n, int k, unsigned char* __restrict__ text) {
    const u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int pb = ((k + 3) >> 2) + 2;
    unsigned char rec[18], line[68];
    for (int j = 0; j < pb; ++j) rec[j] = recs[i * pb + j];
    kc_record_to_line(rec, k, line);
    unsigned char* dst = text + i * (u64)(k + 4);
    for (int j = 0; j < k + 4; ++j) dst[j] = line[j];
}

// ---------------------------------------------------------------- host runtime -------------------------------
struct kh_counter {
    int k = 0, W = 1, device = 0, pb = 0;
    u64 n_slots = 0;
    size_t table_bytes = 0;
    u64* table = nullptr;
    KcCounters* d_ctr = nullptr;
    KcCounters h_ctr = {};
    cudaStream_t stream = nullptr, copy_stream = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr, ev2 = nullptr, ev3 = nullptr, ev_copied[2] = {}, ev_consumed[2] = {};
    unsigned char* stage[2] = {};
    size_t stage_cap = 0;
    unsigned char* out = nullptr;
    size_t out_cap = 0;
    void* scratch = nullptr;
    size_t scratch_cap = 0;
    void* outbox = nullptr;           // kh_count_partition: the slots grouped by owner
    size_t outbox_cap = 0;
    void* inbox = nullptr;            // kh_count_merge_device / kh_count_link_check*: records copied over from another device or the host
    size_t inbox_cap = 0;
    void* cursor = nullptr;           // kh_count_partition: per-owner counts / write cursors
    size_t cursor_cap = 0;
    void* hist = nullptr;             // kh_count_histogram: 256 x u64 bins
    size_t hist_cap = 0;
    void* depth = nullptr;            // kh_count_contig_depth: records | offsets | contig text
    size_t depth_cap = 0;
    void* link = nullptr;             // kh_count_link_check*: the KcLink sums
    size_t link_cap = 0;
    u64 peers_enabled = 0;            // bit d: this counter's device reads device d's memory directly
    u64 n_bytes = 0;
    u32 n_launches = 0;
    float ms_count = 0.f, ms_extract = 0.f;
    bool have_count = false;
    bool may_grow = true;             // KH_COUNT_GROW=0: a full table is an error instead of a reason to grow
    double lf = 0.5;
    u32 n_grows = 0;
    u64 distinct_ub = 0;              // host-side upper bound of the distinct count: every launched position counted as new
    std::string err;
};

namespace {

int kc_fail(kh_counter* c, int status, const std::string& msg) {
    if (c) c->err = msg;
    return status;
}

#define KC_CUDA(c, expr)                                                                          \
    do {                                                                                          \
        cudaError_t e_ = (expr);                                                                  \
        if (e_ != cudaSuccess)                                                                    \
            return kc_fail((c), e_ == cudaErrorMemoryAllocation ? KH_ERR_NOMEM : KH_ERR_CUDA,     \
                           std::string(#expr) + ": " + cudaGetErrorString(e_));                   \
    } while (0)
#define KC_TRY(expr)                  \
    do {                              \
        const int rc_ = (expr);       \
        if (rc_ != KH_OK) return rc_; \
    } while (0)

int kc_grow(kh_counter* c, void** p, size_t* cap, size_t bytes) {
    if (*p && bytes <= *cap) return KH_OK;
    if (*p) { KC_CUDA(c, cudaFree(*p)); *p = nullptr; *cap = 0; }
    const size_t want = std::max<size_t>(256, bytes + bytes / 8);
    KC_CUDA(c, cudaMalloc(p, want));
    *cap = want;
    return KH_OK;
}

// wait for the stream and bring the counters to the host; a full table is reported from here on
int kc_settle(kh_counter* c) {
    KC_CUDA(c, cudaMemcpyAsync(&c->h_ctr, c->d_ctr, sizeof(KcCounters), cudaMemcpyDeviceToHost, c->stream));
    KC_CUDA(c, cudaStreamSynchronize(c->stream));
    if (c->h_ctr.errors & kKcErrFull)
        return kc_fail(c, KH_ERR_TABLE_FULL, "k-mer counter: more distinct k-mers than slots (n_distinct_expected / load_factor)");
    return KH_OK;
}

// How many of the next `want` positions may be counted right now without any risk of running out of slots: every position
// could be a new k-mer, so a launch never gets more positions than the table has room for below kKcMaxLoad.  When that
// room falls under kKcMinLaunch positions the table grows (x2, rehashed on the GPU) -- no occurrence is ever dropped and
// nobody has to know the number of distinct k-mers in advance.  Waits for the stream only when the host-side upper
// bound of the distinct count (every launched position counted as new) says the table might be short.
int kc_grow(kh_counter* c) {
    const u64 new_slots = 2 * c->n_slots;
    const size_t new_bytes = (size_t)new_slots * (c->W == 1 ? 16 : 32);
    u64* fresh = nullptr;
    KC_CUDA(c, cudaMalloc(reinterpret_cast<void**>(&fresh), new_bytes));
    KC_CUDA(c, cudaMemsetAsync(fresh, 0, new_bytes, c->stream));
    const u64 blocks = (c->n_slots + 255) / 256;
    if (c->W == 1) kc_rehash_kernel<1><<<(unsigned)blocks, 256, 0, c->stream>>>(c->table, c->n_slots, fresh, new_slots, c->d_ctr);
    else kc_rehash_kernel<2><<<(unsigned)blocks, 256, 0, c->stream>>>(c->table, c->n_slots, fresh, new_slots, c->d_ctr);
    KC_CUDA(c, cudaGetLastError());
    ++c->n_launches;
    ++c->n_grows;
    KC_CUDA(c, cudaStreamSynchronize(c->stream));
    KC_CUDA(c, cudaFree(c->table));
    c->table = fresh; c->n_slots = new_slots; c->table_bytes = new_bytes;
    return KH_OK;
}
int kc_reserve(kh_counter* c, u64 want, u64* granted) {
    auto room = [&](u64 distinct) {
        const u64 limit = (u64)(kKcMaxLoad * (double)c->n_slots);
        return limit > distinct ? limit - distinct : 0ull;
    };
    if (room(c->distinct_ub) >= want) { *granted = want; return KH_OK; }
    KC_TRY(kc_settle(c));
    c->distinct_ub = c->h_ctr.n_distinct;
    const u64 floor = std::min<u64>(want, kKcMinLaunch);
    while (room(c->distinct_ub) < floor) {
        if (!c->may_grow) {
            if (room(c->distinct_ub) >= 16) break;
            return kc_fail(c, KH_ERR_TABLE_FULL, "k-mer counter: the table is full and growing is disabled (KH_COUNT_GROW=0)");
        }
        KC_TRY(kc_grow(c));
    }
    *granted = std::min<u64>(want, room(c->distinct_ub));
    return KH_OK;
}

int kc_launch_count(kh_counter* c, const unsigned char* buf, u64 n, u64 p_begin, u64 p_end) {
    if (p_end <= p_begin) return KH_OK;
    const u64 span = p_end - (p_begin & ~15ull);
    const u64 blocks = (span + kKcTile - 1) / kKcTile;
    if (blocks > 0x7FFFFFFFull) return kc_fail(c, KH_ERR_ARG, "kh_count_reads_device: at most 2^42 bytes per call");
    const unsigned g = (unsigned)blocks;
    if (c->W == 1) kc_count_kernel<1><<<g, kKcThreads, 0, c->stream>>>(buf, n, p_begin, p_end, c->table, c->n_slots, c->k, c->d_ctr);
    else kc_count_kernel<2><<<g, kKcThreads, 0, c->stream>>>(buf, n, p_begin, p_end, c->table, c->n_slots, c->k, c->d_ctr);
    KC_CUDA(c, cudaGetLastError());
    ++c->n_launches;
    return KH_OK;
}

static_assert(sizeof(KcDepth) == sizeof(kh_contig_depth) && sizeof(KcDepth) == 24, "kh_contig_depth layout");

int kc_depth_check(kh_counter* c, bool null_arg, u64 n, uint32_t world, uint32_t rank, const char* what) {
    if (!c) return KH_ERR_ARG;
    if (n && null_arg) return kc_fail(c, KH_ERR_ARG, std::string(what) + ": null pointer");
    if (world < 1 || world > kKcMaxWorld || rank >= world) return kc_fail(c, KH_ERR_ARG, std::string(what) + ": 1 <= world <= 64 and rank < world");
    return KH_OK;
}

// records initialised, then the tiles of [p_begin, p_begin + span) (seg = the text at p_begin); host waits for both
int kc_launch_depth(kh_counter* c, const unsigned char* seg, u64 span, u64 p_begin, const u64* offsets, u64 n, u32 world, u32 rank, KcDepth* out) {
    const u64 blocks = (span + kKcTile - 1) / kKcTile;
    if (blocks > 0x7FFFFFFFull) return kc_fail(c, KH_ERR_ARG, "kh_count_contig_depth: at most 2^42 bytes of contig text per call");
    kc_depth_init_kernel<<<(unsigned)std::min<u64>((n + 255) / 256, 4096), 256, 0, c->stream>>>(out, n);
    KC_CUDA(c, cudaGetLastError());
    ++c->n_launches;
    if (blocks) {
        const unsigned g = (unsigned)blocks;
        if (c->W == 1) kc_depth_kernel<1><<<g, kKcThreads, 0, c->stream>>>(seg, span, p_begin, offsets, n, c->table, c->n_slots, c->k, world, rank, out);
        else kc_depth_kernel<2><<<g, kKcThreads, 0, c->stream>>>(seg, span, p_begin, offsets, n, c->table, c->n_slots, c->k, world, rank, out);
        KC_CUDA(c, cudaGetLastError());
        ++c->n_launches;
    }
    KC_CUDA(c, cudaStreamSynchronize(c->stream));
    return KH_OK;
}

// Memory of any device of this process handed to a counter call: KH_ERR_ARG unless it is device (or managed) memory.
// *foreign: it lives on another device; this counter's device then reads that device's memory peer to peer where the
// two allow it (the copies below go through the host otherwise).
int kc_device_memory(kh_counter* c, const void* p, const char* what, bool* foreign) {
    cudaPointerAttributes a{};
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess || (a.type != cudaMemoryTypeDevice && a.type != cudaMemoryTypeManaged)) {
        cudaGetLastError();
        return kc_fail(c, KH_ERR_ARG, std::string(what) + " is not device memory");
    }
    *foreign = a.type == cudaMemoryTypeDevice && a.device != c->device;
    if (*foreign && a.device >= 0 && a.device < 64 && !((c->peers_enabled >> a.device) & 1ull)) {
        int can = 0;
        if (cudaDeviceCanAccessPeer(&can, c->device, a.device) == cudaSuccess && can) {
            const cudaError_t e = cudaDeviceEnablePeerAccess(a.device, 0);
            if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) KC_CUDA(c, e);
            cudaGetLastError();
        }
        c->peers_enabled |= 1ull << a.device;
    }
    return KH_OK;
}

// `bytes` at p, readable by this counter's kernels: p itself, or -- another GPU's memory -- one copy into the counter's
// inbox, in stream order
int kc_stage_in(kh_counter* c, const void* p, size_t bytes, const char* what, const void** local) {
    bool foreign = false;
    KC_TRY(kc_device_memory(c, p, what, &foreign));
    *local = p;
    if (!foreign) return KH_OK;
    KC_TRY(kc_grow(c, &c->inbox, &c->inbox_cap, bytes));
    KC_CUDA(c, cudaMemcpyAsync(c->inbox, p, bytes, cudaMemcpyDefault, c->stream));
    *local = c->inbox;
    return KH_OK;
}

int kc_link_check_args(kh_counter* c, bool null_arg, u64 n, u32 min_count, u32 min_ext, u32 world, u32 rank, uint64_t* n_cut_out,
                       const char* what) {
    if (!c || !n_cut_out) return KH_ERR_ARG;
    *n_cut_out = 0;
    if (min_count < 1 || min_count > kKcCountCap || min_ext < 1 || min_ext > kKcExtCap)
        return kc_fail(c, KH_ERR_ARG, std::string(what) + ": 1 <= min_count <= 255 and 1 <= min_ext <= 127");
    return kc_depth_check(c, null_arg, n, world, rank, what);
}

// kc_link_kernel over n records at `in` (this device) into `out` (this device; may be `in`); host waits, *n_cut = its sum
int kc_launch_link(kh_counter* c, const void* in, void* out, u64 n, u32 min_count, u32 min_ext, u32 world, u32 rank, uint64_t* n_cut,
                   const char* what) {
    const u64 blocks = (n + kKcLinkRecs - 1) / kKcLinkRecs;
    if (blocks > 0x7FFFFFFFull) return kc_fail(c, KH_ERR_ARG, std::string(what) + ": at most 2^41 records per call");
    KC_TRY(kc_grow(c, &c->link, &c->link_cap, sizeof(KcLink)));
    KcLink* acc = static_cast<KcLink*>(c->link);
    KC_CUDA(c, cudaMemsetAsync(acc, 0, sizeof(KcLink), c->stream));
    const unsigned char* i = static_cast<const unsigned char*>(in);
    unsigned char* o = static_cast<unsigned char*>(out);
    if (c->W == 1)
        kc_link_kernel<1><<<(unsigned)blocks, kKcLinkThreads, 0, c->stream>>>(i, o, n, c->table, c->n_slots, c->k, min_count, min_ext, world, rank, acc);
    else
        kc_link_kernel<2><<<(unsigned)blocks, kKcLinkThreads, 0, c->stream>>>(i, o, n, c->table, c->n_slots, c->k, min_count, min_ext, world, rank, acc);
    KC_CUDA(c, cudaGetLastError());
    ++c->n_launches;
    KcLink h{};
    KC_CUDA(c, cudaMemcpyAsync(&h, acc, sizeof h, cudaMemcpyDeviceToHost, c->stream));
    KC_CUDA(c, cudaStreamSynchronize(c->stream));
    if (h.bad) return kc_fail(c, KH_ERR_BAD_INPUT, std::string(what) + ": an extension byte is not one of A C G T F");
    *n_cut = h.n_cut;
    return KH_OK;
}

}  // namespace

extern "C" {

int kh_count_create(int k, uint64_t n_distinct_expected, double load_factor, int device, kh_counter** out) {
    if (!out) return KH_ERR_ARG;
    *out = nullptr;
    if (k < 2 || k > 61 || !(load_factor > 0.0) || load_factor > 1.0) return KH_ERR_ARG;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev < 1 || device < 0 || device >= ndev) {
        cudaGetLastError();
        return KH_ERR_CUDA;                                  // no CPU fallback
    }
    kh_counter* c = new kh_counter();
    c->k = k; c->W = kc_slot_words(k); c->device = device; c->pb = (k + 3) / 4 + 2;
    if (const char* e = getenv("KH_COUNT_GROW")) c->may_grow = atoi(e) != 0;
    c->lf = load_factor;
    const double want = (double)std::max<uint64_t>(n_distinct_expected, 1) / load_factor;
    c->n_slots = std::max<u64>(1024, (u64)want + 1);
    c->table_bytes = (size_t)c->n_slots * (c->W == 1 ? 16 : 32);
    auto bail = [&](cudaError_t e) {
        const int rc = e == cudaErrorMemoryAllocation ? KH_ERR_NOMEM : KH_ERR_CUDA;
        cudaGetLastError();
        kh_count_destroy(c);
        return rc;
    };
    cudaError_t e;
    if ((e = cudaSetDevice(device)) != cudaSuccess) return bail(e);
    if ((e = cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking)) != cudaSuccess) return bail(e);
    if ((e = cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking)) != cudaSuccess) return bail(e);
    if ((e = cudaEventCreate(&c->ev0)) != cudaSuccess) return bail(e);
    if ((e = cudaEventCreate(&c->ev1)) != cudaSuccess) return bail(e);
    if ((e = cudaEventCreate(&c->ev2)) != cudaSuccess) return bail(e);
    if ((e = cudaEventCreate(&c->ev3)) != cudaSuccess) return bail(e);
    for (int i = 0; i < 2; ++i) {
        if ((e = cudaEventCreateWithFlags(&c->ev_copied[i], cudaEventDisableTiming)) != cudaSuccess) return bail(e);
        if ((e = cudaEventCreateWithFlags(&c->ev_consumed[i], cudaEventDisableTiming)) != cudaSuccess) return bail(e);
    }
    if ((e = cudaMalloc(reinterpret_cast<void**>(&c->table), c->table_bytes)) != cudaSuccess) return bail(e);
    if ((e = cudaMalloc(reinterpret_cast<void**>(&c->d_ctr), sizeof(KcCounters))) != cudaSuccess) return bail(e);
    if ((e = cudaMemsetAsync(c->table, 0, c->table_bytes, c->stream)) != cudaSuccess) return bail(e);
    if ((e = cudaMemsetAsync(c->d_ctr, 0, sizeof(KcCounters), c->stream)) != cudaSuccess) return bail(e);
    if ((e = cudaStreamSynchronize(c->stream)) != cudaSuccess) return bail(e);
    *out = c;
    return KH_OK;
}

int kh_count_destroy(kh_counter* c) {
    if (!c) return KH_OK;
    cudaSetDevice(c->device);
    if (c->stream) cudaStreamSynchronize(c->stream);
    if (c->copy_stream) cudaStreamSynchronize(c->copy_stream);
    cudaFree(c->table); cudaFree(c->d_ctr); cudaFree(c->stage[0]); cudaFree(c->stage[1]); cudaFree(c->out); cudaFree(c->scratch);
    cudaFree(c->outbox); cudaFree(c->inbox); cudaFree(c->cursor); cudaFree(c->hist); cudaFree(c->depth); cudaFree(c->link);
    if (c->ev0) cudaEventDestroy(c->ev0);
    if (c->ev1) cudaEventDestroy(c->ev1);
    if (c->ev2) cudaEventDestroy(c->ev2);
    if (c->ev3) cudaEventDestroy(c->ev3);
    for (int i = 0; i < 2; ++i) {
        if (c->ev_copied[i]) cudaEventDestroy(c->ev_copied[i]);
        if (c->ev_consumed[i]) cudaEventDestroy(c->ev_consumed[i]);
    }
    if (c->stream) cudaStreamDestroy(c->stream);
    if (c->copy_stream) cudaStreamDestroy(c->copy_stream);
    cudaGetLastError();
    delete c;
    return KH_OK;
}

int kh_count_clear(kh_counter* c) {
    if (!c) return KH_ERR_ARG;
    KC_CUDA(c, cudaSetDevice(c->device));
    KC_CUDA(c, cudaMemsetAsync(c->table, 0, c->table_bytes, c->stream));
    KC_CUDA(c, cudaMemsetAsync(c->d_ctr, 0, sizeof(KcCounters), c->stream));
    c->n_bytes = 0;
    c->distinct_ub = 0;
    c->h_ctr = KcCounters{};
    c->err.clear();
    return KH_OK;
}

int kh_count_reads_device(kh_counter* c, const char* reads_dev, uint64_t n_bytes) {
    if (!c || (n_bytes && !reads_dev)) return KH_ERR_ARG;
    if (n_bytes == 0) return KH_OK;
    KC_CUDA(c, cudaSetDevice(c->device));
    KC_CUDA(c, cudaEventRecord(c->ev0, c->stream));
    KC_TRY(kc_launch_count(c, reinterpret_cast<const unsigned char*>(reads_dev), n_bytes, 0, n_bytes));
    c->distinct_ub += n_bytes;
    KC_CUDA(c, cudaEventRecord(c->ev1, c->stream));
    c->have_count = true;
    c->n_bytes += n_bytes;
    return KH_OK;
}

// Host reads: chunks of 64 M positions, double-buffered -- the copy of chunk i+1 runs beside the kernel of chunk i.
// A chunk travels with 16 bytes in front of it and 64 behind it, so k-mers that straddle a chunk boundary are cut
// exactly as in one piece (the halo of the kernel's first / last tile).
int kh_count_reads(kh_counter* c, const char* reads_host, uint64_t n_bytes) {
    if (!c || (n_bytes && !reads_host)) return KH_ERR_ARG;
    if (n_bytes == 0) return KH_OK;
    KC_CUDA(c, cudaSetDevice(c->device));
    const u64 nchunks = (n_bytes + kKcChunk - 1) / kKcChunk;
    const size_t need = (size_t)std::min<u64>(n_bytes, kKcChunk + kKcHalo);
    if (need > c->stage_cap) {
        KC_CUDA(c, cudaStreamSynchronize(c->stream));
        for (int i = 0; i < 2; ++i) {
            if (c->stage[i]) { KC_CUDA(c, cudaFree(c->stage[i])); c->stage[i] = nullptr; }
        }
        c->stage_cap = 0;
        for (int i = 0; i < (nchunks > 1 ? 2 : 1); ++i) KC_CUDA(c, cudaMalloc(reinterpret_cast<void**>(&c->stage[i]), need));
        c->stage_cap = need;
    } else if (nchunks > 1 && !c->stage[1]) {
        KC_CUDA(c, cudaMalloc(reinterpret_cast<void**>(&c->stage[1]), c->stage_cap));
    }
    auto range = [&](u64 ci, u64& a, u64& b, u64& off, u64& len) { kc_chunk_range(ci, kKcChunk, n_bytes, a, b, off, len); };
    auto issue_copy = [&](u64 ci) -> int {
        u64 a, b, off, len;
        range(ci, a, b, off, len);
        if (ci >= 2) KC_CUDA(c, cudaStreamWaitEvent(c->copy_stream, c->ev_consumed[ci & 1], 0));
        KC_CUDA(c, cudaMemcpyAsync(c->stage[ci & 1], reads_host + a, b - a, cudaMemcpyHostToDevice, c->copy_stream));
        KC_CUDA(c, cudaEventRecord(c->ev_copied[ci & 1], c->copy_stream));
        return KH_OK;
    };
    KC_CUDA(c, cudaEventRecord(c->ev0, c->stream));
    // earlier work on the main stream may still read the staging buffers
    KC_CUDA(c, cudaEventRecord(c->ev_consumed[0], c->stream));
    KC_CUDA(c, cudaStreamWaitEvent(c->copy_stream, c->ev_consumed[0], 0));
    KC_TRY(issue_copy(0));
    for (u64 ci = 0; ci < nchunks; ++ci) {
        if (ci + 1 < nchunks) KC_TRY(issue_copy(ci + 1));
        u64 a, b, off, len;
        range(ci, a, b, off, len);
        KC_CUDA(c, cudaStreamWaitEvent(c->stream, c->ev_copied[ci & 1], 0));
        for (u64 done = 0; done < len;) {                  // normally one launch; several when the table is nearly full
            u64 take = 0;
            KC_TRY(kc_reserve(c, len - done, &take));
            if (take < len - done) take &= ~15ull;         // pieces start on a 16-character boundary
            KC_TRY(kc_launch_count(c, c->stage[ci & 1], b - a, off - a + done, off - a + done + take));
            c->distinct_ub += take;
            done += take;
        }
        KC_CUDA(c, cudaEventRecord(c->ev_consumed[ci & 1], c->stream));
    }
    KC_CUDA(c, cudaEventRecord(c->ev1, c->stream));
    c->have_count = true;
    c->n_bytes += n_bytes;
    return kc_settle(c);                                    // the caller's buffer is free again; errors surface here
}

int kh_count_extract_device(kh_counter* c, uint32_t min_count, uint32_t min_ext, const void** pairs_dev_out, uint64_t* n_out) {
    if (!c || !n_out) return KH_ERR_ARG;
    *n_out = 0;
    if (pairs_dev_out) *pairs_dev_out = nullptr;
    if (min_count < 1 || min_count > kKcCountCap || min_ext < 1 || min_ext > kKcExtCap)
        return kc_fail(c, KH_ERR_ARG, "kh_count_extract: 1 <= min_count <= 255 and 1 <= min_ext <= 127");
    KC_CUDA(c, cudaSetDevice(c->device));
    KC_TRY(kc_settle(c));
    const u64 cap = c->h_ctr.n_distinct;
    KC_TRY(kc_grow(c, reinterpret_cast<void**>(&c->out), &c->out_cap, (size_t)std::max<u64>(cap, 1) * c->pb));
    KC_CUDA(c, cudaMemsetAsync(&c->d_ctr->n_reported, 0, sizeof(u64), c->stream));
    const u64 blocks = (c->n_slots + kKcExtThreads * kKcExtPer - 1) / (kKcExtThreads * kKcExtPer);
    KC_CUDA(c, cudaEventRecord(c->ev2, c->stream));
    if (c->W == 1)
        kc_extract_kernel<1><<<(unsigned)blocks, kKcExtThreads, 0, c->stream>>>(c->table, c->n_slots, c->k, min_count, min_ext, c->out, cap, c->d_ctr);
    else
        kc_extract_kernel<2><<<(unsigned)blocks, kKcExtThreads, 0, c->stream>>>(c->table, c->n_slots, c->k, min_count, min_ext, c->out, cap, c->d_ctr);
    KC_CUDA(c, cudaGetLastError());
    ++c->n_launches;
    KC_CUDA(c, cudaEventRecord(c->ev3, c->stream));
    KC_TRY(kc_settle(c));
    KC_CUDA(c, cudaEventElapsedTime(&c->ms_extract, c->ev2, c->ev3));
    if (c->h_ctr.n_reported > cap) return kc_fail(c, KH_ERR_CUDA, "k-mer counter: extract wrote past the distinct count (internal)");
    *n_out = c->h_ctr.n_reported;
    if (pairs_dev_out) *pairs_dev_out = c->out;
    return KH_OK;
}

int kh_count_extract(kh_counter* c, uint32_t min_count, uint32_t min_ext, void* pairs_host_out, uint64_t capacity, uint64_t* n_out) {
    if (!c || !n_out) return KH_ERR_ARG;
    const void* dev = nullptr;
    KC_TRY(kh_count_extract_device(c, min_count, min_ext, &dev, n_out));
    if (!pairs_host_out) return KH_OK;
    if (capacity < *n_out) return kc_fail(c, KH_ERR_ARG, "kh_count_extract: capacity is smaller than the number of reported k-mers (*n_out)");
    if (*n_out) {
        KC_CUDA(c, cudaMemcpyAsync(pairs_host_out, dev, (size_t)*n_out * c->pb, cudaMemcpyDeviceToHost, c->stream));
        KC_CUDA(c, cudaStreamSynchronize(c->stream));
    }
    return KH_OK;
}

int kh_count_extract_lines(kh_counter* c, uint32_t min_count, uint32_t min_ext, char* lines_host_out, uint64_t capacity_lines, uint64_t* n_out) {
    if (!c || !n_out) return KH_ERR_ARG;
    const void* dev = nullptr;
    KC_TRY(kh_count_extract_device(c, min_count, min_ext, &dev, n_out));
    if (!lines_host_out) return KH_OK;
    if (capacity_lines < *n_out) return kc_fail(c, KH_ERR_ARG, "kh_count_extract_lines: capacity is smaller than the number of reported k-mers (*n_out)");
    const u64 n = *n_out, ll = (u64)c->k + 4;
    if (n == 0) return KH_OK;
    // formatted in pieces of 16 M lines so the device-side text buffer stays small next to the table
    const u64 piece = 16ull << 20;
    KC_TRY(kc_grow(c, &c->scratch, &c->scratch_cap, (size_t)(std::min(n, piece) * ll)));
    for (u64 i0 = 0; i0 < n; i0 += piece) {
        const u64 cnt = std::min(piece, n - i0);
        kc_lines_kernel<<<(unsigned)((cnt + 255) / 256), 256, 0, c->stream>>>(static_cast<const unsigned char*>(dev) + i0 * c->pb, cnt, c->k,
                                                                              static_cast<unsigned char*>(c->scratch));
        KC_CUDA(c, cudaGetLastError());
        ++c->n_launches;
        KC_CUDA(c, cudaMemcpyAsync(lines_host_out + i0 * ll, c->scratch, (size_t)(cnt * ll), cudaMemcpyDeviceToHost, c->stream));
        KC_CUDA(c, cudaStreamSynchronize(c->stream));
    }
    return KH_OK;
}

uint64_t kh_count_record_bytes(int k) { return k < 2 || k > 61 ? 0ull : (kc_slot_words(k) == 1 ? 16ull : 32ull); }

int kh_count_partition(kh_counter* c, int world, const void** records_dev_out, uint64_t* offsets_host_out) {
    if (!c || !records_dev_out || !offsets_host_out) return KH_ERR_ARG;
    *records_dev_out = nullptr;
    if (world < 1 || world > (int)kKcMaxWorld) return kc_fail(c, KH_ERR_ARG, "kh_count_partition: 1 <= world <= 64");
    KC_CUDA(c, cudaSetDevice(c->device));
    KC_TRY(kc_settle(c));                                   // a table that overflowed while counting is reported here
    const u64 n = c->h_ctr.n_distinct, rb = c->W == 1 ? 16 : 32;
    KC_TRY(kc_grow(c, &c->outbox, &c->outbox_cap, (size_t)(std::max<u64>(n, 1) * rb)));
    KC_TRY(kc_grow(c, &c->cursor, &c->cursor_cap, kKcMaxWorld * sizeof(u64)));
    u64* cur = static_cast<u64*>(c->cursor);
    const u64 blocks = (c->n_slots + kKcExtThreads * kKcExtPer - 1) / (kKcExtThreads * kKcExtPer);
    auto launch = [&](bool scatter) -> int {
        if (c->W == 1)
            kc_partition_kernel<1><<<(unsigned)blocks, kKcExtThreads, 0, c->stream>>>(c->table, c->n_slots, (u32)world, scatter, cur, static_cast<u64*>(c->outbox));
        else
            kc_partition_kernel<2><<<(unsigned)blocks, kKcExtThreads, 0, c->stream>>>(c->table, c->n_slots, (u32)world, scatter, cur, static_cast<u64*>(c->outbox));
        KC_CUDA(c, cudaGetLastError());
        ++c->n_launches;
        return KH_OK;
    };
    u64 h[kKcMaxWorld + 1] = {};
    KC_CUDA(c, cudaMemsetAsync(cur, 0, (size_t)world * sizeof(u64), c->stream));
    KC_TRY(launch(false));
    KC_CUDA(c, cudaMemcpyAsync(h + 1, cur, (size_t)world * sizeof(u64), cudaMemcpyDeviceToHost, c->stream));
    KC_CUDA(c, cudaStreamSynchronize(c->stream));
    for (int o = 0; o < world; ++o) h[o + 1] += h[o];      // per-owner counts -> segment offsets
    if (h[world] != n) return kc_fail(c, KH_ERR_CUDA, "k-mer counter: occupied slots differ from the distinct count (internal)");
    KC_CUDA(c, cudaMemcpyAsync(cur, h, (size_t)world * sizeof(u64), cudaMemcpyHostToDevice, c->stream));
    KC_TRY(launch(true));
    KC_CUDA(c, cudaStreamSynchronize(c->stream));
    for (int o = 0; o <= world; ++o) offsets_host_out[o] = h[o];
    *records_dev_out = c->outbox;
    return KH_OK;
}

int kh_count_merge_device(kh_counter* c, const void* records_dev, uint64_t n) {
    if (!c || (n && !records_dev)) return KH_ERR_ARG;
    if (n == 0) return KH_OK;
    KC_CUDA(c, cudaSetDevice(c->device));
    const u64 rb = c->W == 1 ? 16 : 32;
    const void* staged = nullptr;
    KC_TRY(kc_stage_in(c, records_dev, (size_t)(n * rb), "kh_count_merge_device: records_dev", &staged));
    const u64* src = static_cast<const u64*>(staged);
    for (u64 done = 0; done < n;) {                        // like kh_count_reads: every record may be a new k-mer
        u64 take = 0;
        KC_TRY(kc_reserve(c, n - done, &take));
        const u64 blocks = (take + 255) / 256;
        const u64* r = src + done * (rb / 8);
        if (c->W == 1) kc_merge_kernel<1><<<(unsigned)blocks, 256, 0, c->stream>>>(r, take, c->table, c->n_slots, c->d_ctr);
        else kc_merge_kernel<2><<<(unsigned)blocks, 256, 0, c->stream>>>(r, take, c->table, c->n_slots, c->d_ctr);
        KC_CUDA(c, cudaGetLastError());
        ++c->n_launches;
        c->distinct_ub += take;
        done += take;
    }
    return kc_settle(c);
}

int kh_count_histogram(kh_counter* c, uint64_t* hist_host_out) {
    if (!c || !hist_host_out) return KH_ERR_ARG;
    KC_CUDA(c, cudaSetDevice(c->device));
    KC_TRY(kc_settle(c));                                   // a table that overflowed while counting is reported here
    KC_TRY(kc_grow(c, &c->hist, &c->hist_cap, kKcHistBins * sizeof(u64)));
    int sms = 0;
    KC_CUDA(c, cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, c->device));
    const u64 blocks = std::max<u64>(1, std::min<u64>((c->n_slots + kKcHistThreads - 1) / kKcHistThreads, (u64)std::max(sms, 1) * kKcHistBlocksPerSm));
    u64* d = static_cast<u64*>(c->hist);
    KC_CUDA(c, cudaMemsetAsync(d, 0, kKcHistBins * sizeof(u64), c->stream));
    if (c->W == 1) kc_histogram_kernel<1><<<(unsigned)blocks, kKcHistThreads, 0, c->stream>>>(c->table, c->n_slots, d);
    else kc_histogram_kernel<2><<<(unsigned)blocks, kKcHistThreads, 0, c->stream>>>(c->table, c->n_slots, d);
    KC_CUDA(c, cudaGetLastError());
    ++c->n_launches;
    u64 h[kKcHistBins];
    KC_CUDA(c, cudaMemcpyAsync(h, d, sizeof h, cudaMemcpyDeviceToHost, c->stream));
    KC_CUDA(c, cudaStreamSynchronize(c->stream));
    u64 total = 0;
    for (u32 b = 0; b < kKcHistBins; ++b) total += h[b];
    if (h[0] != 0 || total != c->h_ctr.n_distinct)
        return kc_fail(c, KH_ERR_CUDA, "k-mer counter: spectrum bins differ from the distinct count (internal)");
    memcpy(hist_host_out, h, sizeof h);
    return KH_OK;
}

uint32_t kh_count_auto_min_count(const uint64_t* hist) { return kc_auto_min_count(reinterpret_cast<const u64*>(hist)); }

// Host contigs: the records, the offsets and the text [offsets[0], offsets[n]) share one counter-owned buffer.
int kh_count_contig_depth(kh_counter* c, const char* contigs_host, const uint64_t* offsets_host, uint64_t n_contigs, uint32_t world,
                          uint32_t rank, kh_contig_depth* out_host) {
    KC_TRY(kc_depth_check(c, !contigs_host || !offsets_host || !out_host, n_contigs, world, rank, "kh_count_contig_depth"));
    if (n_contigs == 0) return KH_OK;
    for (u64 i = 0; i < n_contigs; ++i)
        if (offsets_host[i + 1] < offsets_host[i]) return kc_fail(c, KH_ERR_ARG, "kh_count_contig_depth: offsets must be non-decreasing");
    KC_CUDA(c, cudaSetDevice(c->device));
    KC_TRY(kc_settle(c));                                   // a table that overflowed while counting is reported here
    const u64 p_begin = offsets_host[0], span = offsets_host[n_contigs] - p_begin;
    const size_t rec_bytes = ((size_t)n_contigs * sizeof(KcDepth) + 15) & ~(size_t)15;
    const size_t off_bytes = ((size_t)(n_contigs + 1) * sizeof(u64) + 15) & ~(size_t)15;
    KC_TRY(kc_grow(c, &c->depth, &c->depth_cap, rec_bytes + off_bytes + (size_t)span));
    unsigned char* base = static_cast<unsigned char*>(c->depth);
    KcDepth* d_out = reinterpret_cast<KcDepth*>(base);
    u64* d_off = reinterpret_cast<u64*>(base + rec_bytes);
    unsigned char* d_text = base + rec_bytes + off_bytes;
    KC_CUDA(c, cudaMemcpyAsync(d_off, offsets_host, (size_t)(n_contigs + 1) * sizeof(u64), cudaMemcpyHostToDevice, c->stream));
    if (span) KC_CUDA(c, cudaMemcpyAsync(d_text, contigs_host + p_begin, (size_t)span, cudaMemcpyHostToDevice, c->stream));
    KC_TRY(kc_launch_depth(c, d_text, span, p_begin, d_off, n_contigs, world, rank, d_out));
    KC_CUDA(c, cudaMemcpyAsync(out_host, d_out, (size_t)n_contigs * sizeof(KcDepth), cudaMemcpyDeviceToHost, c->stream));
    KC_CUDA(c, cudaStreamSynchronize(c->stream));
    return KH_OK;
}

int kh_count_contig_depth_device(kh_counter* c, const char* contigs_dev, const uint64_t* offsets_dev, uint64_t n_contigs, uint32_t world,
                                 uint32_t rank, kh_contig_depth* out_dev) {
    KC_TRY(kc_depth_check(c, !contigs_dev || !offsets_dev || !out_dev, n_contigs, world, rank, "kh_count_contig_depth_device"));
    if (n_contigs == 0) return KH_OK;
    KC_CUDA(c, cudaSetDevice(c->device));
    KC_TRY(kc_settle(c));
    u64 ends[2];                                            // offsets[0] and offsets[n]: the text range and the grid
    KC_CUDA(c, cudaMemcpyAsync(&ends[0], offsets_dev, sizeof(u64), cudaMemcpyDeviceToHost, c->stream));
    KC_CUDA(c, cudaMemcpyAsync(&ends[1], offsets_dev + n_contigs, sizeof(u64), cudaMemcpyDeviceToHost, c->stream));
    KC_CUDA(c, cudaStreamSynchronize(c->stream));
    const u64 span = ends[1] > ends[0] ? ends[1] - ends[0] : 0ull;
    return kc_launch_depth(c, reinterpret_cast<const unsigned char*>(contigs_dev) + ends[0], span, ends[0], reinterpret_cast<const u64*>(offsets_dev),
                           n_contigs, world, rank, reinterpret_cast<KcDepth*>(out_dev));
}

// Unitig extensions.  Host records: one copy to the counter's inbox, checked there in place, one copy back.
int kh_count_link_check(kh_counter* c, void* pairs_host, uint64_t n, uint32_t min_count, uint32_t min_ext, uint32_t world, uint32_t rank,
                        uint64_t* n_cut_out) {
    KC_TRY(kc_link_check_args(c, !pairs_host, n, min_count, min_ext, world, rank, n_cut_out, "kh_count_link_check"));
    if (n == 0) return KH_OK;
    KC_CUDA(c, cudaSetDevice(c->device));
    KC_TRY(kc_settle(c));                                   // a table that overflowed while counting is reported here
    const size_t bytes = (size_t)n * (size_t)c->pb;
    KC_TRY(kc_grow(c, &c->inbox, &c->inbox_cap, bytes));
    KC_CUDA(c, cudaMemcpyAsync(c->inbox, pairs_host, bytes, cudaMemcpyHostToDevice, c->stream));
    KC_TRY(kc_launch_link(c, c->inbox, c->inbox, n, min_count, min_ext, world, rank, n_cut_out, "kh_count_link_check"));
    KC_CUDA(c, cudaMemcpyAsync(pairs_host, c->inbox, bytes, cudaMemcpyDeviceToHost, c->stream));
    KC_CUDA(c, cudaStreamSynchronize(c->stream));
    return KH_OK;
}

// Device records on any device of the process: another device's input is staged into the inbox (kc_stage_in); output
// for another device is written to the inbox and copied over.
int kh_count_link_check_device(kh_counter* c, const void* pairs_in_dev, void* pairs_out_dev, uint64_t n, uint32_t min_count, uint32_t min_ext,
                               uint32_t world, uint32_t rank, uint64_t* n_cut_out) {
    static const char* what = "kh_count_link_check_device";
    KC_TRY(kc_link_check_args(c, !pairs_in_dev || !pairs_out_dev, n, min_count, min_ext, world, rank, n_cut_out, what));
    if (n == 0) return KH_OK;
    KC_CUDA(c, cudaSetDevice(c->device));
    KC_TRY(kc_settle(c));
    const size_t bytes = (size_t)n * (size_t)c->pb;
    bool out_foreign = false;
    KC_TRY(kc_device_memory(c, pairs_out_dev, "kh_count_link_check_device: pairs_out", &out_foreign));
    if (out_foreign) KC_TRY(kc_grow(c, &c->inbox, &c->inbox_cap, bytes));
    const void* src = nullptr;
    KC_TRY(kc_stage_in(c, pairs_in_dev, bytes, "kh_count_link_check_device: pairs_in", &src));
    void* dst = out_foreign ? c->inbox : pairs_out_dev;
    KC_TRY(kc_launch_link(c, src, dst, n, min_count, min_ext, world, rank, n_cut_out, what));
    if (out_foreign) {
        KC_CUDA(c, cudaMemcpyAsync(pairs_out_dev, dst, bytes, cudaMemcpyDefault, c->stream));
        KC_CUDA(c, cudaStreamSynchronize(c->stream));
    }
    return KH_OK;
}

int kh_count_lookup(kh_counter* c, const void* pkmers_host, uint64_t n, uint32_t* counts_host_out) {
    if (!c || (n && (!pkmers_host || !counts_host_out))) return KH_ERR_ARG;
    if (n == 0) return KH_OK;
    KC_CUDA(c, cudaSetDevice(c->device));
    const size_t pl = (size_t)(c->k + 3) / 4, in_bytes = ((size_t)n * pl + 15) & ~(size_t)15, out_bytes = (size_t)n * 9 * sizeof(u32);
    KC_TRY(kc_grow(c, &c->scratch, &c->scratch_cap, in_bytes + out_bytes));
    unsigned char* d_in = static_cast<unsigned char*>(c->scratch);
    u32* d_out = reinterpret_cast<u32*>(d_in + in_bytes);
    KC_CUDA(c, cudaMemcpyAsync(d_in, pkmers_host, (size_t)n * pl, cudaMemcpyHostToDevice, c->stream));
    const unsigned blocks = (unsigned)((n + 255) / 256);
    if (c->W == 1) kc_lookup_kernel<1><<<blocks, 256, 0, c->stream>>>(c->table, c->n_slots, c->k, d_in, n, d_out);
    else kc_lookup_kernel<2><<<blocks, 256, 0, c->stream>>>(c->table, c->n_slots, c->k, d_in, n, d_out);
    KC_CUDA(c, cudaGetLastError());
    ++c->n_launches;
    KC_CUDA(c, cudaMemcpyAsync(counts_host_out, d_out, out_bytes, cudaMemcpyDeviceToHost, c->stream));
    KC_CUDA(c, cudaStreamSynchronize(c->stream));
    return KH_OK;
}

int kh_count_get_stats(kh_counter* c, kh_count_stats* out) {
    if (!c || !out) return KH_ERR_ARG;
    KC_CUDA(c, cudaSetDevice(c->device));
    const int rc = kc_settle(c);
    if (rc != KH_OK && rc != KH_ERR_TABLE_FULL) return rc;
    if (c->have_count) {
        KC_CUDA(c, cudaEventElapsedTime(&c->ms_count, c->ev0, c->ev1));
        c->have_count = false;
    }
    out->n_slots = c->n_slots;
    out->n_distinct = c->h_ctr.n_distinct;
    out->n_occurrences = c->h_ctr.n_occurrences;
    out->n_bytes = c->n_bytes;
    out->n_reported = c->h_ctr.n_reported;
    out->slot_bytes = c->W == 1 ? 16u : 32u;
    out->n_launches = c->n_launches;
    out->n_grows = c->n_grows;
    out->reserved = 0;
    out->ms_count = c->ms_count;
    out->ms_extract = c->ms_extract;
    return rc;
}

const char* kh_count_last_error(kh_counter* c) { return c ? c->err.c_str() : ""; }

}  // extern "C"
