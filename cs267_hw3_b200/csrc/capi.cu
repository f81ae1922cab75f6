// capi.cu -- host runtime behind include/kh_capi.h: owns device memory, streams and the
// kernel sequence for insert (K2+K3), find (K4), assemble (K5+K6) and pack (K1).
//
// Layout in HBM (one handle = one GPU):
//   table        nbuckets x 32 B, one DRAM sector per bucket (4 x u64 or 2 x u128 slots)
//   starts       start-node slot values in input order (grow-only)
//   per insert   start bitmask (n/8 B), per-tile counts/offsets
//   per assemble link[seg] u64, seglen[seg] u8, tmp[seg][seg_chars], contig_len/pre/off, out
// Scratch is grow-only and reused across calls so a steady-state step allocates nothing.
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include <cub/device/device_radix_sort.cuh>

#include "../../include/kh_capi.h"
#include "kernels.cuh"
#include "ctable.cuh"

using namespace kh;

namespace {

struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
};

enum { EV_INS0, EV_INS1, EV_AS0, EV_WALK, EV_RANK, EV_AS1, EV_PACK0, EV_PACK1, EV_CLR0, EV_CLR1, EV_STAGE1, EV_BUILD0, EV_BUILD1, EV_COUNT };

}  // namespace

struct kh_table {
    int k = 0, W = 1, device = 0, pl = 0, pb = 0, slot_bytes = 8, per_bucket = 4;
    double lf = 0.5;
    u64 n_expected = 0, nbuckets = 0;
    cudaStream_t stream = nullptr, own_stream = nullptr, copy_stream = nullptr;
    void* table = nullptr;
    size_t table_bytes = 0;
    DevBuf starts;
    u64 n_starts = 0;
    DevBuf mask, tile_counts, tile_offs, scan_blocks;
    DevBuf part_cursor, grouped;
    DevBuf fine, chunk_cursor, overflow;          // chunked (shared-memory) build
    bool table_dirty = false;         // something was inserted since create/clear
    bool chunk_attr_set = false;
    int debug_cap_pct = 100;          // KH_DEBUG_CAP_PCT: scale the grouping buffers' capacities (tests force the overflow paths)
    bool part_attr_set = false;
    Counters* d_ctr = nullptr;
    Counters* h_ctr = nullptr;
    DevBuf link, seglen, tmp, contig_len, contig_pre, contig_off, out;
    DevBuf stage[2], text_stage, scratch_a, scratch_b, scratch_c;
    DevBuf sort_keys[2], sort_vals[2], sort_tmp;     // kh_sorted_order
    void* h_out = nullptr; size_t h_out_cap = 0;
    void* h_off = nullptr; size_t h_off_cap = 0;
    u32 split_shift = 5, seg_chars = 64;     // every 32nd bucket's first slot is a splitter (tools/probes/sweep_walk.sh)
    cudaEvent_t ev[EV_COUNT] = {};
    cudaEvent_t ev_copied[2] = {}, ev_consumed[2] = {};
    cudaEvent_t ev_built = nullptr, ev_gathered = nullptr;     // chunk table, multi-GPU: the gather of meta words + characters runs beside the link resolution
    bool have_ins = false, have_as = false, have_pack = false, have_clr = false, have_build = false, have_stage = false;
    u64 n_launches = 0;               // kernels launched by this handle since create (kh_get_stats)
    kh_stats stats = {};
    std::string err;
    int sm_count = 148, walk_blocks_per_sm = 0, rank_blocks_per_sm = 0;
    u64 last_contig_bytes = 0, last_n_contigs = 0;
    // ---- chunk table (ctable.cuh): large tables, and every sharded (multi-GPU) handle ----
    struct CtState {
        bool on = false, sealed = false, sharded = false, attr_set = false, connected = false;
        bool assembled = false;           // the segment lists were consumed by a traverse: the next one re-seals
        CtGeom g = {};
        CtCaps caps = {};
        CtPeers pe = {};
        u32 epoch = 0;                    // barriers passed (all ranks call them in lockstep)
        u64 n_local_max = 0, n_total = 0, n_starts_max = 0, out_cap = 0;
        u64 n_starts_host = 0;            // non-sharded handles learn it at every insert (they sync anyway)
        DevBuf xin_vals, xin_chunk, xin_cnt, xin_done, xout_cursor, extra_vals, extra_chunk, extra_cnt, fine, chunk_cursor,
               chunk_base, pool_off, seg_base, ext_key, meta, pool, inbox, inbox_cnt, out_cursor, flags,
               answers, req_seg, g_link, g_meta, g_pool, g_hdr;
        bool slow = false;                // this traverse ranks by pointer jumping (a contig too long for the bounded walk)
        void* ipc_opened[kMaxRanks][24] = {};
    } ct;
    int ct_env = 1;                   // KH_CT: 0 never, 1 tables of >= 2^20 k-mers (and every sharded handle), 2 always
};

namespace {

int fail(kh_table* t, int status, const std::string& msg) {
    if (t) t->err = msg;
    return status;
}

#define KH_CUDA(t, expr)                                                                         \
    do {                                                                                         \
        cudaError_t e_ = (expr);                                                                 \
        if (e_ != cudaSuccess)                                                                   \
            return fail((t), e_ == cudaErrorMemoryAllocation ? KH_ERR_NOMEM : KH_ERR_CUDA,       \
                        std::string(#expr) + ": " + cudaGetErrorString(e_));                     \
    } while (0)

#define KH_TRY(expr)                  \
    do {                              \
        const int rc_ = (expr);       \
        if (rc_ != KH_OK) return rc_; \
    } while (0)

int ensure(kh_table* t, DevBuf& b, size_t bytes, bool keep = false) {
    if (bytes <= b.cap && b.p) return KH_OK;
    const size_t want = std::max<size_t>(256, bytes + bytes / 8);
    void* np = nullptr;
    KH_CUDA(t, cudaMalloc(&np, want));
    if (b.p) {
        if (keep && b.cap) KH_CUDA(t, cudaMemcpyAsync(np, b.p, b.cap, cudaMemcpyDeviceToDevice, t->stream));
        KH_CUDA(t, cudaStreamSynchronize(t->stream));
        KH_CUDA(t, cudaFree(b.p));
    }
    b.p = np;
    b.cap = want;
    return KH_OK;
}

int ensure_pinned(kh_table* t, void*& p, size_t& cap, size_t bytes) {
    if (bytes <= cap && p) return KH_OK;
    if (p) KH_CUDA(t, cudaFreeHost(p));
    p = nullptr; cap = 0;
    const size_t want = std::max<size_t>(4096, bytes + bytes / 8);
    KH_CUDA(t, cudaHostAlloc(&p, want, cudaHostAllocDefault));
    cap = want;
    return KH_OK;
}

int status_from_errors(kh_table* t, u32 e) {
    if (e == 0) return KH_OK;
    if (e & kErrBadInput) return fail(t, KH_ERR_BAD_INPUT, "input contains a base outside ACGT or an extension outside ACGTF");
    if (e & kErrTableFull) return fail(t, KH_ERR_TABLE_FULL, "hash table is full (more distinct k-mers than slots)");
    if (e & kErrNotFound) return fail(t, KH_ERR_NOT_FOUND, "Error: k-mer not found in Distributed HashMap.");
    if (e & kErrCycle) return fail(t, KH_ERR_CYCLE, "a start-rooted chain never reaches forward extension 'F' (cycle)");
    if (e & kErrConverge) return fail(t, KH_ERR_CONVERGE, "two start nodes reach the same end node (chains are not linear)");
    return fail(t, KH_ERR_CUDA, "internal error: segment bookkeeping overflow");
}

// Pull the counters to the host (synchronises the stream).
int read_counters(kh_table* t) {
    KH_CUDA(t, cudaMemcpyAsync(t->h_ctr, t->d_ctr, sizeof(Counters), cudaMemcpyDeviceToHost, t->stream));
    KH_CUDA(t, cudaStreamSynchronize(t->stream));
    return KH_OK;
}
int clear_error_bits(kh_table* t) {
    KH_CUDA(t, cudaMemsetAsync(&t->d_ctr->errors, 0, sizeof(u32), t->stream));
    return KH_OK;
}

// exclusive scan of n u32 -> u64 (out), total -> *total_dev
int device_scan(kh_table* t, const u32* in, u64 n, u64* out, u64* total_dev) {
    const u64 nsb = (n + kScanTile - 1) / kScanTile;
    KH_TRY(ensure(t, t->scan_blocks, (nsb + 1) * sizeof(u64)));
    u64* bs = static_cast<u64*>(t->scan_blocks.p);
    scan_reduce_kernel<<<(unsigned)nsb, kScanThreads, 0, t->stream>>>(in, n, bs);
    scan_spine_kernel<<<1, 1024, 0, t->stream>>>(bs, nsb, total_dev);
    scan_apply_kernel<<<(unsigned)nsb, kScanThreads, 0, t->stream>>>(in, n, bs, out);
    t->n_launches += 3;
    KH_CUDA(t, cudaGetLastError());
    return KH_OK;
}

__global__ void init_assemble_kernel(Counters* c, u32 first_overflow_seg) {
    c->next_walker = 0;
    c->next_seg = first_overflow_seg;
    c->rank_rounds = 0;
    c->n_nodes = 0;
    c->contig_bytes = 0;
    for (int i = 0; i < 40; ++i) c->flags[i] = 0;
}

// from_record_staged reads whole aligned words around a record: keep 16 bytes behind every staging area
constexpr size_t kStageSlack = 16;

static size_t partition_smem(int W, u32 nparts, int pb) {
    const size_t un = std::max<size_t>((size_t)kPartTile * (W == 1 ? 8 : 16), (size_t)kPartTile * pb) + kStageSlack;
    return ((12 * (size_t)nparts + 2 * kPartTile + 15) & ~(size_t)15) + un;
}

// Capacity of a grouping buffer for the records whose home lies in `span` buckets of the table: their expected share
// of n plus 24 binomial sigmas and `slack`, scaled by KH_DEBUG_CAP_PCT.  The hash is uniform, so no histogram pass.
static u64 group_cap(const kh_table* t, u64 n, u64 span, double slack) {
    const double share = (double)n * (double)std::min<u64>(t->nbuckets, span) / (double)t->nbuckets;
    return (u64)(share + 24.0 * std::sqrt(share + 1.0) + slack) * t->debug_cap_pct / 100;
}

template <int W>
int insert_device_impl(kh_table* t, const unsigned char* recs, u64 n, bool record_start) {
    typedef typename Slot<W>::value_t V;
    if (n == 0) return KH_OK;
    if (n >= 0xFFF00000ull) return fail(t, KH_ERR_ARG, "at most 2^32-2^20 records per insert call; split the batch");
    const u64 ntiles = (n + kInsTile - 1) / kInsTile;
    KH_TRY(ensure(t, t->mask, (ntiles + 1) * (kInsTile / 32) * sizeof(u32)));
    KH_TRY(ensure(t, t->tile_counts, (ntiles + 1) * sizeof(u32)));
    KH_TRY(ensure(t, t->tile_offs, (ntiles + 1) * sizeof(u64)));
    // Tables larger than L2 get their records grouped by table region first (see kernels.cuh K2p).
    const bool part = t->table_bytes > (64ull << 20) && n >= (1u << 16);
    // Large batches (>= 1/8 of the table's slots) are built chunk by chunk in shared memory: no global atomics.
    // Measured against insert_slots: faster with 64-bit slots (2.85 vs 3.03 ms), slower with 128-bit slots (4.6 vs
    // 4.1 ms: twice the bytes through the two grouping passes), so the chunked build is the 64-bit path only.
    const bool chunked = W == 1 && part && n * 8 >= t->nbuckets * (u64)t->per_bucket;
    u32 part_shift = 0, nparts = 1;
    u64 part_cap = 0;
    if (part) {
        if (chunked) part_shift = kChunkShift + 7;                     // 128 chunks (8 MB of table) per partition
        else while ((32ull << part_shift) < kPartBytes) ++part_shift;
        while (((t->nbuckets - 1) >> part_shift) + 1 > (u64)kMaxParts) ++part_shift;
        if (chunked && part_shift - kChunkShift > 10) return fail(t, KH_ERR_ARG, "table too large for the chunked build");
        nparts = (u32)(((t->nbuckets - 1) >> part_shift) + 1);
        // rounded to whole insert tiles; overflow falls back to a direct insert (or the chunked build's fix-up list)
        part_cap = (group_cap(t, n, 1ull << part_shift, 64.0) + kInsTile - 1) / kInsTile * kInsTile;
        KH_TRY(ensure(t, t->part_cursor, kMaxParts * sizeof(u32)));
        KH_TRY(ensure(t, t->grouped, (u64)nparts * part_cap * sizeof(V)));
        if (!t->part_attr_set) {
            KH_CUDA(t, cudaFuncSetAttribute(partition_kernel<W>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                            (int)partition_smem(W, kMaxParts, 18)));
            t->part_attr_set = true;
        }
    }
    u32 chunk_cap = 0, overflow_cap = 0;
    u64 nchunks = 0;
    if (chunked) {
        nchunks = (t->nbuckets + kChunkBuckets - 1) >> kChunkShift;
        chunk_cap = std::max(4u, ((u32)group_cap(t, n, kChunkBuckets, 32.0) + 3u) & ~3u);
        overflow_cap = (u32)std::min<u64>(0x7FFFFFFFull, t->debug_cap_pct < 100 ? n + 65536 : n / 32 + 65536);
        KH_TRY(ensure(t, t->fine, nchunks * (u64)chunk_cap * sizeof(V)));
        KH_TRY(ensure(t, t->chunk_cursor, nchunks * sizeof(u32)));
        KH_TRY(ensure(t, t->overflow, (u64)overflow_cap * sizeof(V)));
        if (!t->chunk_attr_set) {
            KH_CUDA(t, cudaFuncSetAttribute(build_chunks_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(kChunkBuckets * 32)));
            t->chunk_attr_set = true;
        }
    }
    if (record_start) KH_CUDA(t, cudaEventRecord(t->ev[EV_INS0], t->stream));
    if (!part) {
        insert_kernel<W><<<(unsigned)ntiles, kInsThreads, (size_t)kInsTile * t->pb + kStageSlack, t->stream>>>(
            recs, n, t->k, static_cast<V*>(t->table), t->nbuckets, static_cast<u32*>(t->mask.p),
            static_cast<u32*>(t->tile_counts.p), t->d_ctr);
    } else if (chunked) {
        if constexpr (W == 1) {
            KH_CUDA(t, cudaMemsetAsync(t->part_cursor.p, 0, kMaxParts * sizeof(u32), t->stream));
            KH_CUDA(t, cudaMemsetAsync(t->chunk_cursor.p, 0, nchunks * sizeof(u32), t->stream));
            KH_CUDA(t, cudaMemsetAsync(&t->d_ctr->n_outbox, 0, sizeof(u32), t->stream));
            const u64 pblocks = (n + kPartTile - 1) / kPartTile;
            partition_kernel<W><<<(unsigned)pblocks, kPartThreads, partition_smem(W, nparts, t->pb), t->stream>>>(
                recs, n, t->k, t->nbuckets, part_shift, nparts, part_cap, static_cast<u32*>(t->part_cursor.p),
                static_cast<V*>(t->grouped.p), static_cast<V*>(t->table), static_cast<u32*>(t->mask.p),
                static_cast<u32*>(t->tile_counts.p), static_cast<V*>(t->overflow.p), overflow_cap, t->d_ctr);
            const u32 bpp = (u32)((part_cap + kSubTile - 1) / kSubTile), nsub = 1u << (part_shift - kChunkShift);
            subpartition_kernel<<<nparts * bpp, kSubThreads, 8 * (size_t)nsub + 16, t->stream>>>(
                static_cast<const V*>(t->grouped.p), static_cast<const u32*>(t->part_cursor.p), part_cap, bpp, kChunkShift,
                nsub, t->nbuckets, chunk_cap, static_cast<u32*>(t->chunk_cursor.p), static_cast<V*>(t->fine.p),
                static_cast<V*>(t->overflow.p), overflow_cap, t->d_ctr);
            build_chunks_kernel<<<(unsigned)nchunks, kBuildThreads, kChunkBuckets * 32, t->stream>>>(
                static_cast<const V*>(t->fine.p), static_cast<const u32*>(t->chunk_cursor.p), chunk_cap, static_cast<V*>(t->table),
                t->nbuckets, t->table_dirty ? 1 : 0, static_cast<V*>(t->overflow.p), overflow_cap, t->d_ctr);
            insert_overflow_kernel<<<64, 256, 0, t->stream>>>(static_cast<const V*>(t->overflow.p), overflow_cap,
                                                             static_cast<V*>(t->table), t->nbuckets, t->d_ctr);
        }
    } else {
        KH_CUDA(t, cudaMemsetAsync(t->part_cursor.p, 0, kMaxParts * sizeof(u32), t->stream));
        const u64 warm_buckets = std::min<u64>(t->nbuckets, (u64)kWarmAhead << part_shift);
        warm_kernel<<<(unsigned)t->sm_count * 4, 256, 0, t->stream>>>(static_cast<const char*>(t->table),
                                                                     (warm_buckets * 32 + 127) >> 7);
        const u64 pblocks = (n + kPartTile - 1) / kPartTile;
        partition_kernel<W><<<(unsigned)pblocks, kPartThreads, partition_smem(W, nparts, t->pb), t->stream>>>(
            recs, n, t->k, t->nbuckets, part_shift, nparts, part_cap, static_cast<u32*>(t->part_cursor.p),
            static_cast<V*>(t->grouped.p), static_cast<V*>(t->table), static_cast<u32*>(t->mask.p),
            static_cast<u32*>(t->tile_counts.p), static_cast<V*>(nullptr), 0u, t->d_ctr);
        const u32 bpp = (u32)(part_cap / kInsTile);
        const unsigned iblocks = nparts * bpp;
        insert_slots_kernel<W><<<iblocks, kInsThreads, 0, t->stream>>>(
            static_cast<const V*>(t->grouped.p), static_cast<const u32*>(t->part_cursor.p), part_cap, bpp, nparts,
            part_shift, static_cast<V*>(t->table), t->nbuckets, t->d_ctr);
    }
    t->table_dirty = true;
    t->n_launches += !part ? 1 : (chunked ? 4 : 3);
    KH_CUDA(t, cudaGetLastError());
    KH_TRY(device_scan(t, static_cast<u32*>(t->tile_counts.p), ntiles, static_cast<u64*>(t->tile_offs.p),
                       &t->d_ctr->scan_total));
    KH_TRY(read_counters(t));     // number of new start nodes (sizes the start list) + error bits
    const u32 e = t->h_ctr->errors;
    if (e) {
        clear_error_bits(t);
        return status_from_errors(t, e);
    }
    const u64 fresh = t->h_ctr->scan_total;
    if (fresh) {
        KH_TRY(ensure(t, t->starts, (t->n_starts + fresh) * sizeof(V), /*keep=*/true));
        const u64 threads = ntiles * 32;
        scatter_starts_kernel<W><<<(unsigned)((threads + 255) / 256), 256, 0, t->stream>>>(
            recs, n, t->k, static_cast<u32*>(t->mask.p), static_cast<u64*>(t->tile_offs.p), ntiles,
            static_cast<V*>(t->starts.p), t->n_starts);
        KH_CUDA(t, cudaGetLastError());
        t->n_starts += fresh;
        ++t->n_launches;
    }
    KH_CUDA(t, cudaEventRecord(t->ev[EV_INS1], t->stream));
    t->have_ins = true;
    return KH_OK;
}

template <int W> int ct_insert_plain(kh_table* t, const unsigned char* recs, u64 n, bool record_start);
template <int W> int ct_assemble_plain(kh_table* t);
template <int W> int ct_seal_plain(kh_table* t);

int insert_device(kh_table* t, const void* recs, u64 n, bool record_start = true) {
    if (t->ct.on) {
        if (t->ct.sharded) return fail(t, KH_ERR_ARG, "sharded handle: use kh_shard_insert");
        return t->W == 1 ? ct_insert_plain<1>(t, static_cast<const unsigned char*>(recs), n, record_start)
                         : ct_insert_plain<2>(t, static_cast<const unsigned char*>(recs), n, record_start);
    }
    return t->W == 1 ? insert_device_impl<1>(t, static_cast<const unsigned char*>(recs), n, record_start)
                     : insert_device_impl<2>(t, static_cast<const unsigned char*>(recs), n, record_start);
}

int pack_device(kh_table* t, const void* text_dev, u64 n_lines, void* pairs_dev) {
    if (n_lines == 0) return KH_OK;
    const u64 nblk = (n_lines + kPackLines - 1) / kPackLines;
    if (nblk > 0x7FFFFFFFull) return fail(t, KH_ERR_ARG, "too many lines in one pack call");
    const size_t smem = (((size_t)kPackLines * (t->k + 4) + 8 + 15) & ~(size_t)15) + (size_t)kPackLines * t->pb;
    pack_lines_kernel<<<(unsigned)nblk, kPackLines, smem, t->stream>>>(
        static_cast<const unsigned char*>(text_dev), n_lines, t->k, static_cast<unsigned char*>(pairs_dev), t->d_ctr);
    KH_CUDA(t, cudaGetLastError());
    ++t->n_launches;
    return KH_OK;
}

template <int W>
int assemble_impl(kh_table* t) {
    typedef typename Slot<W>::value_t V;
    const u64 n_starts = t->n_starts;
    const u64 n_split = ((t->nbuckets - 1) >> t->split_shift) + 1;
    if (n_starts + n_split >= 0xFFF00000ull) return fail(t, KH_ERR_ARG, "too many walk segments for 32-bit ids");
    if (t->walk_blocks_per_sm == 0) {
        KH_CUDA(t, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&t->walk_blocks_per_sm, walk_kernel<W>, kWalkThreads, 0));
        KH_CUDA(t, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&t->rank_blocks_per_sm, rank_kernel, 256, 0));
        if (t->walk_blocks_per_sm < 1 || t->rank_blocks_per_sm < 1) return fail(t, KH_ERR_CUDA, "kernel does not fit on an SM");
    }
    const u64 n_keys = t->h_ctr->n_inserted;     // refreshed by the last insert
    u64 walkers = n_starts + n_split;
    unsigned walk_blocks = (unsigned)std::min<u64>((u64)t->sm_count * t->walk_blocks_per_sm,
                                                    (walkers + kWalkThreads - 1) / kWalkThreads);
    walk_blocks = std::max(walk_blocks, 1u);
    const u64 nwarps = (u64)walk_blocks * (kWalkThreads / 32);
    const u64 seg_cap = walkers + 2 * (n_keys / t->seg_chars + 1) + (u64)kSegBatch * nwarps + 64;
    if (seg_cap >= 0xFFFFFFF0ull) return fail(t, KH_ERR_ARG, "too many walk segments for 32-bit ids");
    KH_TRY(ensure(t, t->link, seg_cap * sizeof(u64)));
    KH_TRY(ensure(t, t->seglen, seg_cap));
    KH_TRY(ensure(t, t->tmp, seg_cap * (u64)t->seg_chars + 16));
    KH_TRY(ensure(t, t->contig_len, (n_starts + 1) * sizeof(u32)));
    KH_TRY(ensure(t, t->contig_pre, (n_starts + 1) * sizeof(u32)));
    KH_TRY(ensure(t, t->contig_off, (n_starts + 1) * sizeof(u64)));
    const u64 out_cap = n_keys + n_starts * (u64)(t->k + 1) + 64;
    KH_TRY(ensure(t, t->out, out_cap));

    KH_CUDA(t, cudaEventRecord(t->ev[EV_AS0], t->stream));
    init_assemble_kernel<<<1, 1, 0, t->stream>>>(t->d_ctr, (u32)walkers);
    KH_CUDA(t, cudaMemsetAsync(static_cast<u32*>(t->contig_len.p) + n_starts, 0, sizeof(u32), t->stream));

    WalkParams wp;
    wp.table = t->table; wp.nbuckets = t->nbuckets; wp.starts = t->starts.p;
    wp.link = static_cast<u64*>(t->link.p); wp.seglen = static_cast<unsigned char*>(t->seglen.p);
    wp.tmp = static_cast<unsigned char*>(t->tmp.p); wp.ctr = t->d_ctr;
    wp.n_starts = (u32)n_starts; wp.n_split = (u32)n_split; wp.split_shift = t->split_shift;
    wp.seg_chars = t->seg_chars; wp.seg_cap = (u32)seg_cap; wp.k = t->k;
    walk_kernel<W><<<walk_blocks, kWalkThreads, 0, t->stream>>>(wp);
    KH_CUDA(t, cudaGetLastError());
    KH_CUDA(t, cudaEventRecord(t->ev[EV_WALK], t->stream));

    RankParams rp;
    rp.link = wp.link; rp.seglen = wp.seglen; rp.ctr = t->d_ctr;
    rp.contig_len = static_cast<u32*>(t->contig_len.p); rp.contig_pre = static_cast<u32*>(t->contig_pre.p);
    rp.n_starts = (u32)n_starts; rp.seg_cap = (u32)seg_cap; rp.k = t->k; rp.max_rounds = 34;
    void* rargs[] = {&rp};
    const unsigned rank_blocks = (unsigned)std::max<u64>(1, std::min<u64>((u64)t->sm_count * t->rank_blocks_per_sm,
                                                                            (seg_cap + 255) / 256));
    KH_CUDA(t, cudaLaunchCooperativeKernel((void*)rank_kernel, dim3(rank_blocks), dim3(256), rargs, 0, t->stream));
    KH_TRY(device_scan(t, rp.contig_len, n_starts + 1, static_cast<u64*>(t->contig_off.p), &t->d_ctr->contig_bytes));
    KH_CUDA(t, cudaEventRecord(t->ev[EV_RANK], t->stream));

    emit_segments_kernel<<<(unsigned)((seg_cap + 255) / 256), 256, 0, t->stream>>>(
        wp.link, wp.seglen, wp.tmp, t->seg_chars, (u32)seg_cap, t->d_ctr, rp.contig_pre,
        static_cast<u64*>(t->contig_off.p), t->k, out_cap, static_cast<char*>(t->out.p));
    if (n_starts) {
        const u64 head_threads = n_starts * (u64)(t->k + 1);
        emit_heads_kernel<W><<<(unsigned)((head_threads + 255) / 256), 256, 0, t->stream>>>(
            static_cast<const V*>(t->starts.p), (u32)n_starts, t->k, rp.contig_len,
            static_cast<u64*>(t->contig_off.p), t->d_ctr, out_cap, static_cast<char*>(t->out.p));
    }
    KH_CUDA(t, cudaGetLastError());
    t->n_launches += 4 + (n_starts ? 1 : 0);        // init, walk, rank, emit_segments (+ emit_heads); the scan counted itself
    KH_CUDA(t, cudaEventRecord(t->ev[EV_AS1], t->stream));
    t->have_as = true;

    KH_TRY(read_counters(t));
    t->stats.n_contigs = n_starts;
    t->stats.n_nodes = t->h_ctr->n_nodes;
    t->stats.contig_bytes = t->h_ctr->contig_bytes;
    t->stats.n_segments = std::min<u64>(t->h_ctr->next_seg, seg_cap);
    t->stats.rank_rounds = t->h_ctr->rank_rounds;
    t->last_contig_bytes = t->h_ctr->contig_bytes;
    t->last_n_contigs = n_starts;
    const u32 e = t->h_ctr->errors;
    if (e) {
        clear_error_bits(t);
        return status_from_errors(t, e);
    }
    if (t->h_ctr->contig_bytes > out_cap)
        return fail(t, KH_ERR_CONVERGE, "contigs cover more k-mers than were inserted (chains share nodes)");
    return KH_OK;
}

int assemble_device(kh_table* t) {
    if (t->ct.on) {
        if (t->ct.sharded) return fail(t, KH_ERR_ARG, "sharded handle: use kh_shard_assemble");
        return t->W == 1 ? ct_assemble_plain<1>(t) : ct_assemble_plain<2>(t);
    }
    return t->W == 1 ? assemble_impl<1>(t) : assemble_impl<2>(t);
}

float elapsed(cudaEvent_t a, cudaEvent_t b) {
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, a, b) != cudaSuccess) { cudaGetLastError(); return 0.f; }
    return ms;
}

int env_int(const char* name, int dflt) {
    const char* v = getenv(name);
    return (v && *v) ? atoi(v) : dflt;
}

int set_option(kh_table* t, const std::string& name, int64_t value) {
    if (name == "split_buckets") {
        if (value < 1 || value > (1 << 20) || (value & (value - 1))) return fail(t, KH_ERR_ARG, "split_buckets must be a power of two in [1, 2^20]");
        u32 s = 0;
        while ((1ll << s) < value) ++s;
        t->split_shift = s;
        return KH_OK;
    }
    if (name == "seg_chars") {
        if (value < 8 || value > 248 || (value & 7)) return fail(t, KH_ERR_ARG, "seg_chars must be a multiple of 8 in [8, 248]");
        t->seg_chars = (u32)value;
        return KH_OK;
    }
    return fail(t, KH_ERR_ARG, "unknown option " + name);
}

}  // namespace

// ============================================================================ chunk table ====
// Host side of ctable.cuh.  A handle is either a plain table (small tables: insert_kernel / walk_kernel above)
// or a chunk table (ct.on).  Every sharded handle is a chunk table; a plain handle with world = 1 uses the very
// same code with itself as its only peer.
namespace {

enum { CTX_XIN_VALS, CTX_XIN_CHUNK, CTX_XIN_CNT, CTX_EXTRA_VALS, CTX_EXTRA_CHUNK, CTX_EXTRA_CNT, CTX_LINK, CTX_META,
       CTX_INBOX, CTX_INBOX_CNT, CTX_PRE, CTX_OFF, CTX_OUT, CTX_FLAGS, CTX_ANSWERS, CTX_GLINK, CTX_GMETA, CTX_GPOOL, CTX_GHDR, CTX_NBUF };

size_t ct_stage_smem(int W, int world) {       // multi-GPU: the remote values of a tile sorted by owner + their chunk ids
    return world > 1 ? (size_t)kStgTile * ((W == 1 ? 8 : 16) + 4) : 0;
}

void ct_set_self(kh_table* t) {
    auto& c = t->ct;
    CtPeers& pe = c.pe;
    const int r = pe.rank;
    pe.xin_vals[r] = c.xin_vals.p; pe.xin_chunk[r] = static_cast<u32*>(c.xin_chunk.p);
    pe.xin_cnt[r] = static_cast<u32*>(c.xin_cnt.p);
    pe.extra_vals[r] = c.extra_vals.p; pe.extra_chunk[r] = static_cast<u32*>(c.extra_chunk.p);
    pe.extra_cnt[r] = static_cast<u32*>(c.extra_cnt.p);
    pe.link[r] = static_cast<u64*>(t->link.p); pe.meta[r] = static_cast<u64*>(c.meta.p);
    pe.inbox[r] = c.inbox.p; pe.inbox_cnt[r] = static_cast<u32*>(c.inbox_cnt.p);
    pe.contig_pre[r] = static_cast<u32*>(t->contig_pre.p); pe.contig_off[r] = static_cast<u64*>(t->contig_off.p);
    pe.out[r] = static_cast<char*>(t->out.p); pe.out_cap[r] = c.out_cap;
    pe.flags[r] = static_cast<u32*>(c.flags.p);
    pe.answers[r] = static_cast<u32*>(c.answers.p);
    pe.g_link[r] = static_cast<u64*>(c.g_link.p); pe.g_meta[r] = static_cast<u64*>(c.g_meta.p);
    pe.g_pool[r] = static_cast<unsigned char*>(c.g_pool.p); pe.g_hdr[r] = static_cast<u32*>(c.g_hdr.p);
}

// empty staging: cursors of the chunk buffers, of the send side and of the receive side
int ct_reset_staging(kh_table* t) {
    auto& c = t->ct;
    KH_CUDA(t, cudaMemsetAsync(c.chunk_cursor.p, 0, ((u64)c.g.chunks_per_rank + 1) * sizeof(u32), t->stream));
    KH_CUDA(t, cudaMemsetAsync(c.xout_cursor.p, 0, kMaxRanks * sizeof(u32), t->stream));
    KH_CUDA(t, cudaMemsetAsync(c.xin_cnt.p, 0, kMaxRanks * sizeof(u32), t->stream));
    KH_CUDA(t, cudaMemsetAsync(c.xin_done.p, 0, (kMaxRanks + 1) * sizeof(u32), t->stream));
    KH_CUDA(t, cudaMemsetAsync(c.extra_cnt.p, 0, 16, t->stream));
    return KH_OK;
}

// Fix the geometry and (re)allocate everything whose size is known up front.  Sharded handles allocate ALL their
// buffers here: nothing inside a step may block the host (another rank's barrier kernel may be waiting for work this
// host thread has not enqueued yet).
template <int W>
int ct_setup(kh_table* t, int rank, int world, u64 n_local_max, u64 n_total, u64 n_starts_max, bool sharded) {
    typedef typename Slot<W>::value_t V;
    auto& c = t->ct;
    const u64 n_exp = std::max<u64>(t->n_expected, 1);
    const u32 slots_max = CtBuild<W>::kMaxSlots, per_bucket = (u32)Slot<W>::kPerBucket;
    const double mu = std::min(t->lf / 1.35, 0.55) * slots_max;                   // mean k-mers per chunk (see chunk_placement_sim.cpp)
    const u64 C64 = std::max<u64>(1, (u64)std::ceil((double)n_exp / mu));
    if (C64 * (u64)world > (1ull << 24)) return fail(t, KH_ERR_ARG, "table too large for the chunk table (more than 2^24 chunks)");
    c.g.k = t->k; c.g.m = ct_minimizer_len(t->k); c.g.win = ct_window(t->k);
    c.g.world = world; c.g.rank = rank;
    c.g.chunks_per_rank = (u32)C64;
    c.g.max_buckets = CtBuild<W>::kMaxBuckets;
    c.g.lf_inv_q16 = (u32)std::min(65536.0 * 64.0, 65536.0 / t->lf + 0.5);
    const u64 C = C64;
    c.n_local_max = n_local_max; c.n_total = n_total; c.n_starts_max = n_starts_max; c.sharded = sharded;
    // table: every chunk gets ceil(load / lf) slots rounded up to whole buckets
    const u64 nb_alloc = (u64)((long double)n_exp / (long double)t->lf / per_bucket) + C + 64;
    if (!t->table || t->table_bytes < nb_alloc * 32) {
        if (t->table) { KH_CUDA(t, cudaStreamSynchronize(t->stream)); KH_CUDA(t, cudaFree(t->table)); t->table = nullptr; }
        KH_CUDA(t, cudaMalloc(&t->table, nb_alloc * 32));
        t->table_bytes = nb_alloc * 32;
    }
    t->nbuckets = nb_alloc;
    c.caps.nbuckets_alloc = nb_alloc;
    // receive buffer for the records other GPUs parse for this one: one part per source rank
    const double share = (double)std::max<u64>(n_local_max, 1) / (double)world;
    u64 xin_cap = world > 1 ? (u64)((share * 1.05 + 64.0 * std::sqrt(share + 1.0) + 4096.0) * t->debug_cap_pct / 100.0) : 8;
    xin_cap = std::max<u64>(8, (xin_cap + 7) & ~7ull);
    if (xin_cap >= 0xFFFFFFF0ull) return fail(t, KH_ERR_ARG, "receive buffer too large");
    c.caps.xin_cap = (u32)xin_cap;
    c.caps.extra_cap = (u32)std::min<u64>(0x7FFFFFF0ull, t->debug_cap_pct < 100 ? n_local_max * (u64)world + 65536 : n_exp / 16 + 65536);
    const u64 hcap = sharded ? std::min<u64>(std::max<u64>(n_starts_max, 1), n_local_max + 1) : 0;     // plain handles size it at seal
    c.caps.hcap = (u32)hcap;
    const u64 seg_cap = hcap + n_exp + 64;
    if (seg_cap >= (u64)kLocalMask - 16 && sharded) return fail(t, KH_ERR_ARG, "too many segments per GPU for 28-bit local ids");
    c.caps.seg_cap = (u32)std::min<u64>(seg_cap, 0xFFFFFF00ull);
    c.caps.pool_cap = n_exp + 16 * C + 64;
    // every rank must arrive at the SAME capacities for the buffers its peers index (staging, extras, inbox): they
    // may depend on n_total, n_local_max, the load factor and K only -- never on this rank's own start-node count
    c.caps.inbox_cap = world > 1 ? (u32)std::min<u64>(0x7FFFFFF0ull, ((n_exp + n_local_max) / world) * 9 / 8 + 4096) : 1;
    c.out_cap = n_total + std::max<u64>(n_starts_max, 1) * (u64)(t->k + 1) + 64;
    KH_TRY(ensure(t, c.xin_vals, (u64)world * xin_cap * sizeof(V)));
    KH_TRY(ensure(t, c.xin_chunk, (u64)world * xin_cap * sizeof(u32)));
    KH_TRY(ensure(t, c.xin_cnt, kMaxRanks * sizeof(u32)));
    KH_TRY(ensure(t, c.xin_done, (kMaxRanks + 1) * sizeof(u32)));          // [kMaxRanks] = extras already filed
    KH_TRY(ensure(t, c.xout_cursor, kMaxRanks * sizeof(u32)));
    KH_TRY(ensure(t, c.extra_vals, (u64)c.caps.extra_cap * sizeof(V)));
    KH_TRY(ensure(t, c.extra_chunk, (u64)c.caps.extra_cap * sizeof(u32)));
    KH_TRY(ensure(t, c.extra_cnt, 16));
    KH_TRY(ensure(t, c.fine, C * (u64)((slots_max + 15) & ~15u) * sizeof(V)));      // position-major groups of a 128-byte line (ct_fine_index)
    KH_TRY(ensure(t, c.chunk_cursor, (C + 1) * sizeof(u32)));
    KH_TRY(ensure(t, c.chunk_base, (C + 2) * sizeof(u32)));
    KH_TRY(ensure(t, c.pool_off, (C + 2) * sizeof(u32)));
    KH_TRY(ensure(t, c.seg_base, (C + 1) * sizeof(u32)));
    KH_TRY(ensure(t, c.pool, c.caps.pool_cap + 64));
    KH_TRY(ensure(t, c.inbox, (u64)world * c.caps.inbox_cap * sizeof(CtReq<W>)));
    KH_TRY(ensure(t, c.inbox_cnt, kMaxRanks * sizeof(u32)));
    KH_TRY(ensure(t, c.out_cursor, kMaxRanks * sizeof(u32)));
    KH_TRY(ensure(t, c.flags, 2 * kMaxRanks * sizeof(u32)));
    // answers to this rank's link requests, and the copies of the other ranks' segment arrays the contig walk reads
    c.caps.g_seg_stride = world > 1 ? ((n_local_max + 1 + n_exp + 64 + 15) & ~15ull) : 0;
    c.caps.g_pool_stride = world > 1 ? ((c.caps.pool_cap + 64 + 15) & ~15ull) : 0;
    KH_TRY(ensure(t, c.answers, std::max<u64>(16, (u64)(world > 1 ? world : 0) * c.caps.inbox_cap * sizeof(u32))));
    KH_TRY(ensure(t, c.req_seg, std::max<u64>(16, (u64)(world > 1 ? world : 0) * c.caps.inbox_cap * sizeof(u32))));
    KH_TRY(ensure(t, c.g_link, std::max<u64>(16, (u64)world * c.caps.g_seg_stride * sizeof(u64))));
    KH_TRY(ensure(t, c.g_meta, std::max<u64>(16, (u64)world * c.caps.g_seg_stride * sizeof(u64))));
    KH_TRY(ensure(t, c.g_pool, std::max<u64>(16, (u64)world * c.caps.g_pool_stride)));
    KH_TRY(ensure(t, c.g_hdr, 2 * kMaxRanks * sizeof(u32)));
    if (sharded) {
        KH_TRY(ensure(t, t->link, seg_cap * sizeof(u64)));
        KH_TRY(ensure(t, c.meta, seg_cap * sizeof(u64)));
        KH_TRY(ensure(t, c.ext_key, seg_cap * sizeof(V)));
        KH_TRY(ensure(t, t->contig_len, (hcap + 2) * sizeof(u32)));
        KH_TRY(ensure(t, t->contig_pre, (hcap + 2) * sizeof(u32)));
        KH_TRY(ensure(t, t->contig_off, (hcap + 2) * sizeof(u64)));
        KH_TRY(ensure(t, t->out, c.out_cap));
        KH_TRY(ensure(t, t->starts, (hcap + 1) * sizeof(V)));
        const u64 ntiles = (n_local_max + kInsTile - 1) / kInsTile + 1;
        KH_TRY(ensure(t, t->mask, (ntiles + 1) * (kInsTile / 32) * sizeof(u32)));
        KH_TRY(ensure(t, t->tile_counts, (ntiles + 1) * sizeof(u32)));
        KH_TRY(ensure(t, t->tile_offs, (ntiles + 1) * sizeof(u64)));
        KH_TRY(ensure(t, t->scan_blocks, ((std::max(ntiles, hcap + 2) + kScanTile - 1) / kScanTile + 2) * sizeof(u64)));
    }
    KH_TRY(ct_reset_staging(t));
    KH_CUDA(t, cudaMemsetAsync(c.inbox_cnt.p, 0, kMaxRanks * sizeof(u32), t->stream));
    KH_CUDA(t, cudaMemsetAsync(c.flags.p, 0, 2 * kMaxRanks * sizeof(u32), t->stream));
    KH_CUDA(t, cudaStreamSynchronize(t->stream));
    if (!c.attr_set) {
        KH_CUDA(t, cudaFuncSetAttribute(ct_build_kernel<W>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)CtBuild<W>::kSmem));
        KH_CUDA(t, cudaFuncSetAttribute(ct_build_kernel<W>, cudaFuncAttributePreferredSharedMemoryCarveout, (int)cudaSharedmemCarveoutMaxShared));
        KH_CUDA(t, cudaFuncSetAttribute(ct_stage_kernel<W>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ct_stage_smem(W, 8)));
        c.attr_set = true;
    }
    memset(&c.pe, 0, sizeof(c.pe));
    c.pe.world = world; c.pe.rank = rank;
    c.epoch = 0;
    ct_set_self(t);
    c.on = true; c.sealed = false;
    return KH_OK;
}

int ct_barrier(kh_table* t, int round = -1) {
    auto& c = t->ct;
    if (c.pe.world <= 1) return KH_OK;
    ++c.epoch;
    ct_barrier_kernel<<<1, 32, 0, t->stream>>>(c.pe, c.epoch & 0x7FFFFFFFu, t->d_ctr, round);
    ++t->n_launches;
    KH_CUDA(t, cudaGetLastError());
    return KH_OK;
}

// K2+K3 on a chunk table: stage the records in their owners' memory, register the start nodes in input order
template <int W>
int ct_stage(kh_table* t, const unsigned char* recs, u64 n) {
    typedef typename Slot<W>::value_t V;
    auto& c = t->ct;
    if (n == 0) return KH_OK;
    if (n >= 0xFFF00000ull) return fail(t, KH_ERR_ARG, "at most 2^32-2^20 records per insert call; split the batch");
    const u64 ntiles = (n + kInsTile - 1) / kInsTile;
    if (!c.sharded) {
        KH_TRY(ensure(t, t->mask, (ntiles + 1) * (kInsTile / 32) * sizeof(u32)));
        KH_TRY(ensure(t, t->tile_counts, (ntiles + 1) * sizeof(u32)));
        KH_TRY(ensure(t, t->tile_offs, (ntiles + 1) * sizeof(u64)));
        KH_TRY(ensure(t, t->scan_blocks, ((ntiles + kScanTile - 1) / kScanTile + 2) * sizeof(u64)));
        // the start list may have to hold every record of this call
        KH_TRY(ensure(t, t->starts, (c.n_starts_host + n + 1) * sizeof(V), /*keep=*/true));
        c.caps.hcap = (u32)std::min<u64>(0xFFFFFF00ull, c.n_starts_host + n + 1);        // bound for this call's start scatter only
    } else if (n > c.n_local_max) {
        return fail(t, KH_ERR_ARG, "more records than kh_shard_init reserved (n_local_max)");
    }
    ct_stage_kernel<W><<<(unsigned)((n + kStgTile - 1) / kStgTile), kStgThreads, ct_stage_smem(W, c.g.world), t->stream>>>(
        recs, n, c.g, c.pe, c.caps, static_cast<u32*>(c.chunk_cursor.p), static_cast<V*>(c.fine.p), static_cast<u32*>(c.xout_cursor.p),
        static_cast<u32*>(t->mask.p), static_cast<u32*>(t->tile_counts.p), t->d_ctr);
    KH_CUDA(t, cudaGetLastError());
    KH_TRY(device_scan(t, static_cast<u32*>(t->tile_counts.p), ntiles, static_cast<u64*>(t->tile_offs.p), &t->d_ctr->scan_total));
    ct_scatter_starts_kernel<W><<<(unsigned)((ntiles * 32 + 255) / 256), 256, 0, t->stream>>>(
        recs, n, t->k, static_cast<u32*>(t->mask.p), static_cast<u64*>(t->tile_offs.p), ntiles, static_cast<V*>(t->starts.p),
        t->d_ctr, c.caps.hcap);
    ct_bump_starts_kernel<<<1, 1, 0, t->stream>>>(t->d_ctr, c.caps.hcap);
    KH_CUDA(t, cudaGetLastError());
    t->n_launches += 3;
    KH_CUDA(t, cudaEventRecord(t->ev[EV_STAGE1], t->stream));
    t->have_stage = true;
    c.sealed = false; c.assembled = false;
    t->table_dirty = true;
    return KH_OK;
}

__global__ void ct_init_seal_kernel(Counters* c, u32 hcap) {
    c->next_seg = hcap;
    c->n_inserted = 0;
    c->n_duplicates = 0;
}
__global__ void ct_init_assemble_kernel(Counters* c) {
    c->n_nodes = 0;
    c->contig_bytes = 0;
    c->rank_rounds = 0;
    c->rank_done = 0;
    c->need_jump = 0;
    c->use_jump = 0;
    for (int i = 0; i < 40; ++i) c->flags[i] = 0;
}
__global__ void ct_reset_nodes_kernel(Counters* c) { c->n_nodes = 0; }

// seal, part 0: tell the owners how much they received (then a barrier); part 1: file it, lay out, build + contract
template <int W>
int ct_seal_publish(kh_table* t) {
    auto& c = t->ct;
    if (c.pe.world > 1) {
        ct_publish_xin_kernel<<<1, 32, 0, t->stream>>>(c.pe, c.caps, static_cast<const u32*>(c.xout_cursor.p));
        ++t->n_launches;
        KH_CUDA(t, cudaGetLastError());
    }
    return ct_barrier(t);
}
template <int W>
int ct_seal_build(kh_table* t) {
    typedef typename Slot<W>::value_t V;
    auto& c = t->ct;
    const u32 C = c.g.chunks_per_rank;
    if (!c.sharded) {                 // plain handle: the host knows the start count (every insert call synchronises)
        const u64 hcap = c.n_starts_host + 1;
        const u64 seg_cap = hcap + std::max<u64>(t->n_expected, 1) + 64;
        if (seg_cap >= 0xFFFFFF00ull) return fail(t, KH_ERR_ARG, "too many segments for 32-bit ids");
        c.caps.hcap = (u32)hcap; c.caps.seg_cap = (u32)seg_cap;
        KH_TRY(ensure(t, t->link, seg_cap * sizeof(u64)));
        KH_TRY(ensure(t, c.meta, seg_cap * sizeof(u64)));
        KH_TRY(ensure(t, c.ext_key, seg_cap * sizeof(V)));
        ct_set_self(t);
    }
    ct_init_seal_kernel<<<1, 1, 0, t->stream>>>(t->d_ctr, c.caps.hcap);
    if (c.pe.world > 1) {
        u32* done = static_cast<u32*>(c.xin_done.p);
        ct_xin_scatter_kernel<W><<<(unsigned)t->sm_count * 8, 256, 0, t->stream>>>(
            static_cast<const V*>(c.xin_vals.p), static_cast<const u32*>(c.xin_chunk.p), static_cast<const u32*>(c.xin_cnt.p), done,
            c.g, c.caps, static_cast<u32*>(c.chunk_cursor.p), static_cast<V*>(c.fine.p), t->d_ctr);
        ct_extra_kernel<W><<<64, 256, 0, t->stream>>>(static_cast<const V*>(c.extra_vals.p), static_cast<const u32*>(c.extra_chunk.p),
                                                      static_cast<const u32*>(c.extra_cnt.p), done + kMaxRanks, c.caps, C,
                                                      static_cast<u32*>(c.chunk_cursor.p), static_cast<V*>(c.fine.p), t->d_ctr);
        ct_mark_filed_kernel<<<1, 32, 0, t->stream>>>(static_cast<const u32*>(c.xin_cnt.p), done, static_cast<const u32*>(c.extra_cnt.p),
                                                      done + kMaxRanks, c.caps, c.pe.world);
        t->n_launches += 3;
    }
    ct_layout_kernel<<<1, 1024, 0, t->stream>>>(static_cast<const u32*>(c.chunk_cursor.p), C, c.g, c.caps, (u32)Slot<W>::kPerBucket,
                                                CtBuild<W>::kMaxSlots, static_cast<u32*>(c.chunk_base.p), static_cast<u32*>(c.pool_off.p), t->d_ctr);
    t->n_launches += 2;
    KH_CUDA(t, cudaEventRecord(t->ev[EV_BUILD0], t->stream));
    ct_build_kernel<W><<<C, kCtBuildThreads, CtBuild<W>::kSmem, t->stream>>>(
        static_cast<const V*>(c.fine.p), static_cast<const u32*>(c.chunk_cursor.p), static_cast<const u32*>(c.chunk_base.p),
        static_cast<const u32*>(c.pool_off.p), static_cast<V*>(t->table), static_cast<u32*>(c.seg_base.p),
        static_cast<u64*>(t->link.p), static_cast<u64*>(c.meta.p), static_cast<V*>(c.ext_key.p),
        static_cast<unsigned char*>(c.pool.p), c.g, c.caps, t->d_ctr);
    KH_CUDA(t, cudaGetLastError());
    KH_CUDA(t, cudaEventRecord(t->ev[EV_BUILD1], t->stream));
    t->have_build = true;
    c.sealed = true;
    return KH_OK;
}

// The traverse, in parts that each end with a barrier across the ranks (kh_shard_assemble runs them all; a host that
// emulates several ranks on ONE device enqueues part p for every rank before part p + 1, see kh_capi.h):
//   0  tell the owners what they received | barrier
//   1  seal (if not sealed) + head stubs + resolve the pending links (local lookups; requests to the owners) | barrier
//   2  answer the requests that arrived (one coalesced run of answers per requester) | barrier
//   3  file the answers; send segment links / meta / characters to every other rank | barrier
//   4  contig lengths by walking each contig's segments (bounded) | barrier that agrees on "some contig is too long"
//   5  fast path, enqueued unconditionally (its kernels look at the agreed flag): offsets, second walk that copies the characters
//   6  [the host reads the flag -- it would wait here anyway, the step is over]  slow path only from here on:
//   6 .. 6+R-1  one pointer-jumping round each | barrier that also agrees on "nobody moved"
//   6+R  (slow path only) contig lengths, claims, offsets | barrier
//   7+R  (slow path only) emit | barrier
constexpr int kCtMaxRounds = 24;            // chains of up to 2^24 segments
constexpr int kCtParts = 8 + kCtMaxRounds;
constexpr u32 kCtWalkMaxSteps = 512;        // segments a lane follows before the step falls back to pointer jumping

template <int W>
int ct_assemble_part(kh_table* t, int part) {
    typedef typename Slot<W>::value_t V;
    auto& c = t->ct;
    const unsigned gb = (unsigned)t->sm_count * 8;
    u64* link = static_cast<u64*>(t->link.p);
    CtGathered gt = {};
    for (int r = 0; r < c.pe.world; ++r) {
        const bool me = r == c.pe.rank;
        gt.link[r] = me ? link : static_cast<const u64*>(c.g_link.p) + (u64)r * c.caps.g_seg_stride;
        gt.meta[r] = me ? static_cast<const u64*>(c.meta.p) : static_cast<const u64*>(c.g_meta.p) + (u64)r * c.caps.g_seg_stride;
        gt.pool[r] = me ? static_cast<const unsigned char*>(c.pool.p) : static_cast<const unsigned char*>(c.g_pool.p) + (u64)r * c.caps.g_pool_stride;
    }
    switch (part) {
    case 0:
        if (c.assembled) { c.sealed = false; c.assembled = false; }      // claims and jumped links of a slow traverse: rebuild
        c.slow = false;
        KH_CUDA(t, cudaEventRecord(t->ev[EV_AS0], t->stream));
        if (!c.sealed) return ct_seal_publish<W>(t);
        return ct_barrier(t);
    case 1: {
        if (!c.sealed) { KH_TRY(ct_seal_build<W>(t)); KH_CUDA(t, cudaEventRecord(t->ev[EV_INS1], t->stream)); t->have_ins = true; }
        if (!c.sharded) {
            const u64 hc = c.n_starts_host;
            KH_TRY(ensure(t, t->contig_len, (hc + 3) * sizeof(u32)));
            KH_TRY(ensure(t, t->contig_pre, (hc + 3) * sizeof(u32)));
            KH_TRY(ensure(t, t->contig_off, (hc + 3) * sizeof(u64)));
            c.out_cap = t->h_ctr->n_inserted + c.n_starts_host * (u64)(t->k + 1) + 64;       // n_inserted: refreshed by the seal's sync below
            ct_set_self(t);
        }
        if (c.pe.world > 1) {             // meta words and characters are final: send them while the links are being resolved
            KH_CUDA(t, cudaEventRecord(t->ev_built, t->stream));
            KH_CUDA(t, cudaStreamWaitEvent(t->copy_stream, t->ev_built, 0));
            ct_gather_kernel<<<gb, 256, 0, t->copy_stream>>>(c.pe, c.caps, link, static_cast<const u64*>(c.meta.p), static_cast<const unsigned char*>(c.pool.p),
                                                             static_cast<const u32*>(c.pool_off.p), c.g.chunks_per_rank, t->d_ctr, 0);
            KH_CUDA(t, cudaEventRecord(t->ev_gathered, t->copy_stream));
            ++t->n_launches;
        }
        ct_init_assemble_kernel<<<1, 1, 0, t->stream>>>(t->d_ctr);
        KH_CUDA(t, cudaMemsetAsync(c.out_cursor.p, 0, kMaxRanks * sizeof(u32), t->stream));
        ct_stub_kernel<W><<<std::max(1u, std::min(gb, (c.caps.hcap + 255u) / 256u)), 256, 0, t->stream>>>(
            static_cast<const V*>(t->starts.p), t->d_ctr, c.caps.hcap, link, static_cast<u64*>(c.meta.p), static_cast<V*>(c.ext_key.p));
        ct_resolve_kernel<W><<<gb, 256, 0, t->stream>>>(static_cast<const V*>(t->table), static_cast<const u32*>(c.chunk_base.p),
                                                        static_cast<const u32*>(c.seg_base.p), link, static_cast<const V*>(c.ext_key.p),
                                                        c.g, c.pe, c.caps, static_cast<u32*>(c.out_cursor.p), static_cast<u32*>(c.req_seg.p), t->d_ctr);
        if (c.pe.world > 1) { ct_publish_inbox_kernel<<<1, 32, 0, t->stream>>>(c.pe, c.caps, static_cast<const u32*>(c.out_cursor.p)); ++t->n_launches; }
        t->n_launches += 3;
        KH_CUDA(t, cudaGetLastError());
        return ct_barrier(t);
    }
    case 2:
        if (c.pe.world > 1) {
            ct_answer_kernel<W><<<gb, 256, 0, t->stream>>>(static_cast<const V*>(t->table), static_cast<const u32*>(c.chunk_base.p),
                                                           static_cast<const u32*>(c.seg_base.p), static_cast<const CtReq<W>*>(c.inbox.p),
                                                           static_cast<const u32*>(c.inbox_cnt.p), c.g, c.pe, c.caps);
            KH_CUDA(t, cudaGetLastError());
            ++t->n_launches;
        }
        return ct_barrier(t);
    case 3:
        if (c.pe.world > 1) {
            ct_apply_kernel<<<gb, 256, 0, t->stream>>>(link, static_cast<const u32*>(c.answers.p), static_cast<const u32*>(c.req_seg.p),
                                                       static_cast<const u32*>(c.out_cursor.p), c.caps, c.pe.world, c.pe.rank);
            ct_gather_kernel<<<gb, 256, 0, t->stream>>>(c.pe, c.caps, link, static_cast<const u64*>(c.meta.p), static_cast<const unsigned char*>(c.pool.p),
                                                        static_cast<const u32*>(c.pool_off.p), c.g.chunks_per_rank, t->d_ctr, 1);
            KH_CUDA(t, cudaStreamWaitEvent(t->stream, t->ev_gathered, 0));
            KH_CUDA(t, cudaGetLastError());
            t->n_launches += 2;
        }
        KH_CUDA(t, cudaEventRecord(t->ev[EV_WALK], t->stream));
        return ct_barrier(t);
    case 4:
        ct_walk_len_kernel<<<gb, 256, 0, t->stream>>>(gt, link, c.caps, t->k, kCtWalkMaxSteps, static_cast<u32*>(t->contig_len.p), t->d_ctr);
        KH_CUDA(t, cudaGetLastError());
        ++t->n_launches;
        return ct_barrier(t, -2);
    case 5: {
        // The fast path is enqueued without asking: its kernels return at once if the ranks agreed on pointer jumping
        // (a device-side flag).  No barrier after it: from here on a rank only reads its own memory, and the next
        // step's opening barrier keeps a fast rank from touching a slow one's buffers.
        KH_TRY(device_scan(t, static_cast<u32*>(t->contig_len.p), (u64)c.caps.hcap + 1, static_cast<u64*>(t->contig_off.p), &t->d_ctr->contig_bytes));
        KH_CUDA(t, cudaEventRecord(t->ev[EV_RANK], t->stream));
        ct_walk_emit_kernel<W><<<gb, 256, 0, t->stream>>>(gt, link, static_cast<const V*>(t->starts.p), c.caps, t->k, static_cast<const u32*>(t->contig_len.p),
                                                          static_cast<const u64*>(t->contig_off.p), c.out_cap, static_cast<char*>(t->out.p), t->d_ctr);
        KH_CUDA(t, cudaGetLastError());
        ++t->n_launches;
        KH_CUDA(t, cudaEventRecord(t->ev[EV_AS1], t->stream));
        t->have_as = true;
        return KH_OK;
    }
    case 6: {
        KH_TRY(read_counters(t));                    // which way did all ranks go?  (the host would wait here anyway: the step is over)
        c.slow = (c.pe.world > 1 ? t->h_ctr->use_jump : t->h_ctr->need_jump) != 0;
        if (!c.slow) return KH_OK;
        c.assembled = true;                          // the slow path jumps links in place and claims tails: the next traverse re-seals
        ct_rank_round_kernel<<<gb, 256, 0, t->stream>>>(c.pe, link, c.caps, t->d_ctr, t->d_ctr->flags, 0);
        KH_CUDA(t, cudaGetLastError());
        ++t->n_launches;
        return ct_barrier(t, 0);
    }
    case 6 + kCtMaxRounds: {
        if (!c.slow) return KH_OK;
        ct_reset_nodes_kernel<<<1, 1, 0, t->stream>>>(t->d_ctr);
        ct_lengths_kernel<<<gb, 256, 0, t->stream>>>(c.pe, link, c.caps, t->k, static_cast<u32*>(t->contig_len.p),
                                                     static_cast<u32*>(t->contig_pre.p), t->d_ctr);
        ct_claim_kernel<<<gb, 256, 0, t->stream>>>(c.pe, link, c.caps, static_cast<const u32*>(t->contig_len.p), t->d_ctr);
        KH_CUDA(t, cudaGetLastError());
        t->n_launches += 3;
        KH_TRY(device_scan(t, static_cast<u32*>(t->contig_len.p), (u64)c.caps.hcap + 1, static_cast<u64*>(t->contig_off.p), &t->d_ctr->contig_bytes));
        KH_CUDA(t, cudaEventRecord(t->ev[EV_RANK], t->stream));
        return ct_barrier(t);
    }
    case 7 + kCtMaxRounds:
        if (!c.slow) return KH_OK;
        ct_emit_kernel<<<gb, 256, 0, t->stream>>>(c.pe, link, static_cast<const u64*>(c.meta.p), static_cast<const unsigned char*>(c.pool.p),
                                                  c.caps, t->d_ctr, t->k);
        ct_emit_heads_kernel<W><<<gb, 256, 0, t->stream>>>(static_cast<const V*>(t->starts.p), c.caps, t->k, static_cast<const u32*>(t->contig_len.p),
                                                          static_cast<const u64*>(t->contig_off.p), t->d_ctr, c.out_cap, static_cast<char*>(t->out.p));
        KH_CUDA(t, cudaGetLastError());
        t->n_launches += 2;
        KH_CUDA(t, cudaEventRecord(t->ev[EV_AS1], t->stream));
        t->have_as = true;
        return ct_barrier(t);
    default: {
        if (part < 7 || part >= 6 + kCtMaxRounds) return fail(t, KH_ERR_ARG, "unknown assemble part");
        if (!c.slow) return KH_OK;
        const int r = part - 6;
        ct_rank_round_kernel<<<gb, 256, 0, t->stream>>>(c.pe, link, c.caps, t->d_ctr, t->d_ctr->flags, r);
        KH_CUDA(t, cudaGetLastError());
        ++t->n_launches;
        return ct_barrier(t, r);
    }
    }
}

// wait for the step, collect counters; *bits_out = device error bits (0 = fine)
int ct_finish(kh_table* t, u32* bits_out) {
    auto& c = t->ct;
    KH_TRY(read_counters(t));
    const Counters& h = *t->h_ctr;
    const u64 n_starts = std::min<u64>(h.n_starts_dev, c.caps.hcap);
    t->n_starts = n_starts;
    t->stats.n_contigs = n_starts;
    t->stats.n_nodes = h.n_nodes;
    t->stats.contig_bytes = h.contig_bytes;
    t->stats.n_segments = (h.next_seg > c.caps.hcap ? h.next_seg - c.caps.hcap : 0) + n_starts;
    u32 rounds = 0;
    for (int i = 0; i < kCtMaxRounds; ++i) rounds += h.flags[i] ? 1u : 0u;
    t->stats.rank_rounds = rounds + 1;
    t->last_contig_bytes = h.contig_bytes;
    t->last_n_contigs = n_starts;
    u32 e = h.errors;
    if (e == 0 && h.contig_bytes > c.out_cap) e = kErrConverge;
    if (bits_out) *bits_out = e;
    if (e & kErrInternal) {             // say which capacity or wait it was (rare path: a message on stderr is worth more than silence)
        char msg[512];
        snprintf(msg, sizeof msg, "rank %d/%d internal error, site bits 0x%x (1 barrier wait, 2 start list, 4 segment ids, 8 link inbox, "
                 "16 unresolved head stub, 32 output buffer): starts %llu/%u, segments %u/%u, contig bytes %llu/%llu, epoch %u",
                 c.pe.rank, c.pe.world, h.err_where, (unsigned long long)h.n_starts_dev, c.caps.hcap, h.next_seg, c.caps.seg_cap,
                 (unsigned long long)h.contig_bytes, (unsigned long long)c.out_cap, c.epoch);
        t->err = msg;
        fprintf(stderr, "libkh_b200: %s\n", msg);
    }
    if (h.errors) { clear_error_bits(t); KH_CUDA(t, cudaMemsetAsync(&t->d_ctr->err_where, 0, sizeof(u32), t->stream)); }
    return KH_OK;
}

// plain-handle wrappers -----------------------------------------------------------------------------------------
template <int W>
int ct_insert_plain(kh_table* t, const unsigned char* recs, u64 n, bool record_start) {
    auto& c = t->ct;
    if (record_start) KH_CUDA(t, cudaEventRecord(t->ev[EV_INS0], t->stream));
    KH_TRY(ct_stage<W>(t, recs, n));
    KH_TRY(read_counters(t));                 // start count (sizes the start list of the next call) + input errors
    c.n_starts_host = std::min<u64>(t->h_ctr->n_starts_dev, 0xFFFFFF00ull);
    t->n_starts = c.n_starts_host;
    KH_CUDA(t, cudaEventRecord(t->ev[EV_INS1], t->stream));
    t->have_ins = true;
    const u32 e = t->h_ctr->errors;
    if (e) { clear_error_bits(t); return status_from_errors(t, e); }
    return KH_OK;
}

template <int W>
int ct_seal_plain(kh_table* t) {
    auto& c = t->ct;
    if (c.sealed) return KH_OK;
    KH_TRY(ct_seal_publish<W>(t));
    KH_TRY(ct_seal_build<W>(t));
    KH_CUDA(t, cudaEventRecord(t->ev[EV_INS1], t->stream));
    KH_TRY(read_counters(t));
    const u32 e = t->h_ctr->errors;
    if (e) { clear_error_bits(t); return status_from_errors(t, e); }
    return KH_OK;
}

template <int W>
int ct_assemble_plain(kh_table* t) {
    auto& c = t->ct;
    if (c.assembled) { c.sealed = false; c.assembled = false; }
    KH_TRY(ct_seal_plain<W>(t));              // also refreshes n_inserted on the host (sizes the output)
    KH_TRY(ensure(t, t->out, t->h_ctr->n_inserted + c.n_starts_host * (u64)(t->k + 1) + 64));
    for (int part = 0; part < kCtParts; ++part) KH_TRY(ct_assemble_part<W>(t, part));
    u32 bits = 0;
    KH_TRY(ct_finish(t, &bits));
    if (bits) return status_from_errors(t, bits);
    return KH_OK;
}

}  // namespace

// ============================================================================ C ABI ======
extern "C" {

int kh_abi_version(void) { return 2; }

int kh_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

const char* kh_status_string(int s) {
    switch (s) {
    case KH_OK: return "ok";
    case KH_ERR_ARG: return "bad argument";
    case KH_ERR_CUDA: return "CUDA failure or no CUDA device";
    case KH_ERR_NOT_FOUND: return "Error: k-mer not found in Distributed HashMap.";
    case KH_ERR_TABLE_FULL: return "hash table full";
    case KH_ERR_CYCLE: return "chain never terminates (cycle)";
    case KH_ERR_BAD_INPUT: return "malformed input";
    case KH_ERR_CONVERGE: return "chains are not linear (shared end node)";
    case KH_ERR_NOMEM: return "out of memory";
    default: return "unknown status";
    }
}

uint64_t kh_packed_bytes(int k) { return (uint64_t)((k + 3) / 4); }
uint64_t kh_pair_bytes(int k) { return (uint64_t)((k + 3) / 4 + 2); }

int kh_create(int k, uint64_t n_expected, double load_factor, int device, kh_table** out) {
    if (!out) return KH_ERR_ARG;
    *out = nullptr;
    if (k < 2 || k > 61 || !(load_factor > 0.0) || load_factor > 1.0) return KH_ERR_ARG;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) { cudaGetLastError(); return KH_ERR_CUDA; }
    if (device < 0 || device >= ndev) return KH_ERR_ARG;
    kh_table* t = new kh_table();
    auto bail = [&](int rc) { kh_destroy(t); return rc; };
    t->k = k; t->device = device; t->lf = load_factor; t->n_expected = n_expected;
    t->pl = (k + 3) / 4; t->pb = t->pl + 2;
    // Every sharded handle (kh_shard_init) and large single-GPU tables with long k-mers are chunk tables (ctable.cuh);
    // the others stay plain open-addressing tables.  KH_CT: 0 never, 1 auto, 2 always.
    t->ct_env = env_int("KH_CT", 1);
    // auto: single-GPU tables whose plain form needs 128-bit slots anyway (K >= 30) and that are far larger than L2.
    // With 64-bit slots (K <= 29) the plain table's shared-memory build + walk is the faster single-GPU path
    // (5.6 vs 9.2 ms on the chr14 shape at K=19: short supermers mean ~4 k-mers per segment).
    const bool use_ct = ct_supported(k) && (t->ct_env == 2 || (t->ct_env != 0 && n_expected >= (1ull << 20) && 2 * k + 6 > 64));
    t->W = use_ct ? ct_slot_words(k) : ((2 * k + 6 <= 64) ? 1 : 2);
    t->slot_bytes = t->W == 1 ? 8 : 16;
    t->per_bucket = 32 / t->slot_bytes;
    if (cudaSetDevice(device) != cudaSuccess) return bail(KH_ERR_CUDA);
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return bail(KH_ERR_CUDA);
    if (prop.major < 9) { fprintf(stderr, "libkh_b200: device %d is sm_%d%d; this library is built for sm_100a only\n", device, prop.major, prop.minor); return bail(KH_ERR_CUDA); }
    t->sm_count = prop.multiProcessorCount;
    // One random probe should move one 32-byte sector, not a 64/128-byte L2 fetch.
    const int gran = env_int("KH_L2_FETCH_BYTES", 32);
    if (gran > 0) { cudaDeviceSetLimit(cudaLimitMaxL2FetchGranularity, (size_t)gran); cudaGetLastError(); }

    const long double slots = (long double)std::max<uint64_t>(n_expected, 1) / (long double)load_factor;
    t->nbuckets = std::max<u64>(16, (u64)(slots / t->per_bucket) + 1);
    // Rounded up to a multiple of 16 buckets.  The size is visible to callers (kh_stats n_buckets / n_slots, the slot
    // layout behind kh_get_device_view), so this rounding stays part of the sizing rule.
    t->nbuckets = (t->nbuckets + 15) / 16 * 16;
    t->table_bytes = use_ct ? 0 : (size_t)t->nbuckets * 32;       // a chunk table is allocated by ct_setup
    int rc = KH_OK;
    auto ck = [&](cudaError_t e) { if (e != cudaSuccess && rc == KH_OK) { rc = e == cudaErrorMemoryAllocation ? KH_ERR_NOMEM : KH_ERR_CUDA; t->err = cudaGetErrorString(e); } };
    ck(cudaStreamCreateWithFlags(&t->own_stream, cudaStreamNonBlocking));
    ck(cudaStreamCreateWithFlags(&t->copy_stream, cudaStreamNonBlocking));
    t->stream = t->own_stream;
    if (!use_ct) ck(cudaMalloc(&t->table, t->table_bytes));
    ck(cudaMalloc((void**)&t->d_ctr, sizeof(Counters)));
    ck(cudaHostAlloc((void**)&t->h_ctr, sizeof(Counters), cudaHostAllocDefault));
    for (auto& e : t->ev) ck(cudaEventCreate(&e));
    for (auto& e : t->ev_copied) ck(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    for (auto& e : t->ev_consumed) ck(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    ck(cudaEventCreateWithFlags(&t->ev_built, cudaEventDisableTiming));
    ck(cudaEventCreateWithFlags(&t->ev_gathered, cudaEventDisableTiming));
    if (rc != KH_OK) { fprintf(stderr, "libkh_b200: kh_create: %s\n", t->err.c_str()); return bail(rc); }
    if (!use_ct) ck(cudaMemsetAsync(t->table, 0, t->table_bytes, t->stream));
    ck(cudaMemsetAsync(t->d_ctr, 0, sizeof(Counters), t->stream));
    ck(cudaStreamSynchronize(t->stream));
    if (rc != KH_OK) return bail(rc);
    memset(t->h_ctr, 0, sizeof(Counters));
    int v = env_int("KH_SPLIT_BUCKETS", 0);
    if (v > 0 && set_option(t, "split_buckets", v) != KH_OK) fprintf(stderr, "libkh_b200: ignoring KH_SPLIT_BUCKETS=%d\n", v);
    t->debug_cap_pct = std::max(1, env_int("KH_DEBUG_CAP_PCT", 100));
    v = env_int("KH_SEG_CHARS", 0);
    if (v > 0 && set_option(t, "seg_chars", v) != KH_OK) fprintf(stderr, "libkh_b200: ignoring KH_SEG_CHARS=%d\n", v);
    if (use_ct) {
        rc = t->W == 1 ? ct_setup<1>(t, 0, 1, n_expected, n_expected, n_expected, false)
                       : ct_setup<2>(t, 0, 1, n_expected, n_expected, n_expected, false);
        if (rc != KH_OK) { fprintf(stderr, "libkh_b200: kh_create: %s\n", t->err.c_str()); return bail(rc); }
    }
    t->err.clear();
    *out = t;
    return KH_OK;
}

int kh_destroy(kh_table* t) {
    if (!t) return KH_OK;
    cudaSetDevice(t->device);
    if (t->own_stream) cudaStreamSynchronize(t->own_stream);
    DevBuf* bufs[] = {&t->starts, &t->mask, &t->tile_counts, &t->tile_offs, &t->scan_blocks, &t->link, &t->seglen,
                      &t->tmp, &t->part_cursor, &t->grouped, &t->fine, &t->chunk_cursor, &t->overflow, &t->contig_len, &t->contig_pre, &t->contig_off, &t->out, &t->stage[0], &t->stage[1],
                      &t->text_stage, &t->scratch_a, &t->scratch_b, &t->scratch_c, &t->sort_keys[0], &t->sort_keys[1], &t->sort_vals[0], &t->sort_vals[1], &t->sort_tmp};
    for (DevBuf* b : bufs) if (b->p) cudaFree(b->p);
    for (auto& row : t->ct.ipc_opened) for (void* q : row) if (q) cudaIpcCloseMemHandle(q);
    {
        auto& c = t->ct;
        for (DevBuf* b : {&c.xin_vals, &c.xin_chunk, &c.xin_cnt, &c.xin_done, &c.xout_cursor, &c.extra_vals, &c.extra_chunk, &c.extra_cnt, &c.fine,
                          &c.chunk_cursor, &c.chunk_base, &c.pool_off, &c.seg_base, &c.ext_key, &c.meta, &c.pool, &c.inbox, &c.inbox_cnt,
                          &c.out_cursor, &c.flags, &c.answers, &c.req_seg, &c.g_link, &c.g_meta, &c.g_pool, &c.g_hdr})
            if (b->p) cudaFree(b->p);
    }
    if (t->table) cudaFree(t->table);
    if (t->d_ctr) cudaFree(t->d_ctr);
    if (t->h_ctr) cudaFreeHost(t->h_ctr);
    if (t->h_out) cudaFreeHost(t->h_out);
    if (t->h_off) cudaFreeHost(t->h_off);
    for (auto& e : t->ev) if (e) cudaEventDestroy(e);
    for (auto& e : t->ev_copied) if (e) cudaEventDestroy(e);
    for (auto& e : t->ev_consumed) if (e) cudaEventDestroy(e);
    if (t->ev_built) cudaEventDestroy(t->ev_built);
    if (t->ev_gathered) cudaEventDestroy(t->ev_gathered);
    if (t->own_stream) cudaStreamDestroy(t->own_stream);
    if (t->copy_stream) cudaStreamDestroy(t->copy_stream);
    cudaGetLastError();
    delete t;
    return KH_OK;
}

int kh_clear(kh_table* t) {
    if (!t) return KH_ERR_ARG;
    KH_CUDA(t, cudaSetDevice(t->device));
    KH_CUDA(t, cudaEventRecord(t->ev[EV_CLR0], t->stream));
    if (t->ct.on) {              // a chunk table is rewritten chunk by chunk at the next seal: only the staging cursors go back to zero
        KH_TRY(ct_reset_staging(t));
        t->ct.sealed = false; t->ct.assembled = false;
        t->ct.n_starts_host = 0;
    } else {
        KH_CUDA(t, cudaMemsetAsync(t->table, 0, t->table_bytes, t->stream));
    }
    KH_CUDA(t, cudaMemsetAsync(t->d_ctr, 0, sizeof(Counters), t->stream));
    KH_CUDA(t, cudaEventRecord(t->ev[EV_CLR1], t->stream));
    t->have_clr = true;
    t->table_dirty = false;
    t->n_starts = 0;
    memset(t->h_ctr, 0, sizeof(Counters));
    t->stats.n_contigs = t->stats.n_nodes = t->stats.contig_bytes = t->stats.n_segments = 0;
    t->stats.rank_rounds = 0;
    t->last_contig_bytes = t->last_n_contigs = 0;
    return KH_OK;
}

int kh_set_stream(kh_table* t, void* cuda_stream) {
    if (!t) return KH_ERR_ARG;
    KH_CUDA(t, cudaSetDevice(t->device));
    KH_CUDA(t, cudaStreamSynchronize(t->stream));
    // NULL is CUDA's legacy default stream (what torch.cuda.current_stream() is unless changed); it orders
    // with NCCL work that torch enqueues relative to that stream
    t->stream = cuda_stream ? static_cast<cudaStream_t>(cuda_stream) : cudaStreamLegacy;
    return KH_OK;
}

int kh_sync(kh_table* t) {
    if (!t) return KH_ERR_ARG;
    KH_CUDA(t, cudaSetDevice(t->device));
    KH_CUDA(t, cudaStreamSynchronize(t->stream));
    return KH_OK;
}

int kh_set_option(kh_table* t, const char* name, int64_t value) {
    if (!t || !name) return KH_ERR_ARG;
    return set_option(t, name, value);
}

int kh_pack_lines_device(kh_table* t, const void* text_dev, uint64_t n_lines, void* pairs_dev_out) {
    if (!t || (n_lines && (!text_dev || !pairs_dev_out))) return KH_ERR_ARG;
    KH_CUDA(t, cudaSetDevice(t->device));
    KH_CUDA(t, cudaEventRecord(t->ev[EV_PACK0], t->stream));
    KH_TRY(pack_device(t, text_dev, n_lines, pairs_dev_out));
    KH_CUDA(t, cudaEventRecord(t->ev[EV_PACK1], t->stream));
    t->have_pack = true;
    return KH_OK;
}

static const uint64_t kChunkBytes = 64ull << 20;

int kh_pack_lines(kh_table* t, const char* text_host, uint64_t n_lines, void* pairs_host_out) {
    if (!t || (n_lines && (!text_host || !pairs_host_out))) return KH_ERR_ARG;
    KH_CUDA(t, cudaSetDevice(t->device));
    const u64 ll = t->k + 4;
    const u64 chunk = std::max<u64>(kPackLines, (kChunkBytes / ll) / kPackLines * kPackLines);
    KH_TRY(ensure(t, t->text_stage, std::min<u64>(n_lines, chunk) * ll));
    KH_TRY(ensure(t, t->scratch_a, std::min<u64>(n_lines, chunk) * t->pb));
    KH_CUDA(t, cudaEventRecord(t->ev[EV_PACK0], t->stream));
    for (u64 l0 = 0; l0 < n_lines; l0 += chunk) {
        const u64 cnt = std::min<u64>(chunk, n_lines - l0);
        KH_CUDA(t, cudaMemcpyAsync(t->text_stage.p, text_host + l0 * ll, cnt * ll, cudaMemcpyHostToDevice, t->stream));
        KH_TRY(pack_device(t, t->text_stage.p, cnt, t->scratch_a.p));
        KH_CUDA(t, cudaMemcpyAsync(static_cast<char*>(pairs_host_out) + l0 * t->pb, t->scratch_a.p, cnt * t->pb,
                                   cudaMemcpyDeviceToHost, t->stream));
    }
    KH_CUDA(t, cudaEventRecord(t->ev[EV_PACK1], t->stream));
    t->have_pack = true;
    KH_TRY(read_counters(t));
    const u32 e = t->h_ctr->errors;
    if (e) { clear_error_bits(t); return status_from_errors(t, e); }
    return KH_OK;
}

int kh_insert_pairs_device(kh_table* t, const void* pairs_dev, uint64_t n) {
    if (!t || (n && !pairs_dev)) return KH_ERR_ARG;
    KH_CUDA(t, cudaSetDevice(t->device));
    return insert_device(t, pairs_dev, n);
}

// Host records: double-buffered H2D on a copy stream overlapped with the insert kernels.
int kh_insert_pairs(kh_table* t, const void* pairs_host, uint64_t n) {
    if (!t || (n && !pairs_host)) return KH_ERR_ARG;
    if (n == 0) return KH_OK;
    KH_CUDA(t, cudaSetDevice(t->device));
    const u64 chunk = std::max<u64>(kInsTile, (kChunkBytes / t->pb) / kInsTile * kInsTile);
    const u64 nchunks = (n + chunk - 1) / chunk;
    for (int i = 0; i < (nchunks > 1 ? 2 : 1); ++i) KH_TRY(ensure(t, t->stage[i], std::min<u64>(n, chunk) * t->pb));
    const char* src = static_cast<const char*>(pairs_host);
    auto issue_copy = [&](u64 c) -> int {
        const u64 off = c * chunk, cnt = std::min<u64>(chunk, n - off);
        if (c >= 2) KH_CUDA(t, cudaStreamWaitEvent(t->copy_stream, t->ev_consumed[c & 1], 0));
        KH_CUDA(t, cudaMemcpyAsync(t->stage[c & 1].p, src + off * t->pb, cnt * t->pb, cudaMemcpyHostToDevice, t->copy_stream));
        KH_CUDA(t, cudaEventRecord(t->ev_copied[c & 1], t->copy_stream));
        return KH_OK;
    };
    KH_CUDA(t, cudaEventRecord(t->ev[EV_INS0], t->stream));
    // the copy stream must not start before earlier work on the main stream that may still read the staging buffers
    KH_CUDA(t, cudaEventRecord(t->ev_consumed[0], t->stream));
    KH_CUDA(t, cudaStreamWaitEvent(t->copy_stream, t->ev_consumed[0], 0));
    KH_TRY(issue_copy(0));
    for (u64 c = 0; c < nchunks; ++c) {
        if (c + 1 < nchunks) KH_TRY(issue_copy(c + 1));
        const u64 off = c * chunk, cnt = std::min<u64>(chunk, n - off);
        KH_CUDA(t, cudaStreamWaitEvent(t->stream, t->ev_copied[c & 1], 0));
        KH_TRY(insert_device(t, t->stage[c & 1].p, cnt, /*record_start=*/false));
        KH_CUDA(t, cudaEventRecord(t->ev_consumed[c & 1], t->stream));
    }
    return KH_OK;
}

int kh_insert_lines(kh_table* t, const char* text_host, uint64_t n_lines) {
    if (!t || (n_lines && !text_host)) return KH_ERR_ARG;
    if (n_lines == 0) return KH_OK;
    KH_CUDA(t, cudaSetDevice(t->device));
    const u64 ll = t->k + 4;
    const u64 chunk = std::max<u64>(kInsTile, (kChunkBytes / ll) / kInsTile * kInsTile);
    KH_TRY(ensure(t, t->text_stage, std::min<u64>(n_lines, chunk) * ll));
    KH_TRY(ensure(t, t->scratch_a, std::min<u64>(n_lines, chunk) * t->pb));
    KH_CUDA(t, cudaEventRecord(t->ev[EV_INS0], t->stream));
    for (u64 l0 = 0; l0 < n_lines; l0 += chunk) {
        const u64 cnt = std::min<u64>(chunk, n_lines - l0);
        KH_CUDA(t, cudaMemcpyAsync(t->text_stage.p, text_host + l0 * ll, cnt * ll, cudaMemcpyHostToDevice, t->stream));
        KH_TRY(pack_device(t, t->text_stage.p, cnt, t->scratch_a.p));
        KH_TRY(insert_device(t, t->scratch_a.p, cnt, /*record_start=*/false));
    }
    return KH_OK;
}

int kh_find_device(kh_table* t, const void* pkmers_dev, uint64_t n, void* pairs_dev_out, uint8_t* found_dev_out) {
    if (!t || (n && (!pkmers_dev || !pairs_dev_out || !found_dev_out))) return KH_ERR_ARG;
    if (n == 0) return KH_OK;
    KH_CUDA(t, cudaSetDevice(t->device));
    const unsigned blocks = (unsigned)((n + 255) / 256);
    if (t->ct.on) {
        if (t->ct.pe.world > 1) return fail(t, KH_ERR_ARG, "kh_find on a sharded handle is not supported");
        KH_TRY(t->W == 1 ? ct_seal_plain<1>(t) : ct_seal_plain<2>(t));
        if (t->W == 1)
            ct_find_kernel<1><<<blocks, 256, 0, t->stream>>>(static_cast<const u64*>(t->table), static_cast<const u32*>(t->ct.chunk_base.p), t->ct.g,
                static_cast<const unsigned char*>(pkmers_dev), n, static_cast<unsigned char*>(pairs_dev_out), found_dev_out);
        else
            ct_find_kernel<2><<<blocks, 256, 0, t->stream>>>(static_cast<const u128*>(t->table), static_cast<const u32*>(t->ct.chunk_base.p), t->ct.g,
                static_cast<const unsigned char*>(pkmers_dev), n, static_cast<unsigned char*>(pairs_dev_out), found_dev_out);
        KH_CUDA(t, cudaGetLastError());
        return KH_OK;
    }
    if (t->W == 1)
        find_kernel<1><<<blocks, 256, 0, t->stream>>>(static_cast<const u64*>(t->table), t->nbuckets, t->k,
            static_cast<const unsigned char*>(pkmers_dev), n, static_cast<unsigned char*>(pairs_dev_out), found_dev_out);
    else
        find_kernel<2><<<blocks, 256, 0, t->stream>>>(static_cast<const u128*>(t->table), t->nbuckets, t->k,
            static_cast<const unsigned char*>(pkmers_dev), n, static_cast<unsigned char*>(pairs_dev_out), found_dev_out);
    KH_CUDA(t, cudaGetLastError());
    return KH_OK;
}

int kh_find(kh_table* t, const void* pkmers_host, uint64_t n, void* pairs_host_out, uint8_t* found_host_out) {
    if (!t || (n && (!pkmers_host || !pairs_host_out || !found_host_out))) return KH_ERR_ARG;
    if (n == 0) return KH_OK;
    KH_CUDA(t, cudaSetDevice(t->device));
    KH_TRY(ensure(t, t->scratch_a, n * t->pl));
    KH_TRY(ensure(t, t->scratch_b, n * t->pb));
    KH_TRY(ensure(t, t->scratch_c, n));
    KH_CUDA(t, cudaMemcpyAsync(t->scratch_a.p, pkmers_host, n * t->pl, cudaMemcpyHostToDevice, t->stream));
    KH_TRY(kh_find_device(t, t->scratch_a.p, n, t->scratch_b.p, static_cast<uint8_t*>(t->scratch_c.p)));
    KH_CUDA(t, cudaMemcpyAsync(pairs_host_out, t->scratch_b.p, n * t->pb, cudaMemcpyDeviceToHost, t->stream));
    KH_CUDA(t, cudaMemcpyAsync(found_host_out, t->scratch_c.p, n, cudaMemcpyDeviceToHost, t->stream));
    KH_CUDA(t, cudaStreamSynchronize(t->stream));
    return KH_OK;
}

int kh_assemble_device(kh_table* t, const char** contigs_dev, const uint64_t** offsets_dev,
                       uint64_t* n_contigs, uint64_t* contig_bytes, uint64_t* n_nodes) {
    if (!t) return KH_ERR_ARG;
    KH_CUDA(t, cudaSetDevice(t->device));
    const int rc = assemble_device(t);
    if (contigs_dev) *contigs_dev = static_cast<const char*>(t->out.p);
    if (offsets_dev) *offsets_dev = static_cast<const uint64_t*>(t->contig_off.p);
    if (n_contigs) *n_contigs = t->stats.n_contigs;
    if (contig_bytes) *contig_bytes = rc == KH_OK ? t->stats.contig_bytes : 0;
    if (n_nodes) *n_nodes = t->stats.n_nodes;
    return rc;
}

int kh_assemble(kh_table* t, const char** contigs_host, const uint64_t** offsets_host,
                uint64_t* n_contigs, uint64_t* contig_bytes, uint64_t* n_nodes) {
    if (!t) return KH_ERR_ARG;
    KH_CUDA(t, cudaSetDevice(t->device));
    // size the pinned landing buffers before the timed work so steady-state calls allocate nothing
    const u64 cap_guess = t->h_ctr->n_inserted + t->n_starts * (u64)(t->k + 1) + 64;
    KH_TRY(ensure_pinned(t, t->h_out, t->h_out_cap, cap_guess));
    KH_TRY(ensure_pinned(t, t->h_off, t->h_off_cap, (t->n_starts + 1) * sizeof(u64)));
    const int rc = assemble_device(t);
    if (n_contigs) *n_contigs = t->stats.n_contigs;
    if (n_nodes) *n_nodes = t->stats.n_nodes;
    if (contig_bytes) *contig_bytes = 0;
    if (contigs_host) *contigs_host = static_cast<const char*>(t->h_out);
    if (offsets_host) *offsets_host = static_cast<const uint64_t*>(t->h_off);
    if (rc != KH_OK) return rc;
    const u64 bytes = t->stats.contig_bytes;
    KH_TRY(ensure_pinned(t, t->h_out, t->h_out_cap, bytes));                    // a chunk table learns its size at the seal
    KH_TRY(ensure_pinned(t, t->h_off, t->h_off_cap, (t->n_starts + 1) * sizeof(u64)));
    if (contigs_host) *contigs_host = static_cast<const char*>(t->h_out);
    if (offsets_host) *offsets_host = static_cast<const uint64_t*>(t->h_off);
    if (bytes) KH_CUDA(t, cudaMemcpyAsync(t->h_out, t->out.p, bytes, cudaMemcpyDeviceToHost, t->stream));
    KH_CUDA(t, cudaMemcpyAsync(t->h_off, t->contig_off.p, (t->n_starts + 1) * sizeof(u64), cudaMemcpyDeviceToHost, t->stream));
    KH_CUDA(t, cudaStreamSynchronize(t->stream));
    if (contig_bytes) *contig_bytes = bytes;
    return KH_OK;
}

int kh_get_stats(kh_table* t, kh_stats* out) {
    if (!t || !out) return KH_ERR_ARG;
    KH_CUDA(t, cudaSetDevice(t->device));
    if (t->ct.on && !t->ct.sharded && !t->ct.sealed && t->table_dirty) KH_TRY(t->W == 1 ? ct_seal_plain<1>(t) : ct_seal_plain<2>(t));
    KH_CUDA(t, cudaStreamSynchronize(t->stream));
    kh_stats& s = t->stats;
    s.n_buckets = t->nbuckets;
    s.n_slots = t->nbuckets * t->per_bucket;
    s.n_inserted = t->h_ctr->n_inserted;
    s.n_duplicates = t->h_ctr->n_duplicates;
    s.n_starts = t->n_starts;
    s.slot_bits = t->W == 1 ? 64 : 128;
    if (t->ct.on) s.n_starts = std::min<u64>(t->h_ctr->n_starts_dev, 0xFFFFFFFFull);
    if (t->have_ins) s.ms_insert = elapsed(t->ev[EV_INS0], t->ev[EV_INS1]);
    if (t->have_as) {
        s.ms_assemble = elapsed(t->ev[EV_AS0], t->ev[EV_AS1]);
        s.ms_walk = elapsed(t->ev[EV_AS0], t->ev[EV_WALK]);
        s.ms_rank = elapsed(t->ev[EV_WALK], t->ev[EV_RANK]);
        s.ms_emit = elapsed(t->ev[EV_RANK], t->ev[EV_AS1]);
    }
    if (t->have_pack) s.ms_pack = elapsed(t->ev[EV_PACK0], t->ev[EV_PACK1]);
    if (t->have_clr) s.ms_clear = elapsed(t->ev[EV_CLR0], t->ev[EV_CLR1]);
    if (t->have_build) s.ms_build = elapsed(t->ev[EV_BUILD0], t->ev[EV_BUILD1]);
    if (t->have_stage && t->have_ins) s.ms_stage = elapsed(t->ev[EV_INS0], t->ev[EV_STAGE1]);
    s.n_launches = t->n_launches;
    *out = s;
    return KH_OK;
}

// ---- output side (scripts/check_it.sh:47-48: `cat test*.dat | sort`) ------------------------------------------
// sort key of a contig: its first 21 characters, 3 bits each (0 = the line ended, 1..4 = A C G T), most significant
// first -- bytewise (LC_ALL=C) order of the lines as far as 21 characters decide it
__global__ void __launch_bounds__(256)
contig_sort_keys_kernel(const char* __restrict__ text, const u64* __restrict__ off, u64 n, u64* __restrict__ keys, u32* __restrict__ idx) {
    const u64 c = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= n) return;
    const u64 b = off[c], len = off[c + 1] - b - 1;                 // without the newline
    u64 key = 0;
    for (u32 j = 0; j < 21; ++j) {
        u32 code = 0;
        if (j < len) code = base_code_fast((unsigned char)text[b + j]) + 1u;
        key = (key << 3) | code;
    }
    keys[c] = key;
    idx[c] = (u32)c;
}

int kh_sorted_order(kh_table* t, uint64_t* order_host_out, uint64_t* n_contigs_out) {
    if (!t || !order_host_out) return KH_ERR_ARG;
    KH_CUDA(t, cudaSetDevice(t->device));
    const u64 n = t->last_n_contigs, bytes = t->last_contig_bytes;
    if (n_contigs_out) *n_contigs_out = n;
    if (n == 0) return KH_OK;
    if (n >= 0xFFFFFFFFull) return fail(t, KH_ERR_ARG, "kh_sorted_order: more than 2^32 contigs");
    for (int i = 0; i < 2; ++i) { KH_TRY(ensure(t, t->sort_keys[i], n * sizeof(u64))); KH_TRY(ensure(t, t->sort_vals[i], n * sizeof(u32))); }
    const char* text = static_cast<const char*>(t->out.p);
    const u64* off = static_cast<const u64*>(t->contig_off.p);
    contig_sort_keys_kernel<<<(unsigned)((n + 255) / 256), 256, 0, t->stream>>>(text, off, n, static_cast<u64*>(t->sort_keys[0].p), static_cast<u32*>(t->sort_vals[0].p));
    size_t tmp_bytes = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, tmp_bytes, static_cast<const u64*>(t->sort_keys[0].p), static_cast<u64*>(t->sort_keys[1].p),
                                    static_cast<const u32*>(t->sort_vals[0].p), static_cast<u32*>(t->sort_vals[1].p), (int)n, 0, 63, t->stream);
    KH_TRY(ensure(t, t->sort_tmp, tmp_bytes + 16));
    KH_CUDA(t, cub::DeviceRadixSort::SortPairs(t->sort_tmp.p, tmp_bytes, static_cast<const u64*>(t->sort_keys[0].p), static_cast<u64*>(t->sort_keys[1].p),
                                               static_cast<const u32*>(t->sort_vals[0].p), static_cast<u32*>(t->sort_vals[1].p), (int)n, 0, 63, t->stream));
    t->n_launches += 4;
    std::vector<u64> keys(n);
    std::vector<u32> idx(n);
    KH_CUDA(t, cudaMemcpyAsync(keys.data(), t->sort_keys[1].p, n * sizeof(u64), cudaMemcpyDeviceToHost, t->stream));
    KH_CUDA(t, cudaMemcpyAsync(idx.data(), t->sort_vals[1].p, n * sizeof(u32), cudaMemcpyDeviceToHost, t->stream));
    KH_CUDA(t, cudaStreamSynchronize(t->stream));
    for (u64 i = 0; i < n; ++i) order_host_out[i] = idx[i];
    // contigs that agree on their first 21 characters (rare): finish those runs on the host with the whole lines
    std::vector<char> host_text;
    std::vector<u64> host_off;
    for (u64 i = 0; i < n;) {
        u64 j = i + 1;
        while (j < n && keys[j] == keys[i]) ++j;
        if (j - i > 1) {
            if (host_off.empty()) {
                host_text.resize(bytes); host_off.resize(n + 1);
                KH_CUDA(t, cudaMemcpy(host_text.data(), text, bytes, cudaMemcpyDeviceToHost));
                KH_CUDA(t, cudaMemcpy(host_off.data(), off, (n + 1) * sizeof(u64), cudaMemcpyDeviceToHost));
            }
            std::stable_sort(order_host_out + i, order_host_out + j, [&](uint64_t a, uint64_t b) {
                const u64 la = host_off[a + 1] - host_off[a], lb = host_off[b + 1] - host_off[b];      // incl. '\n' (0x0A < 'A'): a prefix sorts first
                const int c = memcmp(host_text.data() + host_off[a], host_text.data() + host_off[b], std::min(la, lb));
                return c != 0 ? c < 0 : la < lb;
            });
        }
        i = j;
    }
    return KH_OK;
}

int kh_get_device_view(kh_table* t, kh_device_view* out) {
    if (!t || !out) return KH_ERR_ARG;
    if (t->ct.on) return fail(t, KH_ERR_ARG, "kh_get_device_view: a chunk table has no single-record device interface (KH_CT=0 forces a plain table)");
    out->table = t->table; out->n_buckets = t->nbuckets; out->k = t->k; out->slot_bytes = t->slot_bytes;
    out->placement_m = 0; out->device = t->device;
    t->table_dirty = true;              // the caller may insert behind our back: the next bulk insert must not assume an empty table
    return KH_OK;
}

const char* kh_last_error(kh_table* t) { return t ? t->err.c_str() : "null handle"; }

int kh_host_alloc(void** ptr, uint64_t bytes) {
    if (!ptr) return KH_ERR_ARG;
    if (cudaHostAlloc(ptr, bytes ? bytes : 1, cudaHostAllocDefault) != cudaSuccess) { cudaGetLastError(); *ptr = nullptr; return KH_ERR_NOMEM; }
    return KH_OK;
}
int kh_host_free(void* ptr) {
    if (ptr && cudaFreeHost(ptr) != cudaSuccess) { cudaGetLastError(); return KH_ERR_CUDA; }
    return KH_OK;
}

int kh_measure_random_sector_rate(int device, uint64_t footprint_bytes, uint64_t n_probes, double* sectors_per_s) {
    if (!sectors_per_s || footprint_bytes < 4096) return KH_ERR_ARG;
    if (cudaSetDevice(device) != cudaSuccess) { cudaGetLastError(); return KH_ERR_CUDA; }
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return KH_ERR_CUDA;
    const int gran = env_int("KH_L2_FETCH_BYTES", 32);
    if (gran > 0) { cudaDeviceSetLimit(cudaLimitMaxL2FetchGranularity, (size_t)gran); cudaGetLastError(); }
    void* buf = nullptr; u64* sink = nullptr;
    if (cudaMalloc(&buf, footprint_bytes) != cudaSuccess) { cudaGetLastError(); return KH_ERR_NOMEM; }
    cudaMalloc((void**)&sink, 8);
    cudaMemset(buf, 1, footprint_bytes);
    const unsigned blocks = (unsigned)prop.multiProcessorCount * 8;
    const u64 threads = (u64)blocks * 256;
    const u64 per = std::max<u64>(4, (n_probes / threads + 3) / 4 * 4);
    cudaEvent_t a, b;
    cudaEventCreate(&a); cudaEventCreate(&b);
    random_sector_kernel<<<blocks, 256>>>(static_cast<const u64*>(buf), footprint_bytes / 32, per, sink);   // warm-up
    cudaEventRecord(a);
    random_sector_kernel<<<blocks, 256>>>(static_cast<const u64*>(buf), footprint_bytes / 32, per, sink);
    cudaEventRecord(b);
    const cudaError_t e = cudaEventSynchronize(b);
    float ms = 0.f;
    cudaEventElapsedTime(&ms, a, b);
    cudaEventDestroy(a); cudaEventDestroy(b);
    cudaFree(buf); cudaFree(sink);
    if (e != cudaSuccess || ms <= 0.f) { cudaGetLastError(); return KH_ERR_CUDA; }
    *sectors_per_s = (double)(per * threads) / (ms * 1e-3);
    return KH_OK;
}


// ---------------------------------------------------------------- sharded (multi-GPU) ------
int kh_shard_init(kh_table* t, int rank, int world, uint64_t n_local_max, uint64_t n_total, uint64_t n_starts_max) {
    if (!t) return KH_ERR_ARG;
    if (world < 1 || world > kMaxRanks || rank < 0 || rank >= world) return fail(t, KH_ERR_ARG, "1 <= world <= 8 and 0 <= rank < world");
    if (!ct_supported(t->k)) return fail(t, KH_ERR_ARG, "the sharded path supports 17 <= K <= 54");
    if (t->ct.connected) return fail(t, KH_ERR_ARG, "kh_shard_init after kh_shard_connect: set options, init, then export and connect");
    KH_CUDA(t, cudaSetDevice(t->device));
    const int W = ct_slot_words(t->k);
    if (W != t->W) {                       // created as a plain table with narrower slots: it is empty, switch
        t->W = W; t->slot_bytes = W == 1 ? 8 : 16; t->per_bucket = 32 / t->slot_bytes;
    }
    return t->W == 1 ? ct_setup<1>(t, rank, world, n_local_max, n_total, n_starts_max, /*sharded=*/true)
                     : ct_setup<2>(t, rank, world, n_local_max, n_total, n_starts_max, /*sharded=*/true);
}

static int shard_require(kh_table* t) {
    if (!t->ct.on || !t->ct.sharded) return fail(t, KH_ERR_ARG, "handle is not in sharded mode (call kh_shard_init first)");
    return KH_OK;
}

int kh_shard_export_count(void) { return CTX_NBUF; }

// everything two ranks must agree on to index each other's buffers
static uint64_t ct_geometry_signature(kh_table* t) {
    const auto& c = t->ct;
    u64 h = fmix64((u64)c.g.chunks_per_rank + 0x9E3779B97F4A7C15ull);
    h = fmix64(h ^ c.caps.xin_cap); h = fmix64(h ^ c.caps.extra_cap); h = fmix64(h ^ c.caps.inbox_cap);
    h = fmix64(h ^ c.caps.g_seg_stride); h = fmix64(h ^ c.caps.g_pool_stride);
    return fmix64(h ^ (u64)c.pe.world);
}

static void ct_export_list(kh_table* t, void* (&bufs)[CTX_NBUF]) {
    auto& c = t->ct;
    bufs[CTX_XIN_VALS] = c.xin_vals.p; bufs[CTX_XIN_CHUNK] = c.xin_chunk.p; bufs[CTX_XIN_CNT] = c.xin_cnt.p;
    bufs[CTX_EXTRA_VALS] = c.extra_vals.p; bufs[CTX_EXTRA_CHUNK] = c.extra_chunk.p; bufs[CTX_EXTRA_CNT] = c.extra_cnt.p;
    bufs[CTX_LINK] = t->link.p; bufs[CTX_META] = c.meta.p; bufs[CTX_INBOX] = c.inbox.p; bufs[CTX_INBOX_CNT] = c.inbox_cnt.p;
    bufs[CTX_PRE] = t->contig_pre.p; bufs[CTX_OFF] = t->contig_off.p; bufs[CTX_OUT] = t->out.p; bufs[CTX_FLAGS] = c.flags.p;
    bufs[CTX_ANSWERS] = c.answers.p; bufs[CTX_GLINK] = c.g_link.p; bufs[CTX_GMETA] = c.g_meta.p; bufs[CTX_GPOOL] = c.g_pool.p; bufs[CTX_GHDR] = c.g_hdr.p;
}
static void ct_import_list(kh_table* t, int r, void* const (&p)[CTX_NBUF], u64 out_cap) {
    CtPeers& pe = t->ct.pe;
    pe.xin_vals[r] = p[CTX_XIN_VALS]; pe.xin_chunk[r] = static_cast<u32*>(p[CTX_XIN_CHUNK]);
    pe.xin_cnt[r] = static_cast<u32*>(p[CTX_XIN_CNT]);
    pe.extra_vals[r] = p[CTX_EXTRA_VALS]; pe.extra_chunk[r] = static_cast<u32*>(p[CTX_EXTRA_CHUNK]);
    pe.extra_cnt[r] = static_cast<u32*>(p[CTX_EXTRA_CNT]);
    pe.link[r] = static_cast<u64*>(p[CTX_LINK]); pe.meta[r] = static_cast<u64*>(p[CTX_META]);
    pe.inbox[r] = p[CTX_INBOX]; pe.inbox_cnt[r] = static_cast<u32*>(p[CTX_INBOX_CNT]);
    pe.contig_pre[r] = static_cast<u32*>(p[CTX_PRE]); pe.contig_off[r] = static_cast<u64*>(p[CTX_OFF]);
    pe.out[r] = static_cast<char*>(p[CTX_OUT]); pe.out_cap[r] = out_cap;
    pe.flags[r] = static_cast<u32*>(p[CTX_FLAGS]);
    pe.answers[r] = static_cast<u32*>(p[CTX_ANSWERS]);
    pe.g_link[r] = static_cast<u64*>(p[CTX_GLINK]); pe.g_meta[r] = static_cast<u64*>(p[CTX_GMETA]);
    pe.g_pool[r] = static_cast<unsigned char*>(p[CTX_GPOOL]); pe.g_hdr[r] = static_cast<u32*>(p[CTX_GHDR]);
}

int kh_shard_export(kh_table* t, void* handles_out, uint64_t* meta_out) {
    if (!t || !handles_out || !meta_out) return KH_ERR_ARG;
    KH_TRY(shard_require(t));
    KH_CUDA(t, cudaSetDevice(t->device));
    void* bufs[CTX_NBUF];
    ct_export_list(t, bufs);
    cudaIpcMemHandle_t* h = static_cast<cudaIpcMemHandle_t*>(handles_out);
    for (int i = 0; i < CTX_NBUF; ++i) KH_CUDA(t, cudaIpcGetMemHandle(&h[i], bufs[i]));
    meta_out[0] = ct_geometry_signature(t);
    meta_out[1] = t->ct.out_cap;
    return KH_OK;
}

int kh_shard_connect(kh_table* t, const void* all_handles, const uint64_t* all_meta) {
    if (!t || !all_handles || !all_meta) return KH_ERR_ARG;
    KH_TRY(shard_require(t));
    KH_CUDA(t, cudaSetDevice(t->device));
    auto& c = t->ct;
    const cudaIpcMemHandle_t* h = static_cast<const cudaIpcMemHandle_t*>(all_handles);
    for (int r = 0; r < c.pe.world; ++r) {
        if (r == c.pe.rank) continue;
        if (all_meta[2 * r] != ct_geometry_signature(t)) return fail(t, KH_ERR_ARG, "ranks disagree on the table geometry (same n_total, n_local_max, load factor and K everywhere)");
        void* p[CTX_NBUF];
        for (int i = 0; i < CTX_NBUF; ++i) {
            KH_CUDA(t, cudaIpcOpenMemHandle(&p[i], h[r * CTX_NBUF + i], cudaIpcMemLazyEnablePeerAccess));
            c.ipc_opened[r][i] = p[i];
        }
        ct_import_list(t, r, p, all_meta[2 * r + 1]);
    }
    c.connected = true;
    return KH_OK;
}

// All ranks live in this process (one host thread per GPU, or several ranks emulated on one GPU in the tests)
int kh_shard_connect_local(kh_table* t, kh_table* const* peers, int world) {
    if (!t || !peers) return KH_ERR_ARG;
    KH_TRY(shard_require(t));
    auto& c = t->ct;
    if (world != c.pe.world) return fail(t, KH_ERR_ARG, "world does not match kh_shard_init");
    for (int r = 0; r < world; ++r) {
        kh_table* q = peers[r];
        if (!q || !q->ct.on || !q->ct.sharded || q->k != t->k || q->ct.pe.rank != r || ct_geometry_signature(q) != ct_geometry_signature(t))
            return fail(t, KH_ERR_ARG, "peer handle is not shard r of the same table (same K, n_total, load factor)");
        if (q == t) continue;
        if (q->device != t->device) {
            int can = 0;
            cudaDeviceCanAccessPeer(&can, t->device, q->device);
            if (!can) return fail(t, KH_ERR_CUDA, "no peer access between the GPUs");
            cudaSetDevice(t->device);
            const cudaError_t e = cudaDeviceEnablePeerAccess(q->device, 0);
            if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) return fail(t, KH_ERR_CUDA, cudaGetErrorString(e));
            cudaGetLastError();
        }
        void* p[CTX_NBUF];
        ct_export_list(q, p);
        ct_import_list(t, r, p, q->ct.out_cap);
    }
    c.connected = true;
    return KH_OK;
}

// empty table + barrier: no rank may start writing into a peer before that peer has reset its counters
int kh_shard_begin(kh_table* t) {
    if (!t) return KH_ERR_ARG;
    KH_TRY(shard_require(t));
    KH_TRY(kh_clear(t));
    return ct_barrier(t);
}

int kh_shard_insert(kh_table* t, const void* pairs_dev, uint64_t n) {
    if (!t || (n && !pairs_dev)) return KH_ERR_ARG;
    KH_TRY(shard_require(t));
    KH_CUDA(t, cudaSetDevice(t->device));
    if (!t->have_ins || t->ct.sealed || !t->table_dirty) KH_CUDA(t, cudaEventRecord(t->ev[EV_INS0], t->stream));
    return t->W == 1 ? ct_stage<1>(t, static_cast<const unsigned char*>(pairs_dev), n)
                     : ct_stage<2>(t, static_cast<const unsigned char*>(pairs_dev), n);
}

int kh_shard_assemble_parts(void) { return kCtParts; }

int kh_shard_assemble_part(kh_table* t, int part) {
    if (!t) return KH_ERR_ARG;
    KH_TRY(shard_require(t));
    KH_CUDA(t, cudaSetDevice(t->device));
    return t->W == 1 ? ct_assemble_part<1>(t, part) : ct_assemble_part<2>(t, part);
}

int kh_shard_assemble(kh_table* t) {
    for (int part = 0; part < kCtParts; ++part) KH_TRY(kh_shard_assemble_part(t, part));
    return KH_OK;
}

int kh_shard_finish(kh_table* t, int* error_bits_out) {
    if (!t) return KH_ERR_ARG;
    KH_TRY(shard_require(t));
    KH_CUDA(t, cudaSetDevice(t->device));
    u32 bits = 0;
    KH_TRY(ct_finish(t, &bits));
    if (error_bits_out) *error_bits_out = (int)bits;
    return KH_OK;
}

int kh_shard_result(kh_table* t, const char** contigs_dev, const uint64_t** offsets_dev,
                    uint64_t* n_contigs, uint64_t* contig_bytes, uint64_t* n_nodes) {
    if (!t) return KH_ERR_ARG;
    KH_TRY(shard_require(t));
    if (contigs_dev) *contigs_dev = static_cast<const char*>(t->out.p);
    if (offsets_dev) *offsets_dev = static_cast<const uint64_t*>(t->contig_off.p);
    if (n_contigs) *n_contigs = t->stats.n_contigs;
    if (contig_bytes) *contig_bytes = t->stats.contig_bytes;
    if (n_nodes) *n_nodes = t->stats.n_nodes;
    return KH_OK;
}

// introspection for tests and debugging: device pointer and size of an internal buffer of a chunk table
int kh_debug_buffer(kh_table* t, const char* name, void** ptr_out, uint64_t* bytes_out) {
    if (!t || !name || !ptr_out || !bytes_out) return KH_ERR_ARG;
    auto& c = t->ct;
    const std::string n(name);
    const DevBuf* b = nullptr;
    if (n == "link") b = &t->link; else if (n == "meta") b = &c.meta; else if (n == "ext_key") b = &c.ext_key;
    else if (n == "chunk_base") b = &c.chunk_base; else if (n == "seg_base") b = &c.seg_base; else if (n == "chunk_cursor") b = &c.chunk_cursor;
    else if (n == "inbox_cnt") b = &c.inbox_cnt; else if (n == "out_cursor") b = &c.out_cursor; else if (n == "xin_cnt") b = &c.xin_cnt;
    else if (n == "contig_len") b = &t->contig_len; else if (n == "pool") b = &c.pool;
    else if (n == "counters") { *ptr_out = t->d_ctr; *bytes_out = sizeof(Counters); return KH_OK; }
    else if (n == "caps") {          // host-side numbers: hcap, seg_cap, inbox_cap, cap_rs, chunks_per_rank, regions_per_rank
        static thread_local uint64_t v[8];
        v[0] = c.caps.hcap; v[1] = c.caps.seg_cap; v[2] = c.caps.inbox_cap; v[3] = c.caps.xin_cap; v[4] = c.g.chunks_per_rank; v[5] = 0;
        v[6] = c.epoch; v[7] = 0;
        *ptr_out = v; *bytes_out = sizeof(v); return KH_OK;
    }
    if (!b) return fail(t, KH_ERR_ARG, "unknown buffer " + n);
    *ptr_out = b->p; *bytes_out = b->cap;
    return KH_OK;
}

uint64_t kh_slot_bytes(int k) { return (ct_supported(k) ? ct_slot_words(k) : ((2 * k + 6 <= 64) ? 1 : 2)) * 8; }

// device -> host copy on the handle's stream, synchronous (tests / result collection)
int kh_copy_to_host(kh_table* t, void* dst_host, const void* src_dev, uint64_t bytes) {
    if (!t || (bytes && (!dst_host || !src_dev))) return KH_ERR_ARG;
    KH_CUDA(t, cudaSetDevice(t->device));
    if (bytes) KH_CUDA(t, cudaMemcpyAsync(dst_host, src_dev, bytes, cudaMemcpyDeviceToHost, t->stream));
    KH_CUDA(t, cudaStreamSynchronize(t->stream));
    return KH_OK;
}
int kh_copy_device(kh_table* t, void* dst_dev, const void* src_dev, uint64_t bytes) {
    if (!t || (bytes && (!dst_dev || !src_dev))) return KH_ERR_ARG;
    KH_CUDA(t, cudaSetDevice(t->device));
    if (bytes) KH_CUDA(t, cudaMemcpyAsync(dst_dev, src_dev, bytes, cudaMemcpyDefault, t->stream));
    return KH_OK;
}
int kh_device_alloc(void** ptr, uint64_t bytes) {
    if (!ptr) return KH_ERR_ARG;
    if (cudaMalloc(ptr, bytes ? bytes : 1) != cudaSuccess) { cudaGetLastError(); *ptr = nullptr; return KH_ERR_NOMEM; }
    return KH_OK;
}
int kh_device_alloc_on(int device, void** ptr, uint64_t bytes) {
    if (!ptr) return KH_ERR_ARG;
    if (cudaSetDevice(device) != cudaSuccess) { cudaGetLastError(); *ptr = nullptr; return KH_ERR_CUDA; }
    return kh_device_alloc(ptr, bytes);
}
int kh_device_free(void* ptr) {
    if (ptr && cudaFree(ptr) != cudaSuccess) { cudaGetLastError(); return KH_ERR_CUDA; }
    return KH_OK;
}

}  // extern "C"
