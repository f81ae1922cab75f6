// ctable.cuh -- the chunk table: a batch-built hash table whose build step also contracts every contig into
// one segment per supermer, for any number of GPUs.
//
// Replaces, together with the host code in capi.cu ("ct_*"):
//   DistributedHashMap::insert_all / insert_batch_remote   hash_map.hpp:55-80, 38-46   -> ct_stage / ct_scatter / ct_build
//   DistributedHashMap::find (local + remote branch)        hash_map.hpp:83-107          -> ct_find, ct_resolve (+ inbox)
//   assemble_contigs                                        kmer_hash.cpp:38-55          -> ct_build (in shared memory) + ct_resolve
//                                                                                           + ct_rank_round + ct_lengths/claim + ct_emit
//
// Why: a contig walk over a plainly hashed table costs one random DRAM access per k-mer, and HBM serves only
// ~41 G of those per second whatever their size (profiles/r01_random_access_probe_occ8.txt) -- 2.7 ms for the
// chr14 shape, 0.17 of the bandwidth roofline.  Here the home CHUNK of a k-mer (<= 64-72 KB of table) is chosen
// by a hash of its MINIMIZER and only the bucket inside the chunk by the key (slot.cuh).  Consecutive k-mers of a
// contig share the minimizer for a supermer, so while a block holds a chunk in shared memory to build it, it also
// follows every successor link that stays inside the chunk (an LDS probe instead of a DRAM access) and emits one
// contracted SEGMENT per run: its forward-extension characters, and the key of the k-mer that follows it.  What
// is left for HBM is ONE lookup per segment (every ~4 k-mers at K=19, ~16 at K=51) to chain the segments, then
// pointer jumping over the segment list and the copy of the characters.
//
// The table is static: inserts are only STAGED (grouped by table region, ct_stage_kernel); the first find /
// assemble SEALS it: group by chunk (ct_scatter_kernel), size every chunk for its actual load (ct_layout_kernel:
// each chunk gets load / load_factor slots, so the load factor holds per chunk no matter how lumpy the minimizer
// hash is) and build + contract (ct_build_kernel).  Inserting after a seal re-seals from the staged records.
//
// Multi-GPU: chunk ids are global, rank r owns chunks [r*C, (r+1)*C).  ct_stage_kernel writes a record's slot
// value straight into the staging buffer of the owning GPU through its NVLink peer mapping while it groups
// (the all-to-all of hash_map.hpp:64-77 fused into the grouping pass, no separate exchange step); pending
// segment links travel the same way (ct_resolve_kernel -> the owner's inbox) and are answered with one peer store.
// Phases are separated by an in-stream flag barrier (ct_barrier_kernel); the host never waits inside a step.
//
// Segment ids: global id = (rank << 28) | local id.  Local ids [0, hcap) are the contig HEAD STUBS of the start
// nodes parsed by this rank (zero characters, pending link to the segment that starts with the start k-mer --
// rank r therefore emits exactly the reference's <prefix>_<r>.dat); chunk segments follow from hcap upward.
//   link[seg]  = (next segment gid << 32) | characters between this segment's start and the start of `next`
//                (markers in the high word: kLinkTail / kLinkPending / kLinkMissing / kLinkConverge / kLinkClaimed)
//   meta[seg]  = (offset of the segment's characters in the rank's character pool << 24) | number of characters
#pragma once
#include "kernels.cuh"

namespace kh {

// Build-kernel geometry, overridable at compile time for tuning runs (tools/probes/build_variants.sh): buckets per chunk
// for 128-bit slots, threads per block, blocks per SM.
#ifndef KH_CT_BUCKETS2
#define KH_CT_BUCKETS2 2176
#endif
#ifndef KH_CT_THREADS
#define KH_CT_THREADS 512
#endif
#ifndef KH_CT_MINBLOCKS
#define KH_CT_MINBLOCKS 2
#endif
// pointer-jumping passes between two block-wide barriers in phase 4.  The jumps are in place (a stale read is still a
// valid (ancestor, distance) pair), so several passes per barrier are safe; 3 measured best (build 4.24 -> 4.15 ms at
// K=51: profiles/r02_build_geometry_variants.txt) -- the kernel is as much barrier- as issue-bound.
#ifndef KH_CT_JUMPS
#define KH_CT_JUMPS 3
#endif
// Rounds of phase 4 that settle a chain of n + 1 nodes: the smallest R with (KH_CT_JUMPS + 1)^R >= n.  Between two
// barriers a thread may see every other thread's (ancestor, distance) pair as it stood at the last barrier, so a round
// of J passes multiplies a node's reach by J + 1 (not 2^J); only its own nodes' writes it sees at once.
constexpr int ct_jump_rounds(u32 n, u64 reach = 1) { return reach >= n ? 0 : 1 + ct_jump_rounds(n, reach * (KH_CT_JUMPS + 1)); }
template <int W> struct CtBuild {
    // A chunk = one run of buckets that a thread block builds in shared memory.  Shared memory per block:
    //   table | succ u16[node] (later the characters) | (ancestor, distance) u32[node] | ext code + flags u8[node] | pool offset u16[node]
    // = 104 448 B (64-bit slots) / 108 800 B (128-bit slots): two blocks of 512 threads per SM.
    static constexpr u32 kMaxBuckets = (W == 1) ? 1536u : (u32)KH_CT_BUCKETS2;                 // 48 / 68 KB of table per chunk
    static constexpr u32 kMaxSlots = kMaxBuckets * (u32)Slot<W>::kPerBucket;      // 6144 / 4352: also the most records a chunk can take
    static constexpr u32 kOffSucc = kMaxBuckets * 32u;
    static constexpr u32 kOffPd = kOffSucc + kMaxSlots * 2u;
    static constexpr u32 kOffOff = kOffPd + kMaxSlots * 4u;
    static constexpr u32 kOffCode = kOffOff + kMaxSlots * 2u;
    static constexpr u32 kSmem = kOffCode + kMaxSlots;
    // pointer-jumping rounds of phase 4: enough for one chain through every record of a full chunk
    static constexpr int kJumpRounds = ct_jump_rounds(kMaxSlots - 1);
};
constexpr int kCtBuildThreads = KH_CT_THREADS;
static_assert(CtBuild<1>::kMaxSlots <= 0x8000u && CtBuild<2>::kMaxSlots <= 0x8000u, "node ids stay below kSuccExt");
static_assert(CtBuild<1>::kMaxSlots <= 32u * kCtBuildThreads && CtBuild<2>::kMaxSlots <= 32u * kCtBuildThreads,
              "phase 4 keeps a thread's unsettled nodes in one 32-bit mask");
static_assert(KH_CT_JUMPS != 3 || (CtBuild<1>::kJumpRounds == 7 && CtBuild<2>::kJumpRounds == 7),
              "4^7 >= 6143 > 4^6: seven rounds of three passes settle a chain through a full chunk of either slot width");
// Where record number `at` of chunk `chunk` lives in the chunk buffers: position-major, in groups of one 128-byte
// line (8 or 16 records).  All chunks fill at about the same rate, so at any moment the appends of the staging pass
// land in a window of a few hundred MB instead of being spread over every chunk's own multi-KB buffer (3.7 GB in
// all): far fewer TLB misses (tools/probes/scatter_probe.cu: 1.99 -> 1.42 ms for the chr14 shape).
template <int W>
__host__ __device__ __forceinline__ u64 ct_fine_index(u32 chunk, u32 at, u32 nchunks) {
    constexpr u32 G = 128u / (u32)sizeof(typename Slot<W>::value_t);
    return ((u64)(at / G) * nchunks + chunk) * G + (at % G);
}
// s_succ[node]: successor node (< 0x8000) | kSuccExt + own slot (successor is not in this chunk) | kSuccTail | kSuccDead
constexpr u32 kSuccExt = 0x8000u, kSuccTail = 0xFFFFu, kSuccDead = 0xFFFDu, kPredNone = 0xFFFFu;
// s_code[node]: forward extension code in bits 0..2, then
constexpr u32 kCodeBackF = 8u, kCodeMulti = 16u;

template <int W> struct CtReq;                                                      // a pending link on its way to the owner
template <> struct alignas(16) CtReq<1> { u64 key; u32 src; u32 chunk; };
template <> struct alignas(16) CtReq<2> { u128 key; u32 src; u32 chunk; u64 pad; };

struct CtPeers {
    int world, rank;
    void* xin_vals[kMaxRanks];            // [world][xin_cap] slot values this rank received, by source rank
    u32* xin_chunk[kMaxRanks];            // their local chunk ids, same shape
    u32* xin_cnt[kMaxRanks];              // [world] published fill of each source's part
    void* extra_vals[kMaxRanks];          // records that found their part of xin full
    u32* extra_chunk[kMaxRanks];
    u32* extra_cnt[kMaxRanks];
    u64* link[kMaxRanks];
    u64* meta[kMaxRanks];
    void* inbox[kMaxRanks];               // [world][inbox_cap] link requests, by source rank
    u32* inbox_cnt[kMaxRanks];
    u32* answers[kMaxRanks];              // [world][inbox_cap] on the REQUESTER: answers[o * inbox_cap + i] = owner o's answer to its request i
    u64* g_link[kMaxRanks];               // [world][seg_cap]: every rank's copy of every other rank's segment links ...
    u64* g_meta[kMaxRanks];               //   ... and segment meta words (gather before the contig walk)
    unsigned char* g_pool[kMaxRanks];     // [world][pool_stride]: ... and contig characters
    u32* g_hdr[kMaxRanks];                // [world][2]: segments / pool bytes each rank has sent
    u32* contig_pre[kMaxRanks];
    u64* contig_off[kMaxRanks];
    char* out[kMaxRanks];
    u64 out_cap[kMaxRanks];
    u32* flags[kMaxRanks];                // barrier: flags[r][2 * s + parity] = (epoch << 1 | payload bit) rank s signalled to rank r
};

struct CtCaps {
    u32 xin_cap, extra_cap, inbox_cap, seg_cap, hcap;
    u64 nbuckets_alloc, pool_cap;
    u64 g_seg_stride, g_pool_stride;      // per-rank strides of the gathered copies (the same on every rank)
};

__device__ __forceinline__ void ct_internal(Counters* ctr, u32 site) {
    atomicOr(&ctr->errors, kErrInternal);
    atomicOr(&ctr->err_where, site);
}

// ---- in-stream barrier across the GPUs of one step -------------------------------------------------------
// One warp; lane r signals rank r (a store into ITS flag array) and waits for rank r's signal in ours.  Everything
// the previous kernels of this stream wrote -- including stores into peer memory -- is complete when this kernel
// starts, and the release/acquire pair orders the flag against them.  A peer that never arrives (it failed) ends
// the wait after ~4 s with kErrInternal instead of hanging the GPU.
// The flag carries one payload bit next to the epoch.  The barriers between pointer-jumping rounds (round >= 0)
// use it for "this rank moved a link in this round": every rank sees the same bits, so all of them agree when
// nobody moved -- they set rank_done and the remaining round and barrier kernels of the step return at once.
__global__ void ct_barrier_kernel(const CtPeers pe, u32 epoch, Counters* ctr, int round) {
    const int r = (int)threadIdx.x;
    if (round >= 0 && ctr->rank_done) return;                    // agreed on by all ranks: nobody waits here any more
    const u32 bit = round >= 0 ? (ctr->flags[round] ? 1u : 0u) : (round == -2 ? (ctr->need_jump ? 1u : 0u) : 0u);
    u32 peer_bit = 0;
    if (r < pe.world) {
        __threadfence_system();
        u32* dst = pe.flags[r] + 2 * pe.rank + (epoch & 1u);           // two slots per peer, by epoch parity: a peer that is already
        asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(dst), "r"((epoch << 1) | bit) : "memory");
        const u32* src = pe.flags[pe.rank] + 2 * r + (epoch & 1u);      // one barrier ahead cannot overwrite the value we still have to read
        unsigned long long t0, t1;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
        for (;;) {
            u32 seen;
            asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(seen) : "l"(src) : "memory");
            // A NEWER epoch in this slot: the peer has passed this barrier and at least one more of the same parity.  Between
            // two real barriers parity alternates, so it can only have got there by SKIPPING round barriers (rank_done, the
            // early return above) -- i.e. it saw every rank's bit of this epoch as 0, its own included.  Reading that as 0
            // keeps the ranks in agreement (read as 1, this rank would go on alone and wait at a barrier the others skip).
            if ((int)((seen >> 1) - epoch) >= 0) { peer_bit = ((seen >> 1) == epoch) ? (seen & 1u) : (round >= 0 ? 0u : 1u); break; }
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
            if (t1 - t0 > 4000000000ull) { ct_internal(ctr, kSiteBarrier); peer_bit = 1; break; }
            __nanosleep(200);
        }
        __threadfence_system();
    }
    if (round >= 0) {
        const u32 any = __ballot_sync(kFullMask, peer_bit != 0);
        if (r == 0 && any == 0) ctr->rank_done = 1;
    } else if (round == -2) {                                    // some rank has a contig too long for the bounded walk: all take the slow path
        const u32 any = __ballot_sync(kFullMask, peer_bit != 0);
        if (r == 0) ctr->use_jump = any ? 1u : 0u;
    }
}

// ---- pass A: every record goes to the per-chunk buffer of its home chunk ----------------------------------------
// hash_map.hpp:55-80 (insert_all: bucket by owner, one batch per destination) fused with the grouping the build
// needs.  A block parses a tile of 2048 records (staged through shared memory), computes minimizer -> (owner, chunk)
// and then
//   * records this GPU owns: one atomicAdd on the chunk's cursor, one 8/16-byte store into the chunk's buffer.  The
//     write frontier is one line per chunk (a few MB in all), so L2 merges the stores into full lines: no second
//     grouping pass, no staging copy;
//   * records another GPU owns: block-local counting sort by owner (<= 8 bins), then ONE coalesced run per
//     (block, owner) of values + chunk ids straight into the owner's receive buffer through its NVLink mapping --
//     NVLink wants long runs; small scattered peer stores run at a few G/s.  The owner scatters what it received
//     into its chunk buffers after the barrier (ct_xin_scatter_kernel).
// Also the start bitmask / per-tile start counts for the order-preserving start scan (kmer_hash.cpp:27-31).
// kmer_pair bytes -> slot value from the aligned 32-bit words that cover the record (sh = 8 * (address & 3)):
// kmer_pair::init / packKmer (kmer_t.hpp:67-76, packing.hpp:77-92) read back as one big-endian number
template <int W> __device__ __forceinline__ typename Slot<W>::value_t ct_record_from_words(const u32 (&w)[W == 1 ? 3 : 5], u32 sh, int k, int pl, bool& ok);
template <> __device__ __forceinline__ u64 ct_record_from_words<1>(const u32 (&w)[3], u32 sh, int k, int pl, bool& ok) {
    const u32 b0 = __funnelshift_r(w[0], w[1], sh), b1 = __funnelshift_r(w[1], w[2], sh);      // bytes 0-3, 4-7 of the record
    const u64 be = ((u64)__byte_perm(b0, 0, 0x0123) << 32) | (u64)__byte_perm(b1, 0, 0x0123);
    const u64 key = be >> (64 - 2 * k);
    const u32 ext = (u32)((((u64)b1 << 32) | b0) >> (8 * pl));                                     // pl <= 6: both letters inside the 8 bytes
    const u32 b = ext_code((unsigned char)ext), f = ext_code((unsigned char)(ext >> 8));
    ok = (b != kExtBad) && (f != kExtBad);
    return (key << 6) | ((u64)(b & 7u) << 3) | (u64)((f + 1u) & 7u);
}
template <> __device__ __forceinline__ u128 ct_record_from_words<2>(const u32 (&w)[5], u32 sh, int k, int pl, bool& ok) {
    const u32 b0 = __funnelshift_r(w[0], w[1], sh), b1 = __funnelshift_r(w[1], w[2], sh);
    const u32 b2 = __funnelshift_r(w[2], w[3], sh), b3 = __funnelshift_r(w[3], w[4], sh);
    const u64 hi = ((u64)__byte_perm(b0, 0, 0x0123) << 32) | (u64)__byte_perm(b1, 0, 0x0123);
    const u64 lo = ((u64)__byte_perm(b2, 0, 0x0123) << 32) | (u64)__byte_perm(b3, 0, 0x0123);
    u128 v = Slot<2>::shr_any(u128{lo, hi}, 122 - 2 * k);
    const int wq = pl >> 2;                                                                          // 1..3 (pl = 6..14), uniform
    const u32 e0 = wq == 1 ? b1 : (wq == 2 ? b2 : b3), e1 = wq == 1 ? b2 : (wq == 2 ? b3 : 0u);
    const u32 ext = __funnelshift_r(e0, e1, 8u * (pl & 3));
    const u32 b = ext_code((unsigned char)ext), f = ext_code((unsigned char)(ext >> 8));
    ok = (b != kExtBad) && (f != kExtBad);
    v.lo = (v.lo & ~63ull) | ((u64)(b & 7u) << 3) | (u64)((f + 1u) & 7u);
    return v;
}

constexpr int kStgThreads = 256;
constexpr int kStgPer = 4;
constexpr int kStgTile = kStgThreads * kStgPer;     // 1024 records per block = one tile of the start scan (kInsTile)

template <int W>
__global__ void __launch_bounds__(kStgThreads, 5)
ct_stage_kernel(const unsigned char* __restrict__ recs, u64 n, const CtGeom g, const CtPeers pe, const CtCaps caps,
                u32* __restrict__ chunk_cursor, typename Slot<W>::value_t* __restrict__ fine, u32* __restrict__ xout_cursor,
                u32* __restrict__ start_mask, u32* __restrict__ tile_starts, Counters* ctr) {
    typedef Slot<W> S;
    typedef typename S::value_t V;
    constexpr u32 kMaxSlots = CtBuild<W>::kMaxSlots;
    extern __shared__ __align__(16) unsigned char s_raw[];
    // s_raw (multi-GPU only): the remote values of the tile sorted by owner | their chunk ids
    V* s_sorted = reinterpret_cast<V*>(s_raw);
    u32* s_schunk = reinterpret_cast<u32*>(s_raw + (size_t)kStgTile * sizeof(V));
    __shared__ u32 s_cnt[kMaxRanks], s_off[kMaxRanks + 1], s_gbase[kMaxRanks];
    __shared__ u32 s_starts[kStgTile / kInsTile], s_err;
    const int k = g.k, pl = (k + 3) >> 2, pb = pl + 2;
    const u64 rec0 = (u64)blockIdx.x * kStgTile;
    const u32 cnt = (u32)min((u64)kStgTile, n - rec0);
    const bool multi = g.world > 1;
    if (threadIdx.x < kMaxRanks) s_cnt[threadIdx.x] = 0;
    if (threadIdx.x < kStgTile / kInsTile) s_starts[threadIdx.x] = 0;
    if (threadIdx.x == 0) s_err = 0;
    // Records come straight from global memory into registers: a warp reads 32 consecutive records (a few hundred
    // contiguous bytes) with aligned 32-bit loads, L1 serves the overlap between neighbours.  All loads of a thread are
    // issued before the first record is parsed; no shared-memory staging, no barrier on the single-GPU path.
    constexpr int kWords = W == 1 ? 3 : 5;
    u32 raw[kStgPer][kWords];
    u32 shift[kStgPer];
#pragma unroll
    for (int r = 0; r < kStgPer; ++r) {
        const u32 j = threadIdx.x + r * kStgThreads;
        const u64 addr = reinterpret_cast<u64>(recs) + (rec0 + j) * (u64)pb;
        shift[r] = ((u32)addr & 3u) * 8u;
        const u32* wp = reinterpret_cast<const u32*>(addr & ~3ull);
        // the last records of the array are read word by word only as far as the array goes
        const u64 end = reinterpret_cast<u64>(recs) + n * (u64)pb;
#pragma unroll
        for (int q = 0; q < kWords; ++q)
            raw[r][q] = (j < cnt && reinterpret_cast<u64>(wp + q) < end) ? __ldg(wp + q) : 0u;
    }
    __syncthreads();                                   // the shared counters above
    V v[kStgPer];
    u32 dst[kStgPer];            // local chunk id, or 0xFFFFFFFF for a record that is not placed here
    u32 at[kStgPer];             // position in the chunk's buffer (local) / rank inside the owner's bin (remote)
    u32 own[kStgPer];            // owner rank of a remote record, 0xFFFFFFFF otherwise
    u32 err = 0;
#pragma unroll
    for (int r = 0; r < kStgPer; ++r) {
        const u32 j = threadIdx.x + r * kStgThreads;
        bool ok = true, live = j < cnt;
        dst[r] = 0xFFFFFFFFu; own[r] = 0xFFFFFFFFu; at[r] = 0;
        v[r] = ct_record_from_words<W>(raw[r], shift[r], k, pl, ok);
        if (!live) v[r] = S::zero();
        if (live && !ok) { err |= kErrBadInput; live = false; }
        if (live) {
            u32 owner, chunk;
            ct_place(ct_min_hash<W>(v[r], g.m, g.win), g, owner, chunk);
            dst[r] = chunk;
            if (!multi || owner == (u32)g.rank) at[r] = atomicAdd(&chunk_cursor[chunk], 1u);
            else own[r] = owner;
        }
        if (multi) {                                   // rank of a remote record inside its owner's bin of this tile
            const unsigned same = __match_any_sync(kFullMask, own[r]);
            const int leader = __ffs(same) - 1;
            u32 first = 0;
            if ((int)lane_id() == leader && own[r] != 0xFFFFFFFFu) first = atomicAdd(&s_cnt[own[r]], (u32)__popc(same));
            first = __shfl_sync(kFullMask, first, leader);
            if (own[r] != 0xFFFFFFFFu) at[r] = first + (u32)__popc(same & ((1u << lane_id()) - 1u));
        }
        const u32 bal = __ballot_sync(kFullMask, live && S::back(v[r]) == kExtF);
        const u64 first_rec = rec0 + (u64)r * kStgThreads + (threadIdx.x & ~31u);
        if (lane_id() == 0 && first_rec < n) {
            start_mask[first_rec >> 5] = bal;
            if (bal) atomicAdd(&s_starts[(r * kStgThreads + threadIdx.x) / kInsTile], (u32)__popc(bal));
        }
    }
    // records of this GPU: straight into their chunk's buffer
#pragma unroll
    for (int r = 0; r < kStgPer; ++r) {
        if (dst[r] == 0xFFFFFFFFu || own[r] != 0xFFFFFFFFu) continue;
        if (at[r] < kMaxSlots) fine[ct_fine_index<W>(dst[r], at[r], g.chunks_per_rank)] = v[r];
        else { err |= kErrTableFull; atomicOr(&ctr->err_where, kSiteChunkFull); }      // more k-mers share this chunk than it can hold
    }
    err = __reduce_or_sync(kFullMask, err);
    if (lane_id() == 0 && err) atomicOr(&s_err, err);
    if (multi) {
        __syncthreads();                               // s_cnt complete
        if (threadIdx.x == 0) {
            u32 run = 0;
            for (int d = 0; d < g.world; ++d) {
                s_off[d] = run;
                s_gbase[d] = s_cnt[d] ? atomicAdd(&xout_cursor[d], s_cnt[d]) : 0u;
                run += s_cnt[d];
            }
            s_off[g.world] = run;
        }
        __syncthreads();
#pragma unroll
        for (int r = 0; r < kStgPer; ++r) {
            if (own[r] == 0xFFFFFFFFu) continue;
            const u32 pos = s_off[own[r]] + at[r];
            s_sorted[pos] = v[r];
            s_schunk[pos] = dst[r];
        }
        __syncthreads();
        const u32 total = s_off[g.world];
        for (u32 pos = threadIdx.x; pos < total; pos += kStgThreads) {
            u32 d = 0;
#pragma unroll
            for (int q = 1; q < kMaxRanks; ++q) d += (q < g.world && pos >= s_off[q]) ? 1u : 0u;
            const u32 i = s_gbase[d] + (pos - s_off[d]);
            if (i < caps.xin_cap) {
                const u64 slot = (u64)g.rank * caps.xin_cap + i;
                static_cast<V*>(pe.xin_vals[d])[slot] = s_sorted[pos];
                pe.xin_chunk[d][slot] = s_schunk[pos];
            } else {                                   // this source's part of the owner's buffer is full: hand it over one by one
                const u32 o = atomicAdd_system(pe.extra_cnt[d], 1u);
                if (o < caps.extra_cap) {
                    static_cast<V*>(pe.extra_vals[d])[o] = s_sorted[pos];
                    pe.extra_chunk[d][o] = s_schunk[pos];
                } else {
                    atomicOr(&s_err, kErrTableFull);    // far more records than the table was sized for
                }
            }
        }
    }
    __syncthreads();
    if (threadIdx.x < kStgTile / kInsTile) {
        const u64 tile = (u64)blockIdx.x * (kStgTile / kInsTile) + threadIdx.x;
        if (tile * kInsTile < n) tile_starts[tile] = s_starts[threadIdx.x];
    }
    if (threadIdx.x == 0 && s_err) atomicOr(&ctr->errors, s_err);
}

// tell every owner how much this source has put into its receive buffer
__global__ void ct_publish_xin_kernel(const CtPeers pe, const CtCaps caps, const u32* __restrict__ xout_cursor) {
    const int d = (int)threadIdx.x;
    if (d < pe.world && d != pe.rank) pe.xin_cnt[d][pe.rank] = min(xout_cursor[d], caps.xin_cap);
}

// start nodes seen so far live on the device (no host round trip per insert call in the sharded path); follows
// ct_scatter_starts_kernel in a sharded insert (a non-sharded handle has read the count and stores it from the host)
__global__ void ct_bump_starts_kernel(Counters* ctr, u32 hcap) {
    const u64 total = ctr->n_starts_dev + ctr->scan_total;
    if (total > hcap) { ct_internal(ctr, kSiteStarts); ctr->n_starts_dev = hcap; }
    else ctr->n_starts_dev = total;
}

// ---- the owner files what it received: receive buffer -> chunk buffers ------------------------------------------
// done[s] = records of source s already filed (an insert after a seal only adds the new ones)
template <int W>
__global__ void __launch_bounds__(256)
ct_xin_scatter_kernel(const typename Slot<W>::value_t* __restrict__ xin_vals, const u32* __restrict__ xin_chunk,
                      const u32* __restrict__ xin_cnt, const u32* __restrict__ xin_done, const CtGeom g, const CtCaps caps,
                      u32* __restrict__ chunk_cursor, typename Slot<W>::value_t* __restrict__ fine, Counters* ctr) {
    constexpr u32 kMaxSlots = CtBuild<W>::kMaxSlots;
    u32 err = 0;
    for (int src = 0; src < g.world; ++src) {
        if (src == g.rank) continue;
        const u32 n = min(xin_cnt[src], caps.xin_cap), n0 = min(xin_done[src], n);
        const u64 base = (u64)src * caps.xin_cap;
        for (u32 i = n0 + blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
            const u32 c = xin_chunk[base + i];
            const u32 at = atomicAdd(&chunk_cursor[c], 1u);
            if (at < kMaxSlots) fine[ct_fine_index<W>(c, at, g.chunks_per_rank)] = xin_vals[base + i];
            else err |= kErrTableFull;
        }
    }
    if (err) { atomicOr(&ctr->errors, err); atomicOr(&ctr->err_where, kSiteChunkFull); }
}

template <int W>
__global__ void __launch_bounds__(256)
ct_extra_kernel(const typename Slot<W>::value_t* __restrict__ extra_vals, const u32* __restrict__ extra_chunk,
                const u32* __restrict__ extra_cnt, const u32* __restrict__ extra_done, const CtCaps caps, u32 nchunks, u32* __restrict__ chunk_cursor,
                typename Slot<W>::value_t* __restrict__ fine, Counters* ctr) {
    constexpr u32 kMaxSlots = CtBuild<W>::kMaxSlots;
    const u32 n = min(*extra_cnt, caps.extra_cap), n0 = min(*extra_done, n);
    for (u32 i = n0 + blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const u32 c = extra_chunk[i];
        const u32 at = atomicAdd(&chunk_cursor[c], 1u);
        if (at < kMaxSlots) fine[ct_fine_index<W>(c, at, nchunks)] = extra_vals[i];
        else { atomicOr(&ctr->errors, kErrTableFull); atomicOr(&ctr->err_where, kSiteChunkFull); }
    }
}

// what has been filed so far (runs after the two kernels above)
__global__ void ct_mark_filed_kernel(const u32* __restrict__ xin_cnt, u32* __restrict__ xin_done, const u32* __restrict__ extra_cnt,
                                     u32* __restrict__ extra_done, const CtCaps caps, int world) {
    const int s = (int)threadIdx.x;
    if (s < world) xin_done[s] = min(xin_cnt[s], caps.xin_cap);
    if (s == 0) *extra_done = min(*extra_cnt, caps.extra_cap);
}

// ---- layout: every chunk gets load / load_factor slots ------------------------------------------------------
// chunk_base[c] = first bucket of chunk c (C + 1 entries), pool_off[c] = offset of its characters (16-byte aligned)
__global__ void __launch_bounds__(1024)
ct_layout_kernel(const u32* __restrict__ chunk_cursor, u32 nchunks, const CtGeom g, const CtCaps caps, u32 per_bucket, u32 max_slots,
                 u32* __restrict__ chunk_base, u32* __restrict__ pool_off, Counters* ctr) {
    __shared__ u64 s_warp[33];
    constexpr u32 kPer = 8;                                       // consecutive chunks per thread: 8192 chunks per block-wide scan
    u64 carry_b = 0, carry_p = 0;
    bool over = false;                                            // a chunk was offered more records than it holds
    for (u32 c0 = 0; c0 < nchunks; c0 += blockDim.x * kPer) {
        const u32 first = c0 + threadIdx.x * kPer;
        u32 capb[kPer], chars[kPer];
        u64 sum_b = 0, sum_p = 0;
#pragma unroll
        for (u32 q = 0; q < kPer; ++q) {
            const u32 c = first + q;
            capb[q] = 0; chars[q] = 0;
            if (c < nchunks) {
                over |= chunk_cursor[c] > max_slots;
                const u32 load = min(chunk_cursor[c], max_slots);
                if (load) {
                    const u64 want_slots = ((u64)load * g.lf_inv_q16 + 65535u) >> 16;
                    capb[q] = (u32)min((u64)g.max_buckets, max((want_slots + per_bucket - 1) / per_bucket, (u64)(load / per_bucket + 1)));
                }
                chars[q] = (load + 15u) & ~15u;
            }
            sum_b += capb[q]; sum_p += chars[q];
        }
        u64 tot_b, tot_p;
        u64 eb = carry_b + block_exclusive_scan(sum_b, s_warp, tot_b);
        u64 ep = carry_p + block_exclusive_scan(sum_p, s_warp, tot_p);
#pragma unroll
        for (u32 q = 0; q < kPer; ++q) {
            const u32 c = first + q;
            if (c < nchunks) { chunk_base[c] = (u32)eb; pool_off[c] = (u32)ep; }
            eb += capb[q]; ep += chars[q];
        }
        carry_b += tot_b; carry_p += tot_p;
    }
    if (threadIdx.x == 0) {
        chunk_base[nchunks] = (u32)carry_b;
        pool_off[nchunks] = (u32)carry_p;
        if (carry_b > caps.nbuckets_alloc || carry_p > caps.pool_cap) atomicOr(&ctr->errors, kErrTableFull);
    }
    if (over) { atomicOr(&ctr->errors, kErrTableFull); atomicOr(&ctr->err_where, kSiteChunkFull); }
}

// ---- pass B: build a chunk in shared memory and contract its chains ------------------------------------------
// Nodes are the chunk's RECORDS (dense ids 0 .. cnt-1), so every phase after the insert runs with full warps at any
// load factor; while the chunk is being built a slot's index bits carry 1 + the node id of the k-mer stored there.
//
// Probing compares 32-bit tags (key bits 0..31; an occupied slot has a non-zero forward field, so "empty" is a test
// of three bits) and touches the rest of a slot only on a tag match: two LDS.64 per 128-bit bucket instead of 32 bytes.
template <int W> __device__ __forceinline__ u32 ct_tag(typename Slot<W>::value_t v);
template <> __device__ __forceinline__ u32 ct_tag<1>(u64 v) { return (u32)(v >> 6); }
template <> __device__ __forceinline__ u32 ct_tag<2>(u128 v) { return (u32)(v.lo >> 6); }

template <int W, bool VOLATILE>
__device__ __forceinline__ void ct_lds_tags(unsigned saddr, u64 (&w)[4]) {        // the word of each slot of a bucket that holds ext bits + low key bits
    if (W == 1) {
        if (VOLATILE) {
            asm volatile("ld.volatile.shared.v2.u64 {%0,%1}, [%2];" : "=l"(w[0]), "=l"(w[1]) : "r"(saddr) : "memory");
            asm volatile("ld.volatile.shared.v2.u64 {%0,%1}, [%2+16];" : "=l"(w[2]), "=l"(w[3]) : "r"(saddr) : "memory");
        } else {
            asm volatile("ld.shared.v2.u64 {%0,%1}, [%2];" : "=l"(w[0]), "=l"(w[1]) : "r"(saddr));
            asm volatile("ld.shared.v2.u64 {%0,%1}, [%2+16];" : "=l"(w[2]), "=l"(w[3]) : "r"(saddr));
        }
    } else {
        if (VOLATILE) {
            asm volatile("ld.volatile.shared.u64 %0, [%1];" : "=l"(w[0]) : "r"(saddr) : "memory");
            asm volatile("ld.volatile.shared.u64 %0, [%1+16];" : "=l"(w[1]) : "r"(saddr) : "memory");
        } else {
            asm volatile("ld.shared.u64 %0, [%1];" : "=l"(w[0]) : "r"(saddr));
            asm volatile("ld.shared.u64 %0, [%1+16];" : "=l"(w[1]) : "r"(saddr));
        }
    }
}
__device__ __forceinline__ u64 ct_lds64(unsigned saddr) {
    u64 x;
    asm volatile("ld.volatile.shared.u64 %0, [%1];" : "=l"(x) : "r"(saddr) : "memory");
    return x;
}
// full comparison of slot i of the bucket at saddr with `key` (extension and index bits ignored), given its low word
template <int W> __device__ __forceinline__ bool ct_verify(unsigned saddr, int i, u64 low, typename Slot<W>::value_t key, u64& idx_word);
template <> __device__ __forceinline__ bool ct_verify<1>(unsigned, int, u64 low, u64 key, u64& idx_word) {
    idx_word = low;
    return CtSlot<1>::same_key(low, key);
}
template <> __device__ __forceinline__ bool ct_verify<2>(unsigned saddr, int i, u64 low, u128 key, u64& idx_word) {
    idx_word = ct_lds64(saddr + 16u * i + 8u);
    return (((idx_word ^ key.hi) << kIdxBits) | ((low ^ key.lo) >> 6)) == 0ull;
}

// insert `val` (slot value with the node id in its index bits) into the chunk held in shared memory; linear probing
// that wraps inside the chunk.  Returns the slot index, or -1 for a duplicate key, -2 if the chunk is full.
template <int W>
__device__ __forceinline__ int ct_smem_insert(typename Slot<W>::value_t* s_tab, unsigned s_base, u32 nb, typename Slot<W>::value_t val) {
    typedef Slot<W> S;
    typedef typename S::value_t V;
    const u32 tag = ct_tag<W>(val);
    u32 b = ct_bucket_in_chunk(CtSlot<W>::hash32(val), nb);
    for (u32 tries = 0; tries < nb;) {
        u64 w[4];
        ct_lds_tags<W, true>(s_base + b * 32u, w);
        int j = -1;
        u32 match = 0;
#pragma unroll
        for (int i = S::kPerBucket - 1; i >= 0; --i) {
            const bool e = ((u32)w[i] & 7u) == 0u;
            j = e ? i : j;
            match |= (!e && (u32)(w[i] >> 6) == tag) ? (1u << i) : 0u;
        }
        if (match) {                                     // rare: the same 32 low key bits -- look at the whole key
#pragma unroll
            for (int i = 0; i < S::kPerBucket; ++i) {
                u64 iw;
                if ((match >> i) & 1u) if (ct_verify<W>(s_base + b * 32u, i, w[i], val, iw)) return -1;
            }
        }
        if (j < 0) { b = (b + 1 == nb) ? 0u : b + 1; ++tries; continue; }
        const V old = S::cas_shared(s_tab + b * S::kPerBucket + j, S::zero(), val);
        if (S::empty(old)) return (int)(b * S::kPerBucket + j);
        if (CtSlot<W>::same_key(old, val)) return -1;
    }
    return -2;
}

// One bucket of a lookup in the finished chunk: node id of `key` (from the index bits of its slot) if it is here,
// kFindMiss if the bucket has a hole (the key is not in the chunk), kFindNext if the probe must go on.
// The whole bucket is loaded (most lookups hit); the comparison is straight-line code, so two lookups of one
// thread can be in flight together.
constexpr int kFindMiss = -1, kFindNext = -2;
template <int W>
__device__ __forceinline__ void ct_lds_bucket(unsigned saddr, u64 (&q)[4]) {
    asm volatile("ld.shared.v2.u64 {%0,%1}, [%2];" : "=l"(q[0]), "=l"(q[1]) : "r"(saddr));
    asm volatile("ld.shared.v2.u64 {%0,%1}, [%2+16];" : "=l"(q[2]), "=l"(q[3]) : "r"(saddr));
}
template <int W> __device__ __forceinline__ int ct_find_step(unsigned saddr, typename Slot<W>::value_t key);
template <> __device__ __forceinline__ int ct_find_step<1>(unsigned saddr, u64 key) {
    u64 q[4];
    ct_lds_bucket<1>(saddr, q);
    int res = kFindNext;
#pragma unroll
    for (int i = 3; i >= 0; --i) {              // slots fill in order: a hit can only sit before the first hole
        const bool e = ((u32)q[i] & 7u) == 0u;
        const bool m = (((q[i] ^ key) << kIdxBits) >> (kIdxBits + 6)) == 0ull;
        res = e ? kFindMiss : (m ? (int)(q[i] >> (64 - kIdxBits)) - 1 : res);
    }
    return res;
}
template <> __device__ __forceinline__ int ct_find_step<2>(unsigned saddr, u128 key) {
    u64 q[4];
    ct_lds_bucket<2>(saddr, q);
    int res = kFindNext;
#pragma unroll
    for (int i = 1; i >= 0; --i) {
        const bool e = ((u32)q[2 * i] & 7u) == 0u;
        const bool m = (((q[2 * i + 1] ^ key.hi) << kIdxBits) | ((q[2 * i] ^ key.lo) >> 6)) == 0ull;
        res = e ? kFindMiss : (m ? (int)(q[2 * i + 1] >> (64 - kIdxBits)) - 1 : res);
    }
    return res;
}

template <int W>
__global__ void __launch_bounds__(kCtBuildThreads, KH_CT_MINBLOCKS)
ct_build_kernel(const typename Slot<W>::value_t* __restrict__ fine, const u32* __restrict__ chunk_cursor,
                const u32* __restrict__ chunk_base, const u32* __restrict__ pool_off,
                typename Slot<W>::value_t* __restrict__ table, u32* __restrict__ seg_base,
                u64* __restrict__ link, u64* __restrict__ meta, typename Slot<W>::value_t* __restrict__ ext_key,
                unsigned char* __restrict__ pool, const CtGeom g, const CtCaps caps, Counters* ctr) {
    typedef Slot<W> S;
    typedef CtSlot<W> CS;
    typedef typename S::value_t V;
    typedef CtBuild<W> B;
    extern __shared__ __align__(128) unsigned char s_bld[];
    unsigned char* const s_raw = s_bld;
    V* s_tab = reinterpret_cast<V*>(s_raw);
    unsigned short* s_succ = reinterpret_cast<unsigned short*>(s_raw + B::kOffSucc);
    unsigned char* s_pool = s_raw + B::kOffSucc;                 // the characters take over s_succ's memory once the links are out
    u32* s_pd = reinterpret_cast<u32*>(s_raw + B::kOffPd);       // (ancestor node << 16) | distance to it; a segment head: (itself << 16) | its segment index
    unsigned short* s_off = reinterpret_cast<unsigned short*>(s_raw + B::kOffOff);
    unsigned char* s_code = s_raw + B::kOffCode;
    __shared__ u32 s_inserted, s_dups, s_nheads, s_seg0, s_chars, s_err;
    const u32 c = blockIdx.x;
    const u32 b0 = chunk_base[c], nb = chunk_base[c + 1] - b0;
    const u32 cnt = min(chunk_cursor[c], B::kMaxSlots);
    if (nb == 0) {                                   // nothing hashed here
        if (threadIdx.x == 0) seg_base[c] = 0;
        return;
    }
    const unsigned s_base = (unsigned)__cvta_generic_to_shared(s_tab);
    const int k = g.k;
    constexpr int kBatch = 4;
    V v[kBatch];
#pragma unroll
    for (int r = 0; r < kBatch; ++r) {
        const u32 i = threadIdx.x + r * kCtBuildThreads;
        v[r] = i < cnt ? fine[ct_fine_index<W>(c, i, g.chunks_per_rank)] : S::zero();
    }
    if (threadIdx.x == 0) { s_inserted = 0; s_dups = 0; s_nheads = 0; s_chars = 0; s_err = 0; }
    {
        uint4* s4 = reinterpret_cast<uint4*>(s_raw);
        for (u32 i = threadIdx.x; i < nb * 2u; i += kCtBuildThreads) s4[i] = make_uint4(0, 0, 0, 0);
        for (u32 i = threadIdx.x; i < cnt; i += kCtBuildThreads) s_pd[i] = (kPredNone << 16) | 1u;
    }
    __syncthreads();
    // ---- 1. insert (hash_map.hpp:33-35): s_succ[node] = the slot the record went to, for phase 2 ----
    u32 inserted = 0, dups = 0, err = 0;
    for (u32 base = 0; base < cnt; base += kCtBuildThreads * kBatch) {
        V nxt[kBatch];
#pragma unroll
        for (int r = 0; r < kBatch; ++r) {
            const u32 i = base + kCtBuildThreads * kBatch + threadIdx.x + r * kCtBuildThreads;
            nxt[r] = i < cnt ? fine[ct_fine_index<W>(c, i, g.chunks_per_rank)] : S::zero();
        }
#pragma unroll
        for (int r = 0; r < kBatch; ++r) {
            const u32 node = base + threadIdx.x + r * kCtBuildThreads;
            if (node >= cnt) continue;
            const int slot = ct_smem_insert<W>(s_tab, s_base, nb, CS::with_idx(v[r], node + 1u));
            inserted += (slot >= 0);
            dups += (slot == -1);
            if (slot == -2) err |= kErrTableFull;
            s_succ[node] = (unsigned short)(slot >= 0 ? (u32)slot : kSuccDead);
        }
#pragma unroll
        for (int r = 0; r < kBatch; ++r) v[r] = nxt[r];
    }
    inserted = __reduce_add_sync(kFullMask, inserted);
    dups = __reduce_add_sync(kFullMask, dups);
    err = __reduce_or_sync(kFullMask, err);
    if (lane_id() == 0) {
        if (inserted) atomicAdd(&s_inserted, inserted);
        if (dups) atomicAdd(&s_dups, dups);
        if (err) atomicOr(&s_err, err);
    }
    __syncthreads();
    // ---- 2. successor of every k-mer, if it lives in this chunk (kmer_hash.cpp:44-51 as an LDS probe) ----
    // Two k-mers per thread and iteration: both first probes are issued before either is looked at.
#pragma unroll 1
    for (u32 base = threadIdx.x; base < cnt; base += 2 * kCtBuildThreads) {
        u32 slot[2], b[2], code[2];
        V key[2];
        int res[2];
#pragma unroll
        for (int q = 0; q < 2; ++q) {
            const u32 node = base + q * kCtBuildThreads;
            slot[q] = node < cnt ? (u32)s_succ[node] : kSuccDead;
        }
#pragma unroll
        for (int q = 0; q < 2; ++q) {
            const V cur = slot[q] != kSuccDead ? s_tab[slot[q]] : S::zero();
            const u32 f = slot[q] != kSuccDead ? S::fwd(cur) : kExtF;       // a duplicate is not in the table and on no chain
            code[q] = f | ((slot[q] != kSuccDead && S::back(cur) == kExtF) ? kCodeBackF : 0u);
            key[q] = S::next_key(CS::strip(cur), k);
            b[q] = ct_bucket_in_chunk(CS::hash32(key[q]), nb);
        }
#pragma unroll
        for (int q = 0; q < 2; ++q) res[q] = (code[q] & 7u) != kExtF ? ct_find_step<W>(s_base + b[q] * 32u, key[q]) : kFindMiss;
#pragma unroll
        for (int q = 0; q < 2; ++q) {
            for (u32 tries = 1; res[q] == kFindNext && tries < nb; ++tries) {      // the home bucket was full of other keys: go on
                b[q] = (b[q] + 1 == nb) ? 0u : b[q] + 1;
                res[q] = ct_find_step<W>(s_base + b[q] * 32u, key[q]);
            }
        }
#pragma unroll
        for (int q = 0; q < 2; ++q) {
            const u32 node = base + q * kCtBuildThreads;
            if (node >= cnt) continue;
            s_code[node] = (unsigned char)code[q];
            u32 sc = slot[q] == kSuccDead ? kSuccDead : kSuccTail;
            if ((code[q] & 7u) != kExtF) {
                if (res[q] < 0) {
                    sc = kSuccExt | slot[q];
                } else {
                    sc = (u32)res[q];
                    s_pd[res[q]] = (node << 16) | 1u;       // plain store: with two predecessors one of them wins, phase 3 notices
                }
            }
            s_succ[node] = (unsigned short)sc;
        }
    }
    __syncthreads();
    // ---- 3. heads: k-mers no chain of this chunk runs into (or that two run into, or with backward ext 'F') ----
#pragma unroll 1
    for (u32 node = threadIdx.x; node < cnt; node += kCtBuildThreads) {
        const u32 s = s_succ[node];
        if (s < kSuccExt && (s_pd[s] >> 16) != node) s_code[s] |= (unsigned char)kCodeMulti;      // rare; every writer stores the same bit
    }
    __syncthreads();
    for (u32 base = 0; base < cnt; base += kCtBuildThreads) {
        const u32 node = base + threadIdx.x;
        bool head = false, dead = true;
        if (node < cnt) {
            dead = s_succ[node] == kSuccDead;
            head = !dead && ((s_pd[node] >> 16) == kPredNone || (s_code[node] & (kCodeBackF | kCodeMulti)));
        }
        const u32 bal = __ballot_sync(kFullMask, head);
        u32 first = 0;
        if (lane_id() == 0 && bal) first = atomicAdd(&s_nheads, (u32)__popc(bal));
        first = __shfl_sync(kFullMask, first, 0);
        if (head) s_pd[node] = (node << 16) | (first + __popc(bal & ((1u << lane_id()) - 1u)));      // a root: (itself, segment index)
        else if (dead && node < cnt) s_pd[node] = node << 16;                                          // never looked at again
    }
    __syncthreads();
    const u32 nheads = s_nheads;
    if (threadIdx.x == 0) {
        u32 seg0 = nheads ? atomicAdd(&ctr->next_seg, nheads) : 0u;
        if (seg0 + nheads > caps.seg_cap) { ct_internal(ctr, kSiteSegCap); seg0 = caps.seg_cap; }
        s_seg0 = seg0;
        seg_base[c] = seg0;
    }
    // ---- 4. pointer jumping in shared memory: every k-mer learns its segment head and its distance from it ----
    // In place: a stale read is still a valid (ancestor, distance) pair.  A root's low half is its segment index, which a
    // child never adds (it stops as soon as its ancestor is a root).  KH_CT_JUMPS passes run between two barriers; a
    // pass may read other threads' pairs as they stood at the last barrier, so a round is only sure to multiply a
    // node's reach by KH_CT_JUMPS + 1.  B::kJumpRounds rounds therefore settle a chain through every record of a full
    // chunk (a repeat can put thousands of k-mers in one chain; random sequence gives <= ~40).  The loop leaves at the
    // first barrier where nothing is unsettled, so only a cycle without a head (no chain enters it: kmer_hash.cpp never
    // visits it) runs all the rounds; it never settles and phases 5 and 6 skip it.
    // A thread keeps a bit per node of its own that has not settled yet: later rounds only touch those.
    u32 active = 0;
#pragma unroll 1
    for (u32 i = 0, node = threadIdx.x; node < cnt; ++i, node += kCtBuildThreads) {
        const u32 pd = s_pd[node];
        active |= ((pd >> 16) != node) ? (1u << i) : 0u;            // heads and dead nodes are roots already
    }
    for (int round = 0; round < B::kJumpRounds; ++round) {
#pragma unroll 1
        for (int rep = 0; rep < KH_CT_JUMPS; ++rep) {
#pragma unroll 1
            for (u32 m = active; m; m &= m - 1u) {
                const u32 i = (u32)__ffs((int)m) - 1u, node = threadIdx.x + i * kCtBuildThreads;
                const u32 pd = s_pd[node], a = pd >> 16;
                const u32 pa = s_pd[a], a2 = pa >> 16;
                if (a2 == a) { active &= ~(1u << i); continue; }        // the ancestor is a root: this node is done
                s_pd[node] = (a2 << 16) | ((pd + pa) & 0xFFFFu);
            }
        }
        if (!__syncthreads_or(active != 0u)) break;
    }
    __syncthreads();
    const u32 seg0 = s_seg0;
    const u32 my_bits = (u32)g.rank << kRankShift;
    const u64 pool0 = pool_off[c];
    // ---- 5. the last k-mer of every segment writes the segment: link, meta, pending key; reserves its characters ----
    if (seg0 < caps.seg_cap) {
    #pragma unroll 1
    for (u32 node = threadIdx.x; node < cnt; node += kCtBuildThreads) {
            const u32 s = s_succ[node];
            if (s == kSuccDead) continue;
            const u32 pd = s_pd[node], a = pd >> 16;
            const bool root = a == node;
            const u32 pa = root ? pd : s_pd[a];
            if ((pa >> 16) != a) continue;                                   // on a headless cycle
            const u32 f = s_code[node] & 7u;
            bool last = f == kExtF || s >= kSuccExt;
            u32 next_hi = f == kExtF ? kLinkTail : kLinkPending;
            if (!last) {
                const u32 ps = s_pd[s];
                if ((ps >> 16) == s) { last = true; next_hi = my_bits | (seg0 + (ps & 0xFFFFu)); }      // the successor starts its own segment
            }
            if (!last) continue;
            const u32 n = (root ? 0u : (pd & 0xFFFFu)) + (f != kExtF ? 1u : 0u);      // extract_contig (read_kmers.hpp:86-90): no character for 'F'
            const u32 off = atomicAdd(&s_chars, n);
            s_off[a] = (unsigned short)off;
            const u32 gseg = seg0 + (pa & 0xFFFFu);
            link[gseg] = ((u64)next_hi << 32) | (next_hi == kLinkTail ? 0u : n);
            meta[gseg] = ((pool0 + off) << 24) | n;
            if (next_hi == kLinkPending) ext_key[gseg] = S::next_key(CS::strip(s_tab[s & 0x7FFFu]), k);
        }
    }
    __syncthreads();
    // ---- 6. every k-mer drops its forward extension at (segment's characters + distance from the head) ----
#pragma unroll 1
    for (u32 node = threadIdx.x; node < cnt; node += kCtBuildThreads) {
        const u32 code = s_code[node];
        if ((code & 7u) == kExtF) continue;                                  // also the dead ones
        const u32 pd = s_pd[node], a = pd >> 16;
        const bool root = a == node;
        if (!root && (s_pd[a] >> 16) != a) continue;
        s_pool[(u32)s_off[a] + (root ? 0u : (pd & 0xFFFFu))] = ext_char(code & 7u);
    }
    // ---- 7. index bits: node id -> 1 + segment index for the k-mers that start a segment, 0 for the others ----
    {
        const u32 nslots = nb * S::kPerBucket;
        for (u32 i = threadIdx.x; i < nslots; i += kCtBuildThreads) {
            const V cur = s_tab[i];
            if (S::empty(cur)) continue;
            const u32 node = CS::idx(cur) - 1u, pd = s_pd[node];
            s_tab[i] = CS::with_idx(cur, (pd >> 16) == node ? (pd & 0xFFFFu) + 1u : 0u);
        }
    }
    // ---- 8. characters and the finished chunk go to HBM: bulk copies shared -> global (TMA engine), 8 KB pieces ----
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    __syncthreads();
    {
        const u32 tab_bytes = nb * 32u, pool_bytes = (s_chars + 15u) & ~15u;
        constexpr u32 kPiece = 8192u;
        const u32 tab_pieces = (tab_bytes + kPiece - 1u) / kPiece, pool_pieces = (pool_bytes + kPiece - 1u) / kPiece;
        if (lane_id() == 0) {
            unsigned char* g_tab = reinterpret_cast<unsigned char*>(table + (u64)b0 * S::kPerBucket);
            bool any = false;
            for (u32 pc = threadIdx.x >> 5; pc < tab_pieces + pool_pieces; pc += kCtBuildThreads / 32) {
                const bool is_tab = pc < tab_pieces;
                const u32 o = (is_tab ? pc : pc - tab_pieces) * kPiece;
                const u32 bytes = min(kPiece, (is_tab ? tab_bytes : pool_bytes) - o);
                const unsigned src = (unsigned)__cvta_generic_to_shared(is_tab ? s_raw + o : s_pool + o);
                unsigned char* dst = is_tab ? g_tab + o : pool + pool0 + o;
                asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst), "r"(src), "r"(bytes) : "memory");
                any = true;
            }
            if (any) {
                asm volatile("cp.async.bulk.commit_group;" ::: "memory");
                asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
            }
        }
    }
    if (threadIdx.x == 0) {
        if (s_inserted) atomicAdd(&ctr->n_inserted, (u64)s_inserted);
        if (s_dups) atomicAdd(&ctr->n_duplicates, (u64)s_dups);
        if (s_err) { atomicOr(&ctr->errors, s_err); atomicOr(&ctr->err_where, kSiteChunkFull); }      // the only build error: the chunk is full
    }
}

// ---- lookups in the sealed table (HBM) -------------------------------------------------------------------------
// key: ext and index bits 0.  Returns the stored slot value (with its index bits) or false.
template <int W>
__device__ __forceinline__ bool ct_lookup_chunk(const typename Slot<W>::value_t* __restrict__ table, const u32* __restrict__ chunk_base,
                                                u32 chunk, typename Slot<W>::value_t key, typename Slot<W>::value_t& found) {
    typedef Slot<W> S;
    typedef typename S::value_t V;
    const u32 b0 = chunk_base[chunk], nb = chunk_base[chunk + 1] - b0;
    if (nb == 0) return false;
    u32 b = ct_bucket_in_chunk(CtSlot<W>::hash32(key), nb);
    for (u32 tries = 0; tries < nb; ++tries) {
        u64 q[4];
        load256_nc(table + (u64)(b0 + b) * S::kPerBucket, q);
        bool hole = false, hit = false;
#pragma unroll
        for (int i = 0; i < S::kPerBucket; ++i) {                 // branch-free inside the bucket: every lane leaves together
            const V cur = S::from_bucket(q, i);
            const bool e = S::empty(cur);
            if (!hole && !hit && !e && CtSlot<W>::same_key(cur, key)) { found = cur; hit = true; }
            hole = hole || e;
        }
        if (hit) return true;
        if (hole) return false;
        b = (b + 1 == nb) ? 0u : b + 1;
    }
    return false;
}

// batch find (hash_map.hpp:83-92) on a sealed single-GPU chunk table
template <int W>
__global__ void __launch_bounds__(256)
ct_find_kernel(const typename Slot<W>::value_t* __restrict__ table, const u32* __restrict__ chunk_base, const CtGeom g,
               const unsigned char* __restrict__ pkmers, u64 n, unsigned char* __restrict__ pairs_out,
               unsigned char* __restrict__ found_out) {
    typedef Slot<W> S;
    const u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int k = g.k, pl = (k + 3) >> 2, pb = pl + 2;
    unsigned char key[16];
    for (int j = 0; j < pl; ++j) key[j] = pkmers[i * pl + j];
    const typename S::value_t kb = S::from_packed(key, k, pl);
    u32 owner, chunk;
    ct_place(ct_min_hash<W>(kb, g.m, g.win), g, owner, chunk);
    typename S::value_t hit;
    const bool ok = ct_lookup_chunk<W>(table, chunk_base, chunk, kb, hit);
    unsigned char rec[18];
    for (int j = 0; j < pb; ++j) rec[j] = 0;
    if (ok) S::to_record(CtSlot<W>::strip(hit), k, pl, rec);
    for (int j = 0; j < pb; ++j) pairs_out[i * pb + j] = rec[j];
    found_out[i] = ok ? 1 : 0;
}

// ---- contig head stubs: one zero-length segment per start node parsed by this rank ----------------------------
template <int W>
__global__ void __launch_bounds__(256)
ct_stub_kernel(const typename Slot<W>::value_t* __restrict__ starts, const Counters* __restrict__ ctr, u32 hcap,
               u64* __restrict__ link, u64* __restrict__ meta, typename Slot<W>::value_t* __restrict__ ext_key) {
    typedef Slot<W> S;
    const u32 n_starts = (u32)min(ctr->n_starts_dev, (u64)hcap);
    for (u32 c = blockIdx.x * blockDim.x + threadIdx.x; c < hcap; c += gridDim.x * blockDim.x) {
        if (c < n_starts) {
            link[c] = (u64)kLinkPending << 32;
            meta[c] = 0;
            ext_key[c] = S::key_only(starts[c]);
        } else {
            link[c] = (u64)kLinkUnused << 32;
        }
    }
}

// resolve one pending link against THIS rank's table: the segment that starts with `key`
template <int W>
__device__ __forceinline__ u32 ct_resolve_one(const typename Slot<W>::value_t* __restrict__ table, const u32* __restrict__ chunk_base,
                                              const u32* __restrict__ seg_base, u32 chunk, typename Slot<W>::value_t key, u32 my_bits) {
    typename Slot<W>::value_t hit;
    if (!ct_lookup_chunk<W>(table, chunk_base, chunk, key, hit)) return kLinkMissing;      // kmer_hash.cpp:47-49, raised later if start-rooted
    const u32 idx = CtSlot<W>::idx(hit);
    if (idx == 0) return kLinkConverge;                // inside another segment: this k-mer has a second predecessor
    return my_bits | (seg_base[chunk] + idx - 1u);
}

// ---- chain the segments: ONE table lookup per segment -------------------------------------------------------------
// Pending links whose successor lives in this rank's chunks are resolved on the spot; the others are grouped by
// owner (tile-wise, so the peer stores are runs) straight into the owner's inbox.
constexpr int kResPerThread = 4;
constexpr int kResTile = 256 * kResPerThread;
template <int W>
__global__ void __launch_bounds__(256)
ct_resolve_kernel(const typename Slot<W>::value_t* __restrict__ table, const u32* __restrict__ chunk_base,
                  const u32* __restrict__ seg_base, u64* __restrict__ link, const typename Slot<W>::value_t* __restrict__ ext_key,
                  const CtGeom g, const CtPeers pe, const CtCaps caps, u32* __restrict__ out_cursor, u32* __restrict__ req_seg, Counters* ctr) {
    typedef Slot<W> S;
    typedef typename S::value_t V;
    __shared__ u32 s_cnt[kMaxRanks], s_base[kMaxRanks];
    const u32 nseg = min(ctr->next_seg, caps.seg_cap);
    const u32 my_bits = (u32)g.rank << kRankShift;
    const u32 ntiles = (nseg + kResTile - 1) / kResTile;
    for (u32 tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        if (threadIdx.x < kMaxRanks) s_cnt[threadIdx.x] = 0;
        __syncthreads();
        CtReq<W> e[kResPerThread];
        u32 dest[kResPerThread], rk[kResPerThread];
#pragma unroll
        for (int r = 0; r < kResPerThread; ++r) {
            const u32 s = tile * kResTile + r * 256 + threadIdx.x;
            u32 d = 0xFFFFFFFFu;
            if (s < nseg && (u32)(link[s] >> 32) == kLinkPending) {
                const V key = ext_key[s];
                u32 owner, chunk;
                ct_place(ct_min_hash<W>(key, g.m, g.win), g, owner, chunk);
                if (owner == (u32)g.rank) {
                    reinterpret_cast<u32*>(link + s)[1] = ct_resolve_one<W>(table, chunk_base, seg_base, chunk, key, my_bits);
                } else {
                    d = owner;
                    e[r].key = key; e[r].src = my_bits | s; e[r].chunk = chunk;
                }
            }
            dest[r] = d;
            const unsigned same = __match_any_sync(kFullMask, d);
            const int leader = __ffs(same) - 1;
            u32 first = 0;
            if ((int)lane_id() == leader && d != 0xFFFFFFFFu) first = atomicAdd(&s_cnt[d], (u32)__popc(same));
            rk[r] = __shfl_sync(kFullMask, first, leader) + (u32)__popc(same & ((1u << lane_id()) - 1u));
        }
        __syncthreads();
        if (threadIdx.x < kMaxRanks) s_base[threadIdx.x] = s_cnt[threadIdx.x] ? atomicAdd(&out_cursor[threadIdx.x], s_cnt[threadIdx.x]) : 0u;
        __syncthreads();
#pragma unroll
        for (int r = 0; r < kResPerThread; ++r) {
            if (dest[r] == 0xFFFFFFFFu) continue;
            const u32 at = s_base[dest[r]] + rk[r];
            if (at < caps.inbox_cap) {
                static_cast<CtReq<W>*>(pe.inbox[dest[r]])[(u64)g.rank * caps.inbox_cap + at] = e[r];
                req_seg[(u64)dest[r] * caps.inbox_cap + at] = e[r].src & kLocalMask;
            } else {
                ct_internal(ctr, kSiteInbox);
            }
        }
        __syncthreads();
    }
}

__global__ void ct_publish_inbox_kernel(const CtPeers pe, const CtCaps caps, const u32* __restrict__ out_cursor) {
    const int d = (int)threadIdx.x;
    if (d < pe.world) pe.inbox_cnt[d][pe.rank] = min(out_cursor[d], caps.inbox_cap);
}

// the owner answers: local lookup, then the answer goes into the requester's answer array at the request's index --
// consecutive threads, consecutive addresses: NVLink sees long runs instead of one 4-byte store per link
template <int W>
__global__ void __launch_bounds__(256)
ct_answer_kernel(const typename Slot<W>::value_t* __restrict__ table, const u32* __restrict__ chunk_base,
                 const u32* __restrict__ seg_base, const CtReq<W>* __restrict__ inbox, const u32* __restrict__ inbox_cnt,
                 const CtGeom g, const CtPeers pe, const CtCaps caps) {
    const u32 my_bits = (u32)g.rank << kRankShift;
    for (int src = 0; src < g.world; ++src) {
        if (src == g.rank) continue;
        const u32 n = min(inbox_cnt[src], caps.inbox_cap);
        const CtReq<W>* __restrict__ box = inbox + (u64)src * caps.inbox_cap;
        for (u32 i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
            const CtReq<W> e = box[i];
            pe.answers[src][(u64)g.rank * caps.inbox_cap + i] = ct_resolve_one<W>(table, chunk_base, seg_base, e.chunk, e.key, my_bits);
        }
    }
}

// the requester files the answers: link[segment of request i to owner o].high = answers[o][i]
__global__ void __launch_bounds__(256)
ct_apply_kernel(u64* __restrict__ link, const u32* __restrict__ answers, const u32* __restrict__ req_seg, const u32* __restrict__ out_cursor,
                const CtCaps caps, int world, int rank) {
    for (int o = 0; o < world; ++o) {
        if (o == rank) continue;
        const u32 n = min(out_cursor[o], caps.inbox_cap);
        const u64 base = (u64)o * caps.inbox_cap;
        for (u32 i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
            reinterpret_cast<u32*>(link + req_seg[base + i])[1] = answers[base + i];
    }
}

// ---- gather: every rank sends its segment links, meta words and characters to every other rank -----------------------
// After this the contig walk reads local memory only.  What crosses NVLink is one long coalesced stream per peer
// (16 bytes per segment + one byte per k-mer); fine-grained peer reads and writes ran at a few G/s.
__global__ void __launch_bounds__(256)
ct_gather_kernel(const CtPeers pe, const CtCaps caps, const u64* __restrict__ link, const u64* __restrict__ meta,
                 const unsigned char* __restrict__ pool, const u32* __restrict__ pool_off, u32 nchunks, const Counters* __restrict__ ctr,
                 int what) {           // 0: meta words + characters (final once the chunks are built), 1: links (final once they are resolved)
    const u32 nseg = min(ctr->next_seg, caps.seg_cap);
    const u32 first = caps.hcap;                                   // head stubs are only ever read by their own rank
    const u32 cnt = nseg > first ? nseg - first : 0u;
    const u64 pool_vecs = ((u64)pool_off[nchunks] + 15u) >> 4;
    const u64 tid = (u64)blockIdx.x * blockDim.x + threadIdx.x, stride = (u64)gridDim.x * blockDim.x;
    for (int d = 1; d < pe.world; ++d) {
        const int p = (pe.rank + d) % pe.world;                    // every rank starts with a different peer
        u64* gl = pe.g_link[p] + (u64)pe.rank * caps.g_seg_stride;
        u64* gm = pe.g_meta[p] + (u64)pe.rank * caps.g_seg_stride;
        uint4* gp = reinterpret_cast<uint4*>(pe.g_pool[p] + (u64)pe.rank * caps.g_pool_stride);
        if (what == 1) {
            for (u64 i = tid; i < cnt; i += stride) gl[first + i] = link[first + i];
        } else {
            for (u64 i = tid; i < cnt; i += stride) gm[first + i] = meta[first + i];
            const uint4* sp = reinterpret_cast<const uint4*>(pool);
            for (u64 i = tid; i < pool_vecs; i += stride) gp[i] = sp[i];
            if (tid == 0) { pe.g_hdr[p][2 * pe.rank] = nseg; pe.g_hdr[p][2 * pe.rank + 1] = (u32)pool_vecs; }
        }
    }
}

// ---- ranking by walking: one lane per contig follows its segments (kmer_hash.cpp:38-55, a segment per step) ----------
// Contigs are short (~100 k-mers = 4..30 segments), there are hundreds of thousands of them, and every array the walk
// reads is local (own arrays + gathered copies), so a lane per contig keeps the memory system busy with ONE read per
// segment.  A lane counts the links it follows from the contig's first chunk segment, so a contig of more than
// max_steps + 1 chunk segments (its head stub not counted) sets need_jump: the whole step then falls back to pointer jumping.
// max_steps is kCtWalkMaxSteps unless KH_DEBUG_WALK_STEPS lowers it (tests send ordinary inputs down the fallback).
constexpr u32 kCtWalkMaxSteps = 512;
struct CtGathered {
    const u64* link[kMaxRanks];
    const u64* meta[kMaxRanks];
    const unsigned char* pool[kMaxRanks];
};

__global__ void __launch_bounds__(256)
ct_walk_len_kernel(const CtGathered gt, const u64* __restrict__ link, const CtCaps caps, int k, u32 max_steps,
                   u32* __restrict__ contig_len, Counters* ctr) {
    const u32 n_starts = (u32)min(ctr->n_starts_dev, (u64)caps.hcap);
    u64 nodes = 0;
    u32 err = 0, too_long = 0;
    for (u64 c = (u64)blockIdx.x * blockDim.x + threadIdx.x; c <= caps.hcap; c += (u64)gridDim.x * blockDim.x) {
        if (c >= n_starts) { contig_len[c] = 0; continue; }           // the offsets scan runs over hcap + 1 entries
        u32 gid = (u32)(__ldg(link + c) >> 32), chars = 0, e = 0, steps = 0;
        if (gid == kLinkMissing) e = kErrNotFound;                     // the start k-mer itself is not in the table
        else if (gid == kLinkConverge) e = kErrConverge;
        else if (gid >= kLinkCtFirstMarker) e = kErrInternal;
        while (!e) {
            const u64 l = __ldg(gt.link[gid >> kRankShift] + (gid & kLocalMask));
            const u32 hi = (u32)(l >> 32);
            if (hi == kLinkTail) { chars += (u32)(__ldg(gt.meta[gid >> kRankShift] + (gid & kLocalMask)) & 0xFFFFFFu); break; }
            if (hi == kLinkMissing) { e = kErrNotFound; break; }       // kmer_hash.cpp:47-49
            if (hi == kLinkConverge) { e = kErrConverge; break; }
            if (hi >= kLinkCtFirstMarker) { e = kErrInternal; break; }
            chars += (u32)l;
            gid = hi;
            if (++steps > max_steps) { too_long = 1; break; }
        }
        if (e || too_long) { err |= e; contig_len[c] = 0; continue; }
        contig_len[c] = (u32)k + chars + 1u;
        nodes += (u64)chars + 1u;
    }
    nodes = warp_sum_u64(nodes);
    err = __reduce_or_sync(kFullMask, err);
    too_long = __reduce_or_sync(kFullMask, too_long);
    if (lane_id() == 0) {
        if (nodes) atomicAdd(&ctr->n_nodes, nodes);
        if (err) atomicOr(&ctr->errors, err);
        if (err & kErrInternal) atomicOr(&ctr->err_where, kSiteStubOpen);
        if (too_long) atomicOr(&ctr->need_jump, 1u);
    }
}

// copy n bytes (source and destination arbitrarily aligned): destination-aligned 32-bit words built with funnel shifts
__device__ __forceinline__ void ct_copy_chars(char* dst, const unsigned char* src, u32 n) {
    while (n && (reinterpret_cast<uintptr_t>(dst) & 3u)) { *dst++ = (char)*src++; --n; }
    if (n >= 4) {
        const u32 sh = ((u32)reinterpret_cast<uintptr_t>(src) & 3u) * 8u;
        const u32* sw = reinterpret_cast<const u32*>(reinterpret_cast<uintptr_t>(src) & ~(uintptr_t)3);
        u32 w0 = __ldg(sw);
        u32* dw = reinterpret_cast<u32*>(dst);
        const u32 nw = n >> 2;
        for (u32 i = 0; i < nw; ++i) {
            const u32 w1 = __ldg(sw + i + 1);                      // the pools have 64 bytes of slack behind them
            dw[i] = __funnelshift_r(w0, w1, sh);
            w0 = w1;
        }
        dst += 4 * nw; src += 4 * nw; n &= 3u;
    }
    while (n) { *dst++ = (char)*src++; --n; }
}

// second walk: the first k-mer's K characters, then the characters of every segment, then the newline
// (extract_contig, read_kmers.hpp:81-92; kmer_hash.cpp:66)
template <int W>
__global__ void __launch_bounds__(256)
ct_walk_emit_kernel(const CtGathered gt, const u64* __restrict__ link, const typename Slot<W>::value_t* __restrict__ starts,
                    const CtCaps caps, int k, const u32* __restrict__ contig_len, const u64* __restrict__ contig_off, u64 out_cap,
                    char* __restrict__ out, const Counters* __restrict__ ctr) {
    typedef Slot<W> S;
    if (ctr->use_jump || ctr->need_jump || (ctr->errors & (kErrConverge | kErrCycle | kErrInternal | kErrNotFound)) || ctr->contig_bytes > out_cap) return;
    const u32 n_starts = (u32)min(ctr->n_starts_dev, (u64)caps.hcap);
    for (u64 c = (u64)blockIdx.x * blockDim.x + threadIdx.x; c < n_starts; c += (u64)gridDim.x * blockDim.x) {
        const u32 len = contig_len[c];
        if (len == 0) continue;
        char* dst = out + contig_off[c];
        char* const end = dst + len - 1u;
        *end = '\n';
        {                                                              // the start k-mer, four bases per aligned 32-bit store
            const typename S::value_t v0 = starts[c];
            int j = 0;
            while (j < k && (reinterpret_cast<uintptr_t>(dst) & 3u)) { *dst++ = (char)ext_char(S::base_at(v0, k, j)); ++j; }
            for (; j + 4 <= k; j += 4, dst += 4) {
                const u32 w = (u32)ext_char(S::base_at(v0, k, j)) | ((u32)ext_char(S::base_at(v0, k, j + 1)) << 8) |
                              ((u32)ext_char(S::base_at(v0, k, j + 2)) << 16) | ((u32)ext_char(S::base_at(v0, k, j + 3)) << 24);
                *reinterpret_cast<u32*>(dst) = w;
            }
            for (; j < k; ++j) *dst++ = (char)ext_char(S::base_at(v0, k, j));
        }
        u32 gid = (u32)(__ldg(link + c) >> 32);
        for (;;) {
            const u32 r = gid >> kRankShift, i = gid & kLocalMask;
            const u64 l = __ldg(gt.link[r] + i), mt = __ldg(gt.meta[r] + i);
            const u32 n = (u32)(mt & 0xFFFFFFu);
            if (dst + n > end) break;                                  // cannot happen after the length walk; never write outside the contig
            ct_copy_chars(dst, gt.pool[r] + (mt >> 24), n);
            dst += n;
            const u32 hi = (u32)(l >> 32);
            if (hi >= kLinkCtFirstMarker) break;
            gid = hi;
        }
    }
}

// ---- pointer jumping over segment lists that span GPUs --------------------------------------------------------------
// A link is FINAL (top bit of the distance word) once its pointer is the chain's last segment (high word a marker);
// a link that is not final moves when it is visited unless it is already saturated on a self-looping cycle segment,
// so "nothing moved here" means this rank's links will never change again and it only keeps the others company at
// the barriers.  The rounds of all ranks run in lockstep (a barrier
// after each, ct_barrier_kernel): jumping over a peer's link doubles the distance only if the peer jumps too --
// ranks that ran their rounds on their own would walk a chain one remote segment per round.
constexpr int kCtMaxRounds = 24;            // pointer-jumping rounds of a traverse: chains of up to 2^24 segments
__device__ __forceinline__ u64* ct_peer_link(const CtPeers& pe, u32 gid) { return pe.link[gid >> kRankShift] + (gid & kLocalMask); }
__host__ __device__ __forceinline__ bool ct_is_end_marker(u32 hi) { return hi == kLinkTail || hi == kLinkClaimed || hi == kLinkMissing || hi == kLinkConverge; }

// One jump of an open link li (pointer not a marker, not final) over the link lp of the segment it points at.
// The distance saturates at kLinkDistMask: on a cycle it roughly doubles every round, and a sum that carried into the
// final bit would make a cycle's link "final" with a meaningless distance (a start-rooted cycle was then refused as
// KH_ERR_CONVERGE by the claim instead of KH_ERR_CYCLE).  A saturated link is never final, so ct_lengths_kernel
// reports the cycle.  A chain that ends is exact as long as it has fewer than kLinkDistMask characters (contig
// lengths are 32-bit anyway).  Returns li itself when the target is pending or unused: left open, ct_lengths reports it.
__host__ __device__ __forceinline__ u64 ct_jump_link(u64 li, u64 lp) {
    const u32 pp = (u32)(lp >> 32), sp = (u32)lp;
    if (ct_is_end_marker(pp)) return li | kLinkFinalBit;
    if (pp >= kLinkCtFirstMarker) return li;
    const u32 d = ((u32)li & kLinkDistMask) + (sp & kLinkDistMask);      // < 2^32: no wrap
    if (d >= kLinkDistMask) return ((u64)pp << 32) | kLinkDistMask;
    return ((u64)pp << 32) | (d | (sp & kLinkFinalBit));
}

__global__ void __launch_bounds__(256)
ct_rank_round_kernel(const CtPeers pe, u64* __restrict__ link, const CtCaps caps, Counters* ctr, u32* __restrict__ moved, int round) {
    if (ctr->rank_done || (round > 0 && moved[round - 1] == 0)) return;     // everybody / this rank has only final links
    const u32 nseg = min(ctr->next_seg, caps.seg_cap);
    bool any = false;
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < nseg; i += (u64)gridDim.x * blockDim.x) {
        const u64 li = __ldcg(link + i);
        const u32 pi = (u32)(li >> 32), si = (u32)li;
        if (pi >= kLinkCtFirstMarker) continue;               // ends here / unused / still pending (reported by ct_lengths)
        if (si & kLinkFinalBit) continue;
        const u64 lp = __ldcg(ct_peer_link(pe, pi));
        const u64 ln = ct_jump_link(li, lp);
        if (ln == li) continue;
        __stcg(link + i, ln);
        any |= (u32)(lp >> 32) < kLinkCtFirstMarker;          // jumped (a link that only turned final did not move)
    }
    if (__any_sync(kFullMask, any) && lane_id() == 0) moved[round] = 1;
}

// contig lengths for the start nodes of this rank (kmer_hash.cpp:38-55: one contig per start node)
__global__ void __launch_bounds__(256)
ct_lengths_kernel(const CtPeers pe, const u64* __restrict__ link, const CtCaps caps, int k,
                  u32* __restrict__ contig_len, u32* __restrict__ contig_pre, Counters* ctr) {
    const u32 n_starts = (u32)min(ctr->n_starts_dev, (u64)caps.hcap);
    u64 nodes = 0;
    u32 err = 0;
    for (u64 c = (u64)blockIdx.x * blockDim.x + threadIdx.x; c <= caps.hcap; c += (u64)gridDim.x * blockDim.x) {
        if (c >= n_starts) { contig_len[c] = 0; continue; }           // the offsets scan runs over hcap + 1 entries
        const u64 lc = __ldcg(link + c);
        const u32 pc = (u32)(lc >> 32);
        u32 e = 0, tail_hi = 0, chars = 0, pre = 0;
        if (pc == kLinkMissing) e = kErrNotFound;
        else if (pc == kLinkConverge) e = kErrConverge;
        else if (pc >= kLinkCtFirstMarker) { e = kErrInternal; atomicOr(&ctr->err_where, kSiteStubOpen); }                     // a stub is never a tail, and nobody may leave it pending
        else if (!((u32)lc & kLinkFinalBit)) e = kErrCycle;                      // still moving after the last round: kmer_hash.cpp:44 never exits
        else {
            tail_hi = (u32)(__ldcg(ct_peer_link(pe, pc)) >> 32);
            if (tail_hi == kLinkMissing) e = kErrNotFound;                       // kmer_hash.cpp:47-49
            else if (tail_hi == kLinkConverge) e = kErrConverge;
            else {
                pre = (u32)lc & kLinkDistMask;
                chars = pre + (u32)(pe.meta[pc >> kRankShift][pc & kLocalMask] & 0xFFFFFFu);
            }
        }
        if (e) { err |= e; contig_pre[c] = 0; contig_len[c] = 0; continue; }
        contig_pre[c] = pre;
        contig_len[c] = (u32)k + chars + 1u;
        nodes += (u64)chars + 1u;
    }
    nodes = warp_sum_u64(nodes);
    err = __reduce_or_sync(kFullMask, err);
    if (lane_id() == 0) {
        if (nodes) atomicAdd(&ctr->n_nodes, nodes);
        if (err) atomicOr(&ctr->errors, err);
    }
}

// each contig claims its last segment (possibly on another GPU): link[tail] = (CLAIMED, home rank << 28 | contig)
__global__ void __launch_bounds__(256)
ct_claim_kernel(const CtPeers pe, const u64* __restrict__ link, const CtCaps caps, const u32* __restrict__ contig_len, Counters* ctr) {
    const u32 n_starts = (u32)min(ctr->n_starts_dev, (u64)caps.hcap);
    for (u64 c = (u64)blockIdx.x * blockDim.x + threadIdx.x; c < n_starts; c += (u64)gridDim.x * blockDim.x) {
        if (contig_len[c] == 0) continue;
        const u32 tail = (u32)(__ldcg(link + c) >> 32);
        const u64 want = (u64)kLinkTail << 32;
        const u64 old = atomicCAS(ct_peer_link(pe, tail), want, ((u64)kLinkClaimed << 32) | (((u32)pe.rank << kRankShift) | (u32)c));
        if (old != want) atomicOr(&ctr->errors, kErrConverge);       // two start nodes, one end node
    }
}

// ---- emit: every GPU copies the characters of its segments into the output of the contig's home rank ---------------
// One lane resolves a segment's destination (its last segment's claim -> contig -> offset), then the warp copies.
__global__ void __launch_bounds__(256)
ct_emit_kernel(const CtPeers pe, const u64* __restrict__ link, const u64* __restrict__ meta, const unsigned char* __restrict__ pool,
               const CtCaps caps, Counters* ctr, int k) {
    const u32 nseg = min(ctr->next_seg, caps.seg_cap);
    if (ctr->errors & (kErrConverge | kErrCycle | kErrInternal | kErrNotFound)) return;       // the host reports it; write nothing
    const u64 stride = (u64)gridDim.x * blockDim.x;
    for (u64 seg0 = (u64)caps.hcap + (u64)blockIdx.x * blockDim.x + (threadIdx.x & ~31u); seg0 < nseg; seg0 += stride) {   // stubs carry no characters
        const u64 seg = seg0 + lane_id();
        u32 len = 0;
        char* dst = nullptr;
        const unsigned char* src = nullptr;
        if (seg < nseg) {
            const u64 li = link[seg];
            const u32 pi = (u32)(li >> 32);
            const u64 mt = meta[seg];
            u32 cg = 0, dist = 0;
            bool ok = false, is_tail = false;
            if (pi == kLinkClaimed) { cg = (u32)li; ok = true; is_tail = true; }
            else if (pi < kLinkCtFirstMarker && ((u32)li & kLinkFinalBit)) {
                const u64 lt = *ct_peer_link(pe, pi);
                if ((u32)(lt >> 32) == kLinkClaimed) { cg = (u32)lt; dist = (u32)li & kLinkDistMask; ok = true; }
            }
            if (ok) {                                          // otherwise: on no start-rooted chain, ignored like the reference
                const u32 r = cg >> kRankShift, c = cg & kLocalMask;
                const u32 pre = pe.contig_pre[r][c];
                if (!is_tail && dist > pre) { atomicOr(&ctr->errors, kErrConverge); ok = false; }
                if (ok) {
                    const u64 off = pe.contig_off[r][c] + (u64)k + (is_tail ? pre : pre - dist);
                    len = (u32)(mt & 0xFFFFFFu);
                    if (off + len > pe.out_cap[r]) { ct_internal(ctr, kSiteOutCap); len = 0; }
                    dst = pe.out[r] + off;
                    src = pool + (mt >> 24);
                }
            }
        }
        u32 todo = __ballot_sync(kFullMask, len > 0);
        while (todo) {
            const int sl = __ffs(todo) - 1;
            todo &= todo - 1;
            const u32 n = __shfl_sync(kFullMask, len, sl);
            char* d = reinterpret_cast<char*>(__shfl_sync(kFullMask, reinterpret_cast<u64>(dst), sl));
            const unsigned char* s = reinterpret_cast<const unsigned char*>(__shfl_sync(kFullMask, reinterpret_cast<u64>(src), sl));
            for (u32 j = lane_id(); j < n; j += 32) d[j] = (char)s[j];
        }
    }
}

// first k-mer of each contig + '\n' (read_kmers.hpp:84, kmer_hash.cpp:66); n_starts read on the device.
// Both tables: the plain traverse writes its heads with it too.
template <int W>
__global__ void __launch_bounds__(256)
ct_emit_heads_kernel(const typename Slot<W>::value_t* __restrict__ starts, u32 hcap, int k,
                     const u32* __restrict__ contig_len, const u64* __restrict__ contig_off,
                     const Counters* __restrict__ ctr, u64 out_cap, char* __restrict__ out) {
    typedef Slot<W> S;
    if (ctr->errors & (kErrConverge | kErrCycle | kErrInternal | kErrNotFound)) return;
    const u32 n_starts = (u32)min(ctr->n_starts_dev, (u64)hcap);
    const u64 total = (u64)n_starts * (u32)(k + 1);
    for (u64 t = (u64)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (u64)gridDim.x * blockDim.x) {
        const u64 c = t / (u32)(k + 1);
        const u32 j = (u32)(t - c * (u32)(k + 1));
        const u32 len = contig_len[c];
        if (len == 0) continue;
        const u64 off = contig_off[c];
        if (off + len > out_cap) continue;
        if (j < (u32)k) out[off + j] = (char)ext_char(S::base_at(starts[c], k, (int)j));
        else out[off + len - 1] = '\n';
    }
}

// Start list in input order, one warp per insert tile (kInsTile records = 32 mask words), appended behind the
// n_starts_dev already registered and bounded by hcap: the write position comes from the device, so a sharded step
// needs no host round trip.  Both tables register their start nodes with it (register_starts in capi.cu).
template <int W>
__global__ void __launch_bounds__(256)
ct_scatter_starts_kernel(const unsigned char* __restrict__ recs, u64 n, int k, const u32* __restrict__ start_mask,
                         const u64* __restrict__ tile_offsets, u64 ntiles, typename Slot<W>::value_t* __restrict__ starts_out,
                         const Counters* __restrict__ ctr, u32 hcap) {
    typedef Slot<W> S;
    const u64 tile = ((u64)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (tile >= ntiles) return;
    const int pl = (k + 3) >> 2, pb = pl + 2;
    const u64 word = tile * (kInsTile / 32) + lane_id();
    const u64 nwords = (n + 31) >> 5;
    u32 m = word < nwords ? start_mask[word] : 0u;
    u32 inc = __popc(m);
    const u32 mine = inc;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const u32 y = __shfl_up_sync(kFullMask, inc, d);
        if (lane_id() >= (u32)d) inc += y;
    }
    u64 dst = ctr->n_starts_dev + tile_offsets[tile] + (inc - mine);
    while (m) {
        const int bit = __ffs(m) - 1;
        m &= m - 1;
        const u64 rec = (word << 5) + bit;
        bool ok;
        unsigned char tmp[18];
        const unsigned char* src = recs + rec * pb;
        for (int i = 0; i < pb; ++i) tmp[i] = src[i];
        if (dst < hcap) starts_out[dst] = S::from_record(tmp, k, pl, ok);
        ++dst;
    }
}

}  // namespace kh
