// kernels.cuh -- the sm_100a kernels of the single-GPU k-mer hash / contig traversal path.
//
//   K1 pack_lines_kernel      text lines -> kmer_pair records            (read_kmers.hpp:72-76, packing.hpp:50-92)
//   K2 insert_kernel          records -> open-addressing table + start bitmask, direct (tables that fit L2)
//                                                                         (hash_map.hpp:55-72, kmer_hash.cpp:27-31)
//   K2p partition_kernel      records grouped by ~16 MB table region (+ start bitmask)
//       insert_slots_kernel   grouped slot values -> table, CAS-first, region warm-up      (tables larger than L2)
//   K3 scan_* / scatter_starts_kernel   start bitmask -> start list in file order           (kmer_hash.cpp:27-31)
//   K4 find_kernel            batch lookup                                (hash_map.hpp:83-92)
//   K5 walk_kernel            one lane per walk segment                   (kmer_hash.cpp:38-55, kmer_t.hpp:51-53)
//      rank_kernel            pointer jumping over the segment list (cooperative launch)
//   K6 emit_segments_kernel / emit_heads_kernel   contig text             (read_kmers.hpp:81-92)
//
// All of it is HBM-bound integer work: no tensor cores, no floating point.  The multi-GPU path uses the chunk
// table (ctable.cuh).
#pragma once
#include <cooperative_groups.h>

#include "slot.cuh"

namespace kh {
namespace cg = cooperative_groups;

constexpr u32 kFullMask = 0xFFFFFFFFu;

__device__ __forceinline__ u32 lane_id() { return threadIdx.x & 31u; }
__device__ __forceinline__ u64 warp_sum_u64(u64 x) {
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) x += __shfl_xor_sync(kFullMask, x, d);
    return x;
}

// Cooperative copy global -> shared of `bytes` bytes (16-byte vectors when aligned).
__device__ __forceinline__ void stage_in(unsigned char* s_dst, const unsigned char* g_src, u32 bytes) {
    if ((reinterpret_cast<uintptr_t>(g_src) & 15u) == 0) {
        const u32 nv = bytes >> 4;
        const uint4* s4 = reinterpret_cast<const uint4*>(g_src);
        uint4* d4 = reinterpret_cast<uint4*>(s_dst);
        for (u32 i = threadIdx.x; i < nv; i += blockDim.x) d4[i] = load128_stream(s4 + i);
        for (u32 i = (nv << 4) + threadIdx.x; i < bytes; i += blockDim.x) s_dst[i] = g_src[i];
    } else {
        for (u32 i = threadIdx.x; i < bytes; i += blockDim.x) s_dst[i] = g_src[i];
    }
}
__device__ __forceinline__ void stage_out(unsigned char* g_dst, const unsigned char* s_src, u32 bytes) {
    if ((reinterpret_cast<uintptr_t>(g_dst) & 15u) == 0) {
        const u32 nv = bytes >> 4;
        const uint4* s4 = reinterpret_cast<const uint4*>(s_src);
        uint4* d4 = reinterpret_cast<uint4*>(g_dst);
        for (u32 i = threadIdx.x; i < nv; i += blockDim.x) d4[i] = s4[i];
        for (u32 i = (nv << 4) + threadIdx.x; i < bytes; i += blockDim.x) g_dst[i] = s_src[i];
    } else {
        for (u32 i = threadIdx.x; i < bytes; i += blockDim.x) g_dst[i] = s_src[i];
    }
}

// =========================================================================================
// K1  pack: (K+4)-byte text lines -> reference kmer_pair bytes
// =========================================================================================
constexpr int kPackLines = 256;   // lines per block; 256*(K+4) is a multiple of 16 for every K

// Four letters (little-endian in one 32-bit word, first letter in the low byte) -> one packed byte
// (first letter in bits 7..6), branch-free:  code = ((c >> 1) & 3) ^ ((c >> 2) & 1)  maps A,C,G,T to
// 0,1,2,3; the multiply gathers the four 2-bit codes.  `ok` is cleared unless all four are ACGT.
__device__ __forceinline__ u32 pack4(u32 w, bool& ok) {
    const u32 valid = __vcmpeq4(w, 0x41414141u) | __vcmpeq4(w, 0x43434343u) | __vcmpeq4(w, 0x47474747u) |
                      __vcmpeq4(w, 0x54545454u);
    ok = ok && (valid == 0xFFFFFFFFu);
    const u32 codes = ((w >> 1) & 0x03030303u) ^ ((w >> 2) & 0x01010101u);
    return (codes * 0x40100401u) >> 24;
}
// 32-bit word at an arbitrary byte offset of a 4-byte aligned shared array
__device__ __forceinline__ u32 lds_unaligned32(const unsigned char* base, u32 off) {
    const u32* w = reinterpret_cast<const u32*>(base) + (off >> 2);
    return __funnelshift_r(w[0], w[1], (off & 3u) * 8u);
}

__global__ void __launch_bounds__(kPackLines)
pack_lines_kernel(const unsigned char* __restrict__ text, u64 n_lines, int k,
                  unsigned char* __restrict__ pairs, Counters* ctr) {
    extern __shared__ __align__(16) unsigned char smem[];
    const int ll = k + 4, pl = (k + 3) >> 2, pb = pl + 2;
    unsigned char* s_in = smem;                                   // + 8 bytes of slack for the word reads
    unsigned char* s_out = smem + (((u32)kPackLines * ll + 8u + 15u) & ~15u);
    const u64 line0 = (u64)blockIdx.x * kPackLines;
    const u32 cnt = (u32)min((u64)kPackLines, n_lines - line0);
    stage_in(s_in, text + line0 * ll, cnt * ll);
    __syncthreads();
    if (threadIdx.x < cnt) {
        const u32 off = threadIdx.x * ll;
        unsigned char* rec = s_out + threadIdx.x * pb;
        bool ok = true;
        const int full = k >> 2;                                  // whole groups of four bases
        for (int q = 0; q < full; ++q) rec[q] = (unsigned char)pack4(lds_unaligned32(s_in, off + 4 * q), ok);
        if (k & 3) {                                              // packing.hpp:85-91: the tail is padded with 'A'
            u32 w = lds_unaligned32(s_in, off + 4 * full);
            const u32 keep = (1u << (8 * (k & 3))) - 1u;
            w = (w & keep) | (0x41414141u & ~keep);
            rec[full] = (unsigned char)pack4(w, ok);
        }
        const unsigned char b = s_in[off + k + 1], f = s_in[off + k + 2];   // byte k is a separator nobody reads
        ok = ok && ext_code(b) != kExtBad && ext_code(f) != kExtBad;
        rec[pl] = b;
        rec[pl + 1] = f;
        if (!ok) atomicOr(&ctr->errors, kErrBadInput);
    }
    __syncthreads();
    stage_out(pairs + line0 * pb, s_out, cnt * pb);
}

// =========================================================================================
// K2  insert (+ the start-node bitmask K3 consumes)
// =========================================================================================
constexpr int kInsThreads = 256;
constexpr int kInsPerThread = 4;
constexpr int kInsTile = kInsThreads * kInsPerThread;    // 1024 records per block

enum { kInsInserted = 0, kInsDuplicate = 1, kInsFull = 2 };

// Claim the first empty slot of the probe sequence starting at bucket b (q = preloaded bucket b).
// Slots inside a bucket fill in order and are never released, so a reader may stop at the first
// empty slot.  First writer wins on a duplicate key.
template <int W>
__device__ __forceinline__ int insert_one(typename Slot<W>::value_t* table, u64 nbuckets, u64 b,
                                          typename Slot<W>::value_t v, u64 (&q)[4], u64* pos_out = nullptr) {
    typedef Slot<W> S;
    for (u64 tries = 0; tries < nbuckets; ++tries) {
#pragma unroll
        for (int i = 0; i < S::kPerBucket; ++i) {
            typename S::value_t cur = S::from_bucket(q, i);
            if (S::empty(cur)) {
                cur = S::cas(table + b * S::kPerBucket + i, S::zero(), v);
                if (S::empty(cur)) {
                    if (pos_out) *pos_out = b * S::kPerBucket + i;
                    return kInsInserted;
                }
            }
            if (S::same_key(cur, v)) return kInsDuplicate;
        }
        b = (b + 1 == nbuckets) ? 0 : b + 1;
        load256_cg(table + b * S::kPerBucket, q);
    }
    return kInsFull;
}

template <int W>
__global__ void __launch_bounds__(kInsThreads)
insert_kernel(const unsigned char* __restrict__ recs, u64 n, int k,
              typename Slot<W>::value_t* table, u64 nbuckets,
              u32* __restrict__ start_mask, u32* __restrict__ tile_starts, Counters* ctr) {
    typedef Slot<W> S;
    typedef typename S::value_t V;
    extern __shared__ __align__(16) unsigned char s_rec[];
    __shared__ u32 s_starts, s_inserted, s_dups, s_err;
    const int pl = (k + 3) >> 2, pb = pl + 2;
    const u64 rec0 = (u64)blockIdx.x * kInsTile;
    const u32 cnt = (u32)min((u64)kInsTile, n - rec0);
    if (threadIdx.x == 0) { s_starts = 0; s_inserted = 0; s_dups = 0; s_err = 0; }
    stage_in(s_rec, recs + rec0 * pb, cnt * pb);
    __syncthreads();

    V v[kInsPerThread];
    u64 b[kInsPerThread];
    u64 q[kInsPerThread][4];
    bool live[kInsPerThread];
    u32 err = 0, starts = 0;
#pragma unroll
    for (int r = 0; r < kInsPerThread; ++r) {
        const u32 j = threadIdx.x + r * kInsThreads;
        live[r] = j < cnt;
        bool ok = true;
        v[r] = S::zero();
        if (live[r]) v[r] = S::from_record_staged(s_rec + j * pb, k, pl, ok);
        if (!ok) { err |= kErrBadInput; live[r] = false; }
        b[r] = live[r] ? place_bucket<W>(v[r], nbuckets) : 0;
        if (live[r]) load256_cg(table + b[r] * S::kPerBucket, q[r]);      // 4 independent sector reads in flight
        // kmer_hash.cpp:27-31: remember which records start a contig, by position in the input
        const u32 bal = __ballot_sync(kFullMask, live[r] && S::back(v[r]) == kExtF);
        const u64 word = (rec0 + (u64)r * kInsThreads + (threadIdx.x & ~31u)) >> 5;
        if (lane_id() == 0 && (word << 5) < n) { start_mask[word] = bal; starts += __popc(bal); }
    }
    u32 inserted = 0, dups = 0;
#pragma unroll
    for (int r = 0; r < kInsPerThread; ++r) {
        if (!live[r]) continue;
        const int rc = insert_one<W>(table, nbuckets, b[r], v[r], q[r]);
        inserted += (rc == kInsInserted);
        dups += (rc == kInsDuplicate);
        if (rc == kInsFull) err |= kErrTableFull;
    }
    // block totals -> one atomic each
    inserted = __reduce_add_sync(kFullMask, inserted);
    dups = __reduce_add_sync(kFullMask, dups);
    err = __reduce_or_sync(kFullMask, err);
    if (lane_id() == 0) {
        if (starts) atomicAdd(&s_starts, starts);
        if (inserted) atomicAdd(&s_inserted, inserted);
        if (dups) atomicAdd(&s_dups, dups);
        if (err) atomicOr(&s_err, err);
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        tile_starts[blockIdx.x] = s_starts;
        if (s_inserted) atomicAdd(&ctr->n_inserted, (u64)s_inserted);
        if (s_dups) atomicAdd(&ctr->n_duplicates, (u64)s_dups);
        if (s_err) atomicOr(&ctr->errors, s_err);
    }
}

// block-wide exclusive scan helper (also used by the scan kernels below)
__device__ __forceinline__ u64 block_exclusive_scan(u64 x, u64* s_warp, u64& block_total) {
    u64 inc = x;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const u64 y = __shfl_up_sync(kFullMask, inc, d);
        if (lane_id() >= (u32)d) inc += y;
    }
    const u32 warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
    if (lane_id() == 31) s_warp[warp] = inc;
    __syncthreads();
    if (warp == 0) {
        u64 w = lane_id() < nwarps ? s_warp[lane_id()] : 0;
        u64 winc = w;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const u64 y = __shfl_up_sync(kFullMask, winc, d);
            if (lane_id() >= (u32)d) winc += y;
        }
        if (lane_id() < nwarps) s_warp[lane_id()] = winc - w;
        if (lane_id() == 31) s_warp[32] = winc;
    }
    __syncthreads();
    block_total = s_warp[32];
    const u64 r = s_warp[warp] + inc - x;
    __syncthreads();
    return r;
}

// =========================================================================================
// K2p  partitioned insert: prep (histogram + start bitmask) -> partition -> insert_slots
// =========================================================================================
// Random CAS traffic over a multi-GB table is bound by DRAM row activations (~16 G read+CAS/s
// measured, profiles/r01_random_access_probe_occ8.txt); the same traffic against an L2-resident
// region runs at >50-120 G/s.  So for tables larger than L2 the records are first grouped by
// table region ("partition" = 2^part_shift consecutive buckets, ~16 MB of table) with one streaming
// counting-sort pass; the insert kernel then sweeps the grouped array front to back, and the blocks
// in flight at any moment touch only a couple of regions.  The table semantics are unchanged
// (same buckets, same probing) -- only the order of insertion differs.
constexpr u64 kPartBytes = 16ull << 20;    // table bytes per partition (more when the table needs over kMaxParts of them)
constexpr int kMaxParts = 1024;
constexpr int kPartThreads = 256;
constexpr int kPartPerThread = 8;
constexpr int kPartTile = kPartThreads * kPartPerThread;     // 2048 records per block

// pass 1: block-local counting sort by partition, coalesced runs into per-partition buffers of fixed
// capacity (no histogram pass: a partition's expected share is known from the uniform hash; space is
// reserved with one atomicAdd per (block, partition); a record that does not fit -- never in practice
// -- is inserted directly).  Also produces the start bitmask / per-tile start counts that
// scatter_starts_kernel consumes (tiles of kInsTile records, identical to insert_kernel's).
#ifndef KH_PART_MIN_BLOCKS
#define KH_PART_MIN_BLOCKS 4
#endif
template <int W>
__global__ void __launch_bounds__(kPartThreads, KH_PART_MIN_BLOCKS)
partition_kernel(const unsigned char* __restrict__ recs, u64 n, int k, u64 nbuckets, u32 part_shift, u32 nparts,
                 u64 part_cap, u32* __restrict__ cursor, typename Slot<W>::value_t* __restrict__ grouped,
                 typename Slot<W>::value_t* table, u32* __restrict__ start_mask, u32* __restrict__ tile_starts,
                 typename Slot<W>::value_t* __restrict__ overflow, u32 overflow_cap, Counters* ctr) {
    typedef Slot<W> S;
    typedef typename S::value_t V;
    extern __shared__ __align__(16) unsigned char s_raw[];
    // layout: hist u32[nparts] | off u32[nparts] | gbase u32[nparts] | part id per sorted position u16[kPartTile]
    //         | union { record bytes (phase 1), sorted slots (phase 3) }
    u32* s_hist = reinterpret_cast<u32*>(s_raw);
    u32* s_off = s_hist + nparts;
    u32* s_gbase = s_off + nparts;
    unsigned short* s_pid = reinterpret_cast<unsigned short*>(s_raw + 12 * (size_t)nparts);
    unsigned char* s_union = s_raw + ((12 * (size_t)nparts + 2 * kPartTile + 15) & ~(size_t)15);
    unsigned char* s_rec = s_union;
    V* s_sorted = reinterpret_cast<V*>(s_union);
    __shared__ u64 s_warp[33];
    __shared__ u32 s_starts[kPartTile / kInsTile], s_err, s_direct_ins, s_direct_dup;
    const int pl = (k + 3) >> 2, pb = pl + 2;
    const u64 rec0 = (u64)blockIdx.x * kPartTile;
    const u32 cnt = (u32)min((u64)kPartTile, n - rec0);
    for (u32 i = threadIdx.x; i < nparts; i += blockDim.x) s_hist[i] = 0;
    if (threadIdx.x < kPartTile / kInsTile) s_starts[threadIdx.x] = 0;
    if (threadIdx.x == 0) { s_err = 0; s_direct_ins = 0; s_direct_dup = 0; }
    stage_in(s_rec, recs + rec0 * pb, cnt * pb);
    __syncthreads();
    V v[kPartPerThread];
    u32 pid[kPartPerThread], rk[kPartPerThread];
    u32 err = 0;
#pragma unroll
    for (int r = 0; r < kPartPerThread; ++r) {
        const u32 j = threadIdx.x + r * kPartThreads;
        bool ok = true, live = j < cnt;
        pid[r] = 0xFFFFFFFFu;
        v[r] = S::zero();
        if (live) v[r] = S::from_record_staged(s_rec + j * pb, k, pl, ok);
        if (!ok) { err |= kErrBadInput; live = false; }
        if (live) {
            pid[r] = (u32)(place_bucket<W>(v[r], nbuckets) >> part_shift);
            rk[r] = atomicAdd(&s_hist[pid[r]], 1u);
        }
        // kmer_hash.cpp:27-31: which records start a contig, by position in the input
        const u32 bal = __ballot_sync(kFullMask, live && S::back(v[r]) == kExtF);
        const u64 first = rec0 + (u64)r * kPartThreads + (threadIdx.x & ~31u);
        if (lane_id() == 0 && first < n) {
            start_mask[first >> 5] = bal;
            if (bal) atomicAdd(&s_starts[(r * kPartThreads + threadIdx.x) / kInsTile], (u32)__popc(bal));
        }
    }
    err = __reduce_or_sync(kFullMask, err);
    if (lane_id() == 0 && err) atomicOr(&s_err, err);
    __syncthreads();
    // block-local exclusive scan of the histogram (nparts <= 1024 = 4 per thread) + global reservations
    {
        u32 h[4], sum = 0;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const u32 i = threadIdx.x * 4 + q;
            h[q] = i < nparts ? s_hist[i] : 0u;
            sum += h[q];
        }
        u64 total;
        u64 run = block_exclusive_scan((u64)sum, s_warp, total);
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const u32 i = threadIdx.x * 4 + q;
            if (i < nparts) {
                s_off[i] = (u32)run;
                s_gbase[i] = h[q] ? atomicAdd(&cursor[i], h[q]) : 0u;
            }
            run += h[q];
        }
    }
    __syncthreads();
#pragma unroll
    for (int r = 0; r < kPartPerThread; ++r) {
        if (pid[r] != 0xFFFFFFFFu) {
            const u32 pos = s_off[pid[r]] + rk[r];
            s_sorted[pos] = v[r];
            s_pid[pos] = (unsigned short)pid[r];
        }
    }
    __syncthreads();
    const u32 good = s_off[nparts - 1] + s_hist[nparts - 1];
    for (u32 pos = threadIdx.x; pos < good; pos += blockDim.x) {
        const u32 p = s_pid[pos];
        const u64 at = (u64)s_gbase[p] + (pos - s_off[p]);
        if (at < part_cap) {
            grouped[(u64)p * part_cap + at] = s_sorted[pos];
        } else if (overflow) {                             // chunked build: the fix-up pass inserts it after the chunks are final
            const u32 o = atomicAdd(&ctr->n_outbox, 1u);
            if (o < overflow_cap) overflow[o] = s_sorted[pos];
            else atomicOr(&s_err, kErrInternal);
        } else {                                           // partition buffer full: insert right here
            const V val = s_sorted[pos];
            const u64 b = place_bucket<W>(val, nbuckets);
            u64 q[4];
            load256_cg(table + b * S::kPerBucket, q);
            const int rc = insert_one<W>(table, nbuckets, b, val, q);
            if (rc == kInsInserted) atomicAdd(&s_direct_ins, 1u);
            else if (rc == kInsDuplicate) atomicAdd(&s_direct_dup, 1u);
            else atomicOr(&s_err, kErrTableFull);
        }
    }
    __syncthreads();
    if (threadIdx.x < kPartTile / kInsTile) {
        const u64 tile = (u64)blockIdx.x * (kPartTile / kInsTile) + threadIdx.x;
        if (tile * kInsTile < n) tile_starts[tile] = s_starts[threadIdx.x];
    }
    if (threadIdx.x == 0) {
        if (s_err) atomicOr(&ctr->errors, s_err);
        if (s_direct_ins) atomicAdd(&ctr->n_inserted, (u64)s_direct_ins);
        if (s_direct_dup) atomicAdd(&ctr->n_duplicates, (u64)s_direct_dup);
    }
}

// =========================================================================================
// K2c  chunked build (64-bit slots): no global atomics at all
// =========================================================================================
// The path for large batches into tables of 64-bit slots.  With 128-bit slots twice the bytes go through the two
// grouping passes and insert_slots_kernel is faster (capi.cu), so these kernels exist for Slot<1> only.
// The grouped records of one partition (partition_kernel) are split once more by 64 KB table chunk
// (subpartition_kernel); then one block per chunk builds the chunk in SHARED memory with ATOMS.CAS and
// writes it to HBM in one coalesced sweep (build_chunks_kernel).  DRAM sees only streaming traffic
// (7 + 8 + 8 + 8 + 8 + 16 bytes per k-mer), no random row activations.  Probing stays the table's
// ordinary linear probing: a record whose probe sequence would leave its chunk (its home is at the very
// end of the chunk and those buckets are full) goes to a small overflow list that is inserted afterwards
// with the ordinary global insert -- by then every chunk is final, so "first empty slot from home" holds.
constexpr u32 kChunkShift = 11;                       // 2048 buckets = 64 KB per chunk
constexpr u32 kChunkBuckets = 1u << kChunkShift;
constexpr int kSubThreads = 256;
constexpr int kSubPerThread = 8;
constexpr int kSubTile = kSubThreads * kSubPerThread;  // 2048 slot values per block

// After the block-wide rank/reserve each thread writes its values straight to their destination run (L2 merges
// the sector writes); staging a sorted copy in shared memory first was measured slower (2.71 vs 2.52 ms insert).
// The kernel splits input partition `part` (values whose home lies in units [part*nsub, (part+1)*nsub), a unit being
// 2^unit_shift buckets) into one buffer per unit.  Level 2 of the chunked build uses it with unit = chunk.
__global__ void __launch_bounds__(kSubThreads, 4)
subpartition_kernel(const u64* __restrict__ grouped, const u32* __restrict__ part_cursor,
                    u64 part_cap, u32 blocks_per_part, u32 unit_shift, u32 nsub, u64 nbuckets,
                    u32 chunk_cap, u32* __restrict__ chunk_cursor, u64* __restrict__ fine,
                    u64* __restrict__ overflow, u32 overflow_cap, Counters* ctr) {
    typedef Slot<1> S;
    typedef u64 V;
    extern __shared__ __align__(16) unsigned char s_raw[];
    u32* s_hist = reinterpret_cast<u32*>(s_raw);                       // nsub <= 1024 units per input partition
    u32* s_gbase = s_hist + nsub;
    const u32 part = blockIdx.x / blocks_per_part, jblk = blockIdx.x % blocks_per_part;
    const u64 n = min((u64)part_cursor[part], part_cap);
    const u64 base = (u64)jblk * kSubTile;
    if (base >= n) return;
    const V* __restrict__ src = grouped + (u64)part * part_cap;
    const u64 first_chunk = (u64)part * nsub;
    for (u32 i = threadIdx.x; i < nsub; i += blockDim.x) s_hist[i] = 0;
    __syncthreads();
    V v[kSubPerThread];
    u32 sid[kSubPerThread], rk[kSubPerThread];
#pragma unroll
    for (int r = 0; r < kSubPerThread; ++r) {
        const u64 i = base + (u64)r * kSubThreads + threadIdx.x;
        v[r] = i < n ? src[i] : S::zero();
    }
#pragma unroll
    for (int r = 0; r < kSubPerThread; ++r) {
        sid[r] = 0xFFFFFFFFu;
        if (!S::empty(v[r])) {
            const u64 chunk = place_bucket<1>(v[r], nbuckets) >> unit_shift;
            sid[r] = min((u32)(chunk - first_chunk), nsub - 1u);
            rk[r] = atomicAdd(&s_hist[sid[r]], 1u);
        }
    }
    __syncthreads();
    // reserve one run per (block, chunk); s_gbase = position of this block's run inside the chunk's buffer
    for (u32 i = threadIdx.x; i < nsub; i += blockDim.x)
        s_gbase[i] = s_hist[i] ? atomicAdd(&chunk_cursor[first_chunk + i], s_hist[i]) : 0u;
    __syncthreads();
#pragma unroll
    for (int r = 0; r < kSubPerThread; ++r) {
        if (sid[r] == 0xFFFFFFFFu) continue;
        const u32 at = s_gbase[sid[r]] + rk[r];
        if (at < chunk_cap) {
            fine[(first_chunk + sid[r]) * (u64)chunk_cap + at] = v[r];
        } else {                                                     // chunk buffer full: fix-up pass takes it
            const u32 o = atomicAdd(&ctr->n_outbox, 1u);
            if (o < overflow_cap) overflow[o] = v[r];
            else atomicOr(&ctr->errors, kErrInternal);
        }
    }
}

// one block per 64 KB chunk: build it in shared memory, write it out once
constexpr int kBuildThreads = 512;
constexpr int kBuildBatch = 4;          // records a thread fetches before it starts inserting (loads in flight)

// Insert into the chunk in shared memory.  The whole bucket is read at once and the first empty slot is picked
// without branches, then ONE ATOMS.CAS claims it; only a lost race (another thread took that slot meanwhile) or a full
// bucket loops.  Probing slot by slot instead ran with ~7 of 32 lanes active and was 60 % of this kernel's issued
// instructions.  Slots of a bucket fill in order and are never emptied, so every occupied slot precedes every empty one.
__device__ __forceinline__ int build_insert_one(u64* s_tab, u32 nb, u32 b, u64 v) {
    typedef Slot<1> S;
    typedef u64 V;
    const unsigned s_base = (unsigned)__cvta_generic_to_shared(s_tab);
    while (b < nb) {
        u64 q[4];
        lds_bucket(s_base + b * 32u, q);
        int j = -1;
        bool dup = false;
#pragma unroll
        for (int i = S::kPerBucket - 1; i >= 0; --i) {            // descending: the smallest empty index wins
            const V c = S::from_bucket(q, i);
            if (S::empty(c)) j = i;
            else if (S::same_key(c, v)) dup = true;
        }
        if (dup) return kInsDuplicate;
        if (j < 0) { ++b; continue; }                             // bucket full: linear probing, next bucket
        const V old = S::cas_shared(s_tab + b * S::kPerBucket + j, S::zero(), v);
        if (S::empty(old)) return kInsInserted;
        if (S::same_key(old, v)) return kInsDuplicate;
        // lost the slot to another thread: look at the bucket again
    }
    return kInsFull;                      // the probe sequence leaves the chunk
}

__global__ void __launch_bounds__(kBuildThreads)
build_chunks_kernel(const u64* __restrict__ fine, const u32* __restrict__ chunk_cursor, u32 chunk_cap,
                    u64* table, u64 nbuckets, int load_existing,
                    u64* __restrict__ overflow, u32 overflow_cap, Counters* ctr) {
    typedef Slot<1> S;
    typedef u64 V;
    extern __shared__ __align__(16) unsigned char s_raw[];
    V* s_tab = reinterpret_cast<V*>(s_raw);                            // kChunkBuckets * 32 bytes
    __shared__ u32 s_inserted, s_dups;
    const u64 b0 = (u64)blockIdx.x << kChunkShift;
    const u32 nb = (u32)min((u64)kChunkBuckets, nbuckets - b0);
    const u32 nvec = nb * 2;                                           // 16-byte vectors in this chunk
    uint4* s4 = reinterpret_cast<uint4*>(s_raw);
    uint4* g4 = reinterpret_cast<uint4*>(table + b0 * S::kPerBucket);
    const u32 cnt = min(chunk_cursor[blockIdx.x], chunk_cap);
    const V* __restrict__ recs = fine + (u64)blockIdx.x * chunk_cap;
    // first batch of records is on its way while the chunk is zeroed / loaded
    V v[kBuildBatch];
#pragma unroll
    for (int r = 0; r < kBuildBatch; ++r) {
        const u32 i = threadIdx.x + r * kBuildThreads;
        v[r] = i < cnt ? recs[i] : S::zero();
    }
    if (threadIdx.x == 0) { s_inserted = 0; s_dups = 0; }
    if (load_existing) for (u32 i = threadIdx.x; i < nvec; i += blockDim.x) s4[i] = g4[i];
    else for (u32 i = threadIdx.x; i < nvec; i += blockDim.x) s4[i] = make_uint4(0, 0, 0, 0);
    __syncthreads();
    u32 inserted = 0, dups = 0;
    for (u32 base = 0; base < cnt; base += kBuildThreads * kBuildBatch) {
        V nxt[kBuildBatch];
#pragma unroll
        for (int r = 0; r < kBuildBatch; ++r) {                        // prefetch the following batch
            const u32 i = base + kBuildThreads * kBuildBatch + threadIdx.x + r * kBuildThreads;
            nxt[r] = i < cnt ? recs[i] : S::zero();
        }
#pragma unroll
        for (int r = 0; r < kBuildBatch; ++r) {
            if (S::empty(v[r])) continue;
            const u32 b = (u32)(place_bucket<1>(v[r], nbuckets) - b0);      // local bucket, < nb by construction
            const int rc = build_insert_one(s_tab, nb, b, v[r]);
            inserted += (rc == kInsInserted);
            dups += (rc == kInsDuplicate);
            if (rc == kInsFull) {
                const u32 o = atomicAdd(&ctr->n_outbox, 1u);
                if (o < overflow_cap) overflow[o] = v[r];
                else atomicOr(&ctr->errors, kErrInternal);
            }
        }
#pragma unroll
        for (int r = 0; r < kBuildBatch; ++r) v[r] = nxt[r];
    }
    inserted = __reduce_add_sync(kFullMask, inserted);
    dups = __reduce_add_sync(kFullMask, dups);
    if (lane_id() == 0) {
        if (inserted) atomicAdd(&s_inserted, inserted);
        if (dups) atomicAdd(&s_dups, dups);
    }
    __syncthreads();
    for (u32 i = threadIdx.x; i < nvec; i += blockDim.x) g4[i] = s4[i];
    if (threadIdx.x == 0) {
        if (s_inserted) atomicAdd(&ctr->n_inserted, (u64)s_inserted);
        if (s_dups) atomicAdd(&ctr->n_duplicates, (u64)s_dups);
    }
}

// the few records the chunk build could not place: ordinary global insert, after every chunk is final
__global__ void __launch_bounds__(256)
insert_overflow_kernel(const u64* __restrict__ overflow, u32 overflow_cap, u64* table, u64 nbuckets, Counters* ctr) {
    typedef Slot<1> S;
    const u32 n = min(ctr->n_outbox, overflow_cap);
    for (u32 i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const u64 v = overflow[i];
        const u64 b = place_bucket<1>(v, nbuckets);
        u64 q[4];
        load256_cg(table + b * S::kPerBucket, q);
        const int rc = insert_one<1>(table, nbuckets, b, v, q);
        if (rc == kInsInserted) atomicAdd(&ctr->n_inserted, 1ull);
        else if (rc == kInsDuplicate) atomicAdd(&ctr->n_duplicates, 1ull);
        else atomicOr(&ctr->errors, kErrTableFull);
    }
}

// sequential L2 warm-up of the first table regions (the rest is warmed by insert_slots_kernel itself)
__global__ void __launch_bounds__(256)
warm_kernel(const char* __restrict__ base, u64 nlines) {
    for (u64 l = (u64)blockIdx.x * blockDim.x + threadIdx.x; l < nlines; l += (u64)gridDim.x * blockDim.x)
        asm volatile("prefetch.global.L2 [%0];" ::"l"(base + (l << 7)));
}

constexpr int kInsSlotsMinBlocks = 6;      // latency-bound kernel: trade registers for resident warps
constexpr u32 kWarmAhead = 1;              // table regions (partitions) prefetched ahead of the inserts
// pass 3: insert pre-converted slot values (grouped by partition, so the table traffic is L2-resident).  CAS slot 0
// of the home bucket blind (4 independent atomics in flight per thread) and fall back to read + CAS only when it is
// taken.
template <int W>
__global__ void __launch_bounds__(kInsThreads, kInsSlotsMinBlocks)
insert_slots_kernel(const typename Slot<W>::value_t* __restrict__ grouped, const u32* __restrict__ cursor,
                    u64 part_cap, u32 blocks_per_part, u32 nparts, u32 part_shift,
                    typename Slot<W>::value_t* table, u64 nbuckets, Counters* ctr) {
    typedef Slot<W> S;
    typedef typename S::value_t V;
    __shared__ u32 s_inserted, s_dups, s_err;
    if (threadIdx.x == 0) { s_inserted = 0; s_dups = 0; s_err = 0; }
    __syncthreads();
    const u32 part = blockIdx.x / blocks_per_part, jblk = blockIdx.x % blocks_per_part;
    const u64 n = min((u64)cursor[part], part_cap);         // records grouped into this partition
    const V* __restrict__ slots = grouped + (u64)part * part_cap;
    const u64 base = (u64)jblk * kInsTile;
    // Warm the table region kWarmAhead partitions ahead of this block's own with sequential L2
    // prefetches: a first touch by a random CAS costs a DRAM row activation each (the 41 G/s ceiling),
    // a sequential sweep of the same region costs streaming bandwidth.  Non-destructive, so no ordering
    // between blocks is needed.  Each block of partition p warms its share of region p + kWarmAhead.
    if (part + kWarmAhead < nparts) {
        const u32 tp = part + kWarmAhead;
        const u64 b0 = (u64)tp << part_shift, b1 = min(nbuckets, ((u64)tp + 1) << part_shift);
        const u64 nlines = ((b1 - b0) * 32 + 127) >> 7;
        const u64 per = (nlines + blocks_per_part - 1) / blocks_per_part;
        const u64 l0 = (u64)jblk * per, l1 = min(nlines, l0 + per);
        const char* region = reinterpret_cast<const char*>(table) + b0 * 32;
        for (u64 l = l0 + threadIdx.x; l < l1; l += blockDim.x)
            asm volatile("prefetch.global.L2 [%0];" ::"l"(region + (l << 7)));
    }
    if (base >= n) return;
    V v[kInsPerThread], old[kInsPerThread];
    bool live[kInsPerThread];
    u32 inserted = 0, dups = 0, err = 0;
#pragma unroll
    for (int r = 0; r < kInsPerThread; ++r) {
        const u64 i = base + (u64)r * kInsThreads + threadIdx.x;
        live[r] = i < n;
        v[r] = live[r] ? slots[i] : S::zero();
        old[r] = S::zero();
        if (live[r]) old[r] = S::cas(table + place_bucket<W>(v[r], nbuckets) * S::kPerBucket, S::zero(), v[r]);
    }
#pragma unroll
    for (int r = 0; r < kInsPerThread; ++r) {
        if (!live[r]) continue;
        if (S::empty(old[r])) { ++inserted; continue; }
        if (S::same_key(old[r], v[r])) { ++dups; continue; }
        // slot 0 is occupied by another key: general path.  The home bucket is hashed again rather than kept from the
        // first loop: four live bucket numbers do not fit the 40 registers of 6 blocks per SM and were spilled.
        const u64 b = place_bucket<W>(v[r], nbuckets);
        u64 q[4];
        load256_cg(table + b * S::kPerBucket, q);
        const int rc = insert_one<W>(table, nbuckets, b, v[r], q);
        inserted += (rc == kInsInserted);
        dups += (rc == kInsDuplicate);
        if (rc == kInsFull) err |= kErrTableFull;
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
    if (threadIdx.x == 0) {
        if (s_inserted) atomicAdd(&ctr->n_inserted, (u64)s_inserted);
        if (s_dups) atomicAdd(&ctr->n_duplicates, (u64)s_dups);
        if (s_err) atomicOr(&ctr->errors, s_err);
    }
}

// =========================================================================================
// exclusive scan of u32 counts -> u64 offsets (three small kernels)
// =========================================================================================
constexpr int kScanThreads = 256;
constexpr int kScanPerThread = 8;
constexpr int kScanTile = kScanThreads * kScanPerThread;   // 2048

__global__ void __launch_bounds__(kScanThreads)
scan_reduce_kernel(const u32* __restrict__ in, u64 n, u64* __restrict__ block_sums) {
    __shared__ u64 s_warp[33];
    const u64 base = (u64)blockIdx.x * kScanTile;
    u64 sum = 0;
#pragma unroll
    for (int j = 0; j < kScanPerThread; ++j) {
        const u64 i = base + (u64)j * kScanThreads + threadIdx.x;
        if (i < n) sum += in[i];
    }
    u64 total;
    block_exclusive_scan(sum, s_warp, total);
    if (threadIdx.x == 0) block_sums[blockIdx.x] = total;
}

// one block: exclusive scan of block_sums in place; total -> *total_out
__global__ void __launch_bounds__(1024)
scan_spine_kernel(u64* block_sums, u64 nblocks, u64* total_out) {
    __shared__ u64 s_warp[33];
    u64 carry = 0;
    for (u64 base = 0; base < nblocks; base += blockDim.x) {
        const u64 i = base + threadIdx.x;
        const u64 x = i < nblocks ? block_sums[i] : 0;
        u64 total;
        const u64 ex = block_exclusive_scan(x, s_warp, total);
        if (i < nblocks) block_sums[i] = carry + ex;
        carry += total;
    }
    if (threadIdx.x == 0) *total_out = carry;
}

__global__ void __launch_bounds__(kScanThreads)
scan_apply_kernel(const u32* __restrict__ in, u64 n, const u64* __restrict__ block_sums, u64* __restrict__ out) {
    __shared__ u64 s_warp[33];
    const u64 base = (u64)blockIdx.x * kScanTile + (u64)threadIdx.x * kScanPerThread;   // contiguous per thread
    u32 x[kScanPerThread];
    u64 sum = 0;
#pragma unroll
    for (int j = 0; j < kScanPerThread; ++j) {
        x[j] = (base + j < n) ? in[base + j] : 0u;
        sum += x[j];
    }
    u64 total;
    u64 run = block_sums[blockIdx.x] + block_exclusive_scan(sum, s_warp, total);
#pragma unroll
    for (int j = 0; j < kScanPerThread; ++j) {
        if (base + j < n) out[base + j] = run;
        run += x[j];
    }
}

// =========================================================================================
// K3  start nodes: bitmask + per-tile offsets -> slot values in input order
// =========================================================================================
// One warp per insert tile (kInsTile records = 32 mask words).
template <int W>
__global__ void __launch_bounds__(256)
scatter_starts_kernel(const unsigned char* __restrict__ recs, u64 n, int k,
                      const u32* __restrict__ start_mask, const u64* __restrict__ tile_offsets, u64 ntiles,
                      typename Slot<W>::value_t* __restrict__ starts_out, u64 out_base) {
    typedef Slot<W> S;
    const u64 tile = ((u64)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (tile >= ntiles) return;
    const int pl = (k + 3) >> 2, pb = pl + 2;
    const u64 word = tile * (kInsTile / 32) + lane_id();
    const u64 nwords = (n + 31) >> 5;
    u32 m = word < nwords ? start_mask[word] : 0u;
    // exclusive prefix of popcounts across the warp
    u32 inc = __popc(m);
    const u32 mine = inc;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const u32 y = __shfl_up_sync(kFullMask, inc, d);
        if (lane_id() >= (u32)d) inc += y;
    }
    u64 dst = out_base + tile_offsets[tile] + (inc - mine);
    while (m) {
        const int bit = __ffs(m) - 1;
        m &= m - 1;
        const u64 rec = (word << 5) + bit;
        bool ok;
        unsigned char tmp[18];
        const unsigned char* src = recs + rec * pb;
        for (int i = 0; i < pb; ++i) tmp[i] = src[i];
        starts_out[dst++] = S::from_record(tmp, k, pl, ok);
    }
}

// =========================================================================================
// K4  lookup
// =========================================================================================
template <int W>
__device__ __forceinline__ bool lookup(const typename Slot<W>::value_t* __restrict__ table, u64 nbuckets,
                                       typename Slot<W>::value_t keybits, typename Slot<W>::value_t& found,
                                       u64& bucket, int& slot) {
    typedef Slot<W> S;
    u64 b = place_bucket<W>(keybits, nbuckets);
    for (u64 tries = 0; tries < nbuckets; ++tries) {
        u64 q[4];
        load256_nc(table + b * S::kPerBucket, q);
        // Branch-free inside the bucket: every lane of a warp leaves the slot scan at the same instruction (returning
        // from inside the loop made the lanes exit at different slot indices, and everything after the lookup in
        // walk_kernel then ran with ~9 of ~24 live lanes -- profiles/r01_final_lines_walk_kernel.txt).
        bool hole = false, hit = false;
#pragma unroll
        for (int i = 0; i < S::kPerBucket; ++i) {
            const typename S::value_t cur = S::from_bucket(q, i);
            const bool e = S::empty(cur);             // buckets fill in order: the first hole ends the probe
            const bool m_ = !hole && !hit && !e && S::same_key(cur, keybits);
            if (m_) { found = cur; slot = i; }
            hit = hit || m_;
            hole = hole || e;
        }
        if (hit) { bucket = b; return true; }
        if (hole) return false;
        b = (b + 1 == nbuckets) ? 0 : b + 1;
    }
    return false;
}

template <int W>
__global__ void __launch_bounds__(256)
find_kernel(const typename Slot<W>::value_t* __restrict__ table, u64 nbuckets, int k,
            const unsigned char* __restrict__ pkmers, u64 n,
            unsigned char* __restrict__ pairs_out, unsigned char* __restrict__ found_out) {
    typedef Slot<W> S;
    const u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int pl = (k + 3) >> 2, pb = pl + 2;
    unsigned char key[16];
    for (int j = 0; j < pl; ++j) key[j] = pkmers[i * pl + j];
    typename S::value_t hit;
    u64 b; int s;
    const bool ok = lookup<W>(table, nbuckets, S::from_packed(key, k, pl), hit, b, s);
    unsigned char rec[18];
    for (int j = 0; j < pb; ++j) rec[j] = 0;
    if (ok) S::to_record(hit, k, pl, rec);
    for (int j = 0; j < pb; ++j) pairs_out[i * pb + j] = rec[j];
    found_out[i] = ok ? 1 : 0;
}

// =========================================================================================
// K5  walk: every k-mer is visited exactly once, by the lane that owns its segment
// =========================================================================================
// Walkers are (a) the start nodes, ids [0, n_starts), and (b) every `split_buckets`-th bucket's
// first slot ("splitters"), ids [n_starts, n_starts + n_split).  A walker follows successors
// (kmer_hash.cpp:44-51) and stops at forward ext 'F' or when the successor sits in a splitter
// slot -- that node belongs to the splitter's own walker.  So a chain of any length is cut into
// independent pieces of geometric length and no contig serialises on one lane; rank_kernel then
// stitches the pieces with pointer jumping.  Each piece's forward-extension characters go to
// tmp[seg * seg_chars ...]; a piece longer than seg_chars continues in an overflow segment.
//
//   link[seg] = (next segment id << 32) | chars in this segment     (kLinkTail: ends the contig)
struct WalkParams {
    const void* table;
    u64 nbuckets;
    const void* starts;
    u64* link;
    unsigned char* seglen;
    unsigned char* tmp;
    Counters* ctr;
    u32 n_starts;
    u32 n_split;
    u32 split_shift;      // split_buckets = 1 << split_shift
    u32 seg_chars;        // multiple of 8
    u32 seg_cap;          // capacity of link/seglen/tmp in segments
    int k;
};

constexpr u32 kWalkBatch = 128;     // walker ids a warp takes per global atomic
constexpr u32 kSegBatch = 32;       // overflow segment ids a warp takes per global atomic
constexpr int kWalkThreads = 256;

template <int W>
__global__ void __launch_bounds__(kWalkThreads)
walk_kernel(const WalkParams p) {
    typedef Slot<W> S;
    typedef typename S::value_t V;
    const V* __restrict__ table = static_cast<const V*>(p.table);
    const V* __restrict__ starts = static_cast<const V*>(p.starts);
    const u32 total = p.n_starts + p.n_split;
    const u32 lane = lane_id();
    const u32 lt_mask = (1u << lane) - 1u;
    const u64 split_mask = (1ull << p.split_shift) - 1ull;

    // warp-uniform pools
    u32 w_next = 0, w_end = 0;      // walker ids
    bool exhausted = false;
    u32 o_next = 0, o_end = 0;      // overflow segment ids

    // lane state
    bool active = false;
    V cur = S::zero(), chk = S::zero();
    u32 seg = 0, n = 0, steps = 0, limit = 256;
    u64 acc = 0;

    auto close = [&](u32 next) {
        if (n & 7u) *reinterpret_cast<u64*>(p.tmp + (u64)seg * p.seg_chars + (n & ~7u)) = acc;
        p.seglen[seg] = (unsigned char)n;
        p.link[seg] = ((u64)next << 32) | (next >= kLinkCtFirstMarker ? 0u : n);
        active = false;
    };

    for (;;) {
        __syncwarp();
        // ---- hand out new walkers to idle lanes ----
        const u32 idle = __ballot_sync(kFullMask, !active);
        if (idle && !exhausted) {
            if (w_next == w_end) {
                u32 base = 0;
                if (lane == 0) base = atomicAdd(&p.ctr->next_walker, kWalkBatch);
                base = __shfl_sync(kFullMask, base, 0);
                w_next = min(base, total);
                w_end = min(base + kWalkBatch, total);    // base + batch cannot wrap: total < 2^32 - batch*grid
                exhausted = (w_next == w_end);
            }
            const u32 avail = w_end - w_next;
            const u32 rank = __popc(idle & lt_mask);
            if (!active && rank < avail) {
                const u32 w = w_next + rank;
                seg = w; n = 0; acc = 0; steps = 0; limit = 256;
                if (w < p.n_starts) {
                    cur = starts[w];
                    active = true;
                } else {
                    const u64 b = (u64)(w - p.n_starts) << p.split_shift;
                    cur = S::load_one_nc(table + b * S::kPerBucket);
                    if (S::empty(cur)) p.link[seg] = (u64)kLinkUnused << 32;
                    else active = true;
                }
                chk = cur;
            }
            w_next += min((u32)__popc(idle), avail);
        }
        if (__ballot_sync(kFullMask, active) == 0) {
            if (exhausted) break;
            continue;
        }
        // ---- lanes whose segment buffer is full move to an overflow segment ----
        const u32 full = __ballot_sync(kFullMask, active && n == p.seg_chars && S::fwd(cur) != kExtF);
        if (full) {
            const u32 want = __popc(full);
            if (o_end - o_next < want) {
                // return nothing: leftover ids of the old pool are marked unused below
                for (u32 id = o_next + lane; id < o_end; id += 32) p.link[id] = (u64)kLinkUnused << 32;
                u32 base = 0;
                if (lane == 0) base = atomicAdd(&p.ctr->next_seg, kSegBatch);
                base = __shfl_sync(kFullMask, base, 0);
                o_next = base; o_end = base + kSegBatch;
            }
            if (full & (1u << lane)) {
                const u32 ns = o_next + __popc(full & lt_mask);
                if (ns >= p.seg_cap) {            // cannot happen when seg_cap is sized as in capi.cu
                    atomicOr(&p.ctr->errors, kErrInternal);
                    close(kLinkTail);
                } else {
                    close(ns);
                    active = true; seg = ns; n = 0; acc = 0;
                }
            }
            o_next += want;
        }
        // ---- one step of kmer_hash.cpp:44-51 per active lane ----
        if (active) {
            const u32 f = S::fwd(cur);
            if (f == kExtF) {
                close(kLinkTail);
            } else {
                acc |= (u64)ext_char(f) << (8u * (n & 7u));         // extract_contig: read_kmers.hpp:86-90
                ++n;
                if ((n & 7u) == 0) {
                    *reinterpret_cast<u64*>(p.tmp + (u64)seg * p.seg_chars + n - 8) = acc;
                    acc = 0;
                }
                V nxt; u64 b; int s;
                if (!lookup<W>(table, p.nbuckets, S::next_key(cur, p.k), nxt, b, s)) {
                    // kmer_hash.cpp:47-49 throws only for chains it walks: mark the segment, rank_kernel raises the
                    // error if a START-rooted contig ends here (a walker started at a splitter may sit on a chain no
                    // start node reaches, which the reference never visits)
                    close(kLinkMissing);
                } else if (s == 0 && (b & split_mask) == 0) {
                    close(p.n_starts + (u32)(b >> p.split_shift));  // the splitter's walker takes over
                } else {
                    cur = nxt;
                    // Brent: a splitter-free cycle would never end this segment
                    if (S::same_key(cur, chk)) {
                        close(kLinkLoop);                           // reported only if a start-rooted contig runs into it
                    } else if (++steps == limit) {
                        chk = cur; steps = 0; limit <<= 1;
                    }
                }
            }
        }
    }
    // ids left in this warp's overflow pool were never used
    for (u32 id = o_next + lane; id < o_end; id += 32)
        if (id < p.seg_cap) p.link[id] = (u64)kLinkUnused << 32;
}

// =========================================================================================
// rank: pointer jumping over segments, contig lengths, tail claims (cooperative launch)
// =========================================================================================
// Invariant: link[i] = (p, s) means "s characters lie between the start of segment i and the
// start of segment p".  Jumping replaces (p, s) by (link[p].p, s + link[p].s); any stale value
// read for link[p] is still a valid such pair, so the update is safe in place without double
// buffering.  A segment is final once its p is a tail.
struct RankParams {
    u64* link;
    const unsigned char* seglen;
    Counters* ctr;
    u32* contig_len;      // K + chars + 1 ('\n') per contig
    u32* contig_pre;      // characters before the tail segment starts
    u32 n_starts;
    u32 seg_cap;
    int k;
    int max_rounds;
};

__device__ __forceinline__ u64 ld_cg64(const u64* p) { return __ldcg(p); }

__global__ void __launch_bounds__(256)
rank_kernel(const RankParams p) {
    cg::grid_group grid = cg::this_grid();
    const u64 gtid = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    const u64 gsize = (u64)gridDim.x * blockDim.x;
    const u32 nseg = min(p.ctr->next_seg, p.seg_cap);
    int round = 0;
    for (; round < p.max_rounds; ++round) {
        bool changed = false;
        for (u64 i = gtid; i < nseg; i += gsize) {
            const u64 li = ld_cg64(p.link + i);
            const u32 pi = (u32)(li >> 32);
            if (pi >= kLinkCtFirstMarker || pi == (u32)i) continue;       // ends here / unused; a one-segment cycle never moves
            const u64 lp = ld_cg64(p.link + pi);
            const u32 pp = (u32)(lp >> 32);
            if (pp == kLinkTail || pp == kLinkMissing || pp == kLinkLoop) continue;      // final: pi is the chain's last segment
            if (pp >= kLinkCtFirstMarker) { atomicOr(&p.ctr->errors, kErrInternal); continue; }
            __stcg(p.link + i, ((u64)pp << 32) | (u32)((u32)li + (u32)lp));
            changed = true;
        }
        if (changed) p.ctr->flags[round] = 1;
        grid.sync();
        if (__ldcg(&p.ctr->flags[round]) == 0) break;
    }
    if (gtid == 0) p.ctr->rank_rounds = (u32)min(round + 1, p.max_rounds);
    grid.sync();
    // ---- contig lengths (kmer_hash.cpp:38-55: one contig per start node) ----
    u64 nodes = 0;
    for (u64 c = gtid; c < p.n_starts; c += gsize) {
        const u64 lc = ld_cg64(p.link + c);
        const u32 pc = (u32)(lc >> 32);
        u32 tail = (u32)c, pre = 0, end = pc;                // end = marker of the chain's last segment
        if (pc < kLinkCtFirstMarker) {
            tail = pc; pre = (u32)lc;
            end = (u32)(ld_cg64(p.link + pc) >> 32);
        }
        if (end != kLinkTail) {
            // a missing successor on a start-rooted chain (kmer_hash.cpp:47-49), or the chain runs into a cycle / is
            // still open after max_rounds (kmer_hash.cpp:44 never exits)
            atomicOr(&p.ctr->errors, end == kLinkMissing ? kErrNotFound : kErrCycle);
            p.contig_pre[c] = 0; p.contig_len[c] = 0;
            continue;
        }
        const u32 chars = pre + p.seglen[tail];
        p.contig_pre[c] = pre;
        p.contig_len[c] = (u32)p.k + chars + 1u;
        nodes += (u64)chars + 1u;
    }
    nodes = warp_sum_u64(nodes);
    if (lane_id() == 0 && nodes) atomicAdd(&p.ctr->n_nodes, nodes);
    grid.sync();
    // ---- each contig claims its tail so segments can find their contig ----
    for (u64 c = gtid; c < p.n_starts; c += gsize) {
        if (p.contig_len[c] == 0) continue;
        const u32 pc = (u32)(ld_cg64(p.link + c) >> 32);
        const u32 tail = (pc == kLinkTail) ? (u32)c : pc;
        const u64 want = (u64)kLinkTail << 32;
        const u64 old = atomicCAS(p.link + tail, want, ((u64)kLinkClaimed << 32) | (u32)c);
        if (old != want) atomicOr(&p.ctr->errors, kErrConverge);   // two starts, one end: not linear chains
    }
}

// =========================================================================================
// K6  emit
// =========================================================================================
// One thread resolves one segment's destination (32 independent metadata chains in flight per warp:
// link -> tail link -> contig_pre/off), then the warp copies the segments' characters cooperatively,
// one coalesced byte-run per segment, to contig_off[c] + K + position.
__global__ void __launch_bounds__(256)
emit_segments_kernel(const u64* __restrict__ link, const unsigned char* __restrict__ seglen,
                     const unsigned char* __restrict__ tmp, u32 seg_chars, u32 seg_cap, Counters* ctr,
                     const u32* __restrict__ contig_pre, const u64* __restrict__ contig_off,
                     int k, u64 out_cap, char* __restrict__ out) {
    // never write when the layout is not trustworthy (host reports the error)
    if (ctr->contig_bytes > out_cap || (ctr->errors & (kErrConverge | kErrCycle | kErrInternal))) return;
    const u64 seg = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    const u32 nseg = min(ctr->next_seg, seg_cap);
    u32 len = 0;
    u64 dst = 0;
    if (seg < nseg) {
        const u64 li = link[seg];
        const u32 pi = (u32)(li >> 32);
        if (pi < kLinkCtFirstMarker || pi == kLinkClaimed) {      // else: never walked / not on any start-rooted chain
            bool ok = true;
            u32 c = 0, pos = 0;
            if (pi == kLinkClaimed) {
                c = (u32)li;
                pos = contig_pre[c];
            } else {
                const u64 lt = link[pi];
                if ((u32)(lt >> 32) != kLinkClaimed) {
                    ok = false;                             // chain without a start node: ignored like the reference
                } else {
                    c = (u32)lt;
                    const u32 pre = contig_pre[c];
                    if ((u32)li > pre) { atomicOr(&ctr->errors, kErrConverge); ok = false; }
                    else pos = pre - (u32)li;
                }
            }
            if (ok) {
                len = seglen[seg];
                dst = contig_off[c] + (u64)k + pos;
            }
        }
    }
    u32 todo = __ballot_sync(kFullMask, len > 0);
    const u64 seg0 = seg - lane_id();
    while (todo) {
        const int src_lane = __ffs(todo) - 1;
        todo &= todo - 1;
        const u32 n = __shfl_sync(kFullMask, len, src_lane);
        const u64 d = __shfl_sync(kFullMask, dst, src_lane);
        const unsigned char* src = tmp + (seg0 + src_lane) * (u64)seg_chars;
        for (u32 j = lane_id(); j < n; j += 32) out[d + j] = (char)src[j];
    }
}

// first k-mer of each contig + trailing newline (read_kmers.hpp:84, kmer_hash.cpp:66)
template <int W>
__global__ void __launch_bounds__(256)
emit_heads_kernel(const typename Slot<W>::value_t* __restrict__ starts, u32 n_starts, int k,
                  const u32* __restrict__ contig_len, const u64* __restrict__ contig_off,
                  const Counters* __restrict__ ctr, u64 out_cap, char* __restrict__ out) {
    typedef Slot<W> S;
    if (ctr->contig_bytes > out_cap || (ctr->errors & (kErrConverge | kErrCycle | kErrInternal))) return;
    const u64 t = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    const u64 c = t / (u32)(k + 1);
    const u32 j = (u32)(t - c * (u32)(k + 1));
    if (c >= n_starts) return;
    const u32 len = contig_len[c];
    if (len == 0) return;
    if (j < (u32)k) out[contig_off[c] + j] = (char)ext_char(S::base_at(starts[c], k, (int)j));
    else out[contig_off[c] + len - 1] = '\n';
}

// =========================================================================================
// roofline helper: independent random 32-byte sector reads
// =========================================================================================
__global__ void __launch_bounds__(256)
random_sector_kernel(const u64* __restrict__ buf, u64 nsectors, u64 probes_per_thread, u64* sink) {
    const u64 tid = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    u64 x = 0, state = fmix64(tid + 0x1234567ull);
    for (u64 i = 0; i < probes_per_thread; i += 4) {
        u64 q[4][4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            state = state * 6364136223846793005ull + 1442695040888963407ull;
            load256_nc(buf + 4 * bucket_of(fmix64(state), nsectors), q[j]);
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) x ^= q[j][0] ^ q[j][1] ^ q[j][2] ^ q[j][3];
    }
    if (x == 0x9E3779B97F4A7C15ull) *sink = x;    // keep the loads alive
}

}  // namespace kh
