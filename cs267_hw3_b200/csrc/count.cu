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
    void* inbox = nullptr;            // kh_count_merge_device: records copied over from another device
    size_t inbox_cap = 0;
    void* cursor = nullptr;           // kh_count_partition: per-owner counts / write cursors
    size_t cursor_cap = 0;
    void* hist = nullptr;             // kh_count_histogram: 256 x u64 bins
    size_t hist_cap = 0;
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
    cudaFree(c->outbox); cudaFree(c->inbox); cudaFree(c->cursor); cudaFree(c->hist);
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
    cudaPointerAttributes a{};
    if (cudaPointerGetAttributes(&a, records_dev) != cudaSuccess || (a.type != cudaMemoryTypeDevice && a.type != cudaMemoryTypeManaged)) {
        cudaGetLastError();
        return kc_fail(c, KH_ERR_ARG, "kh_count_merge_device: records_dev is not device memory");
    }
    const u64 rb = c->W == 1 ? 16 : 32;
    const u64* src = static_cast<const u64*>(records_dev);
    if (a.type == cudaMemoryTypeDevice && a.device != c->device) {
        // another GPU's records: one copy into this counter's inbox, peer to peer where the devices allow it
        if (a.device >= 0 && a.device < 64 && !((c->peers_enabled >> a.device) & 1ull)) {
            int can = 0;
            if (cudaDeviceCanAccessPeer(&can, c->device, a.device) == cudaSuccess && can) {
                const cudaError_t e = cudaDeviceEnablePeerAccess(a.device, 0);
                if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) KC_CUDA(c, e);
                cudaGetLastError();
            }
            c->peers_enabled |= 1ull << a.device;
        }
        KC_TRY(kc_grow(c, &c->inbox, &c->inbox_cap, (size_t)(n * rb)));
        KC_CUDA(c, cudaMemcpyAsync(c->inbox, records_dev, (size_t)(n * rb), cudaMemcpyDefault, c->stream));
        src = static_cast<const u64*>(c->inbox);
    }
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
