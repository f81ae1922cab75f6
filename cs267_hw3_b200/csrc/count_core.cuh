// count_core.cuh -- k-mer analysis: reads -> unique k-mers with their backward / forward extensions.
//
// The stage BEFORE the reference's path (README.md:19-21: "the output of this first preprocessing stage ... is a set of
// unique DNA sequence fragments of length k ... each k-mer is associated with a forward and backward extension"); its
// output is what read_kmers (read_kmers.hpp:54-79) parses from text.  Produced here on the GPU, in the reference's
// kmer_pair bytes (kmer_t.hpp:6-8), it feeds kh_insert_pairs_device without the text round trip (SURVEY.md 8f-4).
// The reference has no code for this stage; the definition below is restated on the CPU by the test oracle.
//
// Definition.  A base is one of 'A' 'C' 'G' 'T'; any other byte separates reads.  Every position whose K bytes are
// bases is an occurrence of that k-mer; the byte before it / after it, when it is a base, is its backward / forward
// observation.  Per distinct k-mer the table keeps saturating counters in ONE 64-bit word, updated by one
// compare-and-swap per occurrence:
//     bits  0..7    occurrences                (saturates at 255, as k-mer counters conventionally do)
//     bits  8..35   backward A, C, G, T        (7 bits each, saturate at 127)
//     bits 36..63   forward  A, C, G, T
// A k-mer is reported when occurrences >= min_count; an extension is the base that alone reaches min_ext on its side,
// 'F' when none does (a contig begins / ends here: README.md:37) or several do (a fork).  No reverse complements --
// the reference has none either (kmer_t.hpp:51-57).
//
// Table: open addressing, linear probing over slots of 16 bytes (K <= 31: key tag | counters) or 32 bytes = one DRAM
// sector (K <= 61: key lo | key hi + occupied bit | counters | unused).  A slot's key is claimed with one 64- / 128-bit
// CAS and never changes; an occurrence then costs the sector read plus one CAS on the counter word in the same sector.
//
// Everything algorithmic in this file is __host__ __device__: tests/native/count_host_check.cu runs the very same
// functions tile by tile on the CPU (plain memory operations instead of atomics) against the oracle.
#pragma once
#include <cstring>

#include "slot.cuh"

namespace kh {

constexpr int kKcThreads = 256;
constexpr int kKcPer = 8;                                   // positions per thread
constexpr u32 kKcTile = kKcThreads * kKcPer;                // 2048 positions per block
// A tile's characters are packed 16 per 32-bit word (2 bits each, first character in bits 31..30).  Word i covers the
// characters [t0 - 16 + 16 i, t0 + 16 i): one word of left halo (the backward observation of the tile's first
// position), the tile, and four words of right halo (K + 1 <= 62 characters behind the tile's last position).
constexpr u32 kKcWords = kKcTile / 16 + 5;

constexpr u32 kKcCountCap = 255, kKcExtCap = 127;
constexpr u32 kKcErrFull = 1u;
constexpr u64 kKcMaxProbes = 1ull << 16;                     // a probe sequence this long means the table is (as good as) full

struct KcCounters {
    u64 n_occurrences;       // positions counted so far
    u64 n_distinct;          // slots claimed so far
    u64 n_reported;          // records written by the last extract
    u32 errors;
    u32 pad;
};

template <int W> struct KcSlot;
template <> struct KcSlot<1> { static constexpr int kWords = 2; };       // 16 bytes
template <> struct KcSlot<2> { static constexpr int kWords = 4; };       // 32 bytes
__host__ __device__ __forceinline__ int kc_slot_words(int k) { return k <= 31 ? 1 : 2; }

// ---- memory operations: atomics on the device, plain accesses in the serial host check --------------------------
__host__ __device__ __forceinline__ u64 kc_cas64(u64* p, u64 cmp, u64 val) {
#ifdef __CUDA_ARCH__
    return atomicCAS(p, cmp, val);
#else
    const u64 old = *p;
    if (old == cmp) *p = val;
    return old;
#endif
}
__host__ __device__ __forceinline__ u128 kc_cas128(u64* p, u128 cmp, u128 val) {
#ifdef __CUDA_ARCH__
    return cas128(reinterpret_cast<u128*>(p), cmp, val);
#else
    u128 old{p[0], p[1]};
    if (old.lo == cmp.lo && old.hi == cmp.hi) { p[0] = val.lo; p[1] = val.hi; }
    return old;
#endif
}
// a slot while other threads may be claiming / counting it: read at L2, never from a stale L1 line
template <int W> __host__ __device__ __forceinline__ void kc_load_slot(const u64* p, u64 (&q)[4]) {
#ifdef __CUDA_ARCH__
    if (W == 1) {
        asm volatile("ld.global.cg.v2.u64 {%0,%1}, [%2];" : "=l"(q[0]), "=l"(q[1]) : "l"(p) : "memory");
        q[2] = q[3] = 0ull;
    } else {
        load256_cg(p, q);
    }
#else
    for (int i = 0; i < KcSlot<W>::kWords; ++i) q[i] = p[i];
    for (int i = KcSlot<W>::kWords; i < 4; ++i) q[i] = 0ull;
#endif
}
__host__ __device__ __forceinline__ u64 kc_mulhi64(u64 a, u64 b) {
#ifdef __CUDA_ARCH__
    return __umul64hi(a, b);
#else
    return (u64)(((unsigned __int128)a * b) >> 64);
#endif
}
__host__ __device__ __forceinline__ u32 kc_funnel_l(u32 hi, u32 lo, u32 s) {       // top 32 bits of (hi:lo) << s, s in 0..31
#ifdef __CUDA_ARCH__
    return __funnelshift_l(lo, hi, s);
#else
    return s ? (hi << s) | (lo >> (32u - s)) : hi;
#endif
}

// Host-side chunking of a long read buffer: chunk ci covers the positions [off, off + len) and travels as the bytes [a, b)
// -- 16 in front of it (keeps 16-byte alignment of the tile words) and 64 behind it -- so that k-mers straddling a chunk
// boundary are cut exactly as in one piece.  `chunk` is a multiple of the tile.  The kernel then runs on that piece with
// p_begin = off - a, p_end = p_begin + len.
inline void kc_chunk_range(u64 ci, u64 chunk, u64 n_bytes, u64& a, u64& b, u64& off, u64& len) {
    off = ci * chunk;
    len = n_bytes - off < chunk ? n_bytes - off : chunk;
    a = off ? off - 16 : 0;
    b = off + len + 64 < n_bytes ? off + len + 64 : n_bytes;
}

// ---- text -> packed tile ------------------------------------------------------------------------------------
// Word of 16 characters starting at buffer offset c0 (may reach outside [0, n): those positions separate reads).
// code: 2 bits per character, first character in bits 31..30; inv: the same shape, 11 where the byte is not a base.
__host__ __device__ __forceinline__ void kc_pack_word(const unsigned char* buf, u64 n, long long c0, u32& code, u32& inv) {
    u32 w[4];
    if (c0 >= 0 && (u64)c0 + 16u <= n && ((reinterpret_cast<uintptr_t>(buf) + (u64)c0) & 15u) == 0u) {
#ifdef __CUDA_ARCH__
        const uint4 v = load128_stream(reinterpret_cast<const uint4*>(buf + c0));
        w[0] = v.x; w[1] = v.y; w[2] = v.z; w[3] = v.w;
#else
        memcpy(w, buf + c0, 16);
#endif
    } else {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            u32 x = 0;
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const long long p = c0 + 4 * j + i;
                const u32 ch = (p >= 0 && (u64)p < n) ? (u32)buf[p] : (u32)'\n';
                x |= ch << (8 * i);
            }
            w[j] = x;
        }
    }
    code = 0; inv = 0;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const unsigned char ch = (unsigned char)(w[j] >> (8 * i));
            const bool ok = is_base(ch);
            code = (code << 2) | (ok ? base_code_fast(ch) : 0u);
            inv = (inv << 2) | (ok ? 0u : 3u);
        }
    }
}

// 64 characters of a packed stream starting at character s (word s / 16, bit 2 * (s % 16)), first character on top
struct KcWin { u64 hi, lo; };
__host__ __device__ __forceinline__ KcWin kc_window(const u32* w, u32 s) {
    const u32 j = s >> 4, sh = 2u * (s & 15u);
    const u32 y0 = kc_funnel_l(w[j], w[j + 1], sh), y1 = kc_funnel_l(w[j + 1], w[j + 2], sh);
    const u32 y2 = kc_funnel_l(w[j + 2], w[j + 3], sh), y3 = kc_funnel_l(w[j + 3], w[j + 4], sh);
    return KcWin{((u64)y0 << 32) | y1, ((u64)y2 << 32) | y3};
}

// One position of a tile.  `local` = position - t0 (0 .. kKcTile-1); stream character 16 + local is the k-mer's first
// base, the one before it the backward observation, the one K behind it the forward observation.
struct KcOcc {
    u64 key_hi, key_lo;      // the k-mer as a right-justified base-4 number, first base most significant (slot.cuh)
    u32 back, fwd;           // 0..3 = A C G T, 4 = none
};
__host__ __device__ __forceinline__ u32 kc_char_bad(const u32* s_inv, u32 c) { return (s_inv[c >> 4] >> (30u - 2u * (c & 15u))) & 3u; }
// (pass 2; the position is known to hold a k-mer, kc_kmer_valid)
__host__ __device__ __forceinline__ KcOcc kc_position(const u32* s_code, const u32* s_inv, u32 local, int k) {
    const u32 s = 15u + local;
    const KcWin y = kc_window(s_code, s);
    // drop character 0 (the backward observation): the k-mer is on top
    const u64 zh = (y.hi << 2) | (y.lo >> 62), zl = y.lo << 2;
    const int kb = 2 * k;                                   // 4 .. 122
    KcOcc o;
    u32 f;
    if (kb <= 64) {
        o.key_hi = 0ull;
        o.key_lo = zh >> (64 - kb);
    } else {
        const int s2 = 128 - kb;                            // 6 .. 62
        o.key_hi = zh >> s2;
        o.key_lo = (zh << (64 - s2)) | (zl >> s2);
    }
    if (kb <= 62) f = (u32)(zh >> (62 - kb)) & 3u;
    else          f = (u32)(zl >> (126 - kb)) & 3u;
    o.back = kc_char_bad(s_inv, s) ? 4u : (u32)(y.hi >> 62);
    o.fwd = kc_char_bad(s_inv, s + (u32)k + 1u) ? 4u : f;
    return o;
}

// pass 1 of a tile: does position `local` hold a k-mer (all K bytes are bases)?  Only the mask stream is looked at.
__host__ __device__ __forceinline__ bool kc_kmer_valid(const u32* s_inv, u32 local, int k) {
    const KcWin v = kc_window(s_inv, 15u + local);
    const u64 vh = (v.hi << 2) | (v.lo >> 62), vl = v.lo << 2;
    const int kb = 2 * k;
    return kb <= 64 ? (vh >> (64 - kb)) == 0ull : (vh == 0ull && (vl >> (128 - kb)) == 0ull);
}

// ---- the counter word -------------------------------------------------------------------------------------------
__host__ __device__ __forceinline__ u32 kc_total(u64 c) { return (u32)(c & 0xFFu); }
__host__ __device__ __forceinline__ u32 kc_back_count(u64 c, u32 base) { return (u32)(c >> (8u + 7u * base)) & 127u; }
__host__ __device__ __forceinline__ u32 kc_fwd_count(u64 c, u32 base) { return (u32)(c >> (36u + 7u * base)) & 127u; }
__host__ __device__ __forceinline__ u64 kc_bump(u64 c, u32 back, u32 fwd) {
    u64 n = c;
    if (kc_total(c) < kKcCountCap) n += 1ull;
    if (back < 4u && kc_back_count(c, back) < kKcExtCap) n += 1ull << (8u + 7u * back);
    if (fwd < 4u && kc_fwd_count(c, fwd) < kKcExtCap) n += 1ull << (36u + 7u * fwd);
    return n;
}
// saturating update of the counter word at p; `c` = what the slot read saw there
__host__ __device__ __forceinline__ void kc_count(u64* p, u64 c, u32 back, u32 fwd) {
    for (;;) {
        const u64 n = kc_bump(c, back, fwd);
        if (n == c) return;                                 // everything this occurrence touches is saturated
        const u64 old = kc_cas64(p, c, n);
        if (old == c) return;
        c = old;
    }
}
// the extension letter of one side (shift 8: backward, 36: forward)
__host__ __device__ __forceinline__ unsigned char kc_pick(u64 c, u32 shift, u32 min_ext) {
    u32 pick = kExtF, nq = 0;
#pragma unroll
    for (u32 b = 0; b < 4u; ++b) {
        const bool q = ((u32)(c >> (shift + 7u * b)) & 127u) >= min_ext;
        pick = q ? b : pick;
        nq += q ? 1u : 0u;
    }
    return ext_char(nq == 1u ? pick : kExtF);
}

// ---- the table --------------------------------------------------------------------------------------------------
__host__ __device__ __forceinline__ u64 kc_hash(u64 key_hi, u64 key_lo) {
    return fmix64(key_lo ^ (key_hi * 0x9E3779B97F4A7C15ull));          // K <= 32: key_hi = 0, the plain finaliser
}
template <int W> __host__ __device__ __forceinline__ void kc_tag(u64 key_hi, u64 key_lo, u64& t0, u64& t1);
template <> __host__ __device__ __forceinline__ void kc_tag<1>(u64, u64 key_lo, u64& t0, u64& t1) { t0 = (key_lo << 1) | 1ull; t1 = 0ull; }
template <> __host__ __device__ __forceinline__ void kc_tag<2>(u64 key_hi, u64 key_lo, u64& t0, u64& t1) { t0 = key_lo; t1 = key_hi | (1ull << 63); }
template <int W> __host__ __device__ __forceinline__ bool kc_slot_empty(const u64 (&q)[4]) { return W == 1 ? q[0] == 0ull : q[1] == 0ull; }
template <int W> __host__ __device__ __forceinline__ bool kc_slot_is(const u64 (&q)[4], u64 t0, u64 t1) {
    return W == 1 ? q[0] == t0 : (q[0] == t0 && q[1] == t1);
}
template <int W> __host__ __device__ __forceinline__ u64 kc_slot_counters(const u64 (&q)[4]) { return W == 1 ? q[1] : q[2]; }

// the slot a k-mer's probe sequence starts at
__host__ __device__ __forceinline__ u64 kc_home(u64 key_hi, u64 key_lo, u64 n_slots) { return kc_mulhi64(kc_hash(key_hi, key_lo), n_slots); }
// one occurrence: find or claim the k-mer's slot (probing from its home slot s), count.  Returns false when the table is full.
template <int W>
__host__ __device__ __forceinline__ bool kc_upsert(u64* table, u64 n_slots, const KcOcc& o, u64 s, bool& fresh) {
    u64 t0, t1;
    kc_tag<W>(o.key_hi, o.key_lo, t0, t1);
    fresh = false;
    for (u64 tries = 0, lim = n_slots < kKcMaxProbes ? n_slots : kKcMaxProbes; tries < lim; ++tries) {
        u64* p = table + s * (u64)KcSlot<W>::kWords;
        u64 q[4];
        kc_load_slot<W>(p, q);
        if (kc_slot_empty<W>(q)) {                          // claim it; whoever wins the CAS owns the key of this slot for good
            if (W == 1) {
                const u64 old = kc_cas64(p, 0ull, t0);
                if (old == 0ull) { fresh = true; q[0] = t0; } else q[0] = old;
            } else {
                const u128 old = kc_cas128(p, u128{0ull, 0ull}, u128{t0, t1});
                if (old.lo == 0ull && old.hi == 0ull) { fresh = true; q[0] = t0; q[1] = t1; } else { q[0] = old.lo; q[1] = old.hi; }
            }
        }
        if (kc_slot_is<W>(q, t0, t1)) {
            kc_count(p + (W == 1 ? 1 : 2), kc_slot_counters<W>(q), o.back, o.fwd);
            return true;
        }
        s = (s + 1 == n_slots) ? 0ull : s + 1;
    }
    return false;
}

// read-only probe of the finished table: the counter word of a k-mer, 0 when it was never seen
template <int W>
__host__ __device__ __forceinline__ u64 kc_find(const u64* table, u64 n_slots, u64 key_hi, u64 key_lo) {
    u64 t0, t1;
    kc_tag<W>(key_hi, key_lo, t0, t1);
    u64 s = kc_home(key_hi, key_lo, n_slots);
    for (u64 tries = 0, lim = n_slots < kKcMaxProbes ? n_slots : kKcMaxProbes; tries < lim; ++tries) {
        const u64* p = table + s * (u64)KcSlot<W>::kWords;
        u64 q[4] = {p[0], p[1], W == 1 ? 0ull : p[2], 0ull};
        if (kc_slot_empty<W>(q)) return 0ull;
        if (kc_slot_is<W>(q, t0, t1)) return kc_slot_counters<W>(q);
        s = (s + 1 == n_slots) ? 0ull : s + 1;
    }
    return 0ull;
}

// growing the table: slot i of the old table (if occupied) moves to the new one -- its key claims a slot by CAS (other
// keys are moving in at the same time), its counter word is stored (keys are unique: nobody else touches that word).
// Returns false when the new table is full (it is sized so that it cannot be).
template <int W>
__host__ __device__ __forceinline__ bool kc_move_slot(const u64* old_table, u64 i, u64* table, u64 n_slots) {
    const u64* src = old_table + i * (u64)KcSlot<W>::kWords;
    const u64 q0[4] = {src[0], src[1], W == 1 ? 0ull : src[2], 0ull};
    if (kc_slot_empty<W>(q0)) return true;
    const u64 t0 = q0[0], t1 = W == 1 ? 0ull : q0[1], counters = kc_slot_counters<W>(q0);
    const u64 key_lo = W == 1 ? t0 >> 1 : t0, key_hi = W == 1 ? 0ull : t1 & ~(1ull << 63);
    u64 s = kc_home(key_hi, key_lo, n_slots);
    for (u64 tries = 0, lim = n_slots < kKcMaxProbes ? n_slots : kKcMaxProbes; tries < lim; ++tries) {
        u64* p = table + s * (u64)KcSlot<W>::kWords;
        u64 q[4];
        kc_load_slot<W>(p, q);
        if (kc_slot_empty<W>(q)) {
            bool mine;
            if (W == 1) mine = kc_cas64(p, 0ull, t0) == 0ull;
            else { const u128 old = kc_cas128(p, u128{0ull, 0ull}, u128{t0, t1}); mine = old.lo == 0ull && old.hi == 0ull; }
            if (mine) { p[W == 1 ? 1 : 2] = counters; return true; }
        }
        s = (s + 1 == n_slots) ? 0ull : s + 1;
    }
    return false;
}

// ---- merging tables (sharded counting: one table per rank, every k-mer reduced at its owner rank) ----------------
// Every field of the counter word saturates, and min(cap, min(cap, a) + min(cap, b)) = min(cap, a + b): adding the words
// of per-rank tables field by field with saturation gives exactly the word one table over all reads would hold, in any
// order and grouping -- provided nothing was dropped before the merge and no k-mer or observation straddles two ranks.
constexpr u32 kKcMaxWorld = 64;

// Owner rank of a k-mer: a second mix of kc_hash, independent of its top bits (kc_home takes those).  Were the owner
// drawn from the top bits too, the keys of one owner would all have their home slot in 1/world of its table.  Depends
// on the key and world only, never on a table size.
__host__ __device__ __forceinline__ u32 kc_owner(u64 key_hi, u64 key_lo, u32 world) {
    return (u32)kc_mulhi64(fmix64(kc_hash(key_hi, key_lo) ^ 0xD6E8FEB86659FD93ull), (u64)world);
}
// per-field saturating sum of two counter words (occurrences at 255, each of the 8 observation counts at 127); no carry
// crosses a field border
__host__ __device__ __forceinline__ u64 kc_add(u64 a, u64 b) {
    u64 t = (a & 0xFFull) + (b & 0xFFull);
    u64 r = t > kKcCountCap ? kKcCountCap : t;
#pragma unroll
    for (u32 f = 0; f < 8u; ++f) {
        const u32 s = 8u + 7u * f;
        t = ((a >> s) & 127ull) + ((b >> s) & 127ull);
        r |= (t > kKcExtCap ? (u64)kKcExtCap : t) << s;
    }
    return r;
}
__host__ __device__ __forceinline__ void kc_tag_key(int W, u64 t0, u64 t1, u64& key_hi, u64& key_lo) {
    key_lo = W == 1 ? t0 >> 1 : t0;
    key_hi = W == 1 ? 0ull : t1 & ~(1ull << 63);
}
// slot i: its owner rank, or `world` when the slot is empty
template <int W>
__host__ __device__ __forceinline__ u32 kc_slot_owner(const u64* table, u64 i, u32 world) {
    const u64* p = table + i * (u64)KcSlot<W>::kWords;
    const u64 q[4] = {p[0], p[1], 0ull, 0ull};
    if (kc_slot_empty<W>(q)) return world;
    u64 kh_, kl_;
    kc_tag_key(W, q[0], q[1], kh_, kl_);
    return kc_owner(kh_, kl_, world);
}
// One record -- a slot of another table of the same K, copied verbatim -- merged into this table: find or claim the key's
// slot (as kc_move_slot / kc_upsert do), then add the counter word with kc_add in a CAS loop: one launch may carry the
// same key from several source tables.  Returns false when the table is full.
template <int W>
__host__ __device__ __forceinline__ bool kc_merge_slot(u64* table, u64 n_slots, const u64* rec, bool& fresh) {
    const u64 t0 = rec[0], t1 = W == 1 ? 0ull : rec[1], add = rec[W == 1 ? 1 : 2];
    u64 key_hi, key_lo;
    kc_tag_key(W, t0, t1, key_hi, key_lo);
    u64 s = kc_home(key_hi, key_lo, n_slots);
    fresh = false;
    for (u64 tries = 0, lim = n_slots < kKcMaxProbes ? n_slots : kKcMaxProbes; tries < lim; ++tries) {
        u64* p = table + s * (u64)KcSlot<W>::kWords;
        u64 q[4];
        kc_load_slot<W>(p, q);
        if (kc_slot_empty<W>(q)) {
            if (W == 1) {
                const u64 old = kc_cas64(p, 0ull, t0);
                if (old == 0ull) { fresh = true; q[0] = t0; } else q[0] = old;
            } else {
                const u128 old = kc_cas128(p, u128{0ull, 0ull}, u128{t0, t1});
                if (old.lo == 0ull && old.hi == 0ull) { fresh = true; q[0] = t0; q[1] = t1; } else { q[0] = old.lo; q[1] = old.hi; }
            }
        }
        if (kc_slot_is<W>(q, t0, t1)) {
            u64* w = p + (W == 1 ? 1 : 2);
            u64 c = kc_slot_counters<W>(q);
            for (;;) {
                const u64 n = kc_add(c, add);
                if (n == c) return true;
                const u64 old = kc_cas64(w, c, n);
                if (old == c) return true;
                c = old;
            }
        }
        s = (s + 1 == n_slots) ? 0ull : s + 1;
    }
    return false;
}

// ---- k-mer <-> the reference's packed bytes (packing.hpp:77-92: first base in bits 7..6 of byte 0, A-padded tail) ---
__host__ __device__ __forceinline__ void kc_key_to_packed(u64 key_hi, u64 key_lo, int k, unsigned char* out) {
    const int pl = (k + 3) >> 2, sh = 8 * pl - 2 * k;       // 0, 2, 4 or 6 bits of padding
    const u64 hi = sh ? (key_hi << sh) | (key_lo >> (64 - sh)) : key_hi, lo = key_lo << sh;
    for (int i = 0; i < pl; ++i) {
        const int bit = 8 * (pl - 1 - i);
        out[i] = (unsigned char)(bit >= 64 ? hi >> (bit - 64) : lo >> bit);
    }
}
__host__ __device__ __forceinline__ void kc_packed_to_key(const unsigned char* in, int k, u64& key_hi, u64& key_lo) {
    const int pl = (k + 3) >> 2, sh = 8 * pl - 2 * k;
    u64 hi = 0, lo = 0;
    for (int i = 0; i < pl; ++i) {
        hi = (hi << 8) | (lo >> 56);
        lo = (lo << 8) | (u64)in[i];
    }
    key_lo = sh ? (lo >> sh) | (hi << (64 - sh)) : lo;
    key_hi = hi >> sh;
}

// slot i of the finished table: is it a reported k-mer, and its record (kmer_pair bytes: packed k-mer, backward, forward)
template <int W>
__host__ __device__ __forceinline__ bool kc_slot_reported(const u64* table, u64 i, u32 min_count) {
    const u64* p = table + i * (u64)KcSlot<W>::kWords;
    const u64 q[4] = {p[0], p[1], W == 1 ? 0ull : p[2], 0ull};
    return !kc_slot_empty<W>(q) && kc_total(kc_slot_counters<W>(q)) >= min_count;
}
// slot i of the finished table: the occurrences of its k-mer (saturated at 255), 0 for an empty slot -- its spectrum bin
template <int W>
__host__ __device__ __forceinline__ u32 kc_slot_total(const u64* table, u64 i) {
    const u64* p = table + i * (u64)KcSlot<W>::kWords;
    const u64 q[4] = {p[0], p[1], W == 1 ? 0ull : p[2], 0ull};
    return kc_slot_empty<W>(q) ? 0u : kc_total(kc_slot_counters<W>(q));
}

// ---- the k-mer spectrum -----------------------------------------------------------------------------------------
// hist[c] (c = 1..254): distinct k-mers counted exactly c times; hist[255]: those seen 255 times or more; hist[0] = 0.
constexpr u32 kKcHistBins = 256;
constexpr u32 kKcDefaultMinCount = 2;
// The valley rule: reads with sequencing errors give a falling slope of erroneous k-mers (count 1, 2, ...) that meets the
// coverage peak of the true ones; the first c where the spectrum stops falling (hist[c+1] >= hist[c]) separates them.
// That c is the threshold when it is >= 2 and k-mers remain at or above it; otherwise (no falling slope -- error-free reads,
// an empty table -- or a spectrum that falls to zero with no second peak) the default 2.
inline u32 kc_auto_min_count(const u64* hist) {
    if (!hist) return kKcDefaultMinCount;
    for (u32 c = 1; c + 1 < kKcHistBins; ++c) {
        if (hist[c + 1] < hist[c]) continue;
        if (c < 2) return kKcDefaultMinCount;
        u64 above = 0;
        for (u32 d = c; d < kKcHistBins; ++d) above += hist[d];
        return above > 0 ? c : kKcDefaultMinCount;
    }
    return kKcDefaultMinCount;
}
// ---- contig depth (kh_count_contig_depth*) ---------------------------------------------------------------------
// Contig c is the text [offsets[c], offsets[c+1]); a window is a position p with p + K <= offsets[c+1] whose K bytes are
// bases; its value is the k-mer's occurrence count (kc_total, 0 when never seen).  Per contig: windows, sum, min, max --
// the layout of kh_contig_depth.  Partials of disjoint window sets (the owners' of a sharded counter) combine field by
// field: +, +, min, max.
struct KcDepth {
    u64 n_kmers, sum;
    u32 min, max;
};
constexpr u32 kKcDepthNoMin = 0xFFFFFFFFu;
constexpr u64 kKcNoContig = ~0ull;                          // the sentinel contig of a lane without a window

// The contig holding byte p: the largest c in [lo, hi) with offsets[c] <= p (empty contigs share their offset with the
// next one, so the largest is the one the byte belongs to).  Needs offsets[lo] <= p; returns lo when no c qualifies.
__host__ __device__ __forceinline__ u64 kc_contig_of(const u64* offsets, u64 lo, u64 hi, u64 p) {
    while (hi - lo > 1) {
        const u64 mid = lo + (hi - lo) / 2;
        if (offsets[mid] <= p) lo = mid;
        else hi = mid;
    }
    return lo;
}
// the window at byte p (all K bytes are bases) belongs to contig c when it starts inside it and ends by its end
__host__ __device__ __forceinline__ bool kc_window_in_contig(const u64* offsets, u64 c, u64 p, int k) {
    return offsets[c] <= p && p + (u64)k <= offsets[c + 1];
}
// the value of one window: its k-mer's occurrences, read-only
template <int W>
__host__ __device__ __forceinline__ u32 kc_depth_value(const u64* table, u64 n_slots, u64 key_hi, u64 key_lo) {
    return kc_total(kc_find<W>(table, n_slots, key_hi, key_lo));
}

template <int W>
__host__ __device__ __forceinline__ void kc_slot_record(const u64* table, u64 i, int k, u32 min_ext, unsigned char* rec) {
    const u64* p = table + i * (u64)KcSlot<W>::kWords;
    const u64 key_lo = W == 1 ? p[0] >> 1 : p[0], key_hi = W == 1 ? 0ull : p[1] & ~(1ull << 63);
    const u64 c = W == 1 ? p[1] : p[2];
    const int pl = (k + 3) >> 2;
    kc_key_to_packed(key_hi, key_lo, k, rec);
    rec[pl] = kc_pick(c, 8u, min_ext);                      // kmer_t.hpp:43-45: fb_ext[0] backward, [1] forward
    rec[pl + 1] = kc_pick(c, 36u, min_ext);
}

// ---- unitig extensions (kh_count_link_check*) --------------------------------------------------------------------
// S = the k-mers the counter reports at (min_count, min_ext), each with its raw extensions (kc_pick at min_ext).  For a
// record x = (s, b, f): f is kept iff f != 'F', y = s[1..K-1] f is in S and y's raw backward extension is s[0]; b is kept
// iff b != 'F', w = b s[0..K-2] is in S and w's raw forward extension is s[K-1].  Otherwise the side becomes 'F'.  The rule
// is symmetric (x -> y kept iff y <- x kept), so on checked records every k-mer has at most one successor and one
// predecessor, each naming it back: paths (unitigs, one start each) and isolated cycles.  world > 1: only sides whose
// neighbour `rank` owns (kc_owner) are looked at; the others stay as they are.  A cut only ever writes 'F', so the owners'
// partials applied one after another in any order give the world = 1 records.
//
// Split in three so that the kernel can keep both lookups in flight: kc_link_plan (the record -> the neighbour keys to
// look up), kc_find_pair (both lookups, probing side by side), kc_link_apply (the counter words -> the checked sides).
struct KcLinkPlan {
    u64 key_hi[2], key_lo[2];        // [0] = successor y, [1] = predecessor w
    u32 want[2];                     // the base the neighbour must name back: s[0] (for y) and s[K-1] (for w)
    bool look[2];                    // side not 'F' and owned by `rank`: the neighbour is looked up
    bool bad;                        // an extension byte outside ACGTF
};

// the record's K-mer (rec: packed k-mer, backward, forward) -> the plan
__host__ __device__ __forceinline__ KcLinkPlan kc_link_plan(const unsigned char* rec, int k, u32 world, u32 rank) {
    const int pl = (k + 3) >> 2, kb = 2 * k;
    u64 hi, lo;
    kc_packed_to_key(rec, k, hi, lo);
    const u32 b = ext_code(rec[pl]), f = ext_code(rec[pl + 1]);
    KcLinkPlan p;
    p.bad = b > kExtF || f > kExtF;
    p.want[0] = kb - 2 >= 64 ? (u32)(hi >> (kb - 66)) & 3u : (u32)(lo >> (kb - 2)) & 3u;             // s[0]
    p.want[1] = (u32)lo & 3u;                                                                           // s[K-1]
    // y = ((s << 2) | f) mod 4^K
    u64 yh = (hi << 2) | (lo >> 62), yl = (lo << 2) | (f & 3u);
    if (kb <= 64) { yh = 0ull; yl &= kb == 64 ? ~0ull : (1ull << kb) - 1ull; }
    else yh &= (1ull << (kb - 64)) - 1ull;
    // w = (s >> 2) | b 4^(K-1)
    u64 wh = hi >> 2, wl = (lo >> 2) | (hi << 62);
    if (kb - 2 >= 64) wh |= (u64)(b & 3u) << (kb - 66);
    else wl |= (u64)(b & 3u) << (kb - 2);
    p.key_hi[0] = yh; p.key_lo[0] = yl;
    p.key_hi[1] = wh; p.key_lo[1] = wl;
    p.look[0] = !p.bad && f < kExtF && (world == 1 || kc_owner(yh, yl, world) == rank);
    p.look[1] = !p.bad && b < kExtF && (world == 1 || kc_owner(wh, wl, world) == rank);
    return p;
}

// kc_find for the keys the plan looks up (0 for the others), both probe sequences advanced side by side: the two slot
// reads of one step are independent, so a thread has both in flight
template <int W>
__host__ __device__ __forceinline__ void kc_find_pair(const u64* table, u64 n_slots, const KcLinkPlan& p, u64 (&c)[2]) {
    u64 t0[2], t1[2], s[2];
    bool live[2];
#pragma unroll
    for (int j = 0; j < 2; ++j) {
        kc_tag<W>(p.key_hi[j], p.key_lo[j], t0[j], t1[j]);
        s[j] = kc_home(p.key_hi[j], p.key_lo[j], n_slots);
        live[j] = p.look[j];
        c[j] = 0ull;
    }
    for (u64 tries = 0, lim = n_slots < kKcMaxProbes ? n_slots : kKcMaxProbes; tries < lim && (live[0] || live[1]); ++tries) {
        u64 q[2][4];
#pragma unroll
        for (int j = 0; j < 2; ++j) {
            const u64* a = table + (live[j] ? s[j] : 0ull) * (u64)KcSlot<W>::kWords;
            q[j][0] = a[0]; q[j][1] = a[1]; q[j][2] = W == 1 ? 0ull : a[2]; q[j][3] = 0ull;
        }
#pragma unroll
        for (int j = 0; j < 2; ++j) {
            if (!live[j]) continue;
            if (kc_slot_empty<W>(q[j])) live[j] = false;
            else if (kc_slot_is<W>(q[j], t0[j], t1[j])) { c[j] = kc_slot_counters<W>(q[j]); live[j] = false; }
            else s[j] = (s[j] + 1 == n_slots) ? 0ull : s[j] + 1;
        }
    }
}

// The checked sides written into rec (sides not looked up stay); returns the number of sides turned to 'F' (0..2)
__host__ __device__ __forceinline__ u32 kc_link_apply(const KcLinkPlan& p, const u64 (&c)[2], int k, u32 min_count, u32 min_ext,
                                                      unsigned char* rec) {
    const int pl = (k + 3) >> 2;
    u32 cut = 0;
    // y must name s[0] backward; w must name s[K-1] forward
    if (p.look[0] && !(kc_total(c[0]) >= min_count && kc_pick(c[0], 8u, min_ext) == ext_char(p.want[0]))) { rec[pl + 1] = 'F'; ++cut; }
    if (p.look[1] && !(kc_total(c[1]) >= min_count && kc_pick(c[1], 36u, min_ext) == ext_char(p.want[1]))) { rec[pl] = 'F'; ++cut; }
    return cut;
}

}  // namespace kh

#include "../../include/kh/record_line.hpp"
