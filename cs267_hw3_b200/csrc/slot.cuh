// slot.cuh -- device-side key/slot format and the memory primitives every kernel shares.
//
// A table slot holds one reference `kmer_pair` (kmer_t.hpp:6-8) as a single integer so
// that ONE compare-and-swap publishes key and value together:
//
//     slot = (key << 6) | (backward_code << 3) | (forward_code + 1)
//
//   key           the k-mer as a right-justified base-4 number, first base most
//                 significant -- the same ordering as pkmer_t::data read big-endian
//                 (packing.hpp:50-92), minus the A-padding of the last byte
//   codes         A=0 C=1 G=2 T=3 F=4; forward is stored +1 so an occupied slot is
//                 never 0, and 0 means empty
//
// 2K+6 <= 64 for K <= 29 -> 64-bit slots (Slot<1>), 4 per 32-byte bucket;
// 2K+6 <= 128 for K <= 61 -> 128-bit slots (Slot<2>), 2 per 32-byte bucket.
// A bucket is exactly one 32-byte DRAM sector and is always read with one 256-bit load.
//
// kmer_pair::next_kmer() (kmer_t.hpp:51-53: unpack, substr(1)+fwd, repack) becomes
// ((key << 2) | fwd) & (4^K - 1) on this representation.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

namespace kh {

typedef unsigned long long u64;
typedef unsigned int u32;

constexpr u32 kExtF = 4;           // code of 'F'
constexpr u32 kExtBad = 7;

struct alignas(16) u128 {
    u64 lo, hi;
};

// Extension letter -> code, branch-free (a switch here diverges inside every record parse: it was ~24 % of
// partition_kernel's issued instructions).  The low five bits of the letter index a table of 3-bit codes:
// A(1)->0  C(3)->1  F(6)->4  G(7)->2  T(20)->3, kExtBad everywhere else.
constexpr u64 ext_lut_entry(u64 lut, int idx, u64 code) { return (lut & ~(7ull << (3 * idx))) | (code << (3 * idx)); }
constexpr u64 kExtLut = ext_lut_entry(ext_lut_entry(ext_lut_entry(ext_lut_entry(ext_lut_entry(
                            0x7FFFFFFFFFFFFFFFull, 1, 0), 3, 1), 6, 4), 7, 2), 20, 3);
__host__ __device__ __forceinline__ u32 ext_code(unsigned char c) {
    const u32 i = c & 31u;
    const bool letter = (c & 0xE0u) == 0x40u && i <= 20u;
    return letter ? ((u32)(kExtLut >> (3u * i)) & 7u) : kExtBad;
}
#ifdef __CUDACC__
// Eight / sixteen bytes starting at an arbitrarily aligned SHARED-memory address, as big-endian integers (byte 0 most
// significant), from aligned 32-bit loads + funnel shifts.  Reads up to 15 bytes past `p`'s last needed byte's word:
// callers stage records with 16 bytes of slack behind them.
__device__ __forceinline__ u64 lds_be64(const unsigned char* p) {
    const uintptr_t a = reinterpret_cast<uintptr_t>(p);
    const u32* w = reinterpret_cast<const u32*>(a & ~(uintptr_t)3);
    const u32 sh = ((u32)a & 3u) * 8u;
    const u32 w0 = w[0], w1 = w[1], w2 = w[2];
    const u32 b0 = __funnelshift_r(w0, w1, sh), b1 = __funnelshift_r(w1, w2, sh);      // bytes 0-3, 4-7 (little-endian words)
    return ((u64)__byte_perm(b0, 0, 0x0123) << 32) | (u64)__byte_perm(b1, 0, 0x0123);
}
__device__ __forceinline__ void lds_be128(const unsigned char* p, u64& hi, u64& lo) {
    const uintptr_t a = reinterpret_cast<uintptr_t>(p);
    const u32* w = reinterpret_cast<const u32*>(a & ~(uintptr_t)3);
    const u32 sh = ((u32)a & 3u) * 8u;
    const u32 w0 = w[0], w1 = w[1], w2 = w[2], w3 = w[3], w4 = w[4];
    const u32 b0 = __funnelshift_r(w0, w1, sh), b1 = __funnelshift_r(w1, w2, sh);
    const u32 b2 = __funnelshift_r(w2, w3, sh), b3 = __funnelshift_r(w3, w4, sh);
    hi = ((u64)__byte_perm(b0, 0, 0x0123) << 32) | (u64)__byte_perm(b1, 0, 0x0123);
    lo = ((u64)__byte_perm(b2, 0, 0x0123) << 32) | (u64)__byte_perm(b3, 0, 0x0123);
}
#endif
__host__ __device__ __forceinline__ unsigned char ext_char(u32 code) {
    // "ACGTF" packed little-endian
    return (unsigned char)((0x4654474341ull >> (8 * code)) & 0xFF);
}
// base letter -> 2-bit code without a table: (c>>1)&3 maps A,C,G,T to 0,1,3,2
__host__ __device__ __forceinline__ u32 base_code_fast(unsigned char c) {
    const u32 x = (c >> 1) & 3u;
    return x ^ (x >> 1);
}
__host__ __device__ __forceinline__ bool is_base(unsigned char c) {
    return c == 'A' || c == 'C' || c == 'G' || c == 'T';
}

__host__ __device__ __forceinline__ u64 fmix64(u64 z) {
    z ^= z >> 33; z *= 0xFF51AFD7ED558CCDull;
    z ^= z >> 33; z *= 0xC4CEB9FE1A85EC53ull;
    z ^= z >> 33;
    return z;
}

// ---- raw memory primitives -------------------------------------------------------------
// One 32-byte sector in one instruction (LDG.E.256 on sm_100a).
__device__ __forceinline__ void load256_nc(const void* p, u64 (&q)[4]) {   // read-only data, no L1 allocation
    asm volatile("ld.global.nc.L1::no_allocate.v4.u64 {%0,%1,%2,%3}, [%4];"
                 : "=l"(q[0]), "=l"(q[1]), "=l"(q[2]), "=l"(q[3]) : "l"(p));
}
__device__ __forceinline__ void load256_cg(const void* p, u64 (&q)[4]) {   // coherent at L2 (table being built)
    asm volatile("ld.global.cg.v4.u64 {%0,%1,%2,%3}, [%4];"
                 : "=l"(q[0]), "=l"(q[1]), "=l"(q[2]), "=l"(q[3]) : "l"(p) : "memory");
}
__device__ __forceinline__ uint4 load128_stream(const uint4* p) {           // streaming input, read once
    uint4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
    return r;
}
__device__ __forceinline__ u128 cas128(u128* addr, u128 cmp, u128 val) {    // ATOMG.E.CAS.128
    u128 old;
    asm volatile("{\n\t.reg .b128 c, v, o;\n\t"
                 "mov.b128 c, {%2, %3};\n\tmov.b128 v, {%4, %5};\n\t"
                 "atom.global.cas.b128 o, [%6], c, v;\n\t"
                 "mov.b128 {%0, %1}, o;\n\t}"
                 : "=l"(old.lo), "=l"(old.hi)
                 : "l"(cmp.lo), "l"(cmp.hi), "l"(val.lo), "l"(val.hi), "l"(addr) : "memory");
    return old;
}

// one 32-byte bucket of a table chunk held in SHARED memory: two LDS.128, re-read on every call (other threads CAS it)
__device__ __forceinline__ void lds_bucket(unsigned saddr, u64 (&q)[4]) {
    asm volatile("ld.volatile.shared.v2.u64 {%0,%1}, [%2];" : "=l"(q[0]), "=l"(q[1]) : "r"(saddr) : "memory");
    asm volatile("ld.volatile.shared.v2.u64 {%0,%1}, [%2+16];" : "=l"(q[2]), "=l"(q[3]) : "r"(saddr) : "memory");
}

// ---- slot traits -------------------------------------------------------------------------
template <int W> struct Slot;

template <> struct Slot<1> {
    typedef u64 value_t;
    static constexpr int kPerBucket = 4;

    static __host__ __device__ __forceinline__ value_t zero() { return 0ull; }
    static __host__ __device__ __forceinline__ bool empty(value_t v) { return v == 0ull; }
    static __host__ __device__ __forceinline__ u32 fwd(value_t v) { return (u32)(v & 7u) - 1u; }
    static __host__ __device__ __forceinline__ u32 back(value_t v) { return (u32)(v >> 3) & 7u; }
    static __host__ __device__ __forceinline__ bool same_key(value_t a, value_t b) { return ((a ^ b) >> 6) == 0ull; }
    static __host__ __device__ __forceinline__ value_t key_only(value_t v) { return v & ~63ull; }
    static __host__ __device__ __forceinline__ u64 hash(value_t v) { return fmix64(v >> 6); }
    static __device__ __forceinline__ value_t from_bucket(const u64 (&q)[4], int i) { return q[i]; }

    // kmer_pair bytes -> slot.  pl = (k+3)/4.
    static __host__ __device__ __forceinline__ value_t from_record(const unsigned char* rec, int k, int pl, bool& ok) {
        u64 be = 0;
        for (int i = 0; i < pl; ++i) be = (be << 8) | rec[i];
        const u64 key = be >> (8 * pl - 2 * k);
        const u32 b = ext_code(rec[pl]), f = ext_code(rec[pl + 1]);
        ok = (b != kExtBad) && (f != kExtBad);
        return (key << 6) | ((u64)(b & 7u) << 3) | (u64)((f + 1u) & 7u);
    }
#ifdef __CUDACC__
    // same, for a record staged in shared memory with >= 16 bytes of slack behind the staging area: the key comes
    // from three aligned word loads instead of a byte loop (the top 2K bits of the big-endian bytes ARE the key)
    static __device__ __forceinline__ value_t from_record_staged(const unsigned char* rec, int k, int pl, bool& ok) {
        const u64 key = lds_be64(rec) >> (64 - 2 * k);
        const u32 b = ext_code(rec[pl]), f = ext_code(rec[pl + 1]);
        ok = (b != kExtBad) && (f != kExtBad);
        return (key << 6) | ((u64)(b & 7u) << 3) | (u64)((f + 1u) & 7u);
    }
#endif
    // packed k-mer bytes (pkmer_t) -> key bits only (ext field 0)
    static __host__ __device__ __forceinline__ value_t from_packed(const unsigned char* p, int k, int pl) {
        u64 be = 0;
        for (int i = 0; i < pl; ++i) be = (be << 8) | p[i];
        return (be >> (8 * pl - 2 * k)) << 6;
    }
    static __host__ __device__ __forceinline__ void to_record(value_t v, int k, int pl, unsigned char* rec) {
        const u64 be = (v >> 6) << (8 * pl - 2 * k);
        for (int i = 0; i < pl; ++i) rec[i] = (unsigned char)(be >> (8 * (pl - 1 - i)));
        rec[pl] = ext_char(back(v));
        rec[pl + 1] = ext_char(fwd(v));
    }
    // key bits of kmer[1:] + fwd  (ext field 0)
    static __host__ __device__ __forceinline__ value_t next_key(value_t v, int k) {
        const u64 mask = ((2 * k + 6) >= 64) ? ~0ull : ((1ull << (2 * k + 6)) - 1ull);
        return ((((v & ~63ull) << 2) | ((u64)fwd(v) << 6)) & mask);
    }
    // 2-bit code of base i (0 = first)
    static __host__ __device__ __forceinline__ u32 base_at(value_t v, int k, int i) {
        return (u32)(v >> (6 + 2 * (k - 1 - i))) & 3u;
    }
    // key bits of backward_ext + kmer[:-1]  (kmer_pair::last_kmer, kmer_t.hpp:55-57); back must be a base
    static __host__ __device__ __forceinline__ value_t prev_key(value_t v, int k) {
        return ((((v >> 6) >> 2) | ((u64)back(v) << (2 * (k - 1)))) << 6);
    }
    static __device__ __forceinline__ value_t cas(value_t* addr, value_t expect, value_t val) {
        return atomicCAS(addr, expect, val);
    }
    static __device__ __forceinline__ value_t load_one_nc(const value_t* p) { return __ldg(p); }
    static __device__ __forceinline__ value_t cas_shared(value_t* addr, value_t expect, value_t val) {
        return atomicCAS(addr, expect, val);        // ATOMS.CAS.64
    }
};

template <> struct Slot<2> {
    typedef u128 value_t;
    static constexpr int kPerBucket = 2;

    static __host__ __device__ __forceinline__ value_t zero() { return u128{0ull, 0ull}; }
    static __host__ __device__ __forceinline__ bool empty(value_t v) { return (v.lo | v.hi) == 0ull; }
    static __host__ __device__ __forceinline__ u32 fwd(value_t v) { return (u32)(v.lo & 7u) - 1u; }
    static __host__ __device__ __forceinline__ u32 back(value_t v) { return (u32)(v.lo >> 3) & 7u; }
    static __host__ __device__ __forceinline__ bool same_key(value_t a, value_t b) {
        return (((a.lo ^ b.lo) >> 6) | (a.hi ^ b.hi)) == 0ull;
    }
    static __host__ __device__ __forceinline__ value_t key_only(value_t v) { return u128{v.lo & ~63ull, v.hi}; }
    static __host__ __device__ __forceinline__ u64 hash(value_t v) {
        return fmix64((v.lo >> 6) ^ fmix64(v.hi + 0x9E3779B97F4A7C15ull));
    }
    static __device__ __forceinline__ value_t from_bucket(const u64 (&q)[4], int i) { return u128{q[2 * i], q[2 * i + 1]}; }

    static __host__ __device__ __forceinline__ value_t shl(value_t v, int s) {   // 0 <= s < 64
        if (s == 0) return v;
        return u128{v.lo << s, (v.hi << s) | (v.lo >> (64 - s))};
    }
    static __host__ __device__ __forceinline__ value_t shr(value_t v, int s) {   // 0 <= s < 64
        if (s == 0) return v;
        return u128{(v.lo >> s) | (v.hi << (64 - s)), v.hi >> s};
    }
    static __host__ __device__ __forceinline__ value_t shr_any(value_t v, int s) {   // 0 <= s < 128
        return s >= 64 ? u128{v.hi >> (s - 64), 0ull} : shr(v, s);
    }
    static __host__ __device__ __forceinline__ value_t be_bytes(const unsigned char* p, int pl) {
        u128 x{0ull, 0ull};
        for (int i = 0; i < pl; ++i) {
            x.hi = (x.hi << 8) | (x.lo >> 56);
            x.lo = (x.lo << 8) | p[i];
        }
        return x;
    }
    static __host__ __device__ __forceinline__ value_t from_record(const unsigned char* rec, int k, int pl, bool& ok) {
        u128 v = shl(shr(be_bytes(rec, pl), 8 * pl - 2 * k), 6);
        const u32 b = ext_code(rec[pl]), f = ext_code(rec[pl + 1]);
        ok = (b != kExtBad) && (f != kExtBad);
        v.lo |= ((u64)(b & 7u) << 3) | (u64)((f + 1u) & 7u);
        return v;
    }
#ifdef __CUDACC__
    static __device__ __forceinline__ value_t from_record_staged(const unsigned char* rec, int k, int pl, bool& ok) {
        u64 hi, lo;
        lds_be128(rec, hi, lo);
        u128 v = shr_any(u128{lo, hi}, 122 - 2 * k);    // key << 6; 122 - 2K is 0..62 for K >= 30 and up to 88 for the short K a chunk table keeps in 128-bit slots
        const u32 b = ext_code(rec[pl]), f = ext_code(rec[pl + 1]);
        ok = (b != kExtBad) && (f != kExtBad);
        v.lo = (v.lo & ~63ull) | ((u64)(b & 7u) << 3) | (u64)((f + 1u) & 7u);
        return v;
    }
#endif
    static __host__ __device__ __forceinline__ value_t from_packed(const unsigned char* p, int k, int pl) {
        return shl(shr(be_bytes(p, pl), 8 * pl - 2 * k), 6);
    }
    static __host__ __device__ __forceinline__ void to_record(value_t v, int k, int pl, unsigned char* rec) {
        const u128 be = shl(shr(v, 6), 8 * pl - 2 * k);
        for (int i = 0; i < pl; ++i) {
            const int sh = 8 * (pl - 1 - i);
            rec[i] = (unsigned char)(sh >= 64 ? (be.hi >> (sh - 64)) : (be.lo >> sh));
        }
        rec[pl] = ext_char(back(v));
        rec[pl + 1] = ext_char(fwd(v));
    }
    static __host__ __device__ __forceinline__ value_t next_key(value_t v, int k) {
        u128 n = shl(u128{v.lo & ~63ull, v.hi}, 2);
        n.lo |= (u64)fwd(v) << 6;
        const int bits = 2 * k + 6;            // 66..128 for K in 30..61; below 64 for the short K a chunk table keeps in 128-bit slots
        if (bits <= 64) { n.hi = 0ull; if (bits < 64) n.lo &= (1ull << bits) - 1ull; }
        else if (bits < 128) n.hi &= (1ull << (bits - 64)) - 1ull;
        return n;
    }
    static __host__ __device__ __forceinline__ u32 base_at(value_t v, int k, int i) {
        const int sh = 6 + 2 * (k - 1 - i);
        return (u32)(sh >= 64 ? (v.hi >> (sh - 64)) : (v.lo >> sh)) & 3u;
    }
    static __host__ __device__ __forceinline__ value_t prev_key(value_t v, int k) {
        u128 key = shr(shr(v, 6), 2);                       // drop ext bits, drop the last base
        const int sh = 2 * (k - 1);                          // 58..120 for K in 30..61
        if (sh >= 64) key.hi |= (u64)back(v) << (sh - 64); else key.lo |= (u64)back(v) << sh;
        return shl(key, 6);
    }
    static __device__ __forceinline__ value_t cas(value_t* addr, value_t expect, value_t val) {
        return cas128(addr, expect, val);
    }
    static __device__ __forceinline__ value_t load_one_nc(const value_t* p) {
        const uint4 r = load128_stream(reinterpret_cast<const uint4*>(p));
        return u128{(u64)r.x | ((u64)r.y << 32), (u64)r.z | ((u64)r.w << 32)};
    }
    static __device__ __forceinline__ value_t cas_shared(value_t* addr, value_t expect, value_t val) {   // ATOMS.CAS.128
        u128 old;
        const unsigned saddr = (unsigned)__cvta_generic_to_shared(addr);
        asm volatile("{\n\t.reg .b128 c, v, o;\n\tmov.b128 c, {%2, %3};\n\tmov.b128 v, {%4, %5};\n\t"
                     "atom.shared.cas.b128 o, [%6], c, v;\n\tmov.b128 {%0, %1}, o;\n\t}"
                     : "=l"(old.lo), "=l"(old.hi)
                     : "l"(expect.lo), "l"(expect.hi), "l"(val.lo), "l"(val.hi), "r"(saddr) : "memory");
        return old;
    }
};


// ---- placement of the plain table: where a k-mer lives --------------------------------------------
// hash -> bucket without requiring a power-of-two table (load-factor sweeps need exact sizes)
__host__ __device__ __forceinline__ u64 bucket_of(u64 h, u64 nbuckets) {
#ifdef __CUDA_ARCH__
    return __umul64hi(h, nbuckets);
#else
    return (u64)(((unsigned __int128)h * nbuckets) >> 64);
#endif
}

// Home bucket of a k-mer: a hash of the key; probing is linear from there.
template <int W>
__host__ __device__ __forceinline__ u64 place_bucket(typename Slot<W>::value_t v, u64 nbuckets) {
    return bucket_of(Slot<W>::hash(v), nbuckets);
}

// =============================================================================================
// Chunk table ("ctable", ctable.cuh): placement by minimizer at CHUNK granularity
// =============================================================================================
// The home CHUNK of a k-mer -- a run of buckets that one thread block builds in shared memory -- is a hash of
// the k-mer's minimizer; the bucket inside the chunk is a hash of the key.  Consecutive k-mers of a contig
// share their minimizer for a "supermer" (~(w+1)/2 k-mers for a window of w m-mers), so they live in the same
// chunk and their successor links are followed in shared memory while the chunk is built; only one lookup per
// supermer ever goes to HBM (tools/probes/chunk_placement_sim.cpp is the CPU gate for balance and run length).
//
// The minimizer is the m-mer (m <= 16, so it fits 32 bits) with the smallest value of (x ^ seed) * odd among
// the `win` RIGHTMOST m-mers of the k-mer (win <= 32); that value is a bijection of the m-mer, so the minimum
// itself identifies the minimizer and is what gets hashed.
constexpr u32 kIdxBits = 14;                     // top bits of a ctable slot: 1 + index of the segment that STARTS at this k-mer (0: none)
constexpr u32 kMinMul = 0x9E3779B1u;             // odd: x -> x * kMinMul is a bijection of the m-mers
constexpr u32 kMinAdd = 0x7F4A7C15u;             // moves poly-A (x = 0) away from the bottom of the order

__host__ __device__ __forceinline__ int ct_minimizer_len(int k) { return k >= 31 ? 15 : (k >= 23 ? 13 : (k >= 17 ? k - 6 : k)); }
__host__ __device__ __forceinline__ int ct_window(int k) { const int w = k - ct_minimizer_len(k) + 1; return w > 32 ? 32 : w; }
// K range the chunk table supports: the slot must have kIdxBits spare bits above the key, and the window must be worth it
__host__ __device__ __forceinline__ bool ct_supported(int k) { return k >= 17 && k <= 54; }
__host__ __device__ __forceinline__ int ct_slot_words(int k) { return (2 * k + 6 + (int)kIdxBits <= 64) ? 1 : 2; }

__host__ __device__ __forceinline__ u32 ct_funnel_r(u32 lo, u32 hi, u32 s) {          // bits [s, s+32) of hi:lo, 0 <= s < 32
#ifdef __CUDA_ARCH__
    return __funnelshift_r(lo, hi, s);
#else
    return s ? ((lo >> s) | (hi << (32 - s))) : lo;
#endif
}
__host__ __device__ __forceinline__ u32 ct_mulhi32(u32 a, u32 b) {
#ifdef __CUDA_ARCH__
    return __umulhi(a, b);
#else
    return (u32)(((u64)a * b) >> 32);
#endif
}
// Order value of the m-mer in the low 2m bits of a 16-base window w: (w mod 4^m) * odd, moved to the top of the word
// -- the shift drops the bases of the window that are not part of the m-mer, so no mask is needed.  Three
// instructions per window position on the GPU (funnel shift, multiply-add, minimum).
// key words: a = bits 0..31 of the key (the LAST bases), b, c, d the following 32-bit words
__host__ __device__ __forceinline__ u32 ct_min_hash_words(u32 a, u32 b, u32 c, u32 d, int m, int win) {
    const u32 mul = kMinMul << (32 - 2 * m);          // m <= 16
    u32 best = 0xFFFFFFFFu;
    int rem = win;
    for (int it = 0; it < 2; ++it) {
        if (rem >= 16) {
#pragma unroll
            for (int j = 0; j < 16; ++j) {
                const u32 h = ct_funnel_r(a, b, 2u * j) * mul + kMinAdd;
                best = h < best ? h : best;
            }
        } else {
#pragma unroll
            for (int j = 0; j < 16; ++j) {
                u32 h = ct_funnel_r(a, b, 2u * j) * mul + kMinAdd;
                h = (j < rem) ? h : 0xFFFFFFFFu;
                best = h < best ? h : best;
            }
        }
        if (rem <= 16) break;
        rem -= 16; a = b; b = c; c = d; d = 0;
    }
    return best;
}
template <int W> __host__ __device__ __forceinline__ u32 ct_min_hash(typename Slot<W>::value_t v, int m, int win);
template <> __host__ __device__ __forceinline__ u32 ct_min_hash<1>(u64 v, int m, int win) {      // v: key << 6, no index bits
    const u64 key = v >> 6;
    return ct_min_hash_words((u32)key, (u32)(key >> 32), 0u, 0u, m, win);
}
template <> __host__ __device__ __forceinline__ u32 ct_min_hash<2>(u128 v, int m, int win) {
    const u64 lo = (v.lo >> 6) | (v.hi << 58), hi = v.hi >> 6;
    return ct_min_hash_words((u32)lo, (u32)(lo >> 32), (u32)hi, (u32)(hi >> 32), m, win);
}

// slot helpers that know about the index bits
__host__ __device__ __forceinline__ u32 ct_fmix32_hi(u32 h) {       // finaliser whose HIGH bits are used (range reduction by mulhi)
    h ^= h >> 15; h *= 0x85EBCA6Bu;
    h ^= h >> 13; h *= 0xC2B2AE35u;
    return h;
}
template <int W> struct CtSlot;
template <> struct CtSlot<1> {
    typedef u64 V;
    static __host__ __device__ __forceinline__ V strip(V v) { return v & (~0ull >> kIdxBits); }
    static __host__ __device__ __forceinline__ u32 idx(V v) { return (u32)(v >> (64 - kIdxBits)); }
    static __host__ __device__ __forceinline__ V with_idx(V v, u32 i) { return strip(v) | ((u64)i << (64 - kIdxBits)); }
    static __host__ __device__ __forceinline__ bool same_key(V a, V b) { return (((a ^ b) << kIdxBits) >> (kIdxBits + 6)) == 0ull; }
    // bucket hash of the key bits of a slot value (extension and index bits ignored): 32-bit multiplies only
    static __host__ __device__ __forceinline__ u32 hash32(V v) {
        const u32 x0 = (u32)v & ~63u, x1 = (u32)(v >> 32) & (0xFFFFFFFFu >> kIdxBits);
        return ct_fmix32_hi((x0 * 0x9E3779B1u) ^ x1);
    }
};
template <> struct CtSlot<2> {
    typedef u128 V;
    static __host__ __device__ __forceinline__ V strip(V v) { return u128{v.lo, v.hi & (~0ull >> kIdxBits)}; }
    static __host__ __device__ __forceinline__ u32 idx(V v) { return (u32)(v.hi >> (64 - kIdxBits)); }
    static __host__ __device__ __forceinline__ V with_idx(V v, u32 i) { return u128{v.lo, (v.hi & (~0ull >> kIdxBits)) | ((u64)i << (64 - kIdxBits))}; }
    static __host__ __device__ __forceinline__ bool same_key(V a, V b) { return (((a.hi ^ b.hi) << kIdxBits) | ((a.lo ^ b.lo) >> 6)) == 0ull; }
    static __host__ __device__ __forceinline__ u32 hash32(V v) {
        const u32 x0 = (u32)v.lo & ~63u, x1 = (u32)(v.lo >> 32), x2 = (u32)v.hi, x3 = (u32)(v.hi >> 32) & (0xFFFFFFFFu >> kIdxBits);
        u32 h = x0 * 0x9E3779B1u;
        h = (h ^ x1) * 0x85EBCA77u;
        h = (h ^ x2) * 0xC2B2AE3Du;
        return ct_fmix32_hi(h ^ x3);
    }
};
// bucket inside a chunk of nb buckets
__host__ __device__ __forceinline__ u32 ct_bucket_in_chunk(u32 h32, u32 nb) { return ct_mulhi32(h32, nb); }

// chunk geometry shared by host and device
struct CtGeom {
    int k, m, win;
    int world, rank;
    u32 chunks_per_rank;        // C: rank r owns the global chunks [r * C, (r + 1) * C)
    u32 max_buckets;            // buckets a chunk may have (shared-memory budget of the build kernel)
    u32 lf_inv_q16;             // 65536 / load factor
};
// minimizer hash -> (owner rank, local chunk) without a division: u * world = owner . fraction, and the global chunk
// floor(u * world * C / 2^32) lies in the owner's range because floor(floor(x C) / C) = floor(x)
__host__ __device__ __forceinline__ void ct_place(u32 minhash, const CtGeom& g, u32& owner, u32& chunk) {
    const u32 u = ct_fmix32_hi(minhash ^ (minhash >> 16));       // the minimum of a window is biased towards 0: remix before reducing
    owner = ct_mulhi32(u, (u32)g.world);
    chunk = ct_mulhi32(u, (u32)g.world * g.chunks_per_rank) - owner * g.chunks_per_rank;
}

// multi-GPU: global segment id = (rank << kRankShift) | local id
constexpr int kMaxRanks = 8;
constexpr u32 kRankShift = 28;
constexpr u32 kLocalMask = (1u << kRankShift) - 1u;
// pointer jumping: a link whose pointer already is its chain's last segment is flagged in the top bit of the distance
// word, so later rounds do not pay a (possibly remote) read for it
constexpr u32 kLinkFinalBit = 0x80000000u;
constexpr u32 kLinkDistMask = 0x7FFFFFFFu;
constexpr u32 kLinkMissing = 0xFFFFFFFBu;   // ctable: the successor k-mer is in no table (raised only if a start-rooted contig ends here)
constexpr u32 kLinkConverge = 0xFFFFFFFAu;  // ctable: the successor k-mer sits in the middle of another segment (it has two predecessors)
constexpr u32 kLinkLoop = kLinkConverge;        // plain table: the walker found itself on a cycle (same value, different path)
constexpr u32 kLinkCtFirstMarker = kLinkConverge;

// Error bits accumulated on the device (Counters::errors)
enum : u32 {
    kErrNotFound = 1u, kErrTableFull = 2u, kErrCycle = 4u, kErrBadInput = 8u,
    kErrConverge = 16u, kErrInternal = 32u
};

constexpr u32 kLinkTail = 0xFFFFFFFFu;      // segment ends a contig (forward ext 'F')
constexpr u32 kLinkUnused = 0xFFFFFFFEu;    // id never walked
constexpr u32 kLinkClaimed = 0xFFFFFFFDu;   // tail claimed by a contig; low word = contig id
constexpr u32 kLinkPending = 0xFFFFFFFCu;   // sharded walk: successor lives on another GPU, link not resolved yet

// where a kErrInternal came from (Counters::err_where)
enum : u32 { kSiteBarrier = 1u, kSiteStarts = 2u, kSiteSegCap = 4u, kSiteInbox = 8u, kSiteStubOpen = 16u, kSiteOutCap = 32u };

struct Counters {
    u32 next_walker;
    u32 next_seg;
    u32 errors;
    u32 rank_rounds;
    u64 n_inserted;
    u64 n_duplicates;
    u64 scan_total;       // result of the last device scan (start nodes of the last insert call)
    u64 n_nodes;
    u64 contig_bytes;
    u32 n_outbox;         // plain table, chunked build: records the chunks could not place (the overflow list)
    u32 flags[40];
    u32 rank_done;        // ctable: no rank moved a link in the last pointer-jumping round (agreed on by all ranks)
    u32 err_where;        // ctable: which capacity / wait raised kErrInternal (CtSite bits), for the error message
    u64 n_starts_dev;     // ctable: start nodes registered so far (kept on the device: no host round trip per insert)
    u32 need_jump;        // ctable: a contig of this rank is too long for the bounded walk
    u32 use_jump;         // ctable: some rank said so (agreed on at a barrier): rank by pointer jumping instead
};

}  // namespace kh
