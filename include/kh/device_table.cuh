// kh/device_table.cuh -- device-side find / insert on a libkh_b200 table, for CUDA code that wants the table inside its
// own kernels instead of through batch calls (SURVEY.md 8(f) rank 3; the per-k-mer HashMap::insert / find of the
// assignment text, README.md:95-99, as __device__ functions).
//
//     kh_device_view v;  kh_get_device_view(table, &v);          // host, include/kh_capi.h
//     my_kernel<<<...>>>(v, ...);                                  // pass it by value
//     __device__: kh::device_find(v, pkmer_bytes, pair_out)        // DistributedHashMap::find   (hash_map.hpp:83-92)
//                 kh::device_insert(v, kmer_pair_bytes)            // DistributedHashMap::insert_locally (hash_map.hpp:33-35)
//
// Keys and records cross in the reference's byte layouts (pkmer_t / kmer_pair, kmer_t.hpp:6-8, packing.hpp:50-92), the
// same as on the C ABI.  Works on PLAIN tables (every table that is not a chunk table: kh_get_device_view says so);
// a chunk table is built in one piece when it is sealed and has no single-record insert -- use kh_find / kh_insert_pairs.
// Inserts made here are visible to kh_find and to other device_find calls at once; start nodes are NOT recorded
// (kh_assemble walks from the start nodes that kh_insert_pairs / kh_insert_lines saw), and the host-side counters
// (kh_stats.n_inserted) do not include them.
#pragma once
#include "../kh_capi.h"
#include "../../cs267_hw3_b200/csrc/kernels.cuh"

namespace kh {

enum { kDevInserted = 0, kDevDuplicate = 1, kDevFull = 2, kDevBadInput = 3 };

template <int W>
__device__ __forceinline__ bool device_find_w(const kh_device_view& v, const unsigned char* pkmer, unsigned char* pair_out) {
    typedef Slot<W> S;
    const int pl = (v.k + 3) >> 2;
    const typename S::value_t key = S::from_packed(pkmer, v.k, pl);
    typename S::value_t hit;
    u64 b;
    int s;
    if (!lookup<W>(static_cast<const typename S::value_t*>(v.table), v.n_buckets, key, hit, b, s)) return false;
    if (pair_out) S::to_record(hit, v.k, pl, pair_out);
    return true;
}
template <int W>
__device__ __forceinline__ int device_insert_w(const kh_device_view& v, const unsigned char* pair) {
    typedef Slot<W> S;
    typedef typename S::value_t V;
    const int pl = (v.k + 3) >> 2;
    bool ok = true;
    const V val = S::from_record(pair, v.k, pl, ok);
    if (!ok) return kDevBadInput;
    V* table = static_cast<V*>(v.table);
    const u64 b = place_bucket<W>(val, v.n_buckets);
    u64 q[4];
    load256_cg(table + b * S::kPerBucket, q);
    const int rc = insert_one<W>(table, v.n_buckets, b, val, q);
    return rc == kInsInserted ? kDevInserted : (rc == kInsDuplicate ? kDevDuplicate : kDevFull);
}

// pkmer: (K+3)/4 packed bytes; pair_out: (K+3)/4 + 2 bytes or nullptr
__device__ __forceinline__ bool device_find(const kh_device_view& v, const unsigned char* pkmer, unsigned char* pair_out) {
    return v.slot_bytes == 8 ? device_find_w<1>(v, pkmer, pair_out) : device_find_w<2>(v, pkmer, pair_out);
}
// pair: (K+3)/4 + 2 bytes (kmer_pair).  First record of a k-mer wins, as everywhere in this library.
__device__ __forceinline__ int device_insert(const kh_device_view& v, const unsigned char* pair) {
    return v.slot_bytes == 8 ? device_insert_w<1>(v, pair) : device_insert_w<2>(v, pair);
}

}  // namespace kh
