/* kh_capi.h -- C ABI of the B200 k-mer hash table + contig traversal library
 * (libkh_b200.so, built from cs267_hw3_b200/csrc/ for sm_100a).
 *
 * This is the drop-in boundary for ONE stage of fractalclockwork/CS267_HW3: the timed
 * region of kmer_hash.cpp:129-137 (insert all k-mers, find the start nodes, walk every
 * contig) plus the packing that feeds it.  Plain C: opaque handle, pointers and sizes,
 * int status codes, no C++ types, no exceptions, no torch types.  The C++ headers in
 * include/ (hash_map.hpp, kmer_t.hpp, ...) and the kmer_hash CLI are thin host code
 * over these calls; INTEGRATION.md shows the binding a reference maintainer would add.
 *
 * Record format on the wire is the reference's own `kmer_pair` bytes (kmer_t.hpp:6-8):
 *   (K+3)/4 packed bytes  -- 2 bits per base, A=0 C=1 G=2 T=3, first base in bits 7..6
 *                            of byte 0, tail padded with A (packing.hpp:50-92)
 *   1 byte backward ext, 1 byte forward ext, ASCII in {A,C,G,T,F} (kmer_t.hpp:43-45)
 * i.e. 7 / 10 / 15 bytes for K = 19 / 31 / 51, alignment 1.  The device-side slot
 * format is private.  Supported K: 2..61 (64-bit or 128-bit slots, chosen by the library).
 *
 * There is no CPU fallback: every entry point that computes needs a CUDA device and
 * returns KH_ERR_CUDA without one.
 *
 * Threading: a handle is not re-entrant; use one handle per host thread / per GPU.
 * Unless stated otherwise calls are synchronous with respect to the host for their
 * host-visible results; *_device variants only enqueue work on the handle's stream.
 */
#ifndef KH_CAPI_H
#define KH_CAPI_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct kh_table kh_table;

enum kh_status {
    KH_OK = 0,
    KH_ERR_ARG = 1,          /* bad argument (null pointer, unsupported K, ...) */
    KH_ERR_CUDA = 2,         /* CUDA runtime failure, or no device; see kh_last_error */
    KH_ERR_NOT_FOUND = 3,    /* a successor k-mer is missing: kmer_hash.cpp:47-49
                                "Error: k-mer not found in Distributed HashMap." */
    KH_ERR_TABLE_FULL = 4,   /* more distinct k-mers than slots */
    KH_ERR_CYCLE = 5,        /* a start-rooted chain never reaches forward ext 'F'
                                (the reference would spin forever, kmer_hash.cpp:44) */
    KH_ERR_BAD_INPUT = 6,    /* base outside ACGT / ext outside ACGTF / malformed line
                                (undefined behaviour in the reference, packing.hpp:52-70) */
    KH_ERR_CONVERGE = 7,     /* two start nodes reach the same end node (not a set of
                                linear chains; violates README.md:33-35) */
    KH_ERR_NOMEM = 8         /* device or pinned-host allocation failed */
};

/* Per-handle counters and stage times of the most recent calls (milliseconds are CUDA-event
 * times on the handle's stream). */
typedef struct kh_stats {
    uint64_t n_slots;          /* table capacity in slots                                   */
    uint64_t n_buckets;        /* 32-byte buckets (4 x 64-bit or 2 x 128-bit slots)         */
    uint64_t n_inserted;       /* records accepted since create/clear (duplicates excluded) */
    uint64_t n_duplicates;     /* records whose k-mer was already present (first one kept;
                                  the reference keeps the last, hash_map.hpp:34 -- identical
                                  for the unique inputs README.md:33-35 guarantees)         */
    uint64_t n_starts;         /* records seen with backward ext 'F'                        */
    uint64_t n_contigs;        /* last assemble                                             */
    uint64_t n_nodes;          /* last assemble: k-mers on emitted contigs                  */
    uint64_t contig_bytes;     /* last assemble: bytes of contig text incl. '\n' each       */
    uint64_t n_segments;       /* last assemble: walk segments (start + splitter + overflow)*/
    uint32_t rank_rounds;      /* last assemble: pointer-jumping rounds                     */
    uint32_t slot_bits;        /* 64 or 128                                                 */
    float ms_insert;           /* last insert call: insert kernel + start-node compaction   */
    float ms_assemble;         /* last assemble: walk + rank + emit                         */
    float ms_walk, ms_rank, ms_emit;
    float ms_pack;             /* last kh_pack_lines* call                                  */
    float ms_clear;            /* last kh_clear                                             */
    float ms_build;            /* chunk table: the build + contract kernel of the last seal  */
    float ms_stage;            /* chunk table: first insert call .. end of the last staging  */
    uint64_t n_launches;       /* kernels this handle has launched since kh_create          */
} kh_stats;

int kh_abi_version(void);                 /* bumps when this header changes incompatibly */
int kh_device_count(void);                /* 0 when no CUDA device is usable             */
const char* kh_status_string(int status);
uint64_t kh_pair_bytes(int k);            /* sizeof(kmer_pair) for this K: (K+3)/4 + 2   */
uint64_t kh_packed_bytes(int k);          /* sizeof(pkmer_t): (K+3)/4                    */

/* Replaces DistributedHashMap::DistributedHashMap(size_t,int,int) (hash_map.hpp:50-52) and
 * the sizing in kmer_hash.cpp:107-109 (table = n_kmers / load_factor; the reference uses
 * load factor 0.5).  `device` is the CUDA ordinal that owns this table. */
int kh_create(int k, uint64_t n_expected, double load_factor, int device, kh_table** out);
int kh_destroy(kh_table* t);
/* Empty the table and forget the start nodes (a fresh DistributedHashMap). Stream-ordered. */
int kh_clear(kh_table* t);
/* Run on an existing CUDA stream (cudaStream_t) instead of the handle's own; NULL = the legacy
 * default stream.  Work the caller orders against this handle (NCCL, copies) must use the same stream. */
int kh_set_stream(kh_table* t, void* cuda_stream);
int kh_sync(kh_table* t);
/* Tuning knobs (also read from the environment at create: KH_SPLIT_BUCKETS, KH_SEG_CHARS):
 *   "split_buckets": every split_buckets-th bucket's first slot ends a walk segment
 *   "seg_chars"    : capacity of one segment's character buffer (multiple of 8, <= 248) */
int kh_set_option(kh_table* t, const char* name, int64_t value);

/* K1 -- replaces the parse loop of read_kmers (read_kmers.hpp:72-76) + kmer_pair::init
 * (kmer_t.hpp:67-76) + packKmer/packFourMer (packing.hpp:50-92): n_lines fixed-width lines of
 * K+4 bytes -> n_lines kmer_pair records. */
int kh_pack_lines(kh_table* t, const char* text_host, uint64_t n_lines, void* pairs_host_out);
int kh_pack_lines_device(kh_table* t, const void* text_dev, uint64_t n_lines, void* pairs_dev_out);

/* K2+K3 -- replaces initialize_kmers (kmer_hash.cpp:21-33): DistributedHashMap::insert_all
 * (hash_map.hpp:55-80) plus the order-preserving scan for backward ext == 'F'
 * (kmer_hash.cpp:27-31).  May be called repeatedly; start nodes accumulate in call order. */
int kh_insert_pairs(kh_table* t, const void* pairs_host, uint64_t n);
int kh_insert_pairs_device(kh_table* t, const void* pairs_dev, uint64_t n);
/* read_kmers + initialize_kmers in one call, straight from text lines (K1 then K2+K3). */
int kh_insert_lines(kh_table* t, const char* text_host, uint64_t n_lines);

/* K4 as a batch -- replaces DistributedHashMap::find (hash_map.hpp:83-107): n packed k-mers
 * (pkmer_t bytes) -> n kmer_pair records and n found flags (1/0; the record is zeroed on a miss). */
int kh_find(kh_table* t, const void* pkmers_host, uint64_t n, void* pairs_host_out, uint8_t* found_host_out);
int kh_find_device(kh_table* t, const void* pkmers_dev, uint64_t n, void* pairs_dev_out, uint8_t* found_dev_out);

/* K3-K6 -- replaces assemble_contigs (kmer_hash.cpp:38-55) + extract_contig
 * (read_kmers.hpp:81-92): one contig per start node, in start-node order, each rendered as
 * its first k-mer's K characters followed by every forward extension != 'F', then '\n'
 * (exactly the bytes output_results writes per contig, kmer_hash.cpp:64-67).
 *   *contigs        : contig text, contig_bytes long  (host / device memory owned by the handle,
 *                     valid until the next assemble, clear or destroy)
 *   *offsets        : n_contigs+1 byte offsets into it
 * Returns KH_ERR_NOT_FOUND / KH_ERR_CYCLE / KH_ERR_CONVERGE as described above. */
int kh_assemble(kh_table* t, const char** contigs_host, const uint64_t** offsets_host,
                uint64_t* n_contigs, uint64_t* contig_bytes, uint64_t* n_nodes);
int kh_assemble_device(kh_table* t, const char** contigs_dev, const uint64_t** offsets_dev,
                       uint64_t* n_contigs, uint64_t* contig_bytes, uint64_t* n_nodes);

/* Output side -- `cat test*.dat | sort` of scripts/check_it.sh:47-48 without the host sort: the contigs of the last
 * kh_assemble / kh_assemble_device / kh_shard_assemble on this handle in bytewise (LC_ALL=C) order of their lines.
 * The sort runs on the GPU over a 21-character prefix key; contigs that agree on it are ordered on the host.
 * order_host_out: room for n_contigs indices into the offsets array. */
int kh_sorted_order(kh_table* t, uint64_t* order_host_out, uint64_t* n_contigs_out);

int kh_get_stats(kh_table* t, kh_stats* out);

/* What a CUDA kernel of the caller needs to use the table directly (include/kh/device_table.cuh: kh::device_find,
 * kh::device_insert -- the per-k-mer HashMap::insert / find of README.md:95-99 as __device__ functions).  Plain tables
 * only: returns KH_ERR_ARG for a chunk table (large K >= 30 tables and sharded handles; create with KH_CT=0 to force a
 * plain one).  The view stays valid until kh_destroy; kh_clear empties the table it points to. */
typedef struct kh_device_view {
    void* table;               /* device pointer: n_buckets x 32 bytes                         */
    uint64_t n_buckets;
    int32_t k;
    int32_t slot_bytes;        /* 8 or 16                                                      */
    int32_t placement_m;       /* reserved, always 0                                           */
    int32_t device;            /* CUDA ordinal that owns the table                             */
} kh_device_view;
int kh_get_device_view(kh_table* t, kh_device_view* out);
const char* kh_last_error(kh_table* t);

/* Pinned host memory for callers that want full-speed host<->device copies. */
int kh_host_alloc(void** ptr, uint64_t bytes);
int kh_host_free(void* ptr);

/* Micro-benchmark used by bench.py for the roofline denominators: `n_probes` independent
 * random 32-byte sector reads over a `footprint_bytes` buffer; returns sectors per second. */
int kh_measure_random_sector_rate(int device, uint64_t footprint_bytes, uint64_t n_probes, double* sectors_per_s);

/* ---------------------------------------------------------------------------------------------
 * Sharded (multi-GPU) path -- replaces the UPC++ side of DistributedHashMap: owner-rank selection
 * (hash_map.hpp:28-30), batched remote inserts (hash_map.hpp:38-46, 64-77), remote finds
 * (hash_map.hpp:93-100) and the barriers (hash_map.hpp:79, kmer_hash.cpp:32, 126, 136).
 * SPMD like the reference: one handle per rank (GPU), every rank makes the same calls in the same
 * order -- from one process per GPU (cs267_hw3_b200/sharded.py under torchrun, CUDA IPC peer mappings)
 * or from one host thread per GPU in one process (include/kh/sharded_host.hpp).  A step is
 *     kh_shard_begin;  kh_shard_insert (any number of times);  kh_shard_assemble;  kh_shard_finish
 * and everything before kh_shard_finish only ENQUEUES work on the handle's stream: the records reach their
 * owner GPU through NVLink peer stores inside the grouping kernel, chain links that leave a GPU and their
 * answers travel the same way, phases are separated by an in-stream barrier kernel.  Nothing in a step
 * allocates or synchronises with the host, so kh_shard_init reserves every buffer.
 * Supported K: 17..54.  Options (kh_set_option / KH_* environment) must be set before kh_shard_init,
 * and kh_shard_init must precede kh_shard_export / kh_shard_connect*.
 * ------------------------------------------------------------------------------------------- */
uint64_t kh_slot_bytes(int k);            /* bytes of one table slot: 8 or 16 */
/* Fix all capacities for this rank: at most n_local_max records (n_starts_max of them start nodes) parsed
 * here, n_total records over all ranks.  kh_create's n_expected is the number of k-mers THIS shard must be
 * able to hold (its share of n_total plus slack, see kh_sharded::shard_capacity). */
int kh_shard_init(kh_table* t, int rank, int world, uint64_t n_local_max, uint64_t n_total, uint64_t n_starts_max);
/* kh_shard_export_count() CUDA IPC handles (64 bytes each) + 2 uint64 of metadata for this rank; gather them
 * from all ranks (rank order) and hand the lot to kh_shard_connect. */
int kh_shard_export_count(void);
int kh_shard_export(kh_table* t, void* handles_out, uint64_t* meta_out);
int kh_shard_connect(kh_table* t, const void* all_handles, const uint64_t* all_meta);
/* all ranks in this process: wire them up directly (peer access is enabled between their devices) */
int kh_shard_connect_local(kh_table* t, kh_table* const* peers, int world);
/* A fresh DistributedHashMap on this rank (kh_clear) + barrier: no rank writes into a peer that has not reset yet. */
int kh_shard_begin(kh_table* t);
/* initialize_kmers (kmer_hash.cpp:21-33) for this rank's block of records (device memory, kmer_pair bytes):
 * stage every record in its owner's memory, register this rank's start nodes in input order. */
int kh_shard_insert(kh_table* t, const void* pairs_dev, uint64_t n);
/* assemble_contigs (kmer_hash.cpp:38-55): build the shard, chain the segments across GPUs, rank, emit.
 * kh_shard_assemble = parts 0 .. kh_shard_assemble_parts()-1 in order; every part ends with the barrier.  A host
 * that drives several ranks on ONE device must enqueue part p for all of them before part p+1 (their streams
 * may share a hardware queue, where a waiting barrier would block the peer's work behind it). */
int kh_shard_assemble(kh_table* t);
int kh_shard_assemble_parts(void);
int kh_shard_assemble_part(kh_table* t, int part);
/* wait for the step; *error_bits_out: 1 k-mer not found, 2 table full, 4 cycle, 8 bad input, 16 converge,
 * 32 internal (a capacity was exceeded / a peer never reached a barrier).  OR the bits of all ranks. */
int kh_shard_finish(kh_table* t, int* error_bits_out);
/* this rank's `<prefix>_<rank>.dat`: the contigs whose start node lies in its block, in input order */
int kh_shard_result(kh_table* t, const char** contigs_dev, const uint64_t** offsets_dev,
                    uint64_t* n_contigs, uint64_t* contig_bytes, uint64_t* n_nodes);

/* ---------------------------------------------------------------------------------------------
 * k-mer analysis -- the stage BEFORE this one: reads -> unique k-mers with their backward / forward
 * extensions (README.md:19-21: "the output of this first preprocessing stage ... is a set of unique DNA
 * sequence fragments of length k", each "associated with a forward and backward extension").  The
 * reference only ever reads that output from a text file (read_kmers.hpp:54-79); here it is produced on
 * the GPU, in the reference's kmer_pair bytes, so it can go straight into kh_insert_pairs_device.
 *
 * Input: a byte buffer of reads.  'A' 'C' 'G' 'T' are bases, every other byte ('\n', 'N', ...) separates
 * reads; each call's buffer is taken to begin and end at a read boundary.  Every position whose K bytes are
 * bases is one occurrence of that k-mer; the byte before / after it, when it is a base, is its backward /
 * forward observation.  Per distinct k-mer the table keeps saturating counters: occurrences (<= 255) and, per
 * side and base, observations (<= 127).  kh_count_extract reports the k-mers with occurrences >= min_count
 * (1..255); an extension is the base that alone reaches min_ext (1..127) on its side, 'F' when none does
 * (a contig begins / ends: README.md:37) or several do (a fork).  No reverse complements, like the reference
 * (kmer_t.hpp:51-57).  Records come out in table order (arbitrary, as k-mer counters' output is).
 * Supported K: 2..61.
 *
 * One GPU per counter, several counters per analysis: every counter field saturates, and saturating sums are
 * associative, so counters that counted disjoint pieces of the reads (cut at a non-base byte) merge field by field
 * into exactly the counters one table over all reads would hold.  kh_count_partition groups a counter's k-mers by
 * owner rank, kh_count_merge_device adds such a group into another counter (on any device of the process): P
 * ranks count their pieces, every owner merges the group addressed to it from every rank, and the union of the
 * owners' extracts is the single-counter result (include/kh/sharded_counter.hpp drives that flow).  Thresholds
 * apply to the merged counters only -- nothing may be dropped before the merge.
 * ------------------------------------------------------------------------------------------- */
typedef struct kh_counter kh_counter;
typedef struct kh_count_stats {
    uint64_t n_slots;          /* table capacity (one k-mer per slot)                              */
    uint64_t n_distinct;       /* distinct k-mers seen since create / clear                        */
    uint64_t n_occurrences;    /* k-mer occurrences counted since create / clear                   */
    uint64_t n_bytes;          /* read bytes consumed since create / clear                         */
    uint64_t n_reported;       /* records of the last kh_count_extract*                            */
    uint32_t slot_bytes;       /* 16 (K <= 31) or 32 (one DRAM sector)                             */
    uint32_t n_launches;       /* kernels launched since create                                    */
    uint32_t n_grows;          /* times the table was doubled and rehashed since create            */
    uint32_t reserved;
    float ms_count;            /* last kh_count_reads*: first byte in .. last kernel out (CUDA events) */
    float ms_extract;          /* last kh_count_extract*: the extract kernel                       */
} kh_count_stats;
/* The table starts with n_distinct_expected / load_factor slots (distinct k-mers of the reads, erroneous ones
 * included).  kh_count_reads never runs out of slots: it hands the kernel no more positions than the table has room
 * for and doubles the table (rehashed on the GPU) when that room gets small -- a good estimate only saves the
 * rehashes (KH_COUNT_GROW=0 turns growing off).  kh_count_reads_device only enqueues and therefore cannot grow:
 * if the table fills up, the next synchronising call returns KH_ERR_TABLE_FULL (until kh_count_clear). */
int kh_count_create(int k, uint64_t n_distinct_expected, double load_factor, int device, kh_counter** out);
int kh_count_destroy(kh_counter* c);
int kh_count_clear(kh_counter* c);
int kh_count_reads(kh_counter* c, const char* reads_host, uint64_t n_bytes);         /* may be called repeatedly */
/* enqueues on the counter's stream: reads_dev (any alignment) must stay valid until the next synchronising call on
 * this counter (kh_count_get_stats, kh_count_extract*, kh_count_lookup, kh_count_reads) */
int kh_count_reads_device(kh_counter* c, const char* reads_dev, uint64_t n_bytes);
/* kmer_pair records (kh_pair_bytes(k) each) of the reported k-mers.  _device: *pairs_dev_out is owned by the
 * counter and valid until its next extract, clear or destroy.  Host variant: pairs_host_out may be NULL to
 * learn *n_out only; with capacity < *n_out nothing is copied and KH_ERR_ARG is returned (*n_out is set). */
int kh_count_extract_device(kh_counter* c, uint32_t min_count, uint32_t min_ext, const void** pairs_dev_out, uint64_t* n_out);
int kh_count_extract(kh_counter* c, uint32_t min_count, uint32_t min_ext, void* pairs_host_out, uint64_t capacity, uint64_t* n_out);
/* The same k-mers as lines of the reference's k-mer file -- K bases, a blank, backward and forward extension, '\n'
 * (K + 4 bytes each; what read_kmers parses, read_kmers.hpp:64-76): the reference's input file, written from reads.
 * lines_host_out may be NULL to learn *n_out; capacity_lines counts lines. */
int kh_count_extract_lines(kh_counter* c, uint32_t min_count, uint32_t min_ext, char* lines_host_out, uint64_t capacity_lines, uint64_t* n_out);
/* The counters of n given k-mers (pkmer_t bytes): 9 x uint32 each -- occurrences, backward A C G T, forward A C G T;
 * all zero for a k-mer that was never seen. */
int kh_count_lookup(kh_counter* c, const void* pkmers_host, uint64_t n, uint32_t* counts_host_out);
int kh_count_get_stats(kh_counter* c, kh_count_stats* out);
const char* kh_count_last_error(kh_counter* c);
/* Merging counters.  A record is one k-mer with its counters, kh_count_record_bytes(k) = 16 or 32 bytes; the format is
 * opaque and meaningful only to a counter of the same K.  The owner rank of a k-mer depends on the k-mer and world only.
 * kh_count_partition: every k-mer of this counter, grouped by owner rank (0..world-1), in a counter-owned device buffer
 * valid until the next partition or destroy; offsets_host_out: world+1 record offsets (group o = records
 * [offsets[o], offsets[o+1])).  1 <= world <= 64.  Host-synchronous; returns KH_ERR_TABLE_FULL after a count that
 * overflowed the table.
 * kh_count_merge_device: saturating merge of n records into this counter.  records_dev may live on any device of this
 * process: if it is not the counter's, it is first copied into a counter-owned inbox (peer to peer where possible).
 * Grows the table like kh_count_reads (KH_COUNT_GROW=0 -> KH_ERR_TABLE_FULL).  Host-synchronous.  Adds the newly seen
 * k-mers to n_distinct; n_occurrences and n_bytes keep counting only what kh_count_reads* consumed here. */
uint64_t kh_count_record_bytes(int k);
int kh_count_partition(kh_counter* c, int world, const void** records_dev_out, uint64_t* offsets_host_out);
int kh_count_merge_device(kh_counter* c, const void* records_dev, uint64_t n);
/* The k-mer spectrum, for choosing min_count (the two-column histogram `jellyfish histo` / GenomeScope use).
 * hist[c], c = 1..254: the number of distinct k-mers counted exactly c times; hist[255]: those seen 255 times or more
 * (the occurrence counter saturates there); hist[0] = 0.  So sum(hist) = n_distinct, and for every m the sum of
 * hist[c] over c >= m is the number of records kh_count_extract*(m, any min_ext) reports.  Counters merged from other
 * counters are covered like counted ones, so the spectrum of a sharded analysis is the bin-by-bin sum of its owners'.
 * kh_count_histogram: hist_host_out has room for 256 uint64; one scan of the table.  Host-synchronous; returns
 * KH_ERR_TABLE_FULL after a count that overflowed the table.
 * kh_count_auto_min_count: the valley rule, a pure function of the 256 bins that needs no device.  Let v be the
 * smallest c in 1..254 with hist[c+1] >= hist[c] (where the falling slope of erroneous k-mers stops).  The result is v
 * when v >= 2 and some k-mer is counted v times or more; otherwise 2 (no falling slope, as for error-free reads or an
 * empty table; or a spectrum that falls to zero without a second peak).  hist = NULL gives 2.  kh_count_extract* take
 * the result like any other min_count. */
int kh_count_histogram(kh_counter* c, uint64_t* hist_host_out);
uint32_t kh_count_auto_min_count(const uint64_t* hist);

/* Introspection for tests and debugging: device pointer and capacity of an internal buffer of a chunk table
 * ("link", "meta", "chunk_base", "seg_base", "chunk_cursor", "counters", ...; "caps" returns HOST numbers). */
int kh_debug_buffer(kh_table* t, const char* name, void** ptr_out, uint64_t* bytes_out);

/* small device-memory helpers for hosts without their own CUDA binding */
int kh_device_alloc(void** ptr, uint64_t bytes);                 /* on the current device */
int kh_device_alloc_on(int device, void** ptr, uint64_t bytes);
int kh_device_free(void* ptr);
int kh_copy_to_host(kh_table* t, void* dst_host, const void* src_dev, uint64_t bytes);
int kh_copy_device(kh_table* t, void* dst_dev, const void* src_dev, uint64_t bytes);

#ifdef __cplusplus
}
#endif
#endif /* KH_CAPI_H */
