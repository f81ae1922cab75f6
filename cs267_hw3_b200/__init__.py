"""cs267_hw3_b200 -- B200-native k-mer hash table + contig traversal (one stage of CS267 HW3).

The product is ``libkh_b200.so`` (hand-written CUDA for sm_100a behind the C ABI in
``include/kh_capi.h``) plus the C++ drop-in headers/CLI in ``include/`` and ``src/``.
This Python package is only a ctypes view of that C ABI for tests, ``bench.py`` and
``__graft_entry__.py``.  There is no CPU path: without the library or without a CUDA device
every call raises.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

from . import build as _build

PKG = os.path.dirname(os.path.abspath(__file__))
# KH_LIB_PATH: load another build of the library (tuning runs with other compile-time geometry, tools/probes/build_variants.sh)
LIB_PATH = os.environ.get("KH_LIB_PATH") or os.path.join(PKG, "libkh_b200.so")

KH_OK, KH_ERR_ARG, KH_ERR_CUDA, KH_ERR_NOT_FOUND, KH_ERR_TABLE_FULL = 0, 1, 2, 3, 4
KH_ERR_CYCLE, KH_ERR_BAD_INPUT, KH_ERR_CONVERGE, KH_ERR_NOMEM = 5, 6, 7, 8

# every symbol include/kh_capi.h declares (tests/test_boundary.py checks header <-> library <-> this list)
ABI_SYMBOLS = [
    "kh_abi_version", "kh_device_count", "kh_status_string", "kh_pair_bytes", "kh_packed_bytes",
    "kh_create", "kh_destroy", "kh_clear", "kh_set_stream", "kh_sync", "kh_set_option",
    "kh_pack_lines", "kh_pack_lines_device", "kh_insert_pairs", "kh_insert_pairs_device", "kh_insert_lines",
    "kh_find", "kh_find_device", "kh_assemble", "kh_assemble_device", "kh_get_stats", "kh_last_error",
    "kh_host_alloc", "kh_host_free", "kh_measure_random_sector_rate",
    # sharded (multi-GPU) path
    "kh_slot_bytes", "kh_shard_init", "kh_shard_export_count", "kh_shard_export", "kh_shard_connect", "kh_shard_connect_local",
    "kh_shard_begin", "kh_shard_insert", "kh_shard_assemble", "kh_shard_assemble_parts", "kh_shard_assemble_part",
    "kh_shard_finish", "kh_shard_result", "kh_debug_buffer", "kh_get_device_view", "kh_sorted_order",
    "kh_device_alloc", "kh_device_alloc_on", "kh_device_free", "kh_copy_to_host", "kh_copy_device",
    # k-mer analysis (reads -> k-mers with extensions), the stage before this one
    "kh_count_create", "kh_count_destroy", "kh_count_clear", "kh_count_reads", "kh_count_reads_device",
    "kh_count_extract", "kh_count_extract_device", "kh_count_extract_lines", "kh_count_lookup", "kh_count_get_stats", "kh_count_last_error",
    "kh_count_record_bytes", "kh_count_partition", "kh_count_merge_device", "kh_count_histogram", "kh_count_auto_min_count",
]


class KhError(RuntimeError):
    def __init__(self, status: int, message: str):
        super().__init__(f"[kh status {status}] {message}")
        self.status = status


class Stats(C.Structure):
    _fields_ = [
        ("n_slots", C.c_uint64), ("n_buckets", C.c_uint64), ("n_inserted", C.c_uint64),
        ("n_duplicates", C.c_uint64), ("n_starts", C.c_uint64), ("n_contigs", C.c_uint64),
        ("n_nodes", C.c_uint64), ("contig_bytes", C.c_uint64), ("n_segments", C.c_uint64),
        ("rank_rounds", C.c_uint32), ("slot_bits", C.c_uint32),
        ("ms_insert", C.c_float), ("ms_assemble", C.c_float), ("ms_walk", C.c_float),
        ("ms_rank", C.c_float), ("ms_emit", C.c_float), ("ms_pack", C.c_float), ("ms_clear", C.c_float),
        ("ms_build", C.c_float), ("ms_stage", C.c_float), ("n_launches", C.c_uint64),
    ]

    def as_dict(self) -> dict:
        return {n: getattr(self, n) for n, _ in self._fields_}


class CountStats(C.Structure):
    _fields_ = [
        ("n_slots", C.c_uint64), ("n_distinct", C.c_uint64), ("n_occurrences", C.c_uint64), ("n_bytes", C.c_uint64),
        ("n_reported", C.c_uint64), ("slot_bytes", C.c_uint32), ("n_launches", C.c_uint32),
        ("n_grows", C.c_uint32), ("reserved", C.c_uint32), ("ms_count", C.c_float), ("ms_extract", C.c_float),
    ]

    def as_dict(self) -> dict:
        return {n: getattr(self, n) for n, _ in self._fields_}


_lib = None


def lib() -> C.CDLL:
    """Load libkh_b200.so (building it in-tree first if it is missing or stale). Raises if impossible."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.environ.get("KH_LIB_PATH") and (not os.path.exists(LIB_PATH) or _build._stale(LIB_PATH, _build.lib_sources())):
        _build.build_lib()
    L = C.CDLL(LIB_PATH)
    u64, vp, i32 = C.c_uint64, C.c_void_p, C.c_int
    pu64 = C.POINTER(u64)
    L.kh_abi_version.restype = i32
    L.kh_device_count.restype = i32
    L.kh_status_string.argtypes = [i32]
    L.kh_status_string.restype = C.c_char_p
    L.kh_pair_bytes.argtypes = [i32]
    L.kh_pair_bytes.restype = u64
    L.kh_packed_bytes.argtypes = [i32]
    L.kh_packed_bytes.restype = u64
    L.kh_create.argtypes = [i32, u64, C.c_double, i32, C.POINTER(vp)]
    L.kh_destroy.argtypes = [vp]
    L.kh_clear.argtypes = [vp]
    L.kh_set_stream.argtypes = [vp, vp]
    L.kh_sync.argtypes = [vp]
    L.kh_set_option.argtypes = [vp, C.c_char_p, C.c_int64]
    L.kh_pack_lines.argtypes = [vp, vp, u64, vp]
    L.kh_pack_lines_device.argtypes = [vp, vp, u64, vp]
    L.kh_insert_pairs.argtypes = [vp, vp, u64]
    L.kh_insert_pairs_device.argtypes = [vp, vp, u64]
    L.kh_insert_lines.argtypes = [vp, vp, u64]
    L.kh_find.argtypes = [vp, vp, u64, vp, vp]
    L.kh_find_device.argtypes = [vp, vp, u64, vp, vp]
    L.kh_assemble.argtypes = [vp, C.POINTER(vp), C.POINTER(vp), pu64, pu64, pu64]
    L.kh_assemble_device.argtypes = [vp, C.POINTER(vp), C.POINTER(vp), pu64, pu64, pu64]
    L.kh_get_stats.argtypes = [vp, C.POINTER(Stats)]
    L.kh_last_error.argtypes = [vp]
    L.kh_last_error.restype = C.c_char_p
    L.kh_host_alloc.argtypes = [C.POINTER(vp), u64]
    L.kh_host_free.argtypes = [vp]
    L.kh_measure_random_sector_rate.argtypes = [i32, u64, u64, C.POINTER(C.c_double)]
    L.kh_device_alloc.argtypes = [C.POINTER(vp), u64]
    L.kh_device_alloc_on.argtypes = [i32, C.POINTER(vp), u64]
    L.kh_device_free.argtypes = [vp]
    L.kh_copy_to_host.argtypes = [vp, vp, vp, u64]
    L.kh_copy_device.argtypes = [vp, vp, vp, u64]
    u32 = C.c_uint32
    L.kh_count_create.argtypes = [i32, u64, C.c_double, i32, C.POINTER(vp)]
    L.kh_count_destroy.argtypes = [vp]
    L.kh_count_clear.argtypes = [vp]
    L.kh_count_reads.argtypes = [vp, vp, u64]
    L.kh_count_reads_device.argtypes = [vp, vp, u64]
    L.kh_count_extract.argtypes = [vp, u32, u32, vp, u64, pu64]
    L.kh_count_extract_device.argtypes = [vp, u32, u32, C.POINTER(vp), pu64]
    L.kh_count_extract_lines.argtypes = [vp, u32, u32, vp, u64, pu64]
    L.kh_count_lookup.argtypes = [vp, vp, u64, vp]
    L.kh_count_get_stats.argtypes = [vp, C.POINTER(CountStats)]
    L.kh_count_last_error.argtypes = [vp]
    L.kh_count_last_error.restype = C.c_char_p
    L.kh_count_record_bytes.argtypes = [i32]
    L.kh_count_record_bytes.restype = u64
    L.kh_count_partition.argtypes = [vp, i32, C.POINTER(vp), pu64]
    L.kh_count_merge_device.argtypes = [vp, vp, u64]
    L.kh_count_histogram.argtypes = [vp, pu64]
    L.kh_count_auto_min_count.argtypes = [pu64]
    L.kh_count_auto_min_count.restype = u32
    _lib = L
    return L


def device_count() -> int:
    return int(lib().kh_device_count())


def pair_bytes(k: int) -> int:
    return (k + 3) // 4 + 2


def packed_bytes(k: int) -> int:
    return (k + 3) // 4


def random_sector_rate(device: int = 0, footprint_bytes: int = 4 << 30, n_probes: int = 1 << 28) -> float:
    out = C.c_double()
    rc = lib().kh_measure_random_sector_rate(device, footprint_bytes, n_probes, C.byref(out))
    if rc != KH_OK:
        raise KhError(rc, lib().kh_status_string(rc).decode())
    return out.value


class PinnedBuffer:
    """Page-locked host memory from the library (kh_host_alloc), viewed as a numpy uint8 array."""

    def __init__(self, nbytes: int):
        self._p = C.c_void_p()
        rc = lib().kh_host_alloc(C.byref(self._p), nbytes)
        if rc != KH_OK:
            raise KhError(rc, "kh_host_alloc failed")
        self.nbytes = nbytes
        self.array = np.ctypeslib.as_array(C.cast(self._p, C.POINTER(C.c_uint8)), shape=(max(nbytes, 1),))[:nbytes]

    @property
    def ptr(self) -> int:
        return self._p.value

    def free(self) -> None:
        if self._p:
            self.array = None
            lib().kh_host_free(self._p)
            self._p = C.c_void_p()

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class KmerHashTable:
    """One GPU's hash table + traversal state (a `kh_table*`).

    Mirrors the stage functions of the reference: ``insert_pairs`` = initialize_kmers
    (kmer_hash.cpp:21-33), ``find`` = DistributedHashMap::find (hash_map.hpp:83-107),
    ``assemble`` = assemble_contigs + extract_contig (kmer_hash.cpp:38-55, read_kmers.hpp:81-92).
    """

    def __init__(self, k: int, n_expected: int, load_factor: float = 0.5, device: int = 0):
        self.k = k
        self._h = C.c_void_p()
        rc = lib().kh_create(k, n_expected, load_factor, device, C.byref(self._h))
        if rc != KH_OK:
            raise KhError(rc, "kh_create: " + lib().kh_status_string(rc).decode())

    # -- plumbing --
    def _check(self, rc: int) -> None:
        if rc != KH_OK:
            msg = lib().kh_last_error(self._h).decode() or lib().kh_status_string(rc).decode()
            raise KhError(rc, msg)

    def close(self) -> None:
        if self._h:
            lib().kh_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def clear(self) -> None:
        self._check(lib().kh_clear(self._h))

    def sync(self) -> None:
        self._check(lib().kh_sync(self._h))

    def set_stream(self, cuda_stream: int | None) -> None:
        self._check(lib().kh_set_stream(self._h, cuda_stream))

    def set_option(self, name: str, value: int) -> None:
        self._check(lib().kh_set_option(self._h, name.encode(), value))

    def stats(self) -> dict:
        s = Stats()
        self._check(lib().kh_get_stats(self._h, C.byref(s)))
        return s.as_dict()

    # -- K1 --
    def pack_lines(self, text) -> np.ndarray:
        t = np.frombuffer(text, dtype=np.uint8) if not isinstance(text, np.ndarray) else np.ascontiguousarray(text)
        ll = self.k + 4
        if t.size % ll:
            raise ValueError("text is not a whole number of (K+4)-byte lines")
        n = t.size // ll
        out = np.empty((n, pair_bytes(self.k)), dtype=np.uint8)
        self._check(lib().kh_pack_lines(self._h, t.ctypes.data, n, out.ctypes.data))
        return out

    def pack_lines_device(self, text_ptr: int, n_lines: int, pairs_ptr: int) -> None:
        self._check(lib().kh_pack_lines_device(self._h, text_ptr, n_lines, pairs_ptr))

    # -- K2 + K3 --
    def insert_pairs(self, pairs) -> None:
        p = np.ascontiguousarray(pairs, dtype=np.uint8)
        n = p.size // pair_bytes(self.k)
        self._check(lib().kh_insert_pairs(self._h, p.ctypes.data, n))

    def insert_pairs_ptr(self, host_ptr: int, n: int) -> None:
        self._check(lib().kh_insert_pairs(self._h, host_ptr, n))

    def insert_pairs_device(self, dev_ptr: int, n: int) -> None:
        self._check(lib().kh_insert_pairs_device(self._h, dev_ptr, n))

    def insert_lines(self, text) -> None:
        t = np.frombuffer(text, dtype=np.uint8) if not isinstance(text, np.ndarray) else np.ascontiguousarray(text)
        ll = self.k + 4
        if t.size % ll:
            raise ValueError("text is not a whole number of (K+4)-byte lines")
        self._check(lib().kh_insert_lines(self._h, t.ctypes.data, t.size // ll))

    # -- K4 --
    def find(self, pkmers) -> tuple[np.ndarray, np.ndarray]:
        q = np.ascontiguousarray(pkmers, dtype=np.uint8)
        n = q.size // packed_bytes(self.k)
        pairs = np.zeros((n, pair_bytes(self.k)), dtype=np.uint8)
        found = np.zeros(n, dtype=np.uint8)
        self._check(lib().kh_find(self._h, q.ctypes.data, n, pairs.ctypes.data, found.ctypes.data))
        return pairs, found.astype(bool)

    # -- K3..K6 --
    def assemble(self, copy: bool = True):
        """Returns (contig text as a uint8 array, offsets uint64[n_contigs+1], n_nodes)."""
        cp, op = C.c_void_p(), C.c_void_p()
        nc, nb, nn = C.c_uint64(), C.c_uint64(), C.c_uint64()
        self._check(lib().kh_assemble(self._h, C.byref(cp), C.byref(op), C.byref(nc), C.byref(nb), C.byref(nn)))
        if nb.value:
            buf = np.ctypeslib.as_array(C.cast(cp, C.POINTER(C.c_uint8)), shape=(nb.value,))
        else:
            buf = np.empty(0, dtype=np.uint8)
        offs = np.ctypeslib.as_array(C.cast(op, C.POINTER(C.c_uint64)), shape=(nc.value + 1,))
        if copy:
            buf, offs = buf.copy(), offs.copy()
        return buf, offs, nn.value

    def assemble_device(self):
        """Enqueue + finish on the device; returns (contigs_dev_ptr, offsets_dev_ptr, n_contigs, bytes, n_nodes)."""
        cp, op = C.c_void_p(), C.c_void_p()
        nc, nb, nn = C.c_uint64(), C.c_uint64(), C.c_uint64()
        self._check(lib().kh_assemble_device(self._h, C.byref(cp), C.byref(op), C.byref(nc), C.byref(nb), C.byref(nn)))
        return cp.value, op.value, nc.value, nb.value, nn.value


class KmerCounter:
    """k-mer analysis on one GPU (a `kh_counter*`): reads -> unique k-mers with their backward / forward extensions,
    the stage whose output the reference reads from text (README.md:19-21, read_kmers.hpp:54-79)."""

    def __init__(self, k: int, n_distinct_expected: int, load_factor: float = 0.5, device: int = 0):
        self.k = k
        self._h = C.c_void_p()
        rc = lib().kh_count_create(k, n_distinct_expected, load_factor, device, C.byref(self._h))
        if rc != KH_OK:
            raise KhError(rc, "kh_count_create: " + lib().kh_status_string(rc).decode())

    def _check(self, rc: int) -> None:
        if rc != KH_OK:
            msg = lib().kh_count_last_error(self._h).decode() or lib().kh_status_string(rc).decode()
            raise KhError(rc, msg)

    def close(self) -> None:
        if self._h:
            lib().kh_count_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def clear(self) -> None:
        self._check(lib().kh_count_clear(self._h))

    def count_reads(self, reads) -> None:
        r = np.frombuffer(reads, dtype=np.uint8) if not isinstance(reads, np.ndarray) else np.ascontiguousarray(reads)
        self._check(lib().kh_count_reads(self._h, r.ctypes.data, r.size))

    def count_reads_ptr(self, host_ptr: int, n_bytes: int) -> None:
        self._check(lib().kh_count_reads(self._h, host_ptr, n_bytes))

    def count_reads_device(self, dev_ptr: int, n_bytes: int) -> None:
        self._check(lib().kh_count_reads_device(self._h, dev_ptr, n_bytes))

    def extract(self, min_count: int = 2, min_ext: int = 2) -> np.ndarray:
        """kmer_pair records of the reported k-mers, shape (n, pair_bytes), in table order."""
        n = C.c_uint64()
        self._check(lib().kh_count_extract(self._h, min_count, min_ext, None, 0, C.byref(n)))
        out = np.empty((n.value, pair_bytes(self.k)), dtype=np.uint8)
        self._check(lib().kh_count_extract(self._h, min_count, min_ext, out.ctypes.data, n.value, C.byref(n)))
        return out

    def extract_device(self, min_count: int = 2, min_ext: int = 2) -> tuple[int, int]:
        """(device pointer to the records, number of records); the buffer belongs to the counter."""
        p, n = C.c_void_p(), C.c_uint64()
        self._check(lib().kh_count_extract_device(self._h, min_count, min_ext, C.byref(p), C.byref(n)))
        return p.value or 0, n.value

    def extract_lines(self, min_count: int = 2, min_ext: int = 2) -> np.ndarray:
        """The reported k-mers in the reference's k-mer file format (uint8 buffer of (K+4)-byte lines)."""
        n = C.c_uint64()
        self._check(lib().kh_count_extract_lines(self._h, min_count, min_ext, None, 0, C.byref(n)))
        out = np.empty(n.value * (self.k + 4), dtype=np.uint8)
        self._check(lib().kh_count_extract_lines(self._h, min_count, min_ext, out.ctypes.data, n.value, C.byref(n)))
        return out

    def lookup(self, pkmers) -> np.ndarray:
        """uint32 (n, 9): occurrences, backward A C G T, forward A C G T of the given packed k-mers."""
        q = np.ascontiguousarray(pkmers, dtype=np.uint8)
        n = q.size // packed_bytes(self.k)
        out = np.zeros((n, 9), dtype=np.uint32)
        self._check(lib().kh_count_lookup(self._h, q.ctypes.data, n, out.ctypes.data))
        return out

    def histogram(self) -> np.ndarray:
        """The k-mer spectrum, uint64[256]: [c] = distinct k-mers seen exactly c times, [255] = 255 times or more, [0] = 0."""
        h = np.zeros(HIST_BINS, dtype=np.uint64)
        self._check(lib().kh_count_histogram(self._h, h.ctypes.data_as(C.POINTER(C.c_uint64))))
        return h

    def stats(self) -> dict:
        s = CountStats()
        self._check(lib().kh_count_get_stats(self._h, C.byref(s)))
        return s.as_dict()

    # -- merging counters (sharded counting, kh_count_partition / kh_count_merge_device) --
    def partition(self, world: int) -> tuple[int, np.ndarray]:
        """Every k-mer of this counter grouped by owner rank: (device pointer to the records, uint64 offsets[world + 1]).
        Group o holds records offsets[o] .. offsets[o+1] of record_bytes(k) bytes; the buffer belongs to the counter."""
        p = C.c_void_p()
        offs = np.zeros(world + 1, dtype=np.uint64)
        self._check(lib().kh_count_partition(self._h, world, C.byref(p), offs.ctypes.data_as(C.POINTER(C.c_uint64))))
        return p.value or 0, offs

    def merge_device(self, dev_ptr: int, n: int) -> None:
        """Add n records (a group of another counter's partition, on any device) to this counter."""
        self._check(lib().kh_count_merge_device(self._h, dev_ptr, n))

    def merge(self, other: "KmerCounter") -> None:
        """Add all k-mers of `other` (same K) to this counter: its counters become those of one counter over both inputs."""
        ptr, offs = other.partition(1)
        self.merge_device(ptr, int(offs[1]))


HIST_BINS = 256


def auto_min_count(hist) -> int:
    """min_count at the valley of a k-mer spectrum (256 bins, KmerCounter.histogram()): kh_count_auto_min_count.
    None gives the default, 2."""
    if hist is None:
        return int(lib().kh_count_auto_min_count(None))
    h = np.ascontiguousarray(hist, dtype=np.uint64)
    if h.shape != (HIST_BINS,):
        raise ValueError(f"a spectrum has {HIST_BINS} bins, got shape {h.shape}")
    return int(lib().kh_count_auto_min_count(h.ctypes.data_as(C.POINTER(C.c_uint64))))


def record_bytes(k: int) -> int:
    """Bytes of one record of kh_count_partition: a counter slot, 16 (K <= 31) or 32."""
    return 16 if k <= 31 else 32
