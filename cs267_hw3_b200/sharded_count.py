"""k-mer analysis over several ranks (GPUs) in this process: the Python twin of kh_sharded::CountCluster
(include/kh/sharded_counter.hpp).

Every rank counts its reads into a batch counter; reduce() partitions every batch by owner rank (kh_count_partition),
every owner merges the group addressed to it from every rank into its owned counter (kh_count_merge_device: one peer
copy per group), and clears the batches.  Counters saturate field by field, and saturating sums are associative, so the
union of the owned extracts is exactly what one counter over all reads reports -- when every rank's reads begin and end
at a non-base byte (split_reads) and nothing is thresholded before the reduce.  Rank r lives on device r % device_count().
"""
from __future__ import annotations

import time
from concurrent.futures import ThreadPoolExecutor

import numpy as np

from .sharded import _fmix64

_M64 = (1 << 64) - 1
_BASES = np.frombuffer(b"ACGT", dtype=np.uint8)


def count_owner(key_hi: int, key_lo: int, world: int) -> int:
    """Mirror of kc_owner() (csrc/count_core.cuh): the rank that owns a k-mer (right-justified base-4 key)."""
    h = _fmix64(key_lo ^ ((key_hi * 0x9E3779B97F4A7C15) & _M64))
    return (_fmix64(h ^ 0xD6E8FEB86659FD93) * world) >> 64


def owner_of_record(rec: bytes, k: int, world: int) -> int:
    """Owner rank of a kmer_pair record (packed k-mer first, as kh_count_extract writes it)."""
    pl = (k + 3) // 4
    key = int.from_bytes(bytes(rec[:pl]), "big") >> (8 * pl - 2 * k)
    return count_owner(key >> 64, key & _M64, world)


def split_reads(text, world: int) -> list[int]:
    """world + 1 cut points splitting text into world pieces of about equal size.  A cut lies at 0, at the end or right
    behind a byte that is not a base, so no k-mer and no extension observation spans two pieces (kh_sharded::split_reads)."""
    t = np.frombuffer(text, dtype=np.uint8) if not isinstance(text, np.ndarray) else text
    n = t.size
    sep = np.flatnonzero(~np.isin(t, _BASES)) + 1            # positions right behind a non-base byte
    cuts = [0]
    for r in range(1, world):
        c = max(cuts[-1], n * r // world)
        if 0 < c < n and t[c - 1] in _BASES:
            i = int(np.searchsorted(sep, c))
            c = int(sep[i]) if i < sep.size else n
        cuts.append(c)
    cuts.append(n)
    return cuts


class ShardedCounter:
    """k-mer analysis of one read set on `world` ranks; rank r on device r % device_count().  Ranks with a device of
    their own run side by side on host threads, ranks that share one run in turn (every step is host-synchronous)."""

    def __init__(self, k: int, world: int, n_distinct_expected_total: int, load_factor: float = 0.5):
        import cs267_hw3_b200 as kh

        ndev = kh.device_count()
        if ndev < 1:
            raise kh.KhError(kh.KH_ERR_CUDA, "ShardedCounter: no CUDA device (there is no CPU fallback)")
        if not 1 <= world <= 64:
            raise ValueError("world must be between 1 and 64")
        self.k, self.world = k, world
        self.devices = [r % ndev for r in range(world)]
        share = n_distinct_expected_total // world + n_distinct_expected_total // (8 * world) + 4096
        self.batch, self.owned = [], []
        for r in range(world):
            self.batch.append(kh.KmerCounter(k, n_distinct_expected_total, load_factor, self.devices[r]))
            self.owned.append(kh.KmerCounter(k, share, load_factor, self.devices[r]))
        self._occ = [0] * world
        self._bytes = [0] * world
        self._pool = ThreadPoolExecutor(world) if 1 < world <= ndev else None
        self.last_reduce = {}

    def _each(self, fn) -> list:
        if self._pool is None:
            return [fn(r) for r in range(self.world)]
        return list(self._pool.map(fn, range(self.world)))

    def close(self) -> None:
        if self._pool is not None:
            self._pool.shutdown()
            self._pool = None
        for c in self.batch + self.owned:
            c.close()

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    # -- counting: reads must begin and end at a non-base byte --
    def count(self, rank: int, reads) -> None:
        self.batch[rank].count_reads(reads)

    def count_device(self, rank: int, dev_ptr: int, n_bytes: int) -> None:
        """Reads in memory of device `self.devices[rank]`; only enqueued, the buffer must live until the next reduce."""
        self.batch[rank].count_reads_device(dev_ptr, n_bytes)

    def reduce(self) -> None:
        """Every rank's batch into the owners' counters, then clear the batches.  self.last_reduce: records exchanged
        and the host-clock times of the two steps (each ends host-synchronous)."""
        import cs267_hw3_b200 as kh

        rb = kh.record_bytes(self.k)
        t0 = time.perf_counter()
        parts = self._each(lambda r: self.batch[r].partition(self.world))
        t1 = time.perf_counter()

        def merge_into(o):
            for i in range(self.world):
                r = (o + i) % self.world                        # owners start at different sources
                ptr, offs = parts[r]
                n = int(offs[o + 1] - offs[o])
                if n:
                    self.owned[o].merge_device(ptr + int(offs[o]) * rb, n)

        self._each(merge_into)
        t2 = time.perf_counter()

        def clear(r):
            st = self.batch[r].stats()
            self._occ[r] += st["n_occurrences"]
            self._bytes[r] += st["n_bytes"]
            self.batch[r].clear()

        self._each(clear)
        n_rec = sum(int(offs[-1]) for _, offs in parts)
        n_remote = sum(int(offs[-1]) - int(offs[r + 1] - offs[r]) for r, (_, offs) in enumerate(parts))
        self.last_reduce = {"records": n_rec, "records_to_other_ranks": n_remote, "record_bytes": rb,
                            "ms_partition": (t1 - t0) * 1e3, "ms_exchange_merge": (t2 - t1) * 1e3}

    def clear(self) -> None:
        """Forget everything counted and reduced (the tables keep their size)."""
        for c in self.batch + self.owned:
            c.clear()
        self._occ = [0] * self.world
        self._bytes = [0] * self.world

    # -- after reduce(): what each rank owns --
    def extract(self, rank: int, min_count: int = 2, min_ext: int = 2) -> np.ndarray:
        return self.owned[rank].extract(min_count, min_ext)

    def extract_device(self, rank: int, min_count: int = 2, min_ext: int = 2) -> tuple[int, int]:
        return self.owned[rank].extract_device(min_count, min_ext)

    def extract_lines(self, rank: int, min_count: int = 2, min_ext: int = 2) -> np.ndarray:
        return self.owned[rank].extract_lines(min_count, min_ext)

    def extract_unitigs(self, rank: int, min_count: int = 2, min_ext: int = 2) -> tuple[np.ndarray, int]:
        """After reduce(): rank's records with unitig extensions (KmerCounter.link_check) and the sides cut.  Every owner,
        starting at `rank`, checks the sides whose neighbour it owns; the partials give exactly the one-counter records."""
        pairs, n_cut = self.owned[rank].extract(min_count, min_ext), 0
        for i in range(self.world):
            o = (rank + i) % self.world
            pairs, cut = self.owned[o].link_check(pairs, min_count, min_ext, self.world, o)
            n_cut += cut
        return pairs, n_cut

    def histogram(self) -> np.ndarray:
        """After reduce(): the k-mer spectrum of everything reduced so far, uint64[256] (KmerCounter.histogram()).  Every
        k-mer has one owner and the owned counters equal one counter's, so the sum of the owners' spectra is exact."""
        return np.sum([c.histogram() for c in self.owned], axis=0, dtype=np.uint64)

    def contig_depth(self, text, offsets) -> np.ndarray:
        """After reduce(): KmerCounter.contig_depth against everything reduced so far.  Owner o looks up the windows
        whose k-mer it owns; every k-mer has one owner, so the combined partials are exactly one counter's records."""
        import cs267_hw3_b200 as kh

        return kh.combine_depth(self._each(lambda o: self.owned[o].contig_depth(text, offsets, self.world, o)))

    def lookup(self, rank: int, pkmers) -> np.ndarray:
        return self.owned[rank].lookup(pkmers)

    def stats(self) -> dict:
        """Totals: occurrences and read bytes counted on all ranks, distinct k-mers reduced so far."""
        b = [c.stats() for c in self.batch]
        return {"n_occurrences": sum(self._occ) + sum(s["n_occurrences"] for s in b),
                "n_bytes": sum(self._bytes) + sum(s["n_bytes"] for s in b),
                "n_distinct": sum(c.stats()["n_distinct"] for c in self.owned)}
