"""Unitig extensions (kh_count_link_check_device) on one GPU, over the records extract left on the device.

    python tools/link_bench.py [reps] [out.jsonl]

Per shape, the depth_bench.py recipe: a chr14-shaped contig set of 16 M k-mers, reads tiled over it at 8 passes of 150
bases, counted into a table of twice the distinct k-mers (0.5 GB at K = 31, 1 GB at K = 51 -- far past the 126 MB of
L2), then extract_device(2, 2).  The check reads that extract buffer in place of residence and writes a second device
buffer, so every call sees the same input; it is timed with a host clock around the synchronous call (2 warm-up calls,
median of `reps`).  Rates: records/s, and lookups/s (two per record: successor and predecessor) over the random-sector
rate of a table-sized footprint (kh_measure_random_sector_rate).  `verified`: on the generator's linear chains the rule
cuts nothing, so n_cut = 0 and the output equals the extract byte for byte.  One JSON line per shape, with the GPU's
name and power limit read in the same run."""
import ctypes as C
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from tools.depth_bench import gpu_identity  # noqa: E402

SHAPES = [(31, 16_000_000), (51, 16_000_000)]                # (K, k-mers)


def run(k, n, coverage=8, read_len=150, reps=7, seed=267):
    import cs267_hw3_b200 as kh
    from tools import kmergen, readgen

    c = max(1, round(n * 860329 / 89710742))
    d = kmergen.Dataset(k, n, c, seed=seed)
    reads = readgen.tile_reads(d.solution(), k, read_len=read_len, coverage=coverage, seed=seed)
    L = kh.lib()
    pb = kh.pair_bytes(k)
    out = {"workload": f"link_k{k}", "k": k, "n_kmers": n, "n_contigs": c, "coverage_passes": coverage, "read_len": read_len,
           "read_bytes": int(reads.size), "record_bytes": pb}
    with kh.KmerCounter(k, n, 0.5, device=0) as kc, kh.KmerHashTable(k, 1024, 0.5, device=0) as tab:
        p = C.c_void_p()
        assert L.kh_device_alloc(C.byref(p), reads.size) == 0
        tab._check(L.kh_copy_device(tab._h, p, reads.ctypes.data, reads.size))
        tab.sync()
        kc.count_reads_device(p.value, reads.size)
        st = kc.stats()
        L.kh_device_free(p)
        ptr, n_rec = kc.extract_device(2, 2)
        assert n_rec == n, (n_rec, n)
        dst = C.c_void_p()
        assert L.kh_device_alloc(C.byref(dst), n * pb) == 0
        ms, cuts = [], set()
        n0 = kc.stats()["n_launches"]
        for i in range(reps + 2):
            t0 = time.perf_counter()
            cuts.add(kc.link_check_device(ptr, dst.value, n, 2, 2))
            if i >= 2:
                ms.append((time.perf_counter() - t0) * 1e3)
        launches = kc.stats()["n_launches"] - n0
        a = np.empty(n * pb, dtype=np.uint8)
        b = np.empty(n * pb, dtype=np.uint8)
        tab._check(L.kh_copy_to_host(tab._h, a.ctypes.data, C.c_void_p(ptr), n * pb))
        tab._check(L.kh_copy_to_host(tab._h, b.ctypes.data, dst, n * pb))
        L.kh_device_free(dst)
        verified = bool(cuts == {0} and (a == b).all() and launches == reps + 2)
        table_bytes = st["n_slots"] * st["slot_bytes"]
    sector_rate = kh.random_sector_rate(0, table_bytes, 1 << 27)
    t = float(np.median(ms))
    recs_s = n / t * 1e3
    out.update({
        "table_bytes": int(table_bytes), "slot_bytes": int(st["slot_bytes"]),
        "ms_link": t, "ms_link_all": [round(x, 3) for x in ms], "records_per_s": recs_s, "lookups_per_s": 2 * recs_s,
        "random_sectors_per_s": sector_rate, "frac_random_sector_rate": 2 * recs_s / sector_rate,
        "ns_per_record": t * 1e6 / n, "n_cut": sorted(cuts), "verified": verified,
    })
    out.update(gpu_identity())
    return out


if __name__ == "__main__":
    reps = int(sys.argv[1]) if len(sys.argv) > 1 else 7
    sink = open(sys.argv[2], "a") if len(sys.argv) > 2 else None
    for k, n in SHAPES:
        line = json.dumps(run(k, n, reps=reps))
        print(line, flush=True)
        if sink:
            sink.write(line + "\n")
            sink.flush()
