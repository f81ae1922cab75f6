"""Throughput of the k-mer analysis stage (kh_count_*) on one GPU: reads tiled over a chr14-shaped contig set.

    python tools/count_bench.py [K] [n_kmers] [coverage] [read_len]

Prints one JSON line: occurrences/s with the reads resident in HBM (CUDA events around the count kernel, table cleared
before every repetition), through host buffers (H2D inside), the extract pass, and the closed loop into insert + traverse.
Verified against the generator: the reported k-mers are exactly the data set's, the contigs its solution."""
import ctypes as C
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import cs267_hw3_b200 as kh  # noqa: E402
from tools import kmergen, readgen  # noqa: E402


def run(k=51, n=4_000_000, coverage=8, read_len=150, reps=5, seed=267):
    c = max(1, round(n * 860329 / 89710742))
    d = kmergen.Dataset(k, n, c, seed=seed)
    t0 = time.time()
    reads = readgen.tile_reads(d.solution(), k, read_len=read_len, coverage=coverage, seed=seed)
    gen_s = time.time() - t0
    L = kh.lib()
    out = {"workload": f"reads_k{k}", "k": k, "n_kmers": n, "n_contigs": c, "coverage_passes": coverage, "read_len": read_len,
           "read_bytes": int(reads.size), "gen_s": round(gen_s, 2)}
    with kh.KmerCounter(k, n, 0.5, device=0) as kc, kh.KmerHashTable(k, n, 0.5, device=0) as tab:
        p = C.c_void_p()
        assert L.kh_device_alloc(C.byref(p), reads.size) == 0
        tab._check(L.kh_copy_device(tab._h, p, reads.ctypes.data, reads.size))
        tab.sync()
        ms_dev, ms_ext = [], []
        for _ in range(reps):
            kc.clear()
            kc.count_reads_device(p.value, reads.size)
            st = kc.stats()
            ms_dev.append(st["ms_count"])
            ptr, n_rec = kc.extract_device(2, 2)
            ms_ext.append(kc.stats()["ms_extract"])
        occ = st["n_occurrences"]
        assert n_rec == n, (n_rec, n)
        tab.insert_pairs_device(ptr, n_rec)
        buf, offs, nodes = tab.assemble()
        ts = tab.stats()
        lines = sorted(buf.tobytes().split(b"\n")[:-1])
        verified = nodes == n and b"\n".join(lines) + b"\n" == d.solution()
        pin = kh.PinnedBuffer(reads.size)
        pin.array[:] = reads
        ms_host = []
        for _ in range(3):
            kc.clear()
            kc.stats()
            t0 = time.perf_counter()
            kc.count_reads_ptr(pin.ptr, reads.size)
            ms_host.append((time.perf_counter() - t0) * 1e3)
        pin.free()
        L.kh_device_free(p)
    ms = float(np.median(ms_dev[1:]))
    peaks = {}
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            peaks = json.load(f)
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6543.4))
    alg = 65 * occ                                            # 1 character + slot sector read + written back
    out.update({
        "occurrences": int(occ), "distinct": int(st["n_distinct"]), "slot_bytes": int(st["slot_bytes"]),
        "ms_count_device": ms, "occurrences_per_s": occ / ms * 1e3,
        "ms_count_all": [round(x, 3) for x in ms_dev],
        "roofline": {"bound": "hbm", "kernel": "kc_count_kernel", "achieved": alg / ms / 1e6, "peak": peak, "unit": "GB/s",
                     "frac": alg / ms / 1e6 / peak, "alg_bytes_per_occurrence": 65, "traffic": None},
        "ms_extract": float(np.median(ms_ext[1:])), "ms_count_host_buffers": float(np.median(ms_host[1:])),
        "host_gbs": reads.size / float(np.median(ms_host[1:])) / 1e6,
        "then_insert_ms_first_call": ts["ms_insert"], "then_assemble_ms_first_call": ts["ms_assemble"], "verified": bool(verified),
    })
    # a bounded piece of the same reads for bench.py's CPU leg (whole lines, about 8 MB); not part of the JSON record
    cut = int(np.flatnonzero(reads[: 8 << 20] == 10)[-1]) + 1
    out["_sample"] = reads[:cut]
    return out


if __name__ == "__main__":
    rec = run(*[int(x) for x in sys.argv[1:]])
    rec.pop("_sample", None)
    print(json.dumps(rec))
