"""Contig depth (kh_count_contig_depth_device) on one GPU, over contigs resident where the assembly left them.

    python tools/depth_bench.py [reps]

Per shape, the count_bench.py recipe: a chr14-shaped contig set of 16 M k-mers, reads tiled over it at 8 passes of
150 bases, counted (kc_count_kernel, CUDA events) into a table of 0.5 GB (K = 31) / 1 GB (K = 51) -- far past the
126 MB of L2 -- then extract, insert and assemble_device.  The depth call is timed with a host clock around the
synchronous call (warm-up, median of `reps`).  Rates: k-mers/s; bytes at 33 B per k-mer (1 text byte + one slot
sector) over the HBM copy rate; lookups/s over the random-sector rate of a table-sized footprint
(kh_measure_random_sector_rate); and, on the same table, kc_count_kernel's occurrences/s -- the depth kernel does a
strict subset of the count kernel's per-position work, so it should cost no more per k-mer.  `verified`: the records
of ~1000 sampled contigs (the longest among them) against their windows packed on the host and looked up with
KmerCounter.lookup, an independent kernel path.  One JSON line per shape, with the GPU's name and power limit."""
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

SHAPES = [(31, 16_000_000, 0), (51, 16_000_000, 0), (51, 16_000_000, 10 ** 6)]      # (K, k-mers, long_nodes)
_ACGT = np.frombuffer(b"ACGT", dtype=np.uint8)


def pack_windows(s: bytes, k: int) -> np.ndarray:
    """Every window of an ACGT-only byte string, packed like pkmer_t (2 bits per base, first base on top, A-padded)."""
    code = np.zeros(256, dtype=np.uint8)
    code[_ACGT] = np.arange(4, dtype=np.uint8)
    cs = code[np.frombuffer(s, dtype=np.uint8)]
    nw, pl = len(s) - k + 1, (k + 3) // 4
    out = np.zeros((max(nw, 0), pl), dtype=np.uint8)
    for b in range(pl):
        for i in range(4):
            if 4 * b + i < k and nw > 0:
                out[:, b] |= cs[4 * b + i: 4 * b + i + nw] << np.uint8(6 - 2 * i)
    return out


def lookup_depth(kc, text, offs, k, contigs) -> np.ndarray:
    """kh_contig_depth records of ACGT-only contigs (a trailing '\\n' allowed), from their windows packed on the host
    and looked up with KmerCounter.lookup."""
    import cs267_hw3_b200 as kh
    out = np.zeros(len(contigs), dtype=kh.DEPTH_DTYPE)
    for j, c in enumerate(contigs):
        s = bytes(text[int(offs[c]):int(offs[c + 1])]).rstrip(b"\n")
        v = kc.lookup(pack_windows(s, k))[:, 0] if len(s) >= k else np.zeros(0, dtype=np.uint32)
        out[j] = (v.size, int(v.astype(np.uint64).sum()), int(v.min()) if v.size else 0xFFFFFFFF, int(v.max()) if v.size else 0)
    return out


def gpu_identity() -> dict:
    import torch
    info = {"gpu": torch.cuda.get_device_name(0), "power_limit_w": None}
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits", "-i", "0"],
                           capture_output=True, text=True, timeout=30)
        info["power_limit_w"] = float(r.stdout.strip().splitlines()[0])
    except Exception:
        pass
    return info


def run(k, n, long_nodes=0, coverage=8, read_len=150, reps=7, seed=267):
    import cs267_hw3_b200 as kh
    from tools import kmergen, readgen

    c = max(1, round(n * 860329 / 89710742))
    d = kmergen.Dataset(k, n, c, seed=seed, long_nodes=long_nodes)
    reads = readgen.tile_reads(d.solution(), k, read_len=read_len, coverage=coverage, seed=seed)
    L = kh.lib()
    out = {"workload": f"depth_k{k}" + ("_long" if long_nodes else ""), "k": k, "n_kmers": n, "n_contigs": c,
           "long_nodes": long_nodes, "coverage_passes": coverage, "read_len": read_len, "read_bytes": int(reads.size)}
    with kh.KmerCounter(k, n, 0.5, device=0) as kc, kh.KmerHashTable(k, n, 0.5, device=0) as tab:
        p = C.c_void_p()
        assert L.kh_device_alloc(C.byref(p), reads.size) == 0
        tab._check(L.kh_copy_device(tab._h, p, reads.ctypes.data, reads.size))
        tab.sync()
        ms_count = []
        for _ in range(3):
            kc.clear()
            kc.count_reads_device(p.value, reads.size)
            st = kc.stats()
            ms_count.append(st["ms_count"])
        L.kh_device_free(p)
        ptr, n_rec = kc.extract_device(2, 2)
        assert n_rec == n, (n_rec, n)
        tab.insert_pairs_device(ptr, n_rec)
        cp, op, nc, nb, nodes = tab.assemble_device()
        dout = C.c_void_p()
        assert L.kh_device_alloc(C.byref(dout), max(nc, 1) * 24) == 0
        ms = []
        for i in range(reps + 2):
            t0 = time.perf_counter()
            kc.contig_depth_device(cp, op, nc, dout.value)
            if i >= 2:
                ms.append((time.perf_counter() - t0) * 1e3)
        rec = np.zeros(nc, dtype=kh.DEPTH_DTYPE)
        tab._check(L.kh_copy_to_host(tab._h, rec.ctypes.data, dout, nc * 24))
        L.kh_device_free(dout)
        text, offs, _ = tab.assemble()
        rng = np.random.default_rng(seed)
        sample = np.unique(np.concatenate(([int(np.argmax(np.diff(offs)))], rng.choice(nc, size=min(nc, 1000), replace=False))))
        want = lookup_depth(kc, text, offs, k, sample)
        verified = bool((rec[sample] == want).all() and int(rec["n_kmers"].sum()) == nodes == n)
        table_bytes = st["n_slots"] * st["slot_bytes"]
        occ = st["n_occurrences"]
    sector_rate = kh.random_sector_rate(0, table_bytes, 1 << 27)
    peak = 6543.4
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            peak = float(json.load(f).get("hbm_gbs", peak))
    except Exception:
        pass
    t = float(np.median(ms))
    t_count = float(np.median(ms_count[1:]))
    kmers_s = n / t * 1e3
    out.update({
        "table_bytes": int(table_bytes), "slot_bytes": int(st["slot_bytes"]), "contig_bytes": int(nb),
        "ms_depth": t, "ms_depth_all": [round(x, 3) for x in ms], "kmers_per_s": kmers_s,
        "gbs_at_33B_per_kmer": 33 * kmers_s / 1e9, "hbm_gbs": peak, "frac_hbm": 33 * kmers_s / 1e9 / peak,
        "random_sectors_per_s": sector_rate, "frac_random_sector_rate": kmers_s / sector_rate,
        "ms_count_kernel": t_count, "count_occurrences": int(occ), "count_occurrences_per_s": occ / t_count * 1e3,
        "depth_ns_per_kmer": t * 1e6 / n, "count_ns_per_occurrence": t_count * 1e6 / occ,
        "sampled_contigs": int(sample.size), "verified": verified,
    })
    out.update(gpu_identity())
    return out


if __name__ == "__main__":
    reps = int(sys.argv[1]) if len(sys.argv) > 1 else 7
    for k, n, longn in SHAPES:
        print(json.dumps(run(k, n, longn, reps=reps)), flush=True)
