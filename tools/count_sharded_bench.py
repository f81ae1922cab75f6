"""Sharded k-mer analysis (cs267_hw3_b200.sharded_count.ShardedCounter) on P GPUs: the count_bench.py workload (reads
tiled over a chr14-shaped contig set), split into P pieces at read boundaries, each piece resident in its rank's HBM.

    python tools/count_sharded_bench.py [--ranks 1,2,4,8] [--k 51] [--n 4000000] [--coverage 8] [--reps 3] [--shared]

One JSON line per rank count: milliseconds of the count (all ranks' kernels, host clock to the last synchronise), the
partition, the exchange + merge (peer copies + kc_merge_kernel) and the extract; records and bytes that cross to another
rank; `verified` = the union of the owned extracts equals one counter over all reads, record for record.  Rank counts
above the visible GPUs are skipped unless --shared (then ranks share devices: a correctness run, not a measurement)."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import cs267_hw3_b200 as kh  # noqa: E402
from cs267_hw3_b200.sharded_count import ShardedCounter, split_reads  # noqa: E402
from tools import kmergen, readgen  # noqa: E402


def _sorted_rows(a):
    return a[np.lexsort(a.T[::-1])] if a.size else a


def _gpu_info():
    import torch
    info = {"gpu": torch.cuda.get_device_name(0), "gpus_visible": torch.cuda.device_count()}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader"], capture_output=True, text=True, timeout=30)
        info["power_limit"] = q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else None
    except Exception:
        info["power_limit"] = None
    return info


def run(world, reads, k, n, reps, single):
    import torch
    ndev = kh.device_count()
    cuts = split_reads(reads, world)
    with ShardedCounter(k, world, n) as sc:
        dev = [torch.from_numpy(reads[cuts[r]:cuts[r + 1]].copy()).to(f"cuda:{sc.devices[r]}") for r in range(world)]
        torch.cuda.synchronize()
        times = {"ms_count": [], "ms_partition": [], "ms_exchange_merge": [], "ms_extract": []}
        for rep in range(reps + 1):                     # the first repetition warms up
            sc.clear()
            for c in sc.batch + sc.owned:
                c.stats()
            t0 = time.perf_counter()
            for r in range(world):
                sc.count_device(r, dev[r].data_ptr(), dev[r].numel())
            for c in sc.batch:
                c.stats()                               # waits for the rank's kernels
            t1 = time.perf_counter()
            sc.reduce()
            t2 = time.perf_counter()
            got = sc._each(lambda r: sc.extract_device(r, 2, 2))
            t3 = time.perf_counter()
            if rep:
                times["ms_count"].append((t1 - t0) * 1e3)
                times["ms_partition"].append(sc.last_reduce["ms_partition"])
                times["ms_exchange_merge"].append(sc.last_reduce["ms_exchange_merge"])
                times["ms_extract"].append((t3 - t2) * 1e3)
        n_rep = sum(x[1] for x in got)
        union = _sorted_rows(np.concatenate([sc.extract(r, 2, 2) for r in range(world)]))
        verified = bool(n_rep == n and union.shape == single.shape and (union == single).all())
        st = sc.stats()
        lr = sc.last_reduce
        del dev
    med = {key: round(float(np.median(v)), 3) for key, v in times.items()}
    return {"ranks": world, "devices_used": min(world, ndev), "ranks_share_devices": world > ndev, **med,
            "ms_total": round(sum(med.values()), 3), "occurrences": int(st["n_occurrences"]), "distinct": int(st["n_distinct"]),
            "records_partitioned": lr["records"], "records_to_other_ranks": lr["records_to_other_ranks"],
            "bytes_exchanged": lr["records_to_other_ranks"] * lr["record_bytes"], "verified": verified}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--ranks", default="1,2,4,8")
    ap.add_argument("--k", type=int, default=51)
    ap.add_argument("--n", type=int, default=4_000_000)
    ap.add_argument("--coverage", type=int, default=8)
    ap.add_argument("--read-len", type=int, default=150)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--seed", type=int, default=267)
    ap.add_argument("--shared", action="store_true", help="also run rank counts above the visible GPUs (correctness only)")
    a = ap.parse_args()
    if kh.device_count() < 1:
        raise SystemExit("count_sharded_bench: no CUDA device")
    k, n = a.k, a.n
    c = max(1, round(n * 860329 / 89710742))
    d = kmergen.Dataset(k, n, c, seed=a.seed)
    reads = readgen.tile_reads(d.solution(), k, read_len=a.read_len, coverage=a.coverage, seed=a.seed)
    with kh.KmerCounter(k, n, 0.5, 0) as one:
        one.count_reads(reads)
        single = _sorted_rows(one.extract(2, 2))
    base = {"workload": f"reads_k{k}", "k": k, "n_kmers": n, "coverage_passes": a.coverage, "read_len": a.read_len,
            "read_bytes": int(reads.size), **_gpu_info(),
            "timing": "host clock, median of reps after one warm-up; every step ends host-synchronous"}
    for w in [int(x) for x in a.ranks.split(",")]:
        if w > kh.device_count() and not a.shared:
            continue
        print(json.dumps({**base, **run(w, reads, k, n, a.reps, single)}), flush=True)


if __name__ == "__main__":
    main()
