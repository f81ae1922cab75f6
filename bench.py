#!/usr/bin/env python
"""bench.py -- k-mers/s over insert + traverse (the timed region of kmer_hash.cpp:129-137).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]

A "step" is one pass of the hot path over one batch of synthetic input: empty table ->
insert every k-mer + find the start nodes -> walk every contig -> contig text materialised.
The workload is BASELINE.json configs[2]/[3]: the human-chr14 shape at K=51 (89 710 742 unique 51-mers in
860 329 contigs, 4 934 090 810 bytes of text, 128-bit slots), synthetic (tools/kmer_gen.cpp), the same file at
every N (strong scaling).  configs[1] (the same shape re-cut at K=19, 64-bit slots) is measured in the same run
and reported under "shapes".

One JSON line on stdout (rank 0); see README/DESIGN.md for the keys.  `value` has the packed
records resident in HBM when the clock starts (as the reference has them resident in host RAM);
`e2e` runs the same step through the host-buffer C ABI calls (kh_insert_pairs / kh_assemble) with
the H2D of the records and the D2H of the contigs inside the timed region.

--dump-outputs DIR writes what the last timed step of the main workload produced (see dump_outputs) as .npy files, so
that two builds can be compared output for output: the inputs are generated from a fixed seed.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

METRIC = "kmers_per_s_insert_plus_traverse"
UNIT = "k-mers/s"
WORKLOADS = {
    # name: (k, n_kmers, n_contigs, long_nodes)
    "chr14_k19": (19, 89_710_742, 860_329, 0),        # BASELINE.json configs[1]
    "chr14_k51": (51, 89_710_742, 860_329, 0),        # configs[2]
    "chr14_k31": (31, 89_710_742, 860_329, 0),        # per-GPU share of the whole-genome shape (configs[4], K=31)
    "chr14_k51_long": (51, 89_710_742, 8_603, 1_000_000),
    "test_k19": (19, 4_514_197, 5_736, 0),            # test.txt shape
    "small_k19": (19, 977_112, 1_000, 0),             # configs[0] (CPU reference case)
}
SEED = 267


def measured_peak_gbs() -> tuple[float, str]:
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_traffic_bytes(kernel_substr: str):
    """DRAM bytes (read + write) per launch of a kernel from the committed ncu --set full capture
    (profiles/r01_final_ncu_full_summary.csv, chr14_k19 workload); None if the file or the kernel is missing."""
    import csv
    p = os.path.join(ROOT, "profiles", "r01_final_ncu_full_summary.csv")
    try:
        rows = list(csv.reader(open(p)))
        h, units = rows[0], rows[1]
        ir, iw, ik = h.index("dram__bytes_read.sum"), h.index("dram__bytes_write.sum"), h.index("Kernel Name")
        scale = {"Gbyte": 1e9, "Mbyte": 1e6, "Kbyte": 1e3, "byte": 1.0}
        for r in rows[2:]:
            if kernel_substr in r[ik]:
                return float(r[ir]) * scale.get(units[ir], 1e9) + float(r[iw]) * scale.get(units[iw], 1e9)
    except Exception:
        pass
    return None


def alg_bytes_per_kmer(k: int) -> dict:
    pb = (k + 3) // 4 + 2
    # SURVEY.md 8(d): record read + insert sector read+write-back + successor sector read + output byte
    return {"record": pb, "insert": 64, "lookup": 32, "output": 1, "total": pb + 97}


DUMP_BLOCK = 4096                                       # elements per sampled block
DUMP_CAP = {"contigs": 8 << 20, "offsets": 2 << 20}     # elements kept per array: 32 MB as float32 + 16 MB as float64
DUMP_MAX_BYTES = 64 << 20


def dump_sample(n: int, cap: int, seed: int = SEED):
    """Which blocks of an n-element output to keep: None (every element) when n <= cap, else the sorted numbers of a
    fixed, seeded choice of DUMP_BLOCK-element blocks, at most cap elements in all."""
    if n <= cap:
        return None
    n_blocks = (n + DUMP_BLOCK - 1) // DUMP_BLOCK
    return np.sort(np.random.default_rng(seed).choice(n_blocks, cap // DUMP_BLOCK, replace=False))


def dump_outputs(out_dir: str, contigs: np.ndarray, offsets: np.ndarray, n_nodes: int) -> dict:
    """What kh_assemble_device hands its caller: the contig text (ASCII codes of '\\n'-terminated contigs) as contigs.npy
    (float32), the n_contigs + 1 byte offsets into it as offsets.npy (float64), and counts.npy (float64: n_contigs,
    contig bytes, nodes).  An array longer than its DUMP_CAP is replaced by a seeded sample of whole blocks, and
    <name>_blocks.npy holds the numbers of the blocks kept (element i of block b is element b * DUMP_BLOCK + i).
    Returns {file name: bytes written}."""
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"counts": np.array([offsets.size - 1, contigs.size, n_nodes], dtype=np.float64)}
    for name, a, dtype in (("contigs", contigs, np.float32), ("offsets", offsets, np.float64)):
        blocks = dump_sample(a.size, DUMP_CAP[name])
        if blocks is not None:
            idx = (blocks[:, None] * DUMP_BLOCK + np.arange(DUMP_BLOCK)).ravel()
            a = a[idx[idx < a.size]]
            arrays[name + "_blocks"] = blocks.astype(np.float64)
        arrays[name] = a.astype(dtype)
    assert sum(a.nbytes for a in arrays.values()) <= DUMP_MAX_BYTES
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)
    return {name + ".npy": int(a.nbytes) for name, a in arrays.items()}


class ClockSampler:
    """SM clock, power and throttle reasons of one GPU during the timed region.  NVML in a background thread (the
    numbers `nvidia-smi --query-gpu=clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.*` prints; nvidia-smi itself
    needs more than a second to start on an 8-GPU box, longer than a whole timed loop), nvidia-smi as the fallback."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.proc, self.lines, self.samples, self.t, self.stop_flag, self.mode = index, None, [], [], None, False, None

    def _nvml_loop(self, nv, h):
        bits = {"hw_slowdown": nv.nvmlClocksEventReasonHwSlowdown, "hw_thermal_slowdown": nv.nvmlClocksEventReasonHwThermalSlowdown,
                "sw_thermal_slowdown": nv.nvmlClocksEventReasonSwThermalSlowdown, "sw_power_cap": nv.nvmlClocksEventReasonSwPowerCap}
        mx = float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM))
        while not self.stop_flag:
            try:
                sm = float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
                pw = nv.nvmlDeviceGetPowerUsage(h) / 1000.0
                r = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
                self.samples.append((sm, mx, pw, [k for k, b in bits.items() if r & b]))
            except Exception:
                pass
            time.sleep(0.002)

    def start(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            idx = int(vis.split(",")[self.index]) if vis and all(x.strip().isdigit() for x in vis.split(",")) else self.index
            h = nv.nvmlDeviceGetHandleByIndex(idx)
            self.mode = "nvml"
            self.t = threading.Thread(target=self._nvml_loop, args=(nv, h), daemon=True)
            self.t.start()
            return
        except Exception:
            self.mode = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=lambda: self.lines.extend(self.proc.stdout), daemon=True)
            self.t.start()
            self.mode = "nvidia-smi"
        except Exception:
            self.proc = None

    def stop(self) -> dict:
        if self.mode == "nvml":
            self.stop_flag = True
            self.t.join(timeout=2)
            if not self.samples:
                return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
            reasons = sorted({r for s_ in self.samples for r in s_[3]})
            return {"sm_mhz": float(np.median([s_[0] for s_ in self.samples])), "sm_max_mhz": max(s_[1] for s_ in self.samples),
                    "power_w_max": max(s_[2] for s_ in self.samples), "samples": len(self.samples), "reasons": reasons,
                    "source": "NVML (clock, power, clocks-event reasons), 2 ms period"}
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        self.t.join(timeout=2)
        sm, mx, reasons, power = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1])); power.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(names, f[4:8]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": max(mx), "power_w_max": max(power),
                "samples": len(sm), "reasons": sorted(reasons), "source": "nvidia-smi -lms 20"}


# ------------------------------------------------------------------ reference arm ---------
def run_reference_arm(args, k: int, workload: str) -> dict:
    """Times the reference's own CPU implementation of the path: oracle/_ref/kmer_hash_ref_<K>
    (the UNMODIFIED /root/reference/kmer_hash.cpp, single-rank UPC++ stand-in) on a bounded
    sample of the workload; the numbers are the program's own timer lines (same timed region)."""
    import oracle
    from tools import kmergen

    _, n_full, c_full, _ = WORKLOADS[workload]
    if oracle.ref_binary(k) is None:
        raise RuntimeError(f"oracle/_ref/kmer_hash_ref_{k} missing: run `make -C oracle` where /root/reference exists")
    mean_nodes = n_full / c_full
    runs = args.steps + args.warmup
    work = tempfile.mkdtemp(prefix="kh_ref_")

    def make(n):
        d = kmergen.Dataset(k, n, max(1, int(round(n / mean_nodes))), seed=SEED)
        p = os.path.join(work, f"sample_{n}.txt")
        d.text().tofile(p)
        return p

    # calibrate on 200k k-mers, then size the sample so all runs fit in ~150 s
    t_cal = oracle.run_reference(k, make(200_000), work, test=False)[1]
    rate = 200_000 / max(t_cal, 1e-6)
    n_s = int(min(n_full, 4_514_197, max(200_000, rate * 150.0 / max(runs, 1) * 0.6)))
    path = make(n_s)
    ins, tot = [], []
    for i in range(runs):
        a, b = oracle.run_reference(k, path, work, test=False)
        if i >= args.warmup:
            ins.append(a); tot.append(b)
    for f in os.listdir(work):
        os.unlink(os.path.join(work, f))
    os.rmdir(work)
    t = float(np.mean(tot))
    value = n_s / t
    sample = (f"K={k}, {n_s} unique k-mers in {max(1, int(round(n_s / mean_nodes)))} contigs (same mean contig "
              f"length as {workload}), synthetic seed {SEED}; timer lines of the reference binary, mean of {len(tot)} runs")
    return {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": t * 1e3, "higher_is_better": True,
        "scaling": "weak" if args.gpus == 1 else "strong", "vs_baseline": None, "dtype": "u8 (std::string keys)",
        "data": "synthetic",
        "config": {"workload": workload, "k": k, "sample_kmers": n_s, "insert_s": float(np.mean(ins)), "total_s": t},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": 1, "kind": "reference", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }


def cpu_baseline_leg(k: int, workload: str, budget_s: float = 20.0) -> dict:
    import oracle
    from tools import kmergen

    _, n_full, c_full, _ = WORKLOADS[workload]
    if oracle.ref_binary(k) is None:
        return {"value": None, "unit": UNIT, "cores": 1, "kind": "reference", "sample": "oracle/_ref not built"}
    mean_nodes = n_full / c_full
    work = tempfile.mkdtemp(prefix="kh_cpu_")
    try:
        def run(n):
            d = kmergen.Dataset(k, n, max(1, int(round(n / mean_nodes))), seed=SEED)
            p = os.path.join(work, "s.txt")
            d.text().tofile(p)
            return oracle.run_reference(k, p, work, test=False)
        t_cal = run(200_000)[1]
        n_s = int(min(n_full, 4_514_197, max(200_000, 200_000 / max(t_cal, 1e-6) * budget_s)))
        ins, tot = run(n_s)
    finally:
        for f in os.listdir(work):
            os.unlink(os.path.join(work, f))
        os.rmdir(work)
    return {"value": n_s / tot, "unit": UNIT, "cores": 1, "kind": "reference",
            "sample": f"oracle/_ref/kmer_hash_ref_{k} (unmodified reference, 1 rank) on K={k}, {n_s} k-mers / "
                      f"{max(1, int(round(n_s / mean_nodes)))} contigs: insert {ins:.3f} s, total {tot:.3f} s",
            "insert_s": ins, "total_s": tot, "sample_kmers": n_s}


# ------------------------------------------------------------------ B200 arm --------------
def ncu_traffic_for(kernel_substr: str, workload: str):
    """DRAM bytes (read + write) per launch of a kernel from this round's committed ncu --set full capture of the same
    bench command (profiles/r02_ncu_full_summary_<workload>.csv); None if there is none."""
    import csv
    p = os.path.join(ROOT, "profiles", f"r02_ncu_full_summary_{workload}.csv")
    try:
        rows = list(csv.reader(open(p)))
        h, units = rows[0], rows[1]
        ir, iw, ik = h.index("dram__bytes_read.sum"), h.index("dram__bytes_write.sum"), h.index("Kernel Name")
        scale = {"Gbyte": 1e9, "Mbyte": 1e6, "Kbyte": 1e3, "byte": 1.0}
        for r in rows[2:]:
            if kernel_substr in r[ik]:
                return float(r[ir]) * scale.get(units[ir], 1e9) + float(r[iw]) * scale.get(units[iw], 1e9), p
    except Exception:
        pass
    return None, None


def measure_shape_n1(args, workload: str, steps: int, warmup: int, local_rank: int, full: bool,
                     dump_dir: str | None = None) -> dict:
    """One workload on one GPU: `steps` timed steps with the records resident in HBM, then the host-buffer leg.
    With `dump_dir`, the last timed step's output is written there (dump_outputs)."""
    import torch

    import cs267_hw3_b200 as kh
    from tools import kmergen

    k, n, c, longn = WORKLOADS[workload]
    if args.n:
        c = max(1, int(round(args.n * c / n)))
        n = args.n
    pb = kh.pair_bytes(k)
    t_gen = time.time()
    data = kmergen.Dataset(k, n, c, seed=SEED, long_nodes=longn)
    host = kh.PinnedBuffer(n * pb)
    data.pairs_into(host.ptr, 0, n)
    exp_digest = data.digest()
    t_gen = time.time() - t_gen

    stream = torch.cuda.current_stream()
    tab = kh.KmerHashTable(k, n, args.load_factor, device=local_rank)
    tab.set_stream(stream.cuda_stream)
    dev = torch.empty(n * pb, dtype=torch.uint8, device="cuda")
    dev.copy_(torch.from_numpy(host.array))
    torch.cuda.synchronize()

    def step_resident():
        tab.clear()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        tab.insert_pairs_device(dev.data_ptr(), n)
        out = tab.assemble_device()
        e1.record(stream)
        return e0, e1, out

    def step_e2e():
        tab.clear()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        tab.insert_pairs_ptr(host.ptr, n)
        buf, offs, nodes = tab.assemble(copy=False)
        e1.record(stream)
        return e0, e1, (buf, offs, nodes)

    sampler = ClockSampler(local_rank)      # sampled over warm-up + timed steps (the timed loop alone is < 0.1 s)
    sampler.start()
    for _ in range(warmup):
        step_resident()
    torch.cuda.synchronize()
    launches0 = tab.stats()["n_launches"]
    wall0 = time.perf_counter()
    keys = ["ms_insert", "ms_stage", "ms_build", "ms_walk", "ms_rank", "ms_emit", "ms_clear"]
    evs, stage = [], {key: [] for key in keys}
    for _ in range(steps):
        e0, e1, out = step_resident()
        evs.append((e0, e1))
        st = tab.stats()
        for key in stage:
            stage[key].append(st[key])
    torch.cuda.synchronize()
    wall = time.perf_counter() - wall0
    launches = tab.stats()["n_launches"] - launches0
    clocks = sampler.stop()
    ms = [a.elapsed_time(b) for a, b in evs]
    ms_per_step = float(np.mean(ms))
    contigs_dev, offsets_dev, n_contigs, contig_bytes, n_nodes = out
    st_last = tab.stats()
    dumped = None
    if dump_dir:
        contigs_h = np.empty(contig_bytes, dtype=np.uint8)
        offsets_h = np.empty(n_contigs + 1, dtype=np.uint64)
        tab._check(kh.lib().kh_copy_to_host(tab._h, contigs_h.ctypes.data, contigs_dev, contigs_h.nbytes))
        tab._check(kh.lib().kh_copy_to_host(tab._h, offsets_h.ctypes.data, offsets_dev, offsets_h.nbytes))
        dumped = dump_outputs(dump_dir, contigs_h, offsets_h, n_nodes)
        del contigs_h, offsets_h

    # correctness gate: re-run the traversal into host memory and compare the contig set with the generator's own
    # solution (order-independent digest) + node/contig counts
    buf, offs, nodes = tab.assemble(copy=False)
    verified = bool(n_nodes == n and n_contigs == c and nodes == n and kmergen.digest_lines(buf) == exp_digest)

    # end to end through host buffers: kh_insert_pairs (pinned records, chunked H2D overlapped with the staging
    # kernels) + kh_assemble (contigs copied back to pinned host memory)
    e2e = None
    if not args.no_e2e:
        for _ in range(min(warmup, 2)):
            step_e2e()
        torch.cuda.synchronize()
        e2e_ms = []
        for _ in range(max(1, min(steps, 5))):
            e0, e1, (buf, offs, nodes) = step_e2e()
            torch.cuda.synchronize()
            e2e_ms.append(e0.elapsed_time(e1))
        e2e_ms_mean = float(np.mean(e2e_ms))
        verified = verified and bool(nodes == n and kmergen.digest_lines(buf) == exp_digest)
        e2e = {"value": n / (e2e_ms_mean * 1e-3), "unit": UNIT, "ms_per_step": e2e_ms_mean,
               "h2d_bytes_per_step": n * pb, "d2h_bytes_per_step": int(contig_bytes + 8 * (n_contigs + 1))}

    # K1 (north star item a): text lines -> kmer_pair records on the GPU, device-resident text, bounded sample
    pack = None
    if full:
        try:
            n_pack = min(n, 16_000_000)
            text = torch.from_numpy(data.text(0, n_pack)).cuda()
            packed = torch.empty(n_pack * pb, dtype=torch.uint8, device="cuda")
            for _ in range(2):
                tab.pack_lines_device(text.data_ptr(), n_pack, packed.data_ptr())
            p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            p0.record(stream)
            for _ in range(5):
                tab.pack_lines_device(text.data_ptr(), n_pack, packed.data_ptr())
            p1.record(stream)
            torch.cuda.synchronize()
            pms = p0.elapsed_time(p1) / 5
            same = bool(np.array_equal(packed.cpu().numpy(), host.array[: n_pack * pb]))
            pack = {"lines": n_pack, "ms": pms, "lines_per_s": n_pack / (pms * 1e-3),
                    "gbs": n_pack * (k + 4 + pb) / (pms * 1e-3) / 1e9, "matches_generator_records": same}
            del text, packed
        except Exception as e:          # secondary number: never fail the bench line over it
            pack = {"error": str(e)}

    peak, peak_src = measured_peak_gbs()
    alg = alg_bytes_per_kmer(k)
    sm = {k2: float(np.mean(v)) for k2, v in stage.items()}
    chunk_table = sm["ms_build"] > 0
    if chunk_table:
        # The step's dominant kernel is ct_build_kernel: it inserts every k-mer (one table sector read + written back:
        # 64 B), follows every successor link (the 32-B lookup, served from shared memory) and produces the contig
        # characters (1 B) -- SURVEY.md 8(d)'s B_alg minus the record read, which belongs to ct_stage_kernel.
        dom, dom_ms, dom_bytes = "ct_build_kernel", sm["ms_build"], n * (alg["insert"] + alg["lookup"] + alg["output"])
    else:
        dom, dom_ms, dom_bytes = "walk_kernel", sm["ms_walk"], n * (alg["lookup"] + alg["output"])
    traffic, traffic_src = ncu_traffic_for(dom, workload) if not args.n else (None, None)
    achieved = dom_bytes / (dom_ms * 1e-3) / 1e9
    path_gbs = n * alg["total"] / (ms_per_step * 1e-3) / 1e9
    slot_b = st_last["slot_bits"] // 8
    out = {
        "ms_per_step": ms_per_step, "value": n / (ms_per_step * 1e-3), "ms_each_step": ms,
        "ms_per_step_median": float(np.median(ms)), "ms_per_step_best": float(np.min(ms)),
        "config": {"workload": workload, "k": k, "n_kmers": n, "n_contigs": c, "load_factor": args.load_factor, "seed": SEED,
                   "table": ("chunk table (csrc/ctable.cuh): one staging pass into per-chunk buffers, every chunk built + contracted in "
                             "shared memory, one HBM lookup per segment, contigs ranked and emitted by per-contig walks"
                             if chunk_table else "plain open-addressing table (csrc/kernels.cuh): shared-memory chunk build, splitter walk"),
                   "slot_bytes": slot_b,
                   "l2": "inputs (records, staging buffers, table) far larger than L2; every step starts from an empty table",
                   "table_clear": "between steps, outside the per-step event pair (the reference constructs its map "
                                  "before its timer, kmer_hash.cpp:119-129); ms_clear reported in stages",
                   "timing": "CUDA events on the launching stream around each step, mean of steps"},
        "stages_ms": dict(sm, ms_seal_and_links_etc=None) if False else sm,
        "n_segments": int(st_last["n_segments"]), "rank_rounds": int(st_last["rank_rounds"]),
        "assembly_time_s": ms_per_step * 1e-3, "wall_s_timed_loop": wall, "gen_s": t_gen, "verified": verified,
        "roofline": {"bound": "hbm", "kernel": dom, "achieved": achieved, "peak": peak, "unit": "GB/s",
                     "frac": achieved / peak, "traffic": traffic,
                     "traffic_source": ("dram__bytes_read.sum + dram__bytes_write.sum per launch, ncu --set full capture of this "
                                        "command: " + os.path.relpath(traffic_src, ROOT)) if traffic else None,
                     "peak_source": peak_src,
                     "units_per_launch": n, "alg_bytes_per_unit": dom_bytes // n, "kernel_ms": dom_ms,
                     "alg_bytes_per_kmer": alg,
                     "insert_stage": {"kernels": "ct_stage + ct_layout + ct_build (the build also does the traverse's lookups)"
                                      if chunk_table else "partition + subpartition + build_chunks / insert_slots",
                                      "ms": sm["ms_insert"]},
                     "path": {"achieved": path_gbs, "frac": path_gbs / peak,
                              "note": "N x B_alg / t(insert+traverse), SURVEY.md 8(d)"},
                     "probes_per_s": 2 * n / (ms_per_step * 1e-3),
                     "sector_ceiling_per_s": peak * 1e9 / 32},
        "e2e": e2e, "pack_lines": pack, "gpu_launches": int(launches), "clocks": clocks, "dumped": dumped,
    }
    tab.close()
    host.free()
    del dev
    torch.cuda.empty_cache()
    return out


def run_b200_arm(args, workload: str) -> dict | None:
    import torch
    import torch.distributed as dist

    import cs267_hw3_b200 as kh

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available() or kh.device_count() < 1:
        raise RuntimeError("bench.py: no CUDA device; the B200 arm has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    if world != args.gpus:
        raise RuntimeError(f"--gpus {args.gpus} but WORLD_SIZE={world}: launch with torch.distributed.run")
    second = [w for w in (args.also or []) if w != workload]
    if world > 1:
        from cs267_hw3_b200 import sharded
        line = sharded.bench(args, workload, rank, world, local_rank, args.steps, args.warmup)
        shapes = {w: sharded.bench(args, w, rank, world, local_rank, max(3, min(args.steps, 5)), 3) for w in second}
        if rank == 0:
            line["shapes"] = {w: {k2: v[k2] for k2 in ("value", "ms_per_step", "stages_ms", "e2e", "verified", "roofline", "config", "scaling")}
                              for w, v in shapes.items()}
        sharded.shutdown()
        return line if rank == 0 else None

    m = measure_shape_n1(args, workload, args.steps, args.warmup, local_rank, full=True, dump_dir=args.dump_outputs)
    k = WORKLOADS[workload][0]
    line = {
        "metric": METRIC, "value": m["value"], "unit": UNIT, "n_gpus": 1,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": m["ms_per_step"], "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "u64" if m["config"]["slot_bytes"] == 8 else "u128", "data": "synthetic",
    }
    for key in ("ms_per_step_median", "ms_per_step_best", "config", "stages_ms", "n_segments", "rank_rounds", "assembly_time_s",
                "wall_s_timed_loop", "gen_s", "verified", "roofline", "e2e", "pack_lines", "gpu_launches", "clocks"):
        line[key] = m[key]
    if m["dumped"]:
        line["dumped"] = {"dir": os.path.abspath(args.dump_outputs), "files": m["dumped"]}
    if second:
        line["shapes"] = {}
        for w in second:
            s2 = measure_shape_n1(args, w, max(3, min(args.steps, 5)), 3, local_rank, full=False)
            line["shapes"][w] = {k2: s2[k2] for k2 in ("value", "ms_per_step", "stages_ms", "e2e", "verified", "roofline", "config",
                                                       "n_segments", "rank_rounds", "gpu_launches")}
    if args.workload is None and not args.n and not args.no_count:
        # SURVEY.md 8(f)-4, a secondary record: the stage BEFORE the timed one (reads -> unique k-mers with extensions,
        # csrc/count.cu) on a bounded sample of the same contig shape; never fail the bench line over it
        try:
            from tools import count_bench
            ka = count_bench.run(k=k, n=4_000_000, coverage=8, read_len=150)
            sample = ka.pop("_sample", None)
            if sample is not None and not args.no_cpu_baseline:
                # the reference has no code for this stage: the CPU number is the oracle's restatement ("port", one core,
                # sort-based) on a bounded piece of the same reads
                import oracle
                t0 = time.perf_counter()
                _, _, occ = oracle.analyse_reads(sample, k, 2, 2)
                dt = time.perf_counter() - t0
                ka["cpu_baseline"] = {"value": occ / dt, "unit": "occurrences/s", "cores": 1, "kind": "port",
                                      "sample": f"oracle/kmer_count_oracle.c on the first {sample.size} bytes of the same reads "
                                                f"({occ} occurrences, {dt:.2f} s)"}
            line["kmer_analysis"] = ka
        except Exception as e:
            line["kmer_analysis"] = {"error": str(e)}
    if not args.no_cpu_baseline:
        line["cpu_baseline"] = cpu_baseline_leg(k, workload)
    else:
        line["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": 1, "kind": "reference", "sample": "skipped"}
    try:        # the same (unmodified) reference on the FULL file, measured once in the build container (tests/golden/make_full_digests.py)
        with open(os.path.join(ROOT, "tests", "golden", "chr14_full.json")) as f:
            full = json.load(f).get(workload)
        if full:
            line["cpu_baseline"]["full_file_run"] = {
                "value": full["n_kmers"] / full["reference_total_s"], "unit": UNIT, "sample_kmers": full["n_kmers"],
                "insert_s": full["reference_insert_s"], "total_s": full["reference_total_s"], "cores": 1,
                "where": full["host"] + " -- NOT this GPU box's host; fixture tests/golden/chr14_full.json"}
    except Exception:
        pass
    return line


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default=None, choices=sorted(WORKLOADS))
    ap.add_argument("--kmers", dest="n", type=int, default=0, help="override the number of k-mers (contigs scale along)")
    ap.add_argument("--load-factor", type=float, default=0.5)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true", help="skip the host-buffer leg (profiling runs)")
    ap.add_argument("--no-count", action="store_true", help="skip the k-mer analysis sub-record (reads -> k-mers)")
    ap.add_argument("--also", nargs="*", default=None, choices=sorted(WORKLOADS),
                    help="further workloads measured in the same run and reported under \"shapes\" (default: chr14_k19)")
    ap.add_argument("--scaling", default="strong", choices=["strong", "weak"],
                    help="N>1 only: strong = the N=1 file split over the GPUs (default); weak = one such file per GPU (K>=31)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the last timed step's output (contigs, offsets, counts) to DIR/<name>.npy (--gpus 1)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.gpus != 1 or args.impl != "b200"):
        ap.error("--dump-outputs needs --gpus 1 and --impl b200")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    # BASELINE.json configs[2]/[3]: the reference's real chr14 shape is K=51 (results/results_parallel_kmer51.txt);
    # the same file at every N (strong scaling over the sharded table).  configs[1] (K=19) rides along as a sub-record.
    workload = args.workload or "chr14_k51"
    if args.also is None:
        args.also = ["chr14_k19"] if (args.workload is None and not args.n) else []
    k = WORKLOADS[workload][0]
    rank = int(os.environ.get("RANK", "0"))
    if args.impl == "reference":
        if rank != 0:
            return
        line = run_reference_arm(args, k, workload)
    else:
        line = run_b200_arm(args, workload)
    if line is not None and rank == 0:
        print(json.dumps(line), flush=True)


if __name__ == "__main__":
    sys.dont_write_bytecode = True      # the tree may be read-only: the bench writes nothing into it
    main()
