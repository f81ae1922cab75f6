"""Contig depth (kh_count_contig_depth*, KmerCounter.contig_depth*, ShardedCounter.contig_depth, kmer_count --depth).

Contig i is the text [offsets[i], offsets[i+1]); a window is a position p with p + K <= offsets[i+1] whose K bytes are
all ACGT, its value the counter's occurrence count of that k-mer (saturated at 255, 0 when never seen).  Per contig:
windows, sum, min, max.  The reference is a numpy restatement of that definition (windows of the reads counted with
np.unique), itself checked against the oracle's counts.
CPU: tests/native/depth_host_check.cu runs the kernel's loops serially against the restatement; the CLI's usage error;
the kernel's register budget.  GPU: both entry points against the restatement, the closed loop reads -> contigs ->
depth, contigs the unmodified reference wrote, the error paths, the sharded combine and the CLI."""
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

import oracle
from tools import kmergen, readgen
from tools.depth_bench import lookup_depth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
KS = [3, 19, 31, 32, 51, 61]
_ACGT = np.frombuffer(b"ACGT", dtype=np.uint8)
NO_MIN = 0xFFFFFFFF


# ------------------------------------------------------------------------------------------- the restatement
def _windows(buf, k):
    """Every K-byte window of buf as an S<k> string, and whether all its bytes are bases."""
    r = np.ascontiguousarray(buf, dtype=np.uint8)
    if r.size < k:
        return np.zeros(0, dtype=f"S{k}"), np.zeros(0, dtype=bool)
    keys = np.ascontiguousarray(np.lib.stride_tricks.sliding_window_view(r, k)).view(f"S{k}").ravel()
    ok = np.lib.stride_tricks.sliding_window_view(np.isin(r, _ACGT), k).all(axis=1)
    return keys, ok


def _counts(reads, k):
    """Distinct k-mers of the reads (sorted) and their occurrence counts saturated at 255."""
    keys, ok = _windows(reads, k)
    uniq, cnt = np.unique(keys[ok], return_counts=True)
    return uniq, np.minimum(cnt, 255).astype(np.uint32)


def _depth_ref(text, offsets, k, table):
    """The definition of kh_contig_depth, restated: per contig its windows, and the sum / min / max of their counts."""
    import cs267_hw3_b200 as kh
    uniq, cnt = table
    t = np.asarray(text, dtype=np.uint8)
    offs = np.asarray(offsets, dtype=np.int64)
    n = offs.size - 1
    out = np.zeros(n, dtype=kh.DEPTH_DTYPE)
    out["min"] = NO_MIN
    if n <= 0:
        return out
    keys, ok = _windows(t[offs[0]:offs[-1]], k)
    pos = offs[0] + np.arange(keys.size)
    c = np.searchsorted(offs[:-1], pos, side="right") - 1
    valid = ok & (pos + k <= offs[np.minimum(c + 1, n)])
    keys, c = keys[valid], c[valid]
    val = np.zeros(keys.size, dtype=np.uint64)
    if uniq.size:
        i = np.minimum(np.searchsorted(uniq, keys), uniq.size - 1)
        val = np.where(uniq[i] == keys, cnt[i], 0).astype(np.uint64)
    np.add.at(out["n_kmers"], c, 1)
    np.add.at(out["sum"], c, val)
    np.minimum.at(out["min"], c, val.astype(np.uint32))
    np.maximum.at(out["max"], c, val.astype(np.uint32))
    return out


def _reads(k, seed, n=20000, c=60, coverage=4, error_rate=0.002, saturate=True):
    """Tiled reads with substitution errors and N / lower-case bytes, plus (saturate) one read repeated 300 times so
    that some k-mers are seen more than 255 times.  Returns (the contigs the reads were cut from, the reads)."""
    rng = np.random.default_rng(seed)
    if k < 8:
        lines = [bytes(_ACGT[rng.integers(0, 4, int(rng.integers(1, 60)))]) for _ in range(300)]
        solution = b"".join(x + b"\n" for x in lines)
        reads = np.frombuffer(solution * 3, dtype=np.uint8).copy()
    else:
        solution = kmergen.Dataset(k, n, c, seed=seed).solution()
        reads = readgen.tile_reads(solution, k, read_len=k + 40, coverage=coverage, seed=seed + 1, error_rate=error_rate)
    pos = rng.choice(reads.size, size=max(1, reads.size // 500), replace=False)
    reads[pos] = np.where(rng.random(pos.size) < 0.5, ord("N"), ord("a")).astype(np.uint8)
    if saturate:
        line = solution.split(b"\n")[0][: k + 8]
        reads = np.concatenate([reads] + [np.frombuffer(line + b"\n", dtype=np.uint8)] * 300)
    return solution, reads


def _contig_case(k, solution, seed):
    """Contig text + offsets that exercise every rule: whole contigs spanning tiles; hundreds of 1-k-mer contigs in a
    tile; empty contigs and contigs shorter than K; runs cut without separators (windows would cross contigs); an N
    inside a contig; contigs of random sequence (missing k-mers).  offsets[0] > 0: the text before it is not read."""
    rng = np.random.default_rng(seed)
    lines = [x for x in solution.split(b"\n") if len(x) >= k]
    pieces = [x + b"\n" for x in lines[:30]]
    for _ in range(400):                                     # one window each, separated or not
        x = lines[int(rng.integers(len(lines)))]
        p = int(rng.integers(0, len(x) - k + 1))
        pieces.append(x[p:p + k] + (b"\n" if rng.random() < 0.5 else b""))
    pieces += [b""] * 30 + [x[: max(1, k - 1)] for x in lines[:20]]
    for x in lines[30:40]:                                   # no separators: cut into pieces of 1 .. 3K bytes
        at = 0
        while at < len(x):
            step = int(rng.integers(1, 3 * k + 1))
            pieces.append(x[at:at + step])
            at += step
    for x in lines[40:45]:                                   # an N in the middle
        m = len(x) // 2
        pieces.append(x[:m] + b"N" + x[m + 1:] + b"\n")
    pieces += [bytes(_ACGT[rng.integers(0, 4, k + 30)]) + b"\n" for _ in range(20)]
    order = rng.permutation(len(pieces))
    pieces = [pieces[i] for i in order]
    head = b"ACGTACGTACGTA"
    text = head + b"".join(pieces)
    offs = np.concatenate(([0], np.cumsum([len(x) for x in pieces]))).astype(np.uint64) + len(head)
    return np.frombuffer(text, dtype=np.uint8).copy(), offs


@pytest.mark.parametrize("k", [3, 19, 51])
def test_restatement_counts_match_the_oracle(k):
    """The restatement's k-mer counts (np.unique) are the oracle's (sort + run scan in C) at min_count = min_ext = 1."""
    _, reads = _reads(k, 100 + k, n=4000, c=20)
    uniq, cnt = _counts(reads, k)
    pairs, counts, _ = oracle.analyse_reads(reads, k, 1, 1)
    pl = (k + 3) // 4
    got = np.array([oracle.unpack_kmer(bytes(p[:pl]), k).encode() for p in pairs], dtype=f"S{k}")
    order = np.argsort(got)
    assert (got[order] == uniq).all() and (counts[order, 0] == cnt).all()
    assert cnt.max() == 255


# ------------------------------------------------------------------------------- CPU: the kernel's loops, serially
@pytest.fixture(scope="module")
def host_check(tmp_path_factory):
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        pytest.skip("nvcc not available")
    exe = str(tmp_path_factory.mktemp("depth") / "depth_host_check")
    subprocess.run([nvcc, "-std=c++17", "-O1", "-Wno-deprecated-gpu-targets", "-o", exe,
                    os.path.join(ROOT, "tests", "native", "depth_host_check.cu")], check=True, capture_output=True)
    return exe


def _run_host(exe, tmp_path, k, reads, text, offs, world):
    import cs267_hw3_b200 as kh
    np.asarray(reads, dtype=np.uint8).tofile(tmp_path / "reads.bin")
    np.asarray(text, dtype=np.uint8).tofile(tmp_path / "text.bin")
    np.asarray(offs, dtype="<u8").tofile(tmp_path / "offs.bin")
    n_slots = max(1024, 2 * int(np.asarray(reads).size))
    out = subprocess.run([exe, str(k), str(n_slots), str(world), str(tmp_path / "reads.bin"), str(tmp_path / "text.bin"),
                          str(tmp_path / "offs.bin")], capture_output=True, text=True, check=True).stdout
    v = np.array([[int(x) for x in ln.split()] for ln in out.splitlines()], dtype=np.uint64).reshape(-1, 8)
    recs = []
    for cols in (v[:, :4], v[:, 4:]):
        r = np.zeros(len(v), dtype=kh.DEPTH_DTYPE)
        for j, name in enumerate(("n_kmers", "sum", "min", "max")):
            r[name] = cols[:, j]
        recs.append(r)
    return recs


@pytest.mark.parametrize("k", KS)
def test_kernel_loops_match_the_restatement(host_check, tmp_path, k):
    """Every K regime, every contig shape of _contig_case, reads with errors, N and counts past 255; the owners' partials
    for world 1, 2, 3 and 8 combine into the world-1 record."""
    solution, reads = _reads(k, 300 + k)
    text, offs = _contig_case(k, solution, 400 + k)
    want = _depth_ref(text, offs, k, _counts(reads, k))
    assert want["n_kmers"].sum() > 0 and (want["max"] == 255).any()
    assert k < 8 or ((want["n_kmers"] > 0) & (want["min"] == 0)).any()          # 4^3 3-mers: none is missing
    assert (want["n_kmers"] == 0).sum() >= 30
    for world in (1, 2, 3, 8):
        one, combined = _run_host(host_check, tmp_path, k, reads, text, offs, world)
        assert (one == want).all(), np.flatnonzero(one != want)[:10]
        assert (combined == want).all(), (world, np.flatnonzero(combined != want)[:10])


def test_kernel_loops_long_contig_and_crowded_tiles(host_check, tmp_path):
    """A contig spanning dozens of tiles, and tiles of nothing but 1-k-mer contigs (hundreds per tile), K = 31."""
    k = 31
    solution, reads = _reads(k, 77, n=60000, c=2, saturate=False)
    lines = solution.split(b"\n")[:-1]
    rng = np.random.default_rng(5)
    long_one = max(lines, key=len)
    short = []
    for _ in range(2000):
        x = lines[int(rng.integers(len(lines)))]
        p = int(rng.integers(0, len(x) - k + 1))
        short.append(x[p:p + k] + b"\n")
    pieces = [long_one + b"\n"] + short
    text = np.frombuffer(b"".join(pieces), dtype=np.uint8).copy()
    offs = np.concatenate(([0], np.cumsum([len(x) for x in pieces]))).astype(np.uint64)
    assert len(long_one) > 10 * 2048
    want = _depth_ref(text, offs, k, _counts(reads, k))
    assert (want["n_kmers"][1:] == 1).all() and want["n_kmers"][0] == len(long_one) - k + 1
    one, combined = _run_host(host_check, tmp_path, k, reads, text, offs, 3)
    assert (one == want).all() and (combined == want).all()


# ------------------------------------------------------------------------------------------- CPU: CLI and kernel build
def test_kmer_count_cli_depth_needs_contigs(tmp_path):
    from cs267_hw3_b200 import build
    exe = build.build_count_cli()
    (tmp_path / "reads.txt").write_bytes(b"ACGTACGTAC\n")
    for args in (["19", "reads.txt", "--depth"], ["19", "reads.txt", "--depth", "kmers.txt"],
                 ["19", "reads.txt", "--histo", "h.txt", "--depth"], ["19", "reads.txt", "--depth", "--histo", "h.txt", "k.txt", "2"]):
        r = subprocess.run([exe, *args], cwd=tmp_path, capture_output=True, text=True)
        assert r.returncode == 1 and r.stderr.startswith("Usage: kmer_count K reads_file"), (args, r.stderr)
        assert "[--depth]" in r.stderr
    assert sorted(os.listdir(tmp_path)) == ["reads.txt"]


def test_depth_kernel_has_no_spills(tmp_path):
    """kc_depth_kernel for sm_100a: ptxas reports no stack frame and no spills (both slot widths)."""
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        pytest.skip("nvcc not available")
    from cs267_hw3_b200 import build
    r = subprocess.run([nvcc, *build.NVCC_FLAGS, "-Xptxas", "-v", "-c", os.path.join(build.CSRC, "count.cu"),
                        "-o", str(tmp_path / "count.o")], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    blocks = re.findall(r"Function properties for (\S*kc_depth_kernel\S*)\n\s*(.*)", r.stderr)
    assert len(blocks) == 2, r.stderr[-2000:]
    for name, props in blocks:
        assert "0 bytes stack frame, 0 bytes spill stores, 0 bytes spill loads" in props, (name, props)


# --------------------------------------------------------------------------------------------------- GPU
def _dev(a):
    import torch
    t = torch.from_numpy(np.ascontiguousarray(a).view(np.uint8).copy()).to("cuda:0")
    torch.cuda.synchronize()
    return t


def _device_depth(kc, text, offs, world=1, rank=0):
    import torch

    import cs267_hw3_b200 as kh
    n = len(offs) - 1
    dt, do = _dev(text), _dev(np.asarray(offs, dtype=np.uint64))
    out = torch.full((max(n, 1) * 24 + 24,), 0xAB, dtype=torch.uint8, device="cuda:0")   # one record past the end
    torch.cuda.synchronize()
    kc.contig_depth_device(dt.data_ptr(), do.data_ptr(), n, out.data_ptr(), world, rank)
    raw = out.cpu().numpy()
    assert (raw[n * 24:] == 0xAB).all(), "wrote past record n - 1"
    return raw[: n * 24].view(kh.DEPTH_DTYPE).copy()


@pytest.mark.gpu
@pytest.mark.parametrize("k", KS)
def test_gpu_contig_depth_matches_the_restatement(k):
    """Host and device entry points against the restatement: reads with errors, N and counts past 255; every contig
    shape of _contig_case; two launches per call."""
    import cs267_hw3_b200 as kh
    solution, reads = _reads(k, 500 + k)
    text, offs = _contig_case(k, solution, 600 + k)
    want = _depth_ref(text, offs, k, _counts(reads, k))
    with kh.KmerCounter(k, max(1024, reads.size), 0.5, 0) as kc:
        kc.count_reads(reads)
        n0 = kc.stats()["n_launches"]
        got = kc.contig_depth(text, offs)
        assert kc.stats()["n_launches"] == n0 + 2
        assert got.dtype == kh.DEPTH_DTYPE and (got == want).all(), np.flatnonzero(got != want)[:10]
        assert (_device_depth(kc, text, offs) == want).all()
        assert (kc.contig_depth(text, offs) == want).all()                  # records re-initialised on every call
        parts = [kc.contig_depth(text, offs, 3, r) for r in range(3)]
        assert (kh.combine_depth(parts) == want).all()


def _closed_loop(k, n, c, seed, m, long_nodes=0):
    """reads -> count -> extract(m) -> insert -> assemble_device -> contig_depth_device on the resident contigs."""
    import torch

    import cs267_hw3_b200 as kh
    d = kmergen.Dataset(k, n, c, seed=seed, long_nodes=long_nodes)
    reads = readgen.tile_reads(d.solution(), k, read_len=k + 40, coverage=5, seed=seed + 1)
    with kh.KmerCounter(k, 2 * n, 0.5, 0) as kc, kh.KmerHashTable(k, n, 0.5, 0) as tab:
        kc.count_reads(reads)
        ptr, n_rec = kc.extract_device(m, 2)
        assert n_rec == n
        tab.insert_pairs_device(ptr, n_rec)
        cp, op, nc, nb, nodes = tab.assemble_device()
        out = torch.empty(nc * 24, dtype=torch.uint8, device="cuda:0")
        torch.cuda.synchronize()
        kc.contig_depth_device(cp, op, nc, out.data_ptr())
        got = out.cpu().numpy().view(kh.DEPTH_DTYPE)
        recs = kc.extract(m, 2)
        total = int(kc.lookup(recs[:, :(k + 3) // 4])[:, 0].astype(np.uint64).sum())
        text, offs, _ = tab.assemble()
        return got, nodes, total, text, offs, reads, lookup_depth(kc, text, offs, k, range(nc)) if long_nodes else None


@pytest.mark.gpu
@pytest.mark.parametrize("k,m", [(19, 2), (51, 3)])
def test_gpu_closed_loop_reads_contigs_depth(k, m):
    """Sum of n_kmers = n_nodes, every min >= m, sum of sums = the extracted k-mers' counts (every k-mer of the
    generator's data lands on a contig); the records equal the restatement over the same contig text."""
    got, nodes, total, text, offs, reads, _ = _closed_loop(k, 40000, 80, 700 + k, m)
    assert int(got["n_kmers"].sum()) == nodes == 40000
    assert (got["min"] >= m).all() and int(got["sum"].sum()) == total
    assert (got == _depth_ref(text, offs, k, _counts(reads, k))).all()


@pytest.mark.gpu
def test_gpu_long_contig_is_exact():
    """One 10^6-k-mer contig (long_nodes) spread over ~500 tiles: every record equals the windows packed on the host and
    looked up one by one."""
    k = 51
    got, nodes, total, text, offs, reads, want = _closed_loop(k, 1_050_000, 20, 800, 2, long_nodes=10 ** 6)
    assert int(got["n_kmers"].max()) == 10 ** 6
    assert int(got["n_kmers"].sum()) == nodes and int(got["sum"].sum()) == total
    assert (got == want).all()


@pytest.mark.gpu
def test_gpu_golden_contigs_of_the_reference(golden_dir):
    """Reads tiled over the contigs the unmodified reference wrote (tests/golden/<case>.dat): their depth equals the
    restatement."""
    import json

    import cs267_hw3_b200 as kh
    with open(os.path.join(golden_dir, "MANIFEST.json")) as f:
        cases = json.load(f)
    for name, case in sorted(cases.items()):
        k = int(case["k"])
        with open(os.path.join(golden_dir, f"{name}.dat"), "rb") as f:
            dat = f.read()
        reads = readgen.tile_reads(dat, k, read_len=k + 40, coverage=6, seed=len(dat))
        text = np.frombuffer(dat, dtype=np.uint8)
        ends = np.flatnonzero(text == 10) + 1
        offs = np.concatenate(([0], ends)).astype(np.uint64)
        with kh.KmerCounter(k, max(1024, reads.size), 0.5, 0) as kc:
            kc.count_reads(reads)
            got = kc.contig_depth(text, offs)
        want = _depth_ref(text, offs, k, _counts(reads, k))
        assert (got == want).all() and (got["min"] >= 6).all(), name


@pytest.mark.gpu
@pytest.mark.parametrize("k", [19, 51])
def test_gpu_growth_missing_kmers_and_errors(k):
    """A counter that grew gives the records of one sized generously; contigs of another data set give min 0; an
    overflowed table is KH_ERR_TABLE_FULL; n_contigs = 0 launches nothing; bad arguments are KH_ERR_ARG."""
    import ctypes as C

    import cs267_hw3_b200 as kh
    solution, reads = _reads(k, 900 + k, n=60000, c=100, coverage=3, saturate=False)
    text, offs = _contig_case(k, solution, 901 + k)
    other = np.frombuffer(kmergen.Dataset(k, 3000, 10, seed=902 + k).solution(), dtype=np.uint8)
    other_offs = np.concatenate(([0], np.flatnonzero(other == 10) + 1)).astype(np.uint64)
    with kh.KmerCounter(k, 100, 0.5, 0) as small, kh.KmerCounter(k, 4 * reads.size, 0.5, 0) as big:
        small.count_reads(reads)
        big.count_reads(reads)
        assert small.stats()["n_grows"] > 0 and big.stats()["n_grows"] == 0
        want = _depth_ref(text, offs, k, _counts(reads, k))
        assert (small.contig_depth(text, offs) == want).all() and (big.contig_depth(text, offs) == want).all()
        miss = big.contig_depth(other, other_offs)
        assert (miss["min"] == 0).all() and (miss["n_kmers"] > 0).all()
        assert (miss == _depth_ref(other, other_offs, k, _counts(reads, k))).all()
        n0 = big.stats()["n_launches"]
        assert big.contig_depth(text, offs[:1]).size == 0
        L, h = kh.lib(), big._h
        rec = np.zeros(4, dtype=kh.DEPTH_DTYPE)
        assert L.kh_count_contig_depth(h, None, None, 0, 1, 0, None) == kh.KH_OK
        assert L.kh_count_contig_depth_device(h, None, None, 0, 1, 0, None) == kh.KH_OK
        assert big.stats()["n_launches"] == n0
        o4 = offs[:5].copy()
        tp, op, rp = text.ctypes.data, o4.ctypes.data, rec.ctypes.data
        for args in ((None, op, 4, 1, 0, rp), (tp, None, 4, 1, 0, rp), (tp, op, 4, 1, 0, None), (tp, op, 4, 0, 0, rp),
                     (tp, op, 4, 65, 0, rp), (tp, op, 4, 2, 2, rp), (tp, op, 0, 3, 3, rp)):
            assert L.kh_count_contig_depth(h, *args) == kh.KH_ERR_ARG, args
            assert L.kh_count_contig_depth_device(h, *args) == kh.KH_ERR_ARG, args
        bad = o4.copy()
        bad[2] = bad[3] + 1
        assert L.kh_count_contig_depth(h, tp, bad.ctypes.data, 4, 1, 0, rp) == kh.KH_ERR_ARG
        assert L.kh_count_contig_depth(None, tp, op, 4, 1, 0, rp) == kh.KH_ERR_ARG
        assert big.stats()["n_launches"] == n0
    os.environ["KH_COUNT_GROW"] = "0"
    try:
        c = kh.KmerCounter(k, 100, 0.5, 0)
    finally:
        os.environ.pop("KH_COUNT_GROW")
    with c:
        p = C.c_void_p()
        assert L.kh_device_alloc(C.byref(p), reads.size) == 0
        with kh.KmerHashTable(k, 1024) as tab:
            tab._check(L.kh_copy_device(tab._h, p, reads.ctypes.data, reads.size))
            tab.sync()
        c.count_reads_device(p.value, reads.size)
        with pytest.raises(kh.KhError) as e:
            c.contig_depth(text, offs)
        assert e.value.status == kh.KH_ERR_TABLE_FULL
        L.kh_device_free(p)


@pytest.mark.gpu
@pytest.mark.parametrize("world", [1, 2, 3, 8])
@pytest.mark.parametrize("batches", [1, 3])
def test_gpu_sharded_contig_depth_equals_one_counter(world, batches):
    """ShardedCounter.contig_depth: the owners' partials combined are the single counter's records, with one reduce at
    the end or reduces in between (ranks sharing GPU 0 when there are fewer GPUs)."""
    import cs267_hw3_b200 as kh
    from cs267_hw3_b200.sharded_count import ShardedCounter, split_reads
    k = 31
    solution, reads = _reads(k, 1000 + world, n=40000, c=80)
    text, offs = _contig_case(k, solution, 1001 + world)
    with kh.KmerCounter(k, reads.size, 0.5, 0) as one:
        one.count_reads(reads)
        want = one.contig_depth(text, offs)
    assert (want == _depth_ref(text, offs, k, _counts(reads, k))).all()
    cuts = split_reads(reads, world * batches)
    with ShardedCounter(k, world, reads.size) as sc:
        for b in range(batches):
            for r in range(world):
                piece = b * world + r
                sc.count(r, reads[cuts[piece]:cuts[piece + 1]])
            sc.reduce()
        got = sc.contig_depth(text, offs)
        assert got.dtype == kh.DEPTH_DTYPE and (got == want).all()


def _run_cli(tmp_path, args, env=None, timeout=300):
    from cs267_hw3_b200 import build
    exe = build.build_count_cli()
    base = {x: v for x, v in os.environ.items() if x not in ("KH_RANKS", "KH_COUNT_BATCH_BYTES")}
    r = subprocess.run([exe, *args], cwd=tmp_path, capture_output=True, text=True, timeout=timeout, env=dict(base, **(env or {})))
    assert r.returncode == 0, r.stdout + r.stderr
    return r.stdout


@pytest.mark.gpu
@pytest.mark.parametrize("ranks", [1, 2])
def test_gpu_kmer_count_depth(tmp_path, ranks):
    """kmer_count K reads --depth --contigs out auto M: out_r.depth has one `n mean min max` line per line of out_r.dat,
    equal to the restatement; the .dat files hold the contigs of a run without --depth and the other stdout lines are
    that run's.  (Contig order follows the counter's table order, which concurrent slot claims make differ from run to
    run, so the ranks' .dat lines are compared as one set.)"""
    k, min_ext = 19, 5
    d = kmergen.Dataset(k, 30000, 60, seed=7000)
    reads = readgen.tile_reads(d.solution(), k, read_len=k + 40, coverage=20, seed=7100, error_rate=0.01)
    (tmp_path / "reads.txt").write_bytes(bytes(reads))
    env = {"KH_RANKS": str(ranks)}
    plain = _run_cli(tmp_path, [str(k), "reads.txt", "--contigs", "plain", "auto", str(min_ext)], env=env)
    out = _run_cli(tmp_path, [str(k), "reads.txt", "--depth", "--contigs", "out", "auto", str(min_ext)], env=env)
    table = _counts(reads, k)
    n_c = n_k = total = 0
    got_lines, plain_lines = [], []
    for r in range(ranks):
        dat = (tmp_path / f"out_{r}.dat").read_bytes()
        got_lines += dat.splitlines()
        plain_lines += (tmp_path / f"plain_{r}.dat").read_bytes().splitlines()
        text = np.frombuffer(dat, dtype=np.uint8)
        offs = np.concatenate(([0], np.flatnonzero(text == 10) + 1)).astype(np.uint64)
        want = _depth_ref(text, offs, k, table)
        lines = (tmp_path / f"out_{r}.depth").read_text().splitlines()
        assert len(lines) == len(offs) - 1 == dat.count(b"\n")
        assert lines == ["%d %.2f %d %d" % (w["n_kmers"], w["sum"] / w["n_kmers"], w["min"], w["max"]) for w in want]
        n_c, n_k, total = n_c + len(lines), n_k + int(want["n_kmers"].sum()), total + int(want["sum"].sum())
    assert n_k == 30000 and sorted(got_lines) == sorted(plain_lines)
    tail = "Depth of %d contigs (%d k-mers): mean %.2f; wrote out_0.depth .. out_%d.depth\n" % (n_c, n_k, total / n_k, ranks - 1)
    assert out.endswith(tail)
    strip = lambda s: [re.sub(r"[0-9.]+ s\b", "T s", x).replace("out", "plain") for x in s.splitlines()]  # noqa: E731
    assert strip(out)[:-1] == strip(plain)
