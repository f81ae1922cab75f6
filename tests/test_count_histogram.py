"""The k-mer spectrum (kh_count_histogram, kh_count_auto_min_count, KmerCounter.histogram, ShardedCounter.histogram,
kmer_count --histo / auto).

hist[c] = distinct k-mers counted exactly c times (c = 1..254), hist[255] = 255 times or more, hist[0] = 0.  Invariants:
sum(hist) = n_distinct, and the suffix sum from m = the records kh_count_extract(m, any min_ext) reports.
CPU: the valley rule on hand-made spectra and against a restatement of its definition; the oracle's spectrum against
numpy; the closed-loop parameters chosen with the oracle; the CLI's usage errors; the kernel's register budget.
GPU: the kernel against the oracle, the invariants, growth, sharded sums and the CLI."""
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

import oracle
from tools import kmergen, readgen

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# Reads with 1 % substitutions at 20x: at min_count 2 erroneous k-mers survive, at the valley only the true ones do.
# Chosen with the oracle (test_closed_loop_parameters_need_the_valley) so that the GPU runs check the GPU only.
LOOP_K, LOOP_N, LOOP_C, LOOP_SEED, LOOP_ERR, LOOP_MIN_EXT = 19, 30000, 60, 7000, 0.01, 5


def _sorted_rows(a: np.ndarray) -> np.ndarray:
    return a[np.lexsort(a.T[::-1])] if a.size else a


def _loop_reads():
    d = kmergen.Dataset(LOOP_K, LOOP_N, LOOP_C, seed=LOOP_SEED)
    reads = readgen.tile_reads(d.solution(), LOOP_K, read_len=LOOP_K + 40, coverage=20, seed=LOOP_SEED + 100,
                               error_rate=LOOP_ERR)
    return d, reads


def _reads(k, n, c, seed, coverage=4, error_rate=0.002, with_n=True, saturate=False):
    """Tiled reads with substitution errors and N / lower-case separators; saturate: plus one read repeated 300 times,
    so that some k-mers are seen more than 255 times."""
    if k < 8:                                    # few distinct k-mers: random text with separators (counts > 255 too)
        rng = np.random.default_rng(seed)
        reads = np.frombuffer(b"ACGT", dtype=np.uint8)[rng.integers(0, 4, 50000)].copy()
        reads[rng.choice(reads.size, 500, replace=False)] = 10
    else:
        d = kmergen.Dataset(k, n, c, seed=seed)
        reads = readgen.tile_reads(d.solution(), k, read_len=k + 40, coverage=coverage, seed=seed + 1, error_rate=error_rate)
        if with_n:
            rng = np.random.default_rng(seed + 2)
            pos = rng.choice(reads.size, size=max(1, reads.size // 500), replace=False)
            reads[pos] = np.where(rng.random(pos.size) < 0.5, ord("N"), ord("a")).astype(np.uint8)
    if saturate:
        rep = np.frombuffer(b"GATTACACCGTAGGCTTAACGTGCATGCCAGTTAGCAATCGGATCCATGCAGTCCGATAGCTTAGGCATC"[: k + 8] + b"\n",
                            dtype=np.uint8)
        reads = np.concatenate([reads] + [rep] * 300)
    return reads


def _oracle_histogram(reads, k: int) -> np.ndarray:
    """The spectrum from the oracle (oracle/kmer_count_oracle.c: sort the occurrences, scan the runs): at min_count =
    min_ext = 1 every distinct k-mer is a record, and its count column is min(run length, 255) -- its bin."""
    _, counts, _ = oracle.analyse_reads(reads, k, 1, 1)
    return np.bincount(counts[:, 0], minlength=256).astype(np.uint64)


def _valley(hist) -> int:
    """The valley rule as kh_capi.h states it, restated for the property check."""
    h = [int(x) for x in hist]
    for v in range(1, 255):
        if h[v + 1] >= h[v]:
            return v if v >= 2 and sum(h[v:]) > 0 else 2
    return 2


def _numpy_histogram(reads: np.ndarray, k: int) -> np.ndarray:
    """The spectrum stated independently of the oracle: every window of K bases, distinct windows counted with np.unique."""
    r = np.asarray(reads, dtype=np.uint8)
    base = np.isin(r, np.frombuffer(b"ACGT", dtype=np.uint8))
    win = np.lib.stride_tricks.sliding_window_view(r, k)
    ok = np.lib.stride_tricks.sliding_window_view(base, k).all(axis=1)
    rows = np.ascontiguousarray(win[ok]).view(np.dtype((np.void, k))).ravel()
    _, counts = np.unique(rows, return_counts=True)
    return np.bincount(np.minimum(counts, 255), minlength=256).astype(np.uint64)


def _histo_text(hist) -> bytes:
    return b"".join(b"%d %d\n" % (c, int(hist[c])) for c in range(1, 256) if hist[c])


# ------------------------------------------------------------------------------------------- CPU: the valley rule
def _spectrum(**bins):
    h = np.zeros(256, dtype=np.uint64)
    for c, n in bins.items():
        h[int(c[1:])] = n
    return h


@pytest.mark.parametrize("name,hist,want", [
    ("clean: all mass at the coverage peak", _spectrum(c20=1000), 2),
    ("clean with a spread peak", _spectrum(c18=100, c19=400, c20=700, c21=300), 2),
    ("error slope + peak: the valley bin", _spectrum(c1=5000, c2=300, c3=20, c4=5, c5=8, c6=40, c15=900, c16=600), 4),
    ("error slope + peak, valley at 3", _spectrum(c1=9000, c2=500, c3=30, c4=31, c20=800), 3),
    ("tie at the floor", _spectrum(c1=100, c2=100, c10=500), 2),
    ("tie right after the floor", _spectrum(c1=100, c2=10, c3=10, c10=500), 2),
    ("tie later on the slope", _spectrum(c1=100, c2=10, c3=3, c4=3, c10=500), 3),
    ("empty table", _spectrum(), 2),
    ("monotone to zero, no second peak", _spectrum(c1=100, c2=10, c3=1), 2),
    ("falls to zero, mass only in the saturated bin", _spectrum(c1=100, c2=50, c255=1000), 3),
    ("falls all the way, never stops", np.arange(300, 44, -1, dtype=np.uint64), 2),
])
def test_auto_min_count_hand_made_spectra(name, hist, want):
    import cs267_hw3_b200 as kh
    hist[0] = 0
    assert kh.auto_min_count(hist) == want, name
    assert _valley(hist) == want, name


def test_auto_min_count_null_and_shape():
    import cs267_hw3_b200 as kh
    assert kh.auto_min_count(None) == 2
    assert kh.lib().kh_count_auto_min_count(None) == 2
    with pytest.raises(ValueError):
        kh.auto_min_count(np.zeros(255, dtype=np.uint64))


def test_auto_min_count_random_spectra_follow_the_definition():
    """kh_count_auto_min_count (C) against the rule restated from kh_capi.h, on random error-slope + peak spectra."""
    import cs267_hw3_b200 as kh
    rng = np.random.default_rng(31)
    for _ in range(400):
        h = np.zeros(256, dtype=np.uint64)
        slope = int(rng.integers(1, 8))
        h[1:slope + 1] = np.sort(rng.integers(0, 10 ** int(rng.integers(1, 7)), slope))[::-1]
        peak = int(rng.integers(2, 256))
        width = int(rng.integers(1, 12))
        lo, hi = max(1, peak - width), min(255, peak + width)
        h[lo:hi + 1] += rng.integers(0, 1000, hi - lo + 1).astype(np.uint64)
        if rng.random() < 0.2:
            h[255] += np.uint64(rng.integers(0, 50))
        assert kh.auto_min_count(h) == _valley(h), h[:40]


# ------------------------------------------------------------------------------------------- CPU: the oracle
@pytest.mark.parametrize("k", [3, 19, 31, 51])
def test_oracle_spectrum_against_numpy(k):
    """The oracle's spectrum (sort + run scan in C) equals an np.unique statement; the invariants hold on the oracle's own
    records; on 20x reads with 1 % errors the valley lies strictly between the error slope and the coverage peak."""
    import cs267_hw3_b200 as kh
    if k < 8:
        reads = _reads(k, 0, 0, seed=k)
    else:
        d = kmergen.Dataset(k, 8000, 20, seed=800 + k)
        reads = readgen.tile_reads(d.solution(), k, read_len=k + 40, coverage=20, seed=801 + k, error_rate=0.01)
        reads = np.concatenate([reads, np.frombuffer(b"A" * 400 + b"\n", dtype=np.uint8)])    # one k-mer seen > 255 times
    h = _oracle_histogram(reads, k)
    assert h.dtype == np.uint64 and h.shape == (256,) and h[0] == 0
    assert (h == _numpy_histogram(reads, k)).all()
    assert h[255] > 0
    all_p, _, _ = oracle.analyse_reads(reads, k, 1, 1)
    assert int(h.sum()) == len(all_p)
    for m in (2, 3, 7, 255):
        assert int(h[m:].sum()) == len(oracle.analyse_reads(reads, k, m, 2)[0])
    if k >= 8:
        v = kh.auto_min_count(h)
        peak = v + int(np.argmax(h[v:255]))
        assert 1 < v < peak and h[v] < h[1] and h[v] < h[peak], (v, peak, h[:25])


def test_closed_loop_parameters_need_the_valley():
    """The reads the GPU closed loop uses: at the oracle's auto threshold its records are exactly the generator's; at
    today's default min_count 2 erroneous k-mers survive."""
    import cs267_hw3_b200 as kh
    d, reads = _loop_reads()
    h = _oracle_histogram(reads, LOOP_K)
    v = kh.auto_min_count(h)
    assert v > 2
    want = _sorted_rows(d.pairs())
    got, _, _ = oracle.analyse_reads(reads, LOOP_K, v, LOOP_MIN_EXT)
    assert got.shape == want.shape and (got == want).all()
    assert len(oracle.analyse_reads(reads, LOOP_K, 2, LOOP_MIN_EXT)[0]) > len(want)


# ------------------------------------------------------------------------------------------- CPU: CLI and kernel build
def test_kmer_count_cli_usage_errors_for_the_spectrum(tmp_path):
    from cs267_hw3_b200 import build
    exe = build.build_count_cli()
    (tmp_path / "reads.txt").write_bytes(b"ACGTACGTAC\n")
    for args in ([], ["19", "reads.txt"], ["19", "reads.txt", "--histo"], ["19", "reads.txt", "--histo", "h.txt", "--contigs"]):
        r = subprocess.run([exe, *args], cwd=tmp_path, capture_output=True, text=True)
        assert r.returncode == 1 and r.stderr.startswith("Usage: kmer_count K reads_file"), (args, r.stderr)
        assert "--histo HISTO_FILE" in r.stderr and "auto" in r.stderr
    assert not (tmp_path / "h.txt").exists()


def test_histogram_kernel_has_no_spills(tmp_path):
    """kc_histogram_kernel for sm_100a: ptxas reports no stack frame and no spills (both slot widths)."""
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        pytest.skip("nvcc not available")
    from cs267_hw3_b200 import build
    r = subprocess.run([nvcc, *build.NVCC_FLAGS, "-Xptxas", "-v", "-c", os.path.join(build.CSRC, "count.cu"),
                        "-o", str(tmp_path / "count.o")], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    blocks = re.findall(r"Function properties for (\S*kc_histogram_kernel\S*)\n\s*(.*)", r.stderr)
    assert len(blocks) == 2, r.stderr[-2000:]
    for name, props in blocks:
        assert "0 bytes stack frame, 0 bytes spill stores, 0 bytes spill loads" in props, (name, props)


# --------------------------------------------------------------------------------------------------- GPU
@pytest.mark.gpu
@pytest.mark.parametrize("k", [3, 19, 31, 32, 51, 61])
def test_gpu_histogram_matches_the_oracle(k):
    """KmerCounter.histogram() bin for bin against the oracle, reads with errors and k-mers seen more than 255 times;
    sum = n_distinct and every suffix sum = the size of extract(m, any min_ext)."""
    import cs267_hw3_b200 as kh
    reads = _reads(k, 100000, 200, seed=2000 + k, saturate=True)
    want = _oracle_histogram(reads, k)
    assert want[255] > 0
    with kh.KmerCounter(k, max(1024, reads.size), 0.5, 0) as kc:
        kc.count_reads(reads)
        h = kc.histogram()
        assert h.dtype == np.uint64 and h.shape == (256,)
        assert (h == want).all(), np.flatnonzero(h != want)[:10]
        assert int(h.sum()) == kc.stats()["n_distinct"]
        for m, me in ((1, 1), (2, 2), (3, 1), (4, 5), (17, 2), (255, 1)):
            assert int(h[m:].sum()) == len(kc.extract(m, me)), (m, me)
        assert kh.auto_min_count(h) == kh.auto_min_count(want)
        n_launches = kc.stats()["n_launches"]
        assert (kc.histogram() == want).all()                   # the buffer is cleared between calls
        assert kc.stats()["n_launches"] == n_launches + 1


@pytest.mark.gpu
@pytest.mark.parametrize("k", [19, 51])
def test_gpu_histogram_after_growth_and_when_full(k):
    """A counter that grew (n_grows > 0) has the spectrum of one sized generously; an empty counter's is all zero; an
    overflowed table (growing off) is KH_ERR_TABLE_FULL, never a partial spectrum."""
    import ctypes as C

    import cs267_hw3_b200 as kh
    reads = _reads(k, 150000, 200, seed=2100 + k, coverage=3)
    with kh.KmerCounter(k, 100, 0.5, 0) as small, kh.KmerCounter(k, 4 * reads.size, 0.5, 0) as big:
        small.count_reads(reads)
        big.count_reads(reads)
        assert small.stats()["n_grows"] > 0 and big.stats()["n_grows"] == 0
        assert (small.histogram() == big.histogram()).all()
        assert (big.histogram() == _oracle_histogram(reads, k)).all()
        big.clear()
        h = big.histogram()
        assert not h.any() and kh.auto_min_count(h) == 2
    L = kh.lib()
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
            c.histogram()
        assert e.value.status == kh.KH_ERR_TABLE_FULL
        L.kh_device_free(p)


@pytest.mark.gpu
@pytest.mark.parametrize("world", [1, 2, 3, 8])
@pytest.mark.parametrize("batches", [1, 3])
def test_gpu_sharded_histogram_equals_one_counter(world, batches):
    """ShardedCounter.histogram(): the owners' spectra summed bin by bin are the single counter's, with one reduce at
    the end or reduces in between."""
    import cs267_hw3_b200 as kh
    from cs267_hw3_b200.sharded_count import ShardedCounter, split_reads
    k = 31
    reads = _reads(k, 120000, 250, seed=2200 + world, saturate=True)
    with kh.KmerCounter(k, reads.size, 0.5, 0) as one:
        one.count_reads(reads)
        want = one.histogram()
    assert (want == _oracle_histogram(reads, k)).all()
    cuts = split_reads(reads, world * batches)
    with ShardedCounter(k, world, reads.size) as sc:
        for b in range(batches):
            for r in range(world):
                piece = b * world + r
                sc.count(r, reads[cuts[piece]:cuts[piece + 1]])
            sc.reduce()
        h = sc.histogram()
        assert h.dtype == np.uint64 and (h == want).all()
        assert int(h.sum()) == sc.stats()["n_distinct"]


def _run_cli(tmp_path, args, env=None, timeout=300):
    from cs267_hw3_b200 import build
    exe = build.build_count_cli()
    base = {x: v for x, v in os.environ.items() if x not in ("KH_RANKS", "KH_COUNT_BATCH_BYTES")}
    r = subprocess.run([exe, *args], cwd=tmp_path, capture_output=True, text=True, timeout=timeout, env=dict(base, **(env or {})))
    assert r.returncode == 0, r.stdout + r.stderr
    return r.stdout


@pytest.mark.gpu
@pytest.mark.parametrize("ranks", [1, 2])
def test_gpu_kmer_count_histo_alone(tmp_path, ranks):
    """--histo alone: exactly the oracle's spectrum in `c n` lines (255 = 255 or more), no other output file."""
    k = 21
    reads = _reads(k, 60000, 120, seed=2300, coverage=6, error_rate=0.005, saturate=True)
    (tmp_path / "reads.txt").write_bytes(bytes(reads))
    want = _oracle_histogram(reads, k)
    out = _run_cli(tmp_path, [str(k), "reads.txt", "--histo", "spectrum.histo"], env={"KH_RANKS": str(ranks)})
    assert (tmp_path / "spectrum.histo").read_bytes() == _histo_text(want)
    assert sorted(os.listdir(tmp_path)) == ["reads.txt", "spectrum.histo"]
    import cs267_hw3_b200 as kh
    assert (f"Spectrum of {int(want.sum())} distinct {k}-mers written to spectrum.histo: min_count 2, "
            f"auto min_count {kh.auto_min_count(want)}\n") in out


@pytest.mark.gpu
@pytest.mark.parametrize("k,ranks", [(31, 1), (31, 3)])
def test_gpu_kmer_count_auto_threshold_kmer_file(tmp_path, k, ranks):
    """min_count `auto`: the k-mer file is the oracle's records at the oracle's valley; numeric thresholds keep today's
    stdout (no spectrum line)."""
    import cs267_hw3_b200 as kh
    d = kmergen.Dataset(k, 40000, 80, seed=2400 + k)
    reads = readgen.tile_reads(d.solution(), k, read_len=k + 40, coverage=20, seed=2401 + k, error_rate=0.01)
    (tmp_path / "reads.txt").write_bytes(bytes(reads))
    v = kh.auto_min_count(_oracle_histogram(reads, k))
    assert v > 2
    want, _, _ = oracle.analyse_reads(reads, k, v, 2)
    pl = (k + 3) // 4
    want_lines = sorted((oracle.unpack_kmer(bytes(p[:pl]), k) + " " + chr(p[pl]) + chr(p[pl + 1])).encode() for p in want)
    env = {"KH_RANKS": str(ranks)}
    out = _run_cli(tmp_path, [str(k), "reads.txt", "kmers.txt", "auto"], env=env)
    assert f": min_count {v}, auto min_count {v}\n" in out and f"Wrote {len(want)} k-mers (count >= {v}," in out
    assert sorted((tmp_path / "kmers.txt").read_bytes().split(b"\n")[:-1]) == want_lines
    out = _run_cli(tmp_path, [str(k), "reads.txt", "numeric.txt", str(v), "2"], env=env)
    assert "Spectrum" not in out and len(out.splitlines()) == 2
    assert out.splitlines()[0].startswith("Counted ") and out.splitlines()[1].startswith(f"Wrote {len(want)} k-mers")
    assert (tmp_path / "numeric.txt").stat().st_size == (tmp_path / "kmers.txt").stat().st_size


@pytest.mark.gpu
@pytest.mark.parametrize("ranks", [1, 2])
def test_gpu_reads_with_errors_to_contigs_at_the_valley(tmp_path, ranks):
    """Closed loop: 20x reads with 1 % errors -> kmer_count --histo H --contigs out auto M -> the generator's contigs.
    The parameters were chosen with the oracle on the CPU (test_closed_loop_parameters_need_the_valley)."""
    import cs267_hw3_b200 as kh
    d, reads = _loop_reads()
    (tmp_path / "reads.txt").write_bytes(bytes(reads))
    want = _oracle_histogram(reads, LOOP_K)
    out = _run_cli(tmp_path, [str(LOOP_K), "reads.txt", "--histo", "h.histo", "--contigs", "out", "auto", str(LOOP_MIN_EXT)],
                   env={"KH_RANKS": str(ranks)})
    assert (tmp_path / "h.histo").read_bytes() == _histo_text(want)
    v = kh.auto_min_count(want)
    assert f"min_count {v}, auto min_count {v}\n" in out and f"Assembled {LOOP_N} k-mers into" in out
    text = b"".join((tmp_path / f"out_{r}.dat").read_bytes() for r in range(ranks))
    assert b"".join(sorted(text.splitlines(keepends=True))) == d.solution()
