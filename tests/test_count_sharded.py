"""Sharded k-mer analysis: per-rank counters merged at the k-mers' owner ranks (kh_count_partition, kh_count_merge_device,
kh_sharded::CountCluster, cs267_hw3_b200.sharded_count.ShardedCounter, kmer_count with KH_RANKS).

The bar is bit-identity: saturating counter fields add associatively, so records AND all nine counters of the merged
owner tables must equal one counter over all reads -- and the oracle.
CPU: the __host__ __device__ functions (csrc/count_core.cuh) run serially by tests/native/count_merge_host_check.cu.
GPU: the same through the C ABI and the drivers; with one GPU all ranks share device 0, with more they are real peers."""
import os
import shutil
import subprocess

import numpy as np
import pytest

import oracle
from cs267_hw3_b200.sharded_count import count_owner, owner_of_record, split_reads
from tools import kmergen, readgen

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _sorted_rows(a: np.ndarray) -> np.ndarray:
    return a[np.lexsort(a.T[::-1])] if a.size else a


def _reads(k, n, c, seed, coverage=3, error_rate=0.0, with_n=False, read_len=None):
    d = kmergen.Dataset(k, n, c, seed=seed)
    reads = readgen.tile_reads(d.solution(), k, read_len=read_len or (k + 40), coverage=coverage, seed=seed + 1,
                               error_rate=error_rate)
    if with_n:                                   # N and lower case are not bases: they split reads
        rng = np.random.default_rng(seed + 2)
        pos = rng.choice(reads.size, size=max(1, reads.size // 500), replace=False)
        reads[pos] = np.where(rng.random(pos.size) < 0.5, ord("N"), ord("a")).astype(np.uint8)
    return d, reads


def _text_reads(k, seed):
    if k < 8:                                    # few distinct k-mers: random text with separators
        rng = np.random.default_rng(seed)
        reads = np.frombuffer(b"ACGT", dtype=np.uint8)[rng.integers(0, 4, 6000)].copy()
        reads[rng.choice(reads.size, 80, replace=False)] = 10
        return reads
    return _reads(k, 10000, 25, seed=seed, coverage=3, error_rate=0.002, with_n=True)[1]


# ------------------------------------------------------------------------------- CPU: the kernels' functions, serially
@pytest.fixture(scope="module")
def merge_check(tmp_path_factory):
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        pytest.skip("nvcc not available")
    exe = str(tmp_path_factory.mktemp("merge") / "count_merge_host_check")
    subprocess.run([nvcc, "-std=c++17", "-O1", "-Wno-deprecated-gpu-targets", "-o", exe,
                    os.path.join(ROOT, "tests", "native", "count_merge_host_check.cu")], check=True, capture_output=True)
    return exe


def _run_merge(exe, tmp_path, reads, k, world, batches, min_count, min_ext, n_slots=None):
    f = tmp_path / "reads.txt"
    np.asarray(reads, dtype=np.uint8).tofile(f)
    n_slots = n_slots or max(1024, 2 * len(reads))
    out = subprocess.run([exe, "merge", str(k), str(world), str(batches), str(n_slots), str(min_count), str(min_ext), str(f)],
                         capture_output=True, text=True, check=True).stdout.splitlines()
    head = [int(x) for x in out[0].split()]
    pb = (k + 3) // 4 + 2
    rank = np.array([int(ln.split()[0]) for ln in out[1:]], dtype=np.int64)
    recs = np.array([list(bytes.fromhex(ln.split()[1])) for ln in out[1:]], dtype=np.uint8).reshape(-1, pb)
    cnts = np.array([[int(x) for x in ln.split()[2:11]] for ln in out[1:]], dtype=np.uint32).reshape(-1, 9)
    order = np.lexsort(recs.T[::-1]) if recs.size else np.zeros(0, dtype=np.int64)
    return head, rank[order], recs[order], cnts[order]


@pytest.mark.parametrize("world", [1, 2, 3, 8])
@pytest.mark.parametrize("k", [3, 19, 31, 32, 51, 61])
def test_merged_owner_tables_match_the_oracle(merge_check, tmp_path, k, world):
    """P pieces counted into P tables, partitioned by kc_owner, merged with kc_merge_slot: the owner tables together are
    one counter over all reads -- records and all nine counters -- with substitution errors and N / lower-case bytes."""
    reads = _text_reads(k, 700 + k)
    want_p, want_c, n_occ = oracle.analyse_reads(reads, k, 2, 2)
    n_all = len(oracle.analyse_reads(reads, k, 1, 1)[0])
    head, rank, recs, cnts = _run_merge(merge_check, tmp_path, reads, k, world, 1, 2, 2)
    assert head[0] == n_occ and head[1] == n_all and head[2] == len(want_p) and head[3] == 0
    assert recs.shape == want_p.shape and (recs == want_p).all()
    assert (cnts == want_c).all()
    # the Python mirror of kc_owner agrees with where the host functions put every k-mer
    assert all(owner_of_record(r, k, world) == o for r, o in zip(recs, rank))


@pytest.mark.parametrize("k,world,batches", [(19, 3, 4), (32, 2, 3), (51, 8, 2), (61, 3, 5)])
def test_batches_reduce_into_non_empty_owner_tables(merge_check, tmp_path, k, world, batches):
    """Count / reduce repeated: every batch merges into owner tables that already hold earlier batches' k-mers."""
    reads = _text_reads(k, 900 + k)
    want_p, want_c, n_occ = oracle.analyse_reads(reads, k, 1, 1)
    head, _, recs, cnts = _run_merge(merge_check, tmp_path, reads, k, world, batches, 1, 1)
    assert head[0] == n_occ and head[1] == len(want_p) and head[3] == 0
    assert (recs == want_p).all() and (cnts == want_c).all()


def test_merge_saturates_exactly_like_one_counter(merge_check, tmp_path):
    """A read repeated 300 times over 3 ranks: no rank reaches a cap (~100 each), the merged counters stop at exactly 255
    occurrences and 127 observations, as the oracle's single count does."""
    reads = np.frombuffer(b"CGTACGTTAGCATTGACC\n" * 300, dtype=np.uint8).copy()
    want_p, want_c, n_occ = oracle.analyse_reads(reads, 7, 1, 1)
    head, _, recs, cnts = _run_merge(merge_check, tmp_path, reads, 7, 3, 1, 1, 1, n_slots=1024)
    assert head[0] == n_occ and head[3] == 0
    assert head[4] < 255 and head[5] < 127                          # nothing saturated on a rank
    assert (recs == want_p).all() and (cnts == want_c).all()
    assert cnts[:, 0].max() == 255 and cnts[:, 1:].max() == 127


def test_owner_is_independent_of_the_home_slot(merge_check):
    """The keys one rank owns (P = 8) spread evenly over the home slots of its table: in each of 8 equal ranges of slots
    the count stays within 6 standard deviations of the mean.  An owner taken from kc_home's bits would put them all
    into one range."""
    world, n_keys = 8, 800000
    out = subprocess.run([merge_check, "spread", str(world), str(1 << 22), str(n_keys)], capture_output=True, text=True,
                         check=True).stdout.split()
    hist = np.array([int(x) for x in out], dtype=np.float64)
    assert abs(hist.sum() - n_keys / world) < 6 * np.sqrt(n_keys / world)       # rank 0 owns 1/P of the keys
    mean = hist.sum() / world
    assert (np.abs(hist - mean) < 6 * np.sqrt(mean)).all(), hist


def _fields(c):
    return [c & 0xFF] + [(c >> (8 + 7 * f)) & 127 for f in range(8)]


def test_kc_add_saturates_every_field_without_carry(merge_check):
    def add(a, b):
        return int(subprocess.run([merge_check, "add", str(a), str(b)], capture_output=True, text=True, check=True).stdout)

    def word(fields):
        return fields[0] | sum(v << (8 + 7 * f) for f, v in enumerate(fields[1:]))

    rng = np.random.default_rng(5)
    cases = [([255] + [127] * 8, [1] * 9), ([200] + [100] * 8, [100] + [50] * 8), ([254] + [126] * 8, [1] * 9),
             ([0] * 9, [255] + [127] * 8), ([128] + [64] * 8, [127] + [63] * 8)]
    cases += [(list(rng.integers(0, 256, 1)) + list(rng.integers(0, 128, 8)), list(rng.integers(0, 256, 1)) + list(rng.integers(0, 128, 8)))
              for _ in range(6)]
    for fa, fb in cases:
        a, b = word([int(x) for x in fa]), word([int(x) for x in fb])
        want = [min(255, int(fa[0]) + int(fb[0]))] + [min(127, int(x) + int(y)) for x, y in zip(fa[1:], fb[1:])]
        got = add(a, b)
        assert _fields(got) == want and got == word(want), (fa, fb)


def test_split_reads_cuts_only_behind_non_base_bytes():
    rng = np.random.default_rng(8)
    for trial in range(30):
        n = int(rng.integers(0, 3000))
        alpha = np.frombuffer(b"ACGT" * int(rng.integers(1, 40)) + b"N\na", dtype=np.uint8)
        text = alpha[rng.integers(0, alpha.size, n)]
        for world in (1, 2, 3, 8):
            cuts = split_reads(text, world)
            assert len(cuts) == world + 1 and cuts[0] == 0 and cuts[-1] == n
            assert all(a <= b for a, b in zip(cuts, cuts[1:]))
            assert all(c in (0, n) or text[c - 1] not in b"ACGT" for c in cuts), (trial, world, cuts)
    # a single read without separators stays in one piece
    assert split_reads(b"ACGT" * 100, 4) == [0, 400, 400, 400, 400]
    assert split_reads(b"ACG\nTTT\nGGG\nCCC\n", 4) == [0, 4, 8, 12, 16]


def test_count_owner_mirror_spreads_keys():
    """The Python mirror used by the GPU tests: keys spread evenly over the ranks."""
    rng = np.random.default_rng(1)
    keys = rng.integers(0, 1 << 62, 40000, dtype=np.int64)
    for world in (2, 3, 8):
        h = np.bincount([count_owner(0, int(x), world) for x in keys], minlength=world)
        assert (np.abs(h - keys.size / world) < 6 * np.sqrt(keys.size / world)).all()


# --------------------------------------------------------------------------------------------------- GPU
def _half(reads):
    return split_reads(reads, 2)[1]


@pytest.mark.gpu
@pytest.mark.parametrize("k", [19, 31, 51])
def test_gpu_merge_two_counters_is_one_counter(k):
    import cs267_hw3_b200 as kh
    _, reads = _reads(k, 150000, 300, seed=1100 + k, coverage=4, error_rate=0.002, with_n=True)
    cut = _half(reads)
    pl = (k + 3) // 4
    with kh.KmerCounter(k, len(reads), 0.5, 0) as one, kh.KmerCounter(k, len(reads), 0.5, 0) as a, \
            kh.KmerCounter(k, len(reads), 0.5, 0) as b:
        one.count_reads(reads)
        a.count_reads(reads[:cut])
        b.count_reads(reads[cut:])
        a.merge(b)
        want = _sorted_rows(one.extract(1, 1))
        got = _sorted_rows(a.extract(1, 1))
        assert got.shape == want.shape and (got == want).all()
        assert (a.lookup(want[:, :pl]) == one.lookup(want[:, :pl])).all()
        assert a.stats()["n_distinct"] == one.stats()["n_distinct"]
        assert a.stats()["n_occurrences"] == one.stats()["n_occurrences"] - b.stats()["n_occurrences"]   # counted here only
        w, wc, _ = oracle.analyse_reads(reads, k, 2, 2)
        assert (_sorted_rows(a.extract(2, 2)) == w).all() and (a.lookup(w[:, :pl]) == wc).all()


@pytest.mark.gpu
@pytest.mark.parametrize("world", [1, 2, 3, 4, 8])
def test_gpu_sharded_counter_equals_one_counter(world):
    import cs267_hw3_b200 as kh
    from cs267_hw3_b200.sharded_count import ShardedCounter
    k = 31
    _, reads = _reads(k, 120000, 250, seed=1200 + world, coverage=4, error_rate=0.002, with_n=True)
    want_p, want_c, n_occ = oracle.analyse_reads(reads, k, 2, 2)
    pl = (k + 3) // 4
    with kh.KmerCounter(k, len(reads), 0.5, 0) as one:
        one.count_reads(reads)
        single = _sorted_rows(one.extract(2, 2))
        n_distinct = one.stats()["n_distinct"]
    assert (single == want_p).all()
    cuts = split_reads(reads, world)
    with ShardedCounter(k, world, len(reads)) as sc:
        for r in range(world):
            sc.count(r, reads[cuts[r]:cuts[r + 1]])
        sc.reduce()
        parts = [sc.extract(r, 2, 2) for r in range(world)]
        union = _sorted_rows(np.concatenate(parts))
        assert union.shape == want_p.shape and (union == want_p).all()
        owner = np.array([owner_of_record(x, k, world) for x in want_p])
        for r, p in enumerate(parts):
            assert all(owner_of_record(x, k, world) == r for x in p)
            assert (sc.lookup(r, want_p[owner == r, :pl]) == want_c[owner == r]).all()
        st = sc.stats()
        assert st["n_distinct"] == n_distinct and st["n_occurrences"] == n_occ and st["n_bytes"] == reads.size
        shares = np.array([len(p) for p in parts], dtype=np.float64)
        assert (np.abs(shares - shares.sum() / world) < 6 * np.sqrt(shares.sum() / world) + 1).all(), shares


@pytest.mark.gpu
def test_gpu_owner_tables_grow_during_merge():
    """Owner tables created far too small grow while merging (kc_reserve / kc_grow) with the same result; with growing
    off a merge that does not fit is KH_ERR_TABLE_FULL, never a silent loss."""
    import cs267_hw3_b200 as kh
    from cs267_hw3_b200.sharded_count import ShardedCounter
    k = 51
    _, reads = _reads(k, 150000, 200, seed=1300, coverage=3, error_rate=0.002)
    want_p, want_c, _ = oracle.analyse_reads(reads, k, 2, 2)
    cuts = split_reads(reads, 2)
    with ShardedCounter(k, 2, 100) as sc:
        for r in range(2):
            sc.count(r, reads[cuts[r]:cuts[r + 1]])
        sc.reduce()
        assert all(c.stats()["n_grows"] > 0 for c in sc.owned)
        assert (_sorted_rows(np.concatenate([sc.extract(r, 2, 2) for r in range(2)])) == want_p).all()
    with kh.KmerCounter(k, len(reads), 0.5, 0) as src:
        src.count_reads(reads)
        os.environ["KH_COUNT_GROW"] = "0"
        try:
            dst = kh.KmerCounter(k, 1000, 1.0, 0)
        finally:
            os.environ.pop("KH_COUNT_GROW")
        with dst:
            with pytest.raises(kh.KhError) as e:
                dst.merge(src)
            assert e.value.status == kh.KH_ERR_TABLE_FULL
    # a count that overflowed its table cannot be partitioned
    import ctypes as C
    L = kh.lib()
    with kh.KmerCounter(k, 100, 0.5, 0) as c:
        p = C.c_void_p()
        assert L.kh_device_alloc(C.byref(p), reads.size) == 0
        with kh.KmerHashTable(k, 1024) as tab:
            tab._check(L.kh_copy_device(tab._h, p, reads.ctypes.data, reads.size))
            tab.sync()
        c.count_reads_device(p.value, reads.size)
        with pytest.raises(kh.KhError) as e:
            c.partition(2)
        assert e.value.status == kh.KH_ERR_TABLE_FULL
        L.kh_device_free(p)


@pytest.mark.gpu
@pytest.mark.parametrize("k,world", [(19, 2), (51, 3)])
def test_gpu_reads_to_contigs_over_sharded_counting(k, world):
    """reads -> ShardedCounter -> every rank's records stay on its GPU -> sharded insert + traverse: the union of the
    ranks' contigs is the generator's solution."""
    import ctypes as C  # noqa: F401

    from cs267_hw3_b200 import sharded as sh
    from cs267_hw3_b200.sharded_count import ShardedCounter
    n, c = 200000, 500
    d, reads = _reads(k, n, c, seed=1400 + k, coverage=8, error_rate=0.0005)
    cuts = split_reads(reads, world)
    with ShardedCounter(k, world, reads.size // 4) as sc:
        for r in range(world):
            sc.count(r, reads[cuts[r]:cuts[r + 1]])
        sc.reduce()
        blocks = [sc.extract_device(r, 3, 3) for r in range(world)]
        assert sum(b[1] for b in blocks) == n
        n_local_max = max(b[1] for b in blocks)
        shards = [sh.Shard(k, r, world, n_local_max, n, 0.5, device=sc.devices[r]) for r in range(world)]
        comm = sh.LocalComm(shards)
        comm.connect()
        comm.begin()
        sh.sharded_insert(comm, blocks)
        sh.sharded_assemble(comm)
        text = b"".join(s.result_host()[0].tobytes() for s in shards)
        for s in shards:
            s.close()
    assert b"".join(sorted(text.splitlines(keepends=True))) == d.solution()


@pytest.mark.gpu
@pytest.mark.parametrize("k,ranks,batch", [(19, 2, None), (31, 3, None), (51, 3, 200000), (19, 2, 100000)])
def test_gpu_kmer_count_cli_with_ranks(tmp_path, k, ranks, batch):
    """KH_RANKS=P: the same k-mer file up to line order and the same contigs (cat | sort) as P = 1, the same counts in the
    'Counted' line; a small KH_COUNT_BATCH_BYTES forces several reduces."""
    from cs267_hw3_b200 import build
    exe = build.build_count_cli()
    # 8 passes, 0.05 % substitutions, thresholds 3: exactly the generator's k-mers (checked against the oracle for these seeds)
    d, reads = _reads(k, 80000, 150, seed=1500 + k, coverage=8, error_rate=0.0005)
    (tmp_path / "reads.txt").write_bytes(bytes(reads))
    env1 = {x: v for x, v in os.environ.items() if x not in ("KH_RANKS", "KH_COUNT_BATCH_BYTES")}
    envp = dict(env1, KH_RANKS=str(ranks), **({"KH_COUNT_BATCH_BYTES": str(batch)} if batch else {}))

    def run(env, *args):
        r = subprocess.run([exe, str(k), "reads.txt", *args, "3", "3"], cwd=tmp_path, capture_output=True, text=True,
                           timeout=300, env=env)
        assert r.returncode == 0, r.stdout + r.stderr
        return r.stdout

    o1 = run(env1, "one.txt")
    op = run(envp, "many.txt")
    assert o1.split(" in ")[0] == op.split(" in ")[0]                 # "Counted N occurrences, M distinct ..."
    assert sorted((tmp_path / "one.txt").read_bytes().split(b"\n")) == sorted((tmp_path / "many.txt").read_bytes().split(b"\n"))
    run(env1, "--contigs", "c1")
    run(envp, "--contigs", "cp")
    one = sorted((tmp_path / "c1_0.dat").read_bytes().splitlines(keepends=True))
    many = sorted(b"".join((tmp_path / f"cp_{r}.dat").read_bytes() for r in range(ranks)).splitlines(keepends=True))
    assert many == one and b"".join(one) == d.solution()
    if batch:
        assert len(bytes(reads)) > 2 * ranks * batch                     # at least two reduces before the final one
