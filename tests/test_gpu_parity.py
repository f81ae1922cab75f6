"""GPU parity: the CUDA path (through the C ABI, include/kh_capi.h) against the oracle, the
golden vectors written by the unmodified reference, and the generator's own solution.

Bit-exact everywhere: the path is integer/byte work, so there is no tolerance.
"""
import os

import numpy as np
import pytest

import oracle
from conftest import GOLDEN, golden_cases
from tools import kmergen

pytestmark = pytest.mark.gpu

CASES = golden_cases()


@pytest.fixture(scope="module")
def kh():
    import cs267_hw3_b200 as m
    assert m.device_count() >= 1, "libkh_b200.so sees no CUDA device"
    return m


def _read(case, ext):
    with open(os.path.join(GOLDEN, f"{case}.{ext}"), "rb") as f:
        return f.read()


def _assemble_text(kh, text, k, load_factor=0.5, options=None, chunks=1, via="pairs"):
    t = np.frombuffer(text, dtype=np.uint8) if not isinstance(text, np.ndarray) else text
    n = t.size // (k + 4)
    with kh.KmerHashTable(k, n, load_factor) as tab:
        for name, val in (options or {}).items():
            tab.set_option(name, val)
        if via == "lines":
            tab.insert_lines(t)
        else:
            pairs = tab.pack_lines(t)
            step = (n + chunks - 1) // chunks if n else 1
            for lo in range(0, n, max(step, 1)):
                tab.insert_pairs(pairs[lo:lo + step])
        buf, offs, nodes = tab.assemble()
        st = tab.stats()
    return buf.tobytes(), offs, nodes, st


# ---------------------------------------------------------------- K1 pack ----------------
@pytest.mark.parametrize("case", sorted(CASES))
def test_pack_golden(kh, case):
    k = CASES[case]["k"]
    text = _read(case, "txt")
    with kh.KmerHashTable(k, 16) as tab:
        got = tab.pack_lines(text)
    assert (got == oracle.parse_lines(text, k)).all()
    for rec, line in zip(got, _read(case, "probe").decode().split("\n")[:-1]):
        assert rec.tobytes().hex() == line.split(" ")[0]       # the reference's own kmer_pair bytes


@pytest.mark.parametrize("k", [2, 5, 19, 20, 29, 30, 31, 32, 51, 60, 61])
def test_pack_all_widths(kh, k):
    rng = np.random.default_rng(k)
    n = 3001
    bases = np.frombuffer(b"ACGT", dtype=np.uint8)[rng.integers(0, 4, (n, k))]
    ext = np.frombuffer(b"ACGTF", dtype=np.uint8)[rng.integers(0, 5, (n, 2))]
    text = np.concatenate([bases, np.full((n, 1), ord(" "), np.uint8), ext, np.full((n, 1), 10, np.uint8)], axis=1)
    with kh.KmerHashTable(k, 16) as tab:
        got = tab.pack_lines(text.reshape(-1))
    assert (got == oracle.parse_lines(text.reshape(-1), k)).all()


def test_pack_rejects_bad_base(kh):
    with kh.KmerHashTable(19, 16) as tab:
        with pytest.raises(kh.KhError) as e:
            tab.pack_lines(b"ACGTACGTACNTACGTACG AC\n")
        assert e.value.status == kh.KH_ERR_BAD_INPUT
        with pytest.raises(kh.KhError):
            tab.pack_lines(b"ACGTACGTACGTACGTACG AX\n")
        assert (tab.pack_lines(b"ACGTACGTACGTACGTACG AC\n") == oracle.parse_lines(b"ACGTACGTACGTACGTACG AC\n", 19)).all()


# ---------------------------------------------------------------- insert + traverse -------
@pytest.mark.parametrize("case", sorted(CASES))
def test_assemble_golden(kh, case):
    """Same bytes, same order as the unmodified reference's <prefix>_0.dat."""
    k = CASES[case]["k"]
    out, offs, nodes, st = _assemble_text(kh, _read(case, "txt"), k)
    assert out == _read(case, "dat")
    assert nodes == CASES[case]["n"] and len(offs) - 1 == CASES[case]["c"]
    assert st["n_inserted"] == CASES[case]["n"] and st["n_duplicates"] == 0


def test_readme_known_answer(kh):
    out, *_ = _assemble_text(kh, _read("readme_k3", "txt"), 3)
    assert sorted(out.split()) == [b"AACCG", b"AATGC", b"GATCTGA"]      # README.md:27


@pytest.mark.parametrize("k,n,c,longn", [
    (19, 50000, 60, 0), (19, 40000, 40000, 0), (19, 30000, 1, 0), (21, 70000, 700, 0), (29, 20000, 100, 0),
    (30, 20000, 100, 0), (31, 60000, 900, 0), (51, 50000, 400, 0), (51, 30000, 3, 29000), (61, 20000, 50, 0),
])
def test_generated_vs_oracle(kh, k, n, c, longn):
    d = kmergen.Dataset(k, n, c, seed=100 + k, long_nodes=longn)
    text = d.text()
    want = oracle.assemble_text(text, k)[0]
    assert want == d.expected()[0]
    out, offs, nodes, st = _assemble_text(kh, text, k)
    assert out == want
    assert nodes == n and len(offs) - 1 == c
    # offsets delimit '\n'-terminated contigs
    b = np.frombuffer(out, dtype=np.uint8)
    assert (b[offs[1:].astype(np.int64) - 1] == 10).all() and offs[0] == 0 and offs[-1] == len(out)


@pytest.mark.parametrize("options", [
    {"split_buckets": 1}, {"split_buckets": 2, "seg_chars": 8}, {"split_buckets": 64, "seg_chars": 16},
    {"split_buckets": 1 << 20, "seg_chars": 248}, {"split_buckets": 1 << 20, "seg_chars": 8},
])
@pytest.mark.parametrize("k", [19, 51])
def test_segmentation_options_do_not_change_output(kh, k, options):
    """Splitter density and segment capacity only change how the walk is cut up."""
    d = kmergen.Dataset(k, 60000, 30, seed=9, long_nodes=20000)
    out, _, nodes, st = _assemble_text(kh, d.text(), k, options=options)
    assert out == d.expected()[0] and nodes == 60000


@pytest.mark.parametrize("lf", [0.3, 0.5, 0.7, 0.9, 0.98])
@pytest.mark.parametrize("k", [19, 51])
def test_load_factors(kh, k, lf):
    d = kmergen.Dataset(k, 80000, 500, seed=int(lf * 100))
    out, *_ = _assemble_text(kh, d.text(), k, load_factor=lf)
    assert out == d.expected()[0]


def test_insert_in_chunks_keeps_start_order(kh):
    d = kmergen.Dataset(19, 50000, 2000, seed=77)
    out, *_ = _assemble_text(kh, d.text(), 19, chunks=7)
    assert out == d.expected()[0]


@pytest.fixture(scope="module")
def large_set():
    """(records, expected output) of a kmergen set, made once per (k, n) for the large plain-table cases below: seed 267
    and the contig density of the test.txt shape (4 514 197 k-mers in 5 736 contigs)."""
    made = {}

    def get(k, n):
        if (k, n) not in made:
            d = kmergen.Dataset(k, n, round(n / 787), seed=267)
            made[k, n] = d.pairs(), d.expected()[0]
            d.close()
        return made[k, n]
    return get


# Kernels a plain-table insert call launches on each path.  The call adds 3 for the start-list scan, and 1 more when it
# brings new start nodes.
_PATH_OF_LAUNCHES = {1: "direct", 3: "insert_slots", 4: "chunked"}


def _insert_paths(tab, pairs, batches):
    """Insert `pairs` from the host in `batches` calls, each within one 64 MB staging piece; the path each call took."""
    paths, step = [], -(-len(pairs) // batches)
    for lo in range(0, len(pairs), step):
        before = tab.stats()
        tab.insert_pairs(pairs[lo:lo + step])
        after = tab.stats()
        launches = after["n_launches"] - before["n_launches"] - 3 - int(after["n_starts"] > before["n_starts"])
        paths.append(_PATH_OF_LAUNCHES.get(launches, launches))
    return paths


def _large_plain(kh, monkeypatch, large_set, k, n, lf, batches):
    """Build a plain table (KH_CT=0) of n k-mers in `batches` calls and check its output; the paths the calls took."""
    monkeypatch.setenv("KH_CT", "0")
    pairs, want = large_set(k, n)
    with kh.KmerHashTable(k, n, lf) as tab:
        paths = _insert_paths(tab, pairs, batches)
        buf, _, nodes = tab.assemble()
        st = tab.stats()
    assert buf.tobytes() == want and nodes == n
    assert st["n_inserted"] == n and st["n_duplicates"] == 0
    return paths


# (k, load factor, batches) -> (k-mers, path of every batch).  Every table is over 64 MiB (n / lf above 8.39 M for
# 64-bit slots, 4.19 M for 128-bit slots), so each call of >= 65 536 records is grouped by table region.
_LARGE_PLAIN = {
    (19, 0.5, 1): (4514197, "chunked"),
    (19, 0.5, 3): (4514197, "chunked"),            # batches after the first load the existing chunks back in
    (19, 0.5, 5): (4514197, "insert_slots"),       # each batch under 1/8 of the table's slots
    (19, 0.9, 1): (8_000_000, "chunked"),
    (19, 0.97, 2): (8_200_000, "chunked"),
    (19, 0.97, 8): (8_200_000, "insert_slots"),
    (51, 0.5, 1): (2_200_000, "insert_slots"),     # 128-bit slots always take insert_slots
    (51, 0.8, 3): (3_500_000, "insert_slots"),
    (31, 0.6, 2): (2_600_000, "insert_slots"),
}


@pytest.mark.parametrize("k,lf,chunks", list(_LARGE_PLAIN))
def test_chunked_shared_memory_build(kh, monkeypatch, large_set, k, lf, chunks):
    """Into a table larger than L2, a batch of at least 1/8 of its 64-bit slots is built chunk by chunk in shared memory
    (no global atomics); smaller batches and 128-bit slots go through the atomic insert_slots path.  Each case reaches
    its path through table and batch size, and all must give the reference's bytes."""
    n, path = _LARGE_PLAIN[k, lf, chunks]
    assert _large_plain(kh, monkeypatch, large_set, k, n, lf, chunks) == [path] * chunks


@pytest.mark.parametrize("chunked", [1, 0])
@pytest.mark.parametrize("pct", ["70", "20"])
def test_grouping_buffer_overflow_paths(kh, monkeypatch, large_set, chunked, pct):
    """The grouping buffers are sized for the expected share plus slack; the rare record that does not fit goes through
    the fix-up list (chunked build) or is inserted directly by partition_kernel (insert_slots path).  KH_DEBUG_CAP_PCT
    shrinks the buffers so a large part of the input takes those paths -- the result must not change."""
    monkeypatch.setenv("KH_DEBUG_CAP_PCT", pct)
    cases = [(19, 4514197, 2, "chunked")] if chunked else [(19, 4514197, 5, "insert_slots"), (51, 2_200_000, 2, "insert_slots")]
    for k, n, batches, path in cases:
        assert _large_plain(kh, monkeypatch, large_set, k, n, 0.5, batches) == [path] * batches


def test_chunked_build_counts_duplicates(kh, large_set):
    """Records already in the table are counted as duplicates by the chunked build and by insert_slots."""
    n = 4514197
    pairs, _ = large_set(19, n)
    with kh.KmerHashTable(19, n) as tab:
        assert _insert_paths(tab, pairs, 1) == ["chunked"]
        assert _insert_paths(tab, pairs[:3_000_000], 1) == ["chunked"]          # a second large batch, all present
        st = tab.stats()
        assert st["n_inserted"] == n and st["n_duplicates"] == 3_000_000
        assert _insert_paths(tab, pairs[:900_000], 1) == ["insert_slots"]
        st = tab.stats()
        assert st["n_inserted"] == n and st["n_duplicates"] == 3_900_000


def test_insert_lines_path(kh):
    d = kmergen.Dataset(31, 50000, 300, seed=78)
    out, *_ = _assemble_text(kh, d.text(), 31, via="lines")
    assert out == d.expected()[0]


def test_per_rank_blocks(kh):
    """rank r emits the contigs whose start line lies in its block (read_kmers.hpp:55-58, kmer_hash.cpp:27-31):
    insert everything, but register start nodes only from the rank's block -- here by inserting the block last
    into a fresh handle that already holds the other records as non-starts is not possible, so emulate ranks
    the way the reference does: one table with all records, starts taken from the block."""
    k, n, c, P = 19, 30000, 300, 3
    d = kmergen.Dataset(k, n, c, seed=5)
    pairs = d.pairs()
    split = (n + P - 1) // P
    for r in range(P):
        lo, hi = split * r, min(n, split * (r + 1))
        others = np.concatenate([pairs[:lo], pairs[hi:]]).copy()
        pl = (k + 3) // 4
        others[others[:, pl] == ord("F"), pl] = ord("A")      # not start nodes for this rank
        with kh.KmerHashTable(k, n) as tab:
            tab.insert_pairs(others)
            tab.insert_pairs(pairs[lo:hi])
            buf, offs, nodes = tab.assemble()
        assert buf.tobytes() == d.expected(P, r)[0]


def test_empty_and_tiny(kh):
    with kh.KmerHashTable(19, 0) as tab:
        buf, offs, nodes = tab.assemble()
        assert buf.size == 0 and list(offs) == [0] and nodes == 0
        tab.insert_pairs(np.empty((0, 7), np.uint8))
        buf, offs, nodes = tab.assemble()
        assert buf.size == 0 and nodes == 0
    out, offs, nodes, _ = _assemble_text(kh, b"ACGTACGTACGTACGTACG FF\n", 19)
    assert out == b"ACGTACGTACGTACGTACG\n" and nodes == 1


def test_clear_gives_a_fresh_table(kh):
    d1, d2 = kmergen.Dataset(19, 20000, 50, seed=1), kmergen.Dataset(19, 15000, 70, seed=2)
    with kh.KmerHashTable(19, 20000) as tab:
        for d in (d1, d2, d1):
            tab.clear()
            tab.insert_pairs(d.pairs())
            buf, _, nodes = tab.assemble()
            assert buf.tobytes() == d.expected()[0] and nodes == d.n
        # assembling twice gives the same answer
        buf2, _, _ = tab.assemble()
        assert buf2.tobytes() == d1.expected()[0]


# ---------------------------------------------------------------- K4 find -----------------
@pytest.mark.parametrize("k", [19, 31, 51])
def test_find_parity(kh, k):
    d = kmergen.Dataset(k, 40000, 200, seed=3 * k)
    pairs = d.pairs()
    pl = (k + 3) // 4
    absent = kmergen.Dataset(k, 5000, 50, seed=999).pairs()[:, :pl]
    queries = np.concatenate([pairs[::3, :pl], absent])
    ref = oracle.Table(k, d.n)
    ref.insert_pairs(pairs)
    with kh.KmerHashTable(k, d.n) as tab:
        tab.insert_pairs(pairs)
        got, found = tab.find(queries)
    for q, g, f in zip(queries, got, found):
        want = ref.find(q.tobytes())
        assert f == (want is not None)
        assert g.tobytes() == (want if want is not None else bytes(pl + 2))


def test_duplicate_keys_are_counted(kh):
    d = kmergen.Dataset(19, 10000, 30, seed=12)
    pairs = d.pairs()
    with kh.KmerHashTable(19, 20000) as tab:
        tab.insert_pairs(pairs)
        tab.insert_pairs(pairs[:1234])
        st = tab.stats()
        assert st["n_inserted"] == 10000 and st["n_duplicates"] == 1234


# ---------------------------------------------------------------- error behaviour ---------
def test_missing_successor(kh):
    # kmer_hash.cpp:47-49: the reference throws this exact text
    with kh.KmerHashTable(19, 16) as tab:
        tab.insert_lines(b"ACGTACGTACGTACGTACG FC\n")
        with pytest.raises(kh.KhError) as e:
            tab.assemble()
        assert e.value.status == kh.KH_ERR_NOT_FOUND
        assert "k-mer not found in Distributed HashMap" in str(e.value)
    with pytest.raises(RuntimeError, match="not found"):
        oracle.assemble_text(b"ACGTACGTACGTACGTACG FC\n", 19)


def _cycle_text(k, tail_len, cyc_len, seed):
    rng = np.random.default_rng(seed)
    while True:
        cyc = "".join("ACGT"[i] for i in rng.integers(0, 4, cyc_len))
        pre = "".join("ACGT"[i] for i in rng.integers(0, 4, tail_len))
        s = pre + cyc + cyc[:k]               # windows of pre+cyc, wrapping around the cycle once
        kmers = [s[i:i + k] for i in range(tail_len + cyc_len)]
        if len(set(kmers)) == len(kmers):
            break
    lines = []
    for i, km in enumerate(kmers):
        back = s[i - 1] if i > 0 else ("F" if tail_len > 0 else cyc[-1])   # a start node only when there is a tail
        fwd = s[i + k]                        # never 'F': the chain runs into the cycle and stays there
        lines.append(f"{km} {back}{fwd}\n")
    rng.shuffle(lines)
    return "".join(lines).encode()


@pytest.mark.parametrize("split", [1, 1 << 20])
def test_cycle_is_reported_not_spun_on(kh, split):
    text = _cycle_text(15, 40, 300, seed=split)
    with pytest.raises(RuntimeError, match="cycle"):
        oracle.assemble_text(text, 15)
    with kh.KmerHashTable(15, 400) as tab:
        tab.set_option("split_buckets", split)
        tab.insert_lines(text)
        with pytest.raises(kh.KhError) as e:
            tab.assemble()
        assert e.value.status == kh.KH_ERR_CYCLE


def test_pure_cycles_without_start_are_ignored(kh):
    # SURVEY 5.1-6: k-mers on no start-rooted chain are silently ignored by the reference
    k = 15
    d = kmergen.Dataset(k, 5000, 20, seed=8)
    cyc = _cycle_text(k, 0, 500, seed=4)      # no start node in it
    text = d.text().tobytes() + cyc
    assert oracle.assemble_text(text, k)[0] == d.expected()[0]
    for split in (1, 8, 1 << 20):
        out, _, nodes, _ = _assemble_text(kh, text, k, options={"split_buckets": split})
        assert out == d.expected()[0] and nodes == 5000


def test_table_full(kh):
    d = kmergen.Dataset(19, 5000, 10, seed=2)
    with kh.KmerHashTable(19, 100, 1.0) as tab:
        with pytest.raises(kh.KhError) as e:
            tab.insert_pairs(d.pairs())
        assert e.value.status == kh.KH_ERR_TABLE_FULL


def test_bad_extension_in_records(kh):
    p = oracle.parse_lines(b"ACGTACGTACGTACGTACG FC\n", 19).copy()
    p[0, -1] = ord("N")
    with kh.KmerHashTable(19, 16) as tab:
        with pytest.raises(kh.KhError) as e:
            tab.insert_pairs(p)
        assert e.value.status == kh.KH_ERR_BAD_INPUT


def test_converging_chains(kh):
    """Two start nodes whose chains share a suffix: outside the input contract (README.md:33-35).  The
    reference emits the shared suffix twice.  This library either does exactly the same (no walk-segment
    boundary falls on the shared part) or refuses with KH_ERR_CONVERGE -- it never emits anything else."""
    k = 11
    a = "ACGGTCATTGCAAGTCCGATAGG"
    b = "T" + a[6:6 + k - 1]                   # second start that feeds into a's 7th k-mer
    lines = [f"{a[i:i + k]} {'F' if i == 0 else a[i - 1]}{'F' if i + k == len(a) else a[i + k]}\n" for i in range(len(a) - k + 1)]
    lines.append(f"{b} F{a[6 + k - 1]}\n")
    text = "".join(lines).encode()
    want = oracle.assemble_text(text, k)[0]
    assert want == (a + "\n" + b + a[6 + k - 1:] + "\n").encode()
    outcomes = set()
    for split in (1, 2, 8, 1 << 20):
        with kh.KmerHashTable(k, 64) as tab:
            tab.set_option("split_buckets", split)
            tab.insert_lines(text)
            try:
                buf, _, _ = tab.assemble()
                assert buf.tobytes() == want
                outcomes.add("same")
            except kh.KhError as e:
                assert e.status == kh.KH_ERR_CONVERGE
                outcomes.add("refused")
    assert "refused" in outcomes               # split_buckets=1 puts a segment boundary on the shared part


# ---------------------------------------------------------------- scale -------------------
@pytest.mark.parametrize("k,n,c,longn", [(19, 4514197, 5736, 0), (51, 3000000, 28770, 0), (51, 3000000, 300, 1000000),
                                         (31, 2000000, 19000, 0)])
def test_medium_shapes_exact(kh, k, n, c, longn):
    """test.txt shape (results_serial.txt:7-9) and k=51 shapes incl. one 10^6-node contig: byte-exact in start order."""
    d = kmergen.Dataset(k, n, c, seed=267, long_nodes=longn)
    want, nc = d.expected_array()
    with kh.KmerHashTable(k, n) as tab:
        tab.insert_pairs(d.pairs())
        buf, offs, nodes = tab.assemble(copy=False)
        assert nodes == n and len(offs) - 1 == c == nc
        assert buf.size == want.size and np.array_equal(buf, want)
        assert kmergen.digest_lines(buf) == d.digest()


@pytest.mark.parametrize("k", [19, 51])
def test_full_chr14_shape_properties(kh, k):
    """BASELINE.json configs[1]/[2]: 89 710 742 k-mers, 860 329 contigs.  Too big for the oracle's C restatement in a
    test, so: (1) the exact bytes of the output against the sha256 the UNMODIFIED reference (oracle/_ref) wrote for this
    very file (tests/golden/chr14_full.json, made by tests/golden/make_full_digests.py -- 383 s / 468 s of CPU per K),
    and (2) the size-independent properties: every k-mer on exactly one contig, contig count, and the
    order-independent digest of the contig set against the generator's own solution."""
    import hashlib
    import json
    n, c = 89_710_742, 860_329
    with open(os.path.join(GOLDEN, "chr14_full.json")) as f:
        ref = json.load(f)[f"chr14_k{k}"]
    assert ref["n_kmers"] == n and ref["n_contigs"] == c and ref["seed"] == 267
    d = kmergen.Dataset(k, n, c, seed=267)
    import cs267_hw3_b200 as m
    pb = m.pair_bytes(k)
    host = m.PinnedBuffer(n * pb)
    d.pairs_into(host.ptr, 0, n)
    with kh.KmerHashTable(k, n) as tab:
        tab.insert_pairs_ptr(host.ptr, n)
        buf, offs, nodes = tab.assemble(copy=False)
        st = tab.stats()
        assert st["n_inserted"] == n and st["n_duplicates"] == 0
        assert nodes == n and len(offs) - 1 == c
        assert buf.size == n + c * k == ref["dat_bytes"]          # sum over contigs of (nodes + K - 1) + 1
        assert hashlib.sha256(buf.tobytes()).hexdigest() == ref["dat_sha256"], "differs from what the unmodified reference wrote"
        assert kmergen.digest_lines(buf) == d.digest()
    host.free()


def test_orphan_chains_and_cycles_are_ignored(kh):
    """k-mers on no start-rooted chain (dangling chains with a missing successor, cycles) are never visited by
    the reference (kmer_hash.cpp:41-53): no error, same output (ADVICE r1).  Plain table here (the walkers that start
    at splitter slots land on such chains), chunk table in test_gpu_ctable.py."""
    k = 19
    d = kmergen.Dataset(k, 30000, 80, seed=8)
    rng = np.random.default_rng(3)
    extra = []
    for _ in range(200):
        s = "".join("ACGT"[i] for i in rng.integers(0, 4, k + 12))
        extra += [f"{s[i:i + k]} {s[i - 1] if i else 'C'}{s[i + k]}\n" for i in range(10)]
    text = d.text().tobytes() + "".join(extra).encode() + _cycle_text(k, 0, 500, seed=4)
    want = oracle.assemble_text(text, k)[0]
    assert want == d.expected()[0]
    out, _, nodes, _ = _assemble_text(kh, text, k)
    assert out == want and nodes == d.n
