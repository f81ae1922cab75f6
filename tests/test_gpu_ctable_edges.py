"""The chunk table (csrc/ctable.cuh) at its capacity edges.

A chunk holds every k-mer whose minimizer hashes to it, at most CtBuild<W>::kMaxSlots = 4352 (128-bit slots, K 23-54)
or 6144 (64-bit slots, K 17-22) of them.  Random sequence fills the fullest chunk to about half of that and keeps
every chain inside a chunk short; a tandem repeat with diverged copies does neither: one m-mer is the minimizer of
thousands of k-mers, so they all land in one chunk as one long chain.  These tests build such sets on purpose:

  * X(m), the m-mer with the smallest order value of all, is the minimizer of every k-mer that has it in its window;
  * "X + 10 random bases", repeated, is one K=51 contig whose k-mers all hold X: one chain in one chunk;
  * contigs that each pass through X once crowd X's chunk with short runs (window 7 at K 17-22) that enter and
    leave it through pending links.

CPU: the constructions and the mirrors they rely on, and a model of the build kernel's pointer-jumping phase under
the stale-read schedule (tests/native/ct_jump_model.cu, built against the shipped header).
GPU: bit-exact output against the oracle with the crowded chunk exactly full, one record past it, lookups in a full
chunk, the sharded path, and the bounded contig walk at its 512-link limit.  The per-chunk load is read back from
the table, so a construction that is off by one fails instead of passing a less crowded case.
"""
import ctypes as C
import os
import shutil
import subprocess

import numpy as np
import pytest

import oracle
from cs267_hw3_b200 import sharded as sh
from tools import kmergen

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
M32 = (1 << 32) - 1
MUL, ADD = 0x9E3779B1, 0x7F4A7C15          # the minimizer order (csrc/slot.cuh: kMinMul, kMinAdd)
MAX_SLOTS = {1: 6144, 2: 4352}              # CtBuild<W>::kMaxSlots
LUT = np.full(256, 255, dtype=np.uint8)
for _i, _c in enumerate(b"ACGT"):
    LUT[_c] = _i


# ------------------------------------------------------------------------------------------------ mirrors ----
def order_value(x: int, m: int) -> int:
    """h(x) = ((x * MUL mod 4^m) << (32 - 2m)) + ADD mod 2^32: the order of m-mers that ct_min_hash minimises."""
    return ((((x * MUL) & ((1 << 2 * m) - 1)) << (32 - 2 * m)) + ADD) & M32


def crowding_mmer(m: int) -> str:
    """The m-mer of smallest order value.  h is a bijection; (v << s) + ADD wraps past 2^32 exactly for v >= v0, and
    every wrapped value is below ADD, so the minimum is at v0 = ceil((2^32 - ADD) / 2^s), x = v0 * MUL^-1 mod 4^m."""
    s = 32 - 2 * m
    v0 = -(-((1 << 32) - ADD) // (1 << s))
    x = v0 * pow(MUL, -1, 1 << 2 * m) % (1 << 2 * m)
    return "".join("ACGT"[(x >> (2 * (m - 1 - i))) & 3] for i in range(m))


def _mmer_int(s: str) -> int:
    v = 0
    for ch in s:
        v = (v << 2) | "ACGT".index(ch)
    return v


def _fmix32_hi(h):
    h = h ^ (h >> np.uint64(15))
    h = (h * np.uint64(0x85EBCA6B)) & np.uint64(M32)
    h = h ^ (h >> np.uint64(13))
    return (h * np.uint64(0xC2B2AE35)) & np.uint64(M32)


def min_hash_codes(codes: np.ndarray, k: int) -> np.ndarray:
    """ct_min_hash of every row of an (n, k) array of base codes (vectorised form of sharded.ct_min_hash)."""
    m, win = sh.ct_minimizer_len(k), sh.ct_window(k)
    cols = k - m + 1
    v = np.zeros((codes.shape[0], cols), dtype=np.uint64)
    for t in range(m):
        v = (v << np.uint64(2)) | codes[:, t:t + cols].astype(np.uint64)
    v = v[:, cols - win:]                                        # the win rightmost m-mers
    h = (((v * np.uint64(MUL)) & np.uint64((1 << 2 * m) - 1)) << np.uint64(32 - 2 * m)) + np.uint64(ADD)
    return (h & np.uint64(M32)).min(axis=1)


def place(mh, world: int, chunks: int):
    """ct_place (csrc/slot.cuh): owner rank and GLOBAL chunk id (owner * C + local chunk) of minimizer hashes."""
    u = _fmix32_hi(np.asarray(mh, dtype=np.uint64) ^ (np.asarray(mh, dtype=np.uint64) >> np.uint64(16)))
    owner = (u * np.uint64(world)) >> np.uint64(32)
    return owner, (u * np.uint64(world * chunks)) >> np.uint64(32)


def chunk_of_x(m: int, world: int, chunks: int) -> tuple[int, int]:
    """(owner, local chunk) of X(m)'s chunk."""
    o, g = place([order_value(_mmer_int(crowding_mmer(m)), m)], world, chunks)
    return int(o[0]), int(g[0]) - int(o[0]) * chunks


def codes_of(s: str) -> np.ndarray:
    return LUT[np.frombuffer(s.encode(), dtype=np.uint8)]


def codes_of_pairs(pairs: np.ndarray, k: int) -> np.ndarray:
    pl = (k + 3) // 4
    b = pairs[:, :pl]
    return np.stack([(b >> 6) & 3, (b >> 4) & 3, (b >> 2) & 3, b & 3], axis=2).reshape(b.shape[0], 4 * pl)[:, :k]


def global_chunks(seq: str, k: int, world: int, chunks: int) -> np.ndarray:
    """Global chunk of every k-mer of a base string, in order."""
    w = np.lib.stride_tricks.sliding_window_view(codes_of(seq), k)
    return place(min_hash_codes(w, k), world, chunks)[1]


def count_segments(contigs: list[str], k: int, world: int, chunks: int) -> int:
    """Chunk segments of a set of contigs: a contig has one segment per run of consecutive k-mers in one chunk."""
    return sum(1 + int(np.count_nonzero(np.diff(global_chunks(s, k, world, chunks).astype(np.int64)))) for s in contigs)


def lines_of(seq: str, k: int, open_end: bool = False) -> list[str]:
    """k-mer file lines of one contig (the first backward and last forward extension 'F')."""
    n = len(seq) - k + 1 - (1 if open_end else 0)
    return [f"{seq[i:i + k]} {'F' if i == 0 else seq[i - 1]}{seq[i + k] if i + k < len(seq) else 'F'}\n" for i in range(n)]


def _rand(rng, n: int) -> str:
    return "".join("ACGT"[i] for i in rng.integers(0, 4, n))


# -------------------------------------------------------------------------------------------- constructions ----
def long_chain(k: int, length: int, seed: int, extra: int = 0) -> str:
    """Base string of `length` + `extra` k-mers: X(m) followed by 10 random bases, repeated.  Every window of the
    win rightmost m-mers (46 bases at K=51) holds a whole copy of X, so all the k-mers share its chunk."""
    m = sh.ct_minimizer_len(k)
    x = crowding_mmer(m)
    assert sh.ct_window(k) + m - 1 >= (m + 10) + m - 1           # any window of that many bases holds a whole copy
    rng = np.random.default_rng(seed)
    need = length + extra + k - 1
    parts = []
    while sum(map(len, parts)) < need:
        parts += [x, _rand(rng, 10)]
    return "".join(parts)[:need]


def crowd(k: int, target: int, world: int, chunks: int, seed: int, flank=(1, 12), used=None) -> list[str]:
    """Contigs that each pass through X(m) once, with random flanks of `flank` k-mers on both sides (pending links
    into and out of X's chunk), until X's chunk holds exactly `target` of their k-mers (the flanks' k-mers land there
    too now and then; the mirror counts them).  No k-mer repeats, within the set or with `used`."""
    m, win = sh.ct_minimizer_len(k), sh.ct_window(k)
    x = crowding_mmer(m)
    o, cx = chunk_of_x(m, world, chunks)
    gx = o * chunks + cx
    rng = np.random.default_rng(seed)
    used = set() if used is None else used
    out, count = [], 0
    while count < target:
        a, b = (int(v) for v in rng.integers(flank[0], flank[1] + 1, 2))
        core = [_rand(rng, k - m), x, _rand(rng, win - 1)]            # exactly the win k-mers that hold X in their window
        seq = _rand(rng, a) + "".join(core) + _rand(rng, b)
        add = int(np.count_nonzero(global_chunks(seq, k, world, chunks) == gx))
        if count + add > target:                                  # finish with a contig of core k-mers only
            r = target - count
            seq = core[0] + x + core[2][:r - 1] if r <= win else "".join(core)
            add = len(seq) - k + 1
        kmers = [seq[i:i + k] for i in range(len(seq) - k + 1)]
        if len(set(kmers)) != len(kmers) or used.intersection(kmers):
            continue
        used.update(kmers)
        out.append(seq)
        count += add
    return out


# ------------------------------------------------------------------------------------------------ CPU tests ----
@pytest.mark.parametrize("m", [11, 12, 13, 14, 15, 16])
def test_crowding_mmer_has_the_smallest_order_value(m):
    x = crowding_mmer(m)
    hx = order_value(_mmer_int(x), m)
    rng = np.random.default_rng(m)
    sample = rng.integers(0, 1 << 2 * m, 50000)
    assert all(order_value(int(v), m) > hx for v in sample if int(v) != _mmer_int(x))
    if m == 11:                                                  # small enough to look at every m-mer
        allv = np.arange(1 << 22, dtype=np.uint64)
        h = ((((allv * np.uint64(MUL)) & np.uint64((1 << 22) - 1)) << np.uint64(10)) + np.uint64(ADD)) & np.uint64(M32)
        assert int(h.argmin()) == _mmer_int(x) and int(h.min()) == hx
    # the library's own mirror: a k-mer that holds X in its window has X's order value as its minimizer hash
    for k in [k for k in range(17, 55) if sh.ct_minimizer_len(k) == m]:
        win = sh.ct_window(k)
        for j in (0, win - 1):                                   # X at both ends of the window
            s = _rand(rng, k - m - j) + x + _rand(rng, j)
            slot = sh.slot_from_pair(oracle.pack_kmer(s) + b"AA", k)
            assert sh.ct_min_hash(slot, k) == hx


@pytest.mark.parametrize("k", [19, 22, 23, 31, 51])
def test_vector_mirror_matches_the_library_mirror(k):
    d = kmergen.Dataset(k, 3000, 30, seed=k)
    pairs = d.pairs()
    mh = min_hash_codes(codes_of_pairs(pairs, k), k)
    for world, chunks in ((1, 13), (3, 7), (8, 1000)):
        owner, g = place(mh, world, chunks)
        for i in range(0, pairs.shape[0], 37):
            slot = sh.slot_from_pair(pairs[i].tobytes(), k)
            assert int(mh[i]) == sh.ct_min_hash(slot, k)
            assert int(owner[i]) == sh.owner_of_slot(slot, k, world)
            assert 0 <= int(g[i]) - int(owner[i]) * chunks < chunks


@pytest.mark.parametrize("length", [1025, 4352, 9950])
def test_long_chain_is_one_chain_in_one_chunk(length):
    k = 51
    seq = long_chain(k, length, seed=length)
    kmers = [seq[i:i + k] for i in range(length)]
    assert len(seq) == length + k - 1 and len(set(kmers)) == length
    hx = order_value(_mmer_int(crowding_mmer(15)), 15)
    w = np.lib.stride_tricks.sliding_window_view(codes_of(seq), k)
    assert (min_hash_codes(w, k) == hx).all()
    for world, chunks in ((1, 7), (3, 100)):
        assert count_segments([seq], k, world, chunks) == 1
    text = "".join(lines_of(seq, k)).encode()
    assert oracle.assemble_text(text, k)[0] == (seq + "\n").encode()


@pytest.mark.parametrize("k,target", [(17, 6144), (19, 6144), (22, 6144), (23, 4352), (31, 4352)])
@pytest.mark.parametrize("world,chunks", [(1, 3), (1, 40), (3, 11)])
def test_crowd_fills_one_chunk_exactly(k, target, world, chunks):
    contigs = crowd(k, target, world, chunks, seed=k + chunks)
    o, cx = chunk_of_x(sh.ct_minimizer_len(k), world, chunks)
    allc = np.concatenate([global_chunks(s, k, world, chunks) for s in contigs])
    assert int(np.count_nonzero(allc == o * chunks + cx)) == target
    kmers = [s[i:i + k] for s in contigs for i in range(len(s) - k + 1)]
    assert len(set(kmers)) == len(kmers)
    text = "".join(ln for s in contigs for ln in lines_of(s, k)).encode()
    out = oracle.assemble_text(text, k)[0]
    assert out == "".join(s + "\n" for s in contigs).encode()


@pytest.fixture(scope="module")
def jump_model(tmp_path_factory):
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        pytest.skip("nvcc not available")
    exe = str(tmp_path_factory.mktemp("jump") / "ct_jump_model")
    subprocess.run([nvcc, "-std=c++17", "-O1", "-gencode", "arch=compute_100a,code=sm_100a", "-o", exe,
                    os.path.join(ROOT, "tests", "native", "ct_jump_model.cu")], check=True, capture_output=True)
    return exe


@pytest.mark.parametrize("w", [1, 2])
def test_pointer_jumping_settles_a_full_chunk(jump_model, w):
    """Phase 4 of ct_build_kernel under the schedule that is worst for it (every read of another thread's node sees
    the last barrier's value): a chain through every record of a full chunk settles within the shipped round cap.
    With the earlier cap of (14 + J - 1) / J = 5 rounds of J = 3 passes, chains of more than 4^5 + 1 = 1025 nodes did
    not, and their segment was never written."""
    cap_slots = MAX_SLOTS[w]
    for length in (1025, 1500, 2048, cap_slots):
        for seed in range(6):
            out = subprocess.run([jump_model, str(w), str(length), str(seed)], capture_output=True, text=True, check=True).stdout.split()
            jumps, threads, max_slots, cap, rounds_run, unsettled, needed = (int(v) for v in out)
            assert max_slots == cap_slots and threads == 512
            assert unsettled == 0, f"W={w}: {unsettled} of {length} nodes unsettled after {rounds_run} rounds"
            assert needed <= cap and rounds_run <= cap
            if jumps == 3:                                       # (J + 1)^R >= length - 1, and no fewer rounds do
                assert needed == {1025: 5, 1500: 6, 2048: 6}.get(length, 7)


# ------------------------------------------------------------------------------------------------ GPU tests ----
def _lib():
    import cs267_hw3_b200 as kh

    L = kh.lib()
    L.kh_debug_buffer.argtypes = [C.c_void_p, C.c_char_p, C.POINTER(C.c_void_p), C.POINTER(C.c_uint64)]
    L.kh_copy_to_host.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64]
    return kh, L


def _chunks_per_rank(tab) -> int:
    kh, L = _lib()
    p, b = C.c_void_p(), C.c_uint64()
    tab._check(L.kh_debug_buffer(tab._h, b"caps", C.byref(p), C.byref(b)))
    return int(C.cast(p, C.POINTER(C.c_uint64))[4])


def _chunk_load(tab, chunk: int) -> int:
    kh, L = _lib()
    p, b = C.c_void_p(), C.c_uint64()
    tab._check(L.kh_debug_buffer(tab._h, b"chunk_cursor", C.byref(p), C.byref(b)))
    out = np.zeros(1, dtype=np.uint32)
    tab._check(L.kh_copy_to_host(tab._h, out.ctypes.data, p.value + 4 * chunk, 4))
    return int(out[0])


@pytest.fixture
def ct_always(monkeypatch):
    monkeypatch.setenv("KH_CT", "2")


def _background(k: int, n: int, seed: int):
    d = kmergen.Dataset(k, n, n // 100, seed=seed)
    text = d.text().tobytes()
    contigs = d.expected()[0].decode().split()
    return text, contigs


@pytest.mark.gpu
@pytest.mark.parametrize("length", [1025, 1500, "full"])
@pytest.mark.parametrize("lf", [0.5, 0.9])
@pytest.mark.parametrize("background", [0, 200_000])
def test_one_chain_in_one_chunk(ct_always, length, lf, background):
    """One K=51 contig whose k-mers all share X's chunk, alone or among random contigs; "full": exactly as many
    chain k-mers as the chunk has room for next to the background records the mirror puts there."""
    kh, _ = _lib()
    k = 51
    bg_text, bg_contigs = _background(k, background, seed=7) if background else (b"", [])
    n_max = background + MAX_SLOTS[2]
    with kh.KmerHashTable(k, n_max, lf) as tab:
        chunks = _chunks_per_rank(tab)
        _, cx = chunk_of_x(15, 1, chunks)
        bg_in_x = sum(int(np.count_nonzero(global_chunks(s, k, 1, chunks) == cx)) for s in bg_contigs)
        n_chain = MAX_SLOTS[2] - bg_in_x if length == "full" else length
        seq = long_chain(k, n_chain, seed=n_chain)
        text = bg_text + "".join(lines_of(seq, k)).encode()
        want = oracle.assemble_text(text, k)[0]
        tab.insert_lines(text)
        assert _chunk_load(tab, cx) == bg_in_x + n_chain
        buf, _, nodes = tab.assemble()
        st = tab.stats()
    assert buf.tobytes() == want
    assert st["n_inserted"] == background + n_chain and nodes == background + n_chain
    assert st["n_segments"] == count_segments(bg_contigs, k, 1, chunks) + len(bg_contigs) + 2     # + start stubs


@pytest.mark.gpu
@pytest.mark.parametrize("k", [19, 22, 23])
def test_crowded_chunk_exactly_full(ct_always, k):
    """Many contigs through X, each a short run in X's chunk with pending links into and out of it, until the chunk
    is full to the record (6144 at K=19 and 22, 4352 at K=23)."""
    kh, _ = _lib()
    target = MAX_SLOTS[1 if k <= 22 else 2]
    with kh.KmerHashTable(k, 4 * target) as tab:
        chunks = _chunks_per_rank(tab)
        _, cx = chunk_of_x(sh.ct_minimizer_len(k), 1, chunks)
        contigs = crowd(k, target, 1, chunks, seed=k)
        text = "".join(ln for s in contigs for ln in lines_of(s, k)).encode()
        want = oracle.assemble_text(text, k)[0]
        tab.insert_lines(text)
        assert _chunk_load(tab, cx) == target
        buf, _, nodes = tab.assemble()
        st = tab.stats()
    n = len(text) // (k + 4)
    assert buf.tobytes() == want and nodes == n and st["n_inserted"] == n
    assert st["n_segments"] == count_segments(contigs, k, 1, chunks) + len(contigs)


@pytest.mark.gpu
@pytest.mark.parametrize("k", [51, 19])
def test_one_record_past_capacity_is_refused(ct_always, k):
    """kMaxSlots + 1 k-mers that share a minimizer: KH_ERR_TABLE_FULL with a message that names the per-chunk
    limit, at the insert and again at a traverse tried anyway, and no output; after clear() the handle is whole."""
    kh, _ = _lib()
    w = 2 if k == 51 else 1
    with kh.KmerHashTable(k, 4 * MAX_SLOTS[w]) as tab:
        chunks = _chunks_per_rank(tab)
        if k == 51:
            contigs = [long_chain(k, MAX_SLOTS[w] + 1, seed=3)]
        else:
            contigs = crowd(k, MAX_SLOTS[w] + 1, 1, chunks, seed=3)
        text = "".join(ln for s in contigs for ln in lines_of(s, k)).encode()
        with pytest.raises(kh.KhError) as e:
            tab.insert_lines(text)
        assert e.value.status == kh.KH_ERR_TABLE_FULL
        assert f"more than {MAX_SLOTS[w]} k-mers that share one minimizer" in str(e.value)
        with pytest.raises(kh.KhError) as e:
            tab.assemble()
        assert e.value.status == kh.KH_ERR_TABLE_FULL
        tab.clear()
        if k == 51:                                                   # the same chain one k-mer shorter
            legal = "".join(lines_of(contigs[0][:-1], k)).encode()
        else:
            legal = "".join(ln for s in crowd(k, MAX_SLOTS[w], 1, chunks, seed=4) for ln in lines_of(s, k)).encode()
        tab.insert_lines(legal)
        buf, _, _ = tab.assemble()
        assert buf.tobytes() == oracle.assemble_text(legal, k)[0]


@pytest.mark.gpu
def test_lookups_in_a_full_chunk(ct_always):
    """X's chunk holds 4352 records in 4352 slots: no hole stops a probe.  Present keys are found; absent keys with
    minimizer X are not (the probe wraps the whole chunk and stops); a contig whose successor is such a key fails with
    the reference's message."""
    kh, _ = _lib()
    k, n = 51, MAX_SLOTS[2]
    pl = (k + 3) // 4
    seq = long_chain(k, n, seed=11, extra=50)
    with kh.KmerHashTable(k, n) as tab:
        chunks = _chunks_per_rank(tab)
        _, cx = chunk_of_x(15, 1, chunks)
        text = "".join(lines_of(seq[:n + k - 1], k)).encode()
        tab.insert_lines(text)
        pairs = oracle.parse_lines(text, k)
        got, found = tab.find(pairs[:, :pl])
        assert _chunk_load(tab, cx) == n
        assert found.all() and (got == pairs).all()
        absent = oracle.parse_lines("".join(lines_of(seq[n:], k)).encode(), k)
        got, found = tab.find(absent[:, :pl])
        assert not found.any() and not got.any()
        tab.clear()
        open_text = "".join(lines_of(seq[:n + k], k, open_end=True)).encode()      # the last k-mer's successor is absent
        tab.insert_lines(open_text)
        assert _chunk_load(tab, cx) == n
        with pytest.raises(kh.KhError) as e:
            tab.assemble()
        assert e.value.status == kh.KH_ERR_NOT_FOUND
        assert "k-mer not found in Distributed HashMap" in str(e.value)
    with pytest.raises(RuntimeError, match="not found"):
        oracle.assemble_text(open_text, k)


def _sharded(k: int, world: int, n_total: int, make_contigs):
    """One sharded step through LocalComm on one GPU.  make_contigs(chunks_per_rank) builds the input once the shards
    exist; returns (input text, per-rank outputs, rank 0's rank_rounds, load of X's chunk on the rank that owns it)."""
    import test_gpu_sharded as S
    import cs267_hw3_b200 as kh

    shards = [sh.Shard(k, r, world, n_total, n_total, 0.5, device=0) for r in range(world)]
    comm = sh.LocalComm(shards)
    comm.connect()
    bufs = []
    try:
        chunks = _chunks_per_rank(shards[0].tab)
        contigs = make_contigs(chunks)
        text = "".join(ln for s in contigs for ln in lines_of(s, k)).encode()
        pairs = oracle.parse_lines(text, k)
        blocks, bufs = S._upload(kh, sh, shards, pairs, pairs.shape[0])
        comm.begin()
        sh.sharded_insert(comm, blocks)
        rounds = sh.sharded_assemble(comm)
        outs = [s.result_host()[0].tobytes() for s in shards]
        o, cx = chunk_of_x(sh.ct_minimizer_len(k), world, chunks)
        load = _chunk_load(shards[o].tab, cx)
        return text, outs, rounds, load
    finally:
        comm.close()
        for p in bufs:
            kh.lib().kh_device_free(p)
        for s in shards:
            s.close()


@pytest.mark.gpu
@pytest.mark.parametrize("world", [2, 3, 8])
@pytest.mark.parametrize("k", [51, 19])
def test_sharded_chunk_at_capacity(world, k):
    """The full chain (K=51) and the full crowd (K=19) on `world` ranks: every rank sends its block's share of the
    crowd to the owner of X's chunk, which ends up with exactly a full chunk; every rank's output is the reference's."""
    w = 2 if k == 51 else 1
    cap = MAX_SLOTS[w]
    if k == 51:
        make = lambda chunks: [long_chain(k, cap, seed=world)]           # noqa: E731
    else:
        make = lambda chunks: crowd(k, cap, world, chunks, seed=world)   # noqa: E731
    text, outs, _, load = _sharded(k, world, 4 * cap, make)
    assert load == cap
    assert outs == oracle.assemble_text(text, k, world)


def _walk_contig(k: int, world: int, chunks: int, segments: int, seed: int) -> str:
    """A random contig cut right after the first k-mer of its `segments`-th chunk segment."""
    rng = np.random.default_rng(seed)
    seq = _rand(rng, 40 * segments + k)
    g = global_chunks(seq, k, world, chunks).astype(np.int64)
    starts = np.flatnonzero(np.diff(g)) + 1                        # k-mers that open segments 2, 3, ...
    cut = int(starts[segments - 2]) + 1 + int(rng.integers(0, starts[segments - 1] - starts[segments - 2]))
    return seq[:cut + k - 1]


@pytest.mark.gpu
@pytest.mark.parametrize("world", [1, 2])
@pytest.mark.parametrize("segments", [513, 514])
def test_bounded_walk_at_its_limit(ct_always, world, segments):
    """ct_walk_len_kernel follows at most 512 links, i.e. a contig of 513 chunk segments is walked and one of 514
    falls back to pointer jumping (rank_rounds 1 on the walk, more after jumping).  Both give the exact output."""
    kh, _ = _lib()
    k = 51
    if world == 1:
        with kh.KmerHashTable(k, 40000) as tab:
            chunks = _chunks_per_rank(tab)
            seq = _walk_contig(k, 1, chunks, segments, seed=segments)
            assert count_segments([seq], k, 1, chunks) == segments
            text = "".join(lines_of(seq, k)).encode()
            tab.insert_lines(text)
            buf, _, _ = tab.assemble()
            st = tab.stats()
        assert buf.tobytes() == (seq + "\n").encode()
        assert st["n_segments"] == segments + 1                        # + the head stub
        rounds = st["rank_rounds"]
    else:
        box = {}

        def make(chunks):
            box["seq"] = _walk_contig(k, world, chunks, segments, seed=segments)
            assert count_segments([box["seq"]], k, world, chunks) == segments
            return [box["seq"]]

        text, outs, rounds, _ = _sharded(k, world, 40000, make)
        assert outs == oracle.assemble_text(text, k, world)
        assert b"".join(outs) == (box["seq"] + "\n").encode()
    assert (rounds == 1) == (segments == 513), f"rank_rounds {rounds} for {segments} segments"
