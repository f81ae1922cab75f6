"""The chunk table's pointer-jumping fallback (csrc/ctable.cuh: ct_rank_round_kernel, ct_lengths_kernel,
ct_claim_kernel, ct_emit_kernel, ct_emit_heads_kernel).

A chunk-table traverse ranks its contigs by walking them (ct_walk_len_kernel) unless some contig has more than 513
chunk segments; then the whole step, every contig of it, goes through pointer jumping.  Every start-rooted cycle ends
up there too (the walk gives up after 512 links), so every KH_ERR_CYCLE a chunk table reports comes from it.
KH_DEBUG_WALK_STEPS=0 sends any step with a contig of two or more chunk segments down that path, and the behaviour
suite runs again under it.  Every assemble that emits output asserts rank_rounds >= 2 whenever a contig has two or
more chunk segments, so a case that quietly stayed on the walk fails instead of passing.

CPU: ct_jump_link, the per-link update, run over cycles and chains (tests/native/ct_link_jump_check.cu, built against
the shipped header).
GPU: the parity suite under the knob; headless and start-rooted cycles (exactly KH_ERR_CYCLE, also through a crowded
chunk, where a distance that carried into the final bit used to turn it into KH_ERR_CONVERGE); converging chains
(exactly KH_ERR_CONVERGE); one- and two-k-mer contigs; reuse of one handle; every K; 2, 3 and 8 ranks; and the
fallback reached without the knob.  Bit-exact against the oracle, or the exact status.
"""
import os
import shutil
import subprocess

import numpy as np
import pytest

import oracle
import test_gpu_ctable_edges as E
import test_gpu_parity as P
from cs267_hw3_b200 import sharded as sh
from tools import kmergen

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ERR_NOT_FOUND, ERR_CYCLE, ERR_CONVERGE = 1, 4, 16        # kh_shard_finish error bits


# ------------------------------------------------------------------------------------------------ CPU tests ----
@pytest.fixture(scope="module")
def link_jump_check(tmp_path_factory):
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        pytest.skip("nvcc not available")
    exe = str(tmp_path_factory.mktemp("linkjump") / "ct_link_jump_check")
    subprocess.run([nvcc, "-std=c++17", "-O1", "-gencode", "arch=compute_100a,code=sm_100a", "-o", exe,
                    os.path.join(ROOT, "tests", "native", "ct_link_jump_check.cu")], check=True, capture_output=True)
    return exe


@pytest.mark.parametrize("shape", ["cycle", "chain"])
def test_jump_link_on_the_host(link_jump_check, shape):
    """cycle: a head stub in front of a cycle of 1 .. 1000 segments averaging 1 .. 6000 characters stays open (never
    final) through all kCtMaxRounds rounds.  A sum that carried into the final bit closed it from about 128
    characters per segment on.  chain: exact distances and final bits, up to 2^31 - 128 characters."""
    r = subprocess.run([link_jump_check, shape], capture_output=True, text=True)
    assert r.returncode == 0 and r.stdout.startswith("ok "), r.stdout + r.stderr


def cycle_lines(cyc: str, k: int, start: bool) -> list[str]:
    """k-mer lines of the cyclic sequence `cyc` (k-mer i is cyc[i:i+k] read around the end).  With `start`, k-mer 0
    has backward 'F', so it is a start node whose chain comes back to it: no k-mer has two predecessors."""
    s = cyc + cyc[:k]
    return [f"{s[i:i + k]} {'F' if start and i == 0 else cyc[i - 1]}{s[i + k]}\n" for i in range(len(cyc))]


def cycle_chunks(cyc: str, k: int, world: int, chunks: int) -> np.ndarray:
    """Global chunk of every k-mer of a cyclic sequence, from k-mer 0 on."""
    return E.global_chunks(cyc + cyc[:k - 1], k, world, chunks)


def cycle_segments(cyc: str, k: int, world: int, chunks: int) -> int:
    """Chunk segments of a start-rooted cycle: k-mer 0 opens one (backward 'F'), every change of chunk another."""
    g = cycle_chunks(cyc, k, world, chunks).astype(np.int64)
    return 1 + int(np.count_nonzero(np.diff(g)))


def random_cycle(k: int, n: int, seed: int) -> str:
    rng = np.random.default_rng(seed)
    while True:
        cyc = E._rand(rng, n)
        s = cyc + cyc[:k - 1]
        if len({s[i:i + k] for i in range(n)}) == n:
            return cyc


def crowded_cycle(k: int, length: int, closing: int, seed: int) -> str:
    """`length` k-mers of X(m)'s crowded chain (E.long_chain), closed into a cycle by `closing` random bases."""
    rng = np.random.default_rng(seed)
    chain = E.long_chain(k, length, seed)
    cyc = chain + E._rand(rng, closing)
    s = cyc + cyc[:k - 1]
    assert len({s[i:i + k] for i in range(len(cyc))}) == len(cyc)
    return cyc


@pytest.mark.parametrize("k", [19, 51])
def test_cycle_constructions(k):
    """The pure start-rooted cycle is refused by the oracle as a cycle; the crowded one (K=51) holds X's chain."""
    for cyc in [random_cycle(k, 400, seed=k)] + ([crowded_cycle(k, 1500, 30, seed=1)] if k == 51 else []):
        text = "".join(cycle_lines(cyc, k, start=True)).encode()
        with pytest.raises(RuntimeError, match="cycle"):
            oracle.assemble_text(text, k)
        pairs = oracle.parse_lines(text, k)
        pl = (k + 3) // 4
        assert int(np.count_nonzero(pairs[:, pl] == ord("F"))) == 1 and not (pairs[:, pl + 1] == ord("F")).any()
    if k == 51:
        cyc = crowded_cycle(k, 1500, 30, seed=1)
        hx = E.order_value(E._mmer_int(E.crowding_mmer(15)), 15)
        w = np.lib.stride_tricks.sliding_window_view(E.codes_of(cyc[:1500 + k - 1]), k)
        assert (E.min_hash_codes(w, k) == hx).all()


# ------------------------------------------------------------------------------------------------ GPU tests ----
def _jumping() -> bool:
    return os.environ.get("KH_CT") == "2" and os.environ.get("KH_DEBUG_WALK_STEPS") == "0"


def _multi_segment(contigs, k: int, world: int, chunks: int) -> bool:
    """Does any of these base strings have two or more chunk segments?  Longest first, prefixes first: cheap for
    the 10^6-k-mer contigs of the medium shapes."""
    for s in sorted(contigs, key=len, reverse=True):
        if len(s) <= k:
            break
        for part in (s[:5000 + k - 1], s):
            if E.count_segments([part], k, world, chunks) > 1:
                return True
            if len(part) == len(s):
                break
    return False


def _contigs_of(buf, offs) -> list[str]:
    b = np.asarray(buf).tobytes()
    o = np.asarray(offs, dtype=np.int64)
    return [b[o[i]:o[i + 1] - 1].decode() for i in range(len(o) - 1)]


@pytest.fixture(autouse=True)
def jump(request, monkeypatch):
    """Chunk table, pointer jumping for every contig of two or more chunk segments; every KmerHashTable.assemble of
    a GPU test checks that the step really went that way."""
    monkeypatch.setenv("KH_CT", "2")
    monkeypatch.setenv("KH_DEBUG_WALK_STEPS", "0")
    if request.node.get_closest_marker("gpu") is None:
        return
    import cs267_hw3_b200 as kh

    orig = kh.KmerHashTable.assemble

    def assemble(self, copy=True):
        buf, offs, nodes = orig(self, copy)
        if _jumping() and 17 <= self.k <= 54:
            chunks = E._chunks_per_rank(self)
            if _multi_segment(_contigs_of(buf, offs), self.k, 1, chunks):
                rounds = self.stats()["rank_rounds"]
                assert rounds >= 2, f"K={self.k}: a contig of two or more chunk segments, but rank_rounds {rounds}"
        return buf, offs, nodes

    monkeypatch.setattr(kh.KmerHashTable, "assemble", assemble)


@pytest.fixture(scope="module")
def kh():
    import cs267_hw3_b200 as m
    assert m.device_count() >= 1, "libkh_b200.so sees no CUDA device"
    return m


def run(kh, k: int, n_expected: int, make, lf: float = 0.5):
    """Insert the lines make(chunks_per_rank) returns ((text, base strings whose segments to count)) into one table
    and assemble (chunks_per_rank is None for a plain table).  Returns (output bytes or None, status, stats, text, chunks).  Under the knob a step with a
    string of two or more chunk segments must show rank_rounds >= 2, whether it emitted output or refused."""
    with kh.KmerHashTable(k, n_expected, lf) as tab:
        chunks = E._chunks_per_rank(tab) if os.environ.get("KH_CT") == "2" and 17 <= k <= 54 else None
        text, paths = make(chunks)
        tab.insert_lines(text)
        out, status = None, kh.KH_OK
        try:
            buf, _, _ = tab.assemble()
            out = buf.tobytes()
        except kh.KhError as e:
            status, msg = e.status, str(e)
            if status == kh.KH_ERR_NOT_FOUND:
                assert "k-mer not found in Distributed HashMap" in msg
        st = tab.stats()
    if chunks and _jumping() and _multi_segment(paths, k, 1, chunks):
        assert st["rank_rounds"] >= 2, f"stayed on the bounded walk: rank_rounds {st['rank_rounds']}"
    return out, status, st, text, chunks


def assemble(kh, k: int, n_expected: int, make, lf: float = 0.5):
    """run() for an input that must assemble: (bytes, stats), checked against the oracle here."""
    out, status, st, text, _ = run(kh, k, n_expected, make, lf)
    assert status == kh.KH_OK, f"status {status}"
    assert out == oracle.assemble_text(text, k)[0]
    return out, st


def _lines(seqs, k: int) -> str:
    return "".join(ln for s in seqs for ln in E.lines_of(s, k))


def _background(k: int, n: int, c: int, seed: int):
    d = kmergen.Dataset(k, n, c, seed=seed)
    return d.text().tobytes().decode(), d.expected()[0].decode().split()


# ---- the parity suite under the knob ----
def _params(fn):
    return [m for m in fn.pytestmark if m.name == "parametrize"][0].args[1]


test_assemble_golden = pytest.mark.gpu(P.test_assemble_golden)
test_load_factors = pytest.mark.gpu(P.test_load_factors)
test_insert_in_chunks_keeps_start_order = pytest.mark.gpu(P.test_insert_in_chunks_keeps_start_order)
test_per_rank_blocks = pytest.mark.gpu(P.test_per_rank_blocks)
test_empty_and_tiny = pytest.mark.gpu(P.test_empty_and_tiny)
test_clear_gives_a_fresh_table = pytest.mark.gpu(P.test_clear_gives_a_fresh_table)
test_missing_successor = pytest.mark.gpu(P.test_missing_successor)
test_orphan_chains_and_cycles_are_ignored = pytest.mark.gpu(P.test_orphan_chains_and_cycles_are_ignored)
test_medium_shapes_exact = pytest.mark.gpu(P.test_medium_shapes_exact)


@pytest.mark.gpu
@pytest.mark.parametrize("k,n,c,longn", [p for p in _params(P.test_generated_vs_oracle) if 17 <= p[0] <= 54])
def test_generated_vs_oracle(kh, k, n, c, longn):
    P.test_generated_vs_oracle(kh, k, n, c, longn)


# ---- cycles ----
@pytest.mark.gpu
@pytest.mark.parametrize("k", [19, 51])
def test_headless_cycles_beside_contigs_are_ignored(kh, k):
    """Cycles no start node leads into, each spanning two or more chunks (so they are segment cycles that keep
    jumping through every round), beside start-rooted contigs and orphan chains: the reference's output."""
    bg, contigs = _background(k, 20000, 60, seed=k)
    cycles = [random_cycle(k, 60 + 37 * i, seed=100 + i) for i in range(12)]

    def make(chunks):
        for cyc in cycles:
            assert len(set(cycle_chunks(cyc, k, 1, chunks).tolist())) >= 2
        text = bg + "".join(ln for cyc in cycles for ln in cycle_lines(cyc, k, start=False))
        return text.encode(), contigs
    out, st = assemble(kh, k, 30000, make)
    print(f"rank_rounds with headless cycles (K={k}): {st['rank_rounds']}")


def _pure_cycle_status(kh, k, cyc, crowded: bool):
    def make(chunks):
        if chunks is None:               # plain table
            return "".join(cycle_lines(cyc, k, start=True)).encode(), []
        segs = cycle_segments(cyc, k, 1, chunks)
        assert segs >= 2, "the cycle lies in one chunk"
        if crowded:                      # the carry case: segments average far more than 2^31 / 2^24 = 128 characters
            _, cx = E.chunk_of_x(15, 1, chunks)
            assert cycle_chunks(cyc, k, 1, chunks)[0] == cx and len(cyc) / segs > 200
        return "".join(cycle_lines(cyc, k, start=True)).encode(), [cyc]
    out, status, st, _, _ = run(kh, k, 40000, make)
    assert out is None
    return status, st


@pytest.mark.gpu
@pytest.mark.parametrize("table", ["chunk", "plain"])
@pytest.mark.parametrize("case", ["random_k19", "random_k51", "crowded_k51"])
def test_pure_start_rooted_cycle(kh, monkeypatch, table, case):
    """The start k-mer has backward 'F' and the last k-mer leads back to it: no k-mer has two predecessors, so the
    only right status is KH_ERR_CYCLE ("a start-rooted chain never reaches forward ext 'F'").  crowded: 1500 k-mers
    of X's chain in one segment, closed by a short random stretch; the head stub's distance passes 2^31 within the
    24 rounds."""
    if table == "plain":
        monkeypatch.setenv("KH_CT", "0")
    k = 19 if case == "random_k19" else 51
    cyc = crowded_cycle(k, 1500, 30, seed=1) if case == "crowded_k51" else random_cycle(k, 400, seed=k)
    status, st = _pure_cycle_status(kh, k, cyc, crowded=case == "crowded_k51")
    assert status == kh.KH_ERR_CYCLE, f"status {status}, rank_rounds {st['rank_rounds']}"


@pytest.mark.gpu
@pytest.mark.parametrize("k", [19, 51])
def test_cycle_entered_from_a_tail(kh, k):
    """A start node's chain runs into a cycle (the entry k-mer has two predecessors): KH_ERR_CYCLE or
    KH_ERR_CONVERGE (DESIGN 8), never output."""
    text = P._cycle_text(k, 40, 300, seed=k)
    out, status, _, _, _ = run(kh, k, 40000, lambda chunks: (text, []))
    assert out is None and status in (kh.KH_ERR_CYCLE, kh.KH_ERR_CONVERGE)


# ---- converging chains ----
def _converging(k: int, chunks: int, where: str, seed: int):
    """A long contig a and a one-k-mer start node b whose successor is a's k-mer j: the chains share a's suffix.
    where: "middle" (k-mer j inside a's segment, b in another chunk), "boundary" (k-mer j opens a segment, b in
    another chunk), "apart" (boundary, and a's and b's start k-mers in different chunks)."""
    rng = np.random.default_rng(seed)
    a = E._rand(rng, 300 + k)
    g = E.global_chunks(a, k, 1, chunks)
    for j in range(5, len(a) - k):
        for c in "ACGT":
            if c == a[j - 1]:
                continue
            b = c + a[j:j + k - 1]
            gb = int(E.global_chunks(b, k, 1, chunks)[0])
            if where == "middle" and g[j - 1] == g[j] and gb != g[j]:
                return a, b, j
            if where in ("boundary", "apart") and g[j - 1] != g[j] and gb != g[j] and (where == "boundary" or gb != g[0]):
                return a, b, j
    raise AssertionError(f"no {where} join found")


@pytest.mark.gpu
@pytest.mark.parametrize("knob", ["jump", "walk"])
@pytest.mark.parametrize("where", ["middle", "boundary", "apart"])
def test_converging_chains(kh, monkeypatch, knob, where):
    """Two start nodes, one end node: exactly KH_ERR_CONVERGE on the fallback (the claim of the shared tail, or the
    marker of a link into the middle of a segment).  On the walk the same input gives the reference's bytes (the
    shared suffix twice) or KH_ERR_CONVERGE."""
    if knob == "walk":
        monkeypatch.delenv("KH_DEBUG_WALK_STEPS")
    k = 19
    box = {}

    def make(chunks):
        a, b, j = _converging(k, chunks, where, seed=3)
        assert E.count_segments([a], k, 1, chunks) >= 2
        box["want"] = (a + "\n" + b + a[j + k - 1:] + "\n").encode()
        return (_lines([a], k) + f"{b} F{a[j + k - 1]}\n").encode(), [a]
    out, status, _, text, _ = run(kh, k, 40000, make)
    assert oracle.assemble_text(text, k)[0] == box["want"]
    if knob == "jump":
        assert status == kh.KH_ERR_CONVERGE and out is None
    else:
        assert status == kh.KH_ERR_CONVERGE or out == box["want"]
        if where == "middle":
            assert status == kh.KH_ERR_CONVERGE


# ---- tiny contigs, missing successors ----
def _tiny(k: int, world: int, chunks: int, n1: int, n2: int, seed: int, long_ones: int = 4):
    """n1 one-k-mer contigs (forward 'F'), n2 two-k-mer contigs whose k-mers lie in different chunks, and a few long
    random contigs.  No k-mer repeats."""
    rng = np.random.default_rng(seed)
    seqs, used = [], set()
    def fresh(s):
        km = [s[i:i + k] for i in range(len(s) - k + 1)]
        if len(set(km)) != len(km) or used.intersection(km):
            return False
        used.update(km)
        return True
    while len(seqs) < n1:
        s = E._rand(rng, k)
        if fresh(s):
            seqs.append(s)
    pairs = []
    while len(pairs) < n2:
        cand = [E._rand(rng, k + 1) for _ in range(4 * n2)]
        g = E.global_chunks("".join(cand), k, world, chunks)     # only the windows inside one candidate are used
        for i, s in enumerate(cand):
            at = i * (k + 1)
            if len(pairs) < n2 and g[at] != g[at + 1] and fresh(s):
                pairs.append(s)
    longs = [s for s in (E._rand(rng, 400 + 50 * i) for i in range(long_ones)) if fresh(s)]
    order = rng.permutation(len(seqs) + len(pairs) + len(longs))
    allseqs = seqs + pairs + longs
    return [allseqs[i] for i in order]


@pytest.mark.gpu
@pytest.mark.parametrize("k", [19, 31])
def test_one_and_two_kmer_contigs(kh, k):
    """About 40 000 contigs of one k-mer (zero characters behind the head) and of two k-mers in two chunks, among a
    few long contigs: the reference's output."""
    def make(chunks):
        seqs = _tiny(k, 1, chunks, 20000, 20000, seed=k)
        assert sum(E.count_segments([s], k, 1, chunks) == 2 for s in seqs if len(s) == k + 1) == 20000
        return _lines(seqs, k).encode(), seqs
    assemble(kh, k, 70000, make)


@pytest.mark.gpu
@pytest.mark.parametrize("k", [19, 51])
def test_missing_successor_after_several_segments(kh, k):
    """The last k-mer's successor is in no table, several chunk segments down the contig: the reference's message."""
    rng = np.random.default_rng(k)
    seq = E._rand(rng, 300 + k)

    def make(chunks):
        assert E.count_segments([seq], k, 1, chunks) >= 3
        return "".join(E.lines_of(seq, k, open_end=True)).encode(), [seq]
    out, status, _, text, _ = run(kh, k, 40000, make)
    assert status == kh.KH_ERR_NOT_FOUND and out is None
    with pytest.raises(RuntimeError, match="not found"):
        oracle.assemble_text(text, k)


# ---- one handle, many traverses ----
@pytest.mark.gpu
@pytest.mark.parametrize("k", [19, 51])
def test_one_handle_reused(kh, k):
    """The fallback jumps links in place and claims tails, so the next traverse re-seals: assemble twice, find
    every record, insert more, assemble again, clear, reuse."""
    d1, d2 = kmergen.Dataset(k, 30000, 90, seed=1), kmergen.Dataset(k, 20000, 50, seed=2)
    p1, p2 = d1.pairs(), d2.pairs()
    pl = (k + 3) // 4
    assert not {r.tobytes() for r in p1[:, :pl]} & {r.tobytes() for r in p2[:, :pl]}
    both = oracle.assemble_text(d1.text().tobytes() + d2.text().tobytes(), k)[0]
    with kh.KmerHashTable(k, 50000) as tab:
        tab.insert_pairs(p1)
        for _ in range(2):
            buf, _, nodes = tab.assemble()
            assert buf.tobytes() == d1.expected()[0] and nodes == d1.n
        got, found = tab.find(p1[:, :pl])
        assert found.all() and (got == p1).all()
        got, found = tab.find(p2[:, :pl])
        assert not found.any()
        tab.insert_pairs(p2)
        buf, _, nodes = tab.assemble()
        assert buf.tobytes() == both and nodes == d1.n + d2.n
        got, found = tab.find(np.concatenate([p1, p2])[:, :pl])
        assert found.all()
        tab.clear()
        tab.insert_pairs(p2)
        buf, _, nodes = tab.assemble()
        assert buf.tobytes() == d2.expected()[0] and nodes == d2.n


@pytest.mark.gpu
@pytest.mark.parametrize("k", range(17, 55))
def test_every_k(kh, k):
    """ct_emit_kernel and ct_emit_heads_kernel depend on the slot width and on K."""
    d = kmergen.Dataset(k, 20000, 100, seed=k)
    text = d.text().tobytes()
    out, _ = assemble(kh, k, 20000, lambda chunks: (text, d.expected()[0].decode().split()))
    assert out == d.expected()[0]


@pytest.mark.gpu
def test_load_factor_0_9_with_long_contigs(kh):
    d = kmergen.Dataset(51, 60000, 30, seed=5, long_nodes=20000)
    text = d.text().tobytes()
    out, _ = assemble(kh, 51, 60000, lambda chunks: (text, d.expected()[0].decode().split()), lf=0.9)
    assert out == d.expected()[0]


# ---- sharded ----
def _shard_run(k: int, world: int, n_total: int, make):
    """One sharded step through LocalComm on one GPU.  make(chunks_per_rank) -> (text, base strings to count
    segments of).  Returns (text, per-rank outputs or None, OR of the error bits, rank_rounds of every rank)."""
    import test_gpu_sharded as S
    import cs267_hw3_b200 as kh

    shards = [sh.Shard(k, r, world, n_total, n_total, 0.5, device=0) for r in range(world)]
    comm = sh.LocalComm(shards)
    comm.connect()
    bufs = []
    try:
        chunks = E._chunks_per_rank(shards[0].tab)
        text, paths = make(chunks)
        pairs = oracle.parse_lines(text, k)
        blocks, bufs = S._upload(kh, sh, shards, pairs, pairs.shape[0])
        comm.begin()
        sh.sharded_insert(comm, blocks)
        comm.assemble()
        bits = comm.finish()
        outs = None if bits else [s.result_host()[0].tobytes() for s in shards]
        rounds = [s.tab.stats()["rank_rounds"] for s in shards]
    finally:
        comm.close()
        for p in bufs:
            kh.lib().kh_device_free(p)
        for s in shards:
            s.close()
    if _jumping() and _multi_segment(paths, k, world, chunks):
        assert max(rounds) >= 2, f"stayed on the bounded walk: rank_rounds {rounds}"
    return text, outs, bits, rounds


def _start_ranks(text: bytes, k: int, world: int) -> set:
    pairs = oracle.parse_lines(text, k)
    starts = np.flatnonzero(pairs[:, (k + 3) // 4] == ord("F"))
    return {r for r in range(world) if any(lo <= s < hi for s in starts for lo, hi in [sh.block_of_rank(len(pairs), world, r)])}


def _orphans(k: int, seed: int):
    """Random contigs, orphan chains (no start, missing successor) and headless cycles of several chunks."""
    bg, contigs = _background(k, 20000, 50, seed=seed)
    rng = np.random.default_rng(seed)
    extra = []
    for _ in range(40):
        s = E._rand(rng, k + 12)
        extra += [f"{s[i:i + k]} {s[i - 1] if i else 'A'}{s[i + k]}\n" for i in range(10)]
    cycles = [random_cycle(k, 80 + 13 * i, seed=seed + 50 + i) for i in range(8)]
    extra += [ln for cyc in cycles for ln in cycle_lines(cyc, k, start=False)]
    return bg + "".join(extra), contigs


@pytest.mark.gpu
@pytest.mark.parametrize("world", [2, 3, 8])
@pytest.mark.parametrize("case", ["orphans", "tiny", "pure_cycle", "crowded_cycle", "converge", "missing"])
def test_sharded(world, case):
    """Every rank's output is the reference's <prefix>_<r>.dat, or the exact error bits.  The one-contig inputs
    leave most ranks without a start node."""
    k = 51 if case == "crowded_cycle" else 19
    box = {}

    def make(chunks):
        if case == "orphans":
            text, paths = _orphans(k, seed=world)
        elif case == "tiny":
            paths = _tiny(k, world, chunks, 6000, 6000, seed=world)
            text = _lines(paths, k)
        elif case in ("pure_cycle", "crowded_cycle"):
            cyc = crowded_cycle(k, 1500, 30, seed=1) if case == "crowded_cycle" else random_cycle(k, 400, seed=world)
            assert cycle_segments(cyc, k, world, chunks) >= 2
            text, paths = "".join(cycle_lines(cyc, k, start=True)), [cyc]
        elif case == "converge":
            a = E._rand(np.random.default_rng(world), 300 + k)
            j = 120
            b = ("A" if a[j - 1] != "A" else "C") + a[j:j + k - 1]
            text, paths = _lines([a], k) + f"{b} F{a[j + k - 1]}\n", [a]
        else:
            seq = E._rand(np.random.default_rng(world), 300 + k)
            text, paths = "".join(E.lines_of(seq, k, open_end=True)), [seq]
        box["text"] = text.encode()
        return box["text"], paths

    n_total = 40000
    text, outs, bits, rounds = _shard_run(k, world, n_total, make)
    if case in ("orphans", "tiny"):
        assert bits == 0 and outs == oracle.assemble_text(text, k, world)
        print(f"world {world} {case}: rank_rounds {rounds}")
    else:
        if world == 8:
            assert len(_start_ranks(text, k, world)) < world
        assert bits == {"pure_cycle": ERR_CYCLE, "crowded_cycle": ERR_CYCLE, "converge": ERR_CONVERGE, "missing": ERR_NOT_FOUND}[case], \
            f"error bits {bits}, rank_rounds {rounds}"


@pytest.mark.gpu
@pytest.mark.parametrize("world", [1, 3])
@pytest.mark.parametrize("case", ["orphans", "tiny"])
def test_long_contig_takes_the_fallback_without_the_knob(monkeypatch, world, case):
    """A contig of 514 chunk segments sends the step to pointer jumping on its own: the orphan and tiny-contig
    inputs with it appended give the reference's output there too."""
    monkeypatch.delenv("KH_DEBUG_WALK_STEPS")
    k = 19

    def make(chunks):
        if case == "orphans":
            text, _ = _orphans(k, seed=7)
        else:
            text = _lines(_tiny(k, world, chunks, 6000, 6000, seed=7), k)
        long_one = E._walk_contig(k, world, chunks, 514, seed=world)
        assert E.count_segments([long_one], k, world, chunks) == 514
        full = text + _lines([long_one], k)
        kms = [full[i:i + k] for i in range(0, len(full), k + 4)]
        assert len(set(kms)) == len(kms)
        return full.encode(), []
    text, outs, bits, rounds = _shard_run(k, world, 60000, make)
    assert bits == 0 and outs == oracle.assemble_text(text, k, world)
    assert max(rounds) >= 2, f"rank_rounds {rounds}"
