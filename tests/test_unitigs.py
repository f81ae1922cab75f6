"""Unitig extensions (kh_count_link_check*, KmerCounter.link_check*, ShardedCounter.extract_unitigs, kmer_count --unitigs).

S = the k-mers a counter reports at (min_count, min_ext), each with its raw extensions.  A record's forward extension f
is kept iff f != 'F', y = s[1..K-1] f is in S and y's backward extension is s[0]; its backward extension b is kept iff
b != 'F', w = b s[0..K-2] is in S and w's forward extension is s[K-1]; a side not kept becomes 'F'.
The reference is a numpy restatement of that rule over the oracle's records (oracle.analyse_reads): the keys sorted,
neighbours found with searchsorted; it shares nothing with the kernel.
CPU: the restatement's symmetry and that it cuts nothing on the generator's data; the unmodified traversal (the oracle's
restatement of kmer_hash.cpp, and the reference binary where it is built) on checked and on unchecked records of reads
with repeats and errors; tests/native/link_host_check.cu against the restatement; the CLI's usage errors; the kernel's
register budget.  GPU: both entry points, the error paths, sharded partials, the closed loop through kh_assemble, the
pointer-jumping path and the CLI."""
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

import oracle
from tools import kmergen, readgen

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
KS = [3, 19, 31, 32, 51, 61]
_ACGT = np.frombuffer(b"ACGT", dtype=np.uint8)
_F = ord("F")
_CODE = np.full(256, 0, dtype=np.uint8)
_CODE[_ACGT] = [0, 1, 2, 3]


# ------------------------------------------------------------------------------------------- the restatement
def _codes(pairs, k):
    """kmer_pair records -> the bases of their K-mers, codes 0..3, shape (n, K)."""
    pl = (k + 3) // 4
    p = np.ascontiguousarray(pairs, dtype=np.uint8).reshape(-1, pl + 2)[:, :pl]
    c = (p[:, :, None] >> np.array([6, 4, 2, 0], dtype=np.uint8)) & 3
    return c.reshape(p.shape[0], -1)[:, :k]


def _strs(codes):
    k = codes.shape[1]
    return np.ascontiguousarray(_ACGT[codes]).view(f"S{k}").ravel()


def _fmix64(z):
    z = z ^ (z >> np.uint64(33))
    z = z * np.uint64(0xFF51AFD7ED558CCD)
    z = z ^ (z >> np.uint64(33))
    z = z * np.uint64(0xC4CEB9FE1A85EC53)
    return z ^ (z >> np.uint64(33))


def _owner(codes, world):
    """kc_owner of every row's k-mer, vectorised (checked against sharded_count.count_owner below)."""
    k = codes.shape[1]
    n_lo = min(k, 32)
    lo = np.zeros(codes.shape[0], dtype=np.uint64)
    hi = np.zeros(codes.shape[0], dtype=np.uint64)
    with np.errstate(over="ignore"):
        for j in range(k - n_lo):
            hi = (hi << np.uint64(2)) | codes[:, j].astype(np.uint64)
        for j in range(k - n_lo, k):
            lo = (lo << np.uint64(2)) | codes[:, j].astype(np.uint64)
        h = _fmix64(_fmix64(lo ^ (hi * np.uint64(0x9E3779B97F4A7C15))) ^ np.uint64(0xD6E8FEB86659FD93))
        w = np.uint64(world)                                 # mulhi(h, world) for world < 2^32
        return (((h >> np.uint64(32)) * w + (((h & np.uint64(0xFFFFFFFF)) * w) >> np.uint64(32))) >> np.uint64(32)).astype(np.int64)


def _lookup(s_str, keys):
    if s_str.size == 0:
        return np.zeros(keys.size, dtype=np.int64), np.zeros(keys.size, dtype=bool)
    i = np.minimum(np.searchsorted(s_str, keys), s_str.size - 1)
    return i, s_str[i] == keys


def link_ref(pairs, s_pairs, k, world=1, rank=0):
    """The rule, restated: (checked copy of `pairs`, sides cut).  s_pairs = S with its raw extensions."""
    pl = (k + 3) // 4
    s_codes = _codes(s_pairs, k)
    s_str = _strs(s_codes)
    order = np.argsort(s_str, kind="stable")
    s_str, s_back, s_fwd = s_str[order], s_pairs[order, pl], s_pairs[order, pl + 1]
    x = np.array(pairs, dtype=np.uint8).reshape(-1, pl + 2)
    if x.shape[0] == 0:
        return x, 0
    c = _codes(x, k)
    b, f = x[:, pl], x[:, pl + 1]
    y = np.concatenate([c[:, 1:], _CODE[f][:, None]], axis=1)
    w = np.concatenate([_CODE[b][:, None], c[:, :-1]], axis=1)
    iy, fy = _lookup(s_str, _strs(y))
    iw, fw = _lookup(s_str, _strs(w))
    look_f, look_b = np.isin(f, _ACGT), np.isin(b, _ACGT)
    if world > 1:
        look_f &= _owner(y, world) == rank
        look_b &= _owner(w, world) == rank
    cut_f = look_f & ~(fy & (s_back[iy] == _ACGT[c[:, 0]]))
    cut_b = look_b & ~(fw & (s_fwd[iw] == _ACGT[c[:, -1]]))
    x[cut_f, pl + 1] = _F
    x[cut_b, pl] = _F
    return x, int(cut_f.sum() + cut_b.sum())


def lines_of(pairs, k):
    """Records -> the reference's k-mer file text (sorted by line, for comparing as sets)."""
    pl = (k + 3) // 4
    p = np.asarray(pairs, dtype=np.uint8).reshape(-1, pl + 2)
    rows = np.concatenate([_ACGT[_codes(p, k)], np.full((p.shape[0], 1), 32, np.uint8), p[:, pl:pl + 2],
                           np.full((p.shape[0], 1), 10, np.uint8)], axis=1)
    return np.sort(np.ascontiguousarray(rows).view(f"S{k + 4}").ravel())


def paths_of(checked, k):
    """On checked records: which k-mers lie on a path (reachable from a start, a k-mer with backward 'F') -- the others
    are on isolated cycles."""
    pl = (k + 3) // 4
    n = checked.shape[0]
    c = _codes(checked, k)
    s = _strs(c)
    order = np.argsort(s)
    b = checked[:, pl]
    w = np.concatenate([_CODE[b][:, None], c[:, :-1]], axis=1)
    i, found = _lookup(s[order], _strs(w))
    has = (b != _F) & found
    p = np.where(has, order[i], np.arange(n))
    for _ in range(max(1, int(np.ceil(np.log2(max(n, 2))))) + 1):
        p = p[p]
    return b[p] == _F


def contig_kmers(text, k):
    """Every K-window of every contig line (contigs as '\\n'-terminated lines)."""
    out = []
    for ln in bytes(text).split(b"\n"):
        if len(ln) >= k:
            a = np.frombuffer(ln, dtype=np.uint8)
            out.append(np.ascontiguousarray(np.lib.stride_tricks.sliding_window_view(a, k)).view(f"S{k}").ravel())
    return np.concatenate(out) if out else np.zeros(0, dtype=f"S{k}")


# ------------------------------------------------------------------------------------------- inputs
def genome(length, seed, repeat=0, copies=1):
    """A random genome; with repeat > 0, one `repeat`-base segment written to `copies` places."""
    rng = np.random.default_rng(seed)
    g = _ACGT[rng.integers(0, 4, length)]
    if repeat:
        seg = g[1000:1000 + repeat].copy()
        at = np.linspace(5000, length - repeat - 5000, copies - 1).astype(np.int64) if copies > 1 else []
        for a in at:
            g[a:a + repeat] = seg
    return g.tobytes() + b"\n"


def reads_of(g, k, seed, error_rate=0.0, coverage=20, read_len=150):
    return readgen.tile_reads(g, k, read_len=read_len, coverage=coverage, seed=seed, error_rate=error_rate)


# The cases of the defect: (genome length, repeat, copies, error rate, min_count), K = 31, min_ext = 2
CASES = {
    "errors_mc2": (60000, 0, 1, 0.005, 2),
    "errors_mc4": (60000, 0, 1, 0.005, 4),
    "repeat3_clean": (60000, 600, 3, 0.0, 2),
    "repeat20_errors": (60000, 600, 20, 0.005, 6),
}


def _case(name, k=31):
    length, rep, copies, err, mc = CASES[name]
    g = genome(length, 11 + len(name), rep, copies)
    return reads_of(g, k, 12 + len(name), err), mc


def _assemble_oracle(pairs, k):
    """The oracle's restatement of the reference's traversal (kmer_hash.cpp): (contig text, n_contigs, n_nodes)."""
    t = oracle.Table(k, max(1, pairs.shape[0]))
    try:
        t.insert_pairs(pairs)
        return t.assemble(pairs)
    finally:
        t.close()


# ------------------------------------------------------------------------------------------- CPU: the restatement
def test_owner_restatement_is_kc_owner():
    from cs267_hw3_b200.sharded_count import count_owner
    rng = np.random.default_rng(3)
    for k in (19, 32, 51):
        c = rng.integers(0, 4, (200, k)).astype(np.uint8)
        key = [int("".join("0123"[v] for v in row), 4) for row in c]
        for world in (2, 3, 8):
            assert list(_owner(c, world)) == [count_owner(x >> 64, x & ((1 << 64) - 1), world) for x in key]


@pytest.mark.parametrize("name", sorted(CASES))
def test_restatement_is_symmetric(name):
    """x -> y kept iff y <- x kept: every kept side names a record whose opposite side names it back."""
    k = 31
    reads, mc = _case(name)
    s, _, _ = oracle.analyse_reads(reads, k, mc, 2)
    x, n_cut = link_ref(s, s, k)
    assert n_cut > 0
    pl = (k + 3) // 4
    c = _codes(x, k)
    st = _strs(c)
    order = np.argsort(st)
    for side, other, mk, first in ((pl + 1, pl, lambda e: np.concatenate([c[:, 1:], _CODE[e][:, None]], 1), 0),
                                   (pl, pl + 1, lambda e: np.concatenate([_CODE[e][:, None], c[:, :-1]], 1), -1)):
        keep = x[:, side] != _F
        i, found = _lookup(st[order], _strs(mk(x[:, side])))
        assert found[keep].all()
        assert (x[order[i], other][keep] == _ACGT[c[:, first]][keep]).all()


def test_restatement_cuts_nothing_on_the_generators_data():
    """At the closed-loop parameters of test_count.py and test_count_histogram.py (the latter at its valley) the rule
    keeps every extension: the generator's contigs are linear chains of reported k-mers."""
    import cs267_hw3_b200 as kh
    for k, n, c, seed, cov, err, mc, me in ((19, 400000, 800, 319, 8, 0.0005, 3, 3), (51, 300000, 600, 351, 8, 0.0005, 3, 3),
                                            (19, 30000, 60, 7000, 20, 0.01, None, 5)):
        d = kmergen.Dataset(k, n, c, seed=seed)
        reads = readgen.tile_reads(d.solution(), k, read_len=k + 40, coverage=cov, seed=seed + (100 if mc is None else 1),
                                   error_rate=err)
        if mc is None:
            _, counts, _ = oracle.analyse_reads(reads, k, 1, 1)
            mc = kh.auto_min_count(np.bincount(counts[:, 0], minlength=256)[:256].astype(np.uint64))
        s, _, _ = oracle.analyse_reads(reads, k, mc, me)
        assert s.shape[0] == n
        x, n_cut = link_ref(s, s, k)
        assert n_cut == 0 and (x == s).all()


@pytest.mark.parametrize("name", sorted(CASES))
def test_traversal_on_checked_records_places_every_kmer_once(name, tmp_path):
    """The unmodified traversal on the checked k-mer file: no error, no k-mer twice, every record on a contig except
    those on isolated cycles.  Without the rule the same run loses or duplicates k-mers (or fails)."""
    k = 31
    reads, mc = _case(name)
    s, _, _ = oracle.analyse_reads(reads, k, mc, 2)
    x, _ = link_ref(s, s, k)
    on_path = paths_of(x, k)
    text, nc, nodes = _assemble_oracle(x, k)
    got = contig_kmers(text, k)
    assert nodes == got.size == int(on_path.sum()) and np.unique(got).size == got.size
    assert (np.sort(got) == np.sort(_strs(_codes(x, k))[on_path])).all()
    if oracle.ref_binary(k):
        (tmp_path / "unitigs.txt").write_bytes(b"".join(lines_of(x, k)))
        ref = oracle.run_reference(k, str(tmp_path / "unitigs.txt"), str(tmp_path))
        assert sorted(ref.splitlines()) == sorted(text.splitlines())
    try:
        text0, _, nodes0 = _assemble_oracle(s, k)
    except RuntimeError:
        return                                                 # k-mer not found: the defect as a failure
    got0 = contig_kmers(text0, k)
    assert nodes0 != s.shape[0] or np.unique(got0).size != got0.size


# ------------------------------------------------------------------------------- CPU: the kernel's logic, serially
@pytest.fixture(scope="module")
def host_check(tmp_path_factory):
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        pytest.skip("nvcc not available")
    exe = str(tmp_path_factory.mktemp("link") / "link_host_check")
    subprocess.run([nvcc, "-std=c++17", "-O1", "-Wno-deprecated-gpu-targets", "-o", exe,
                    os.path.join(ROOT, "tests", "native", "link_host_check.cu")], check=True, capture_output=True)
    return exe


def mixed_reads(k, seed):
    """Reads with substitution errors, N and lower-case bytes, repeats longer than K, and two reads of 300 A's (A^K
    follows itself: a self-loop whose counters saturate)."""
    rng = np.random.default_rng(seed)
    if k < 8:
        reads = _ACGT[rng.integers(0, 4, 20000)].copy()
        reads[rng.choice(reads.size, 300, replace=False)] = 10
        return np.concatenate([reads, np.frombuffer(b"\n" + b"A" * 300 + b"\n", dtype=np.uint8)])
    reads = reads_of(genome(6000 + 40 * k, seed, repeat=2 * k + 17, copies=4), k, seed + 1, error_rate=0.004, coverage=8, read_len=k + 40)
    pos = rng.choice(reads.size, size=reads.size // 700, replace=False)
    reads[pos] = np.where(rng.random(pos.size) < 0.5, ord("N"), ord("a")).astype(np.uint8)
    return np.concatenate([reads, np.frombuffer((b"A" * 300 + b"\n") * 2, dtype=np.uint8)])


@pytest.mark.parametrize("k", KS)
def test_kernel_logic_matches_the_restatement(host_check, tmp_path, k):
    """kc_link_plan / kc_find_pair / kc_link_apply over the table's records equal the restatement, records and n_cut;
    the owners' partials for world 2, 3 and 8, in forward and reverse owner order, give the world-1 records."""
    reads = mixed_reads(k, 40 + k)
    reads.tofile(tmp_path / "reads.bin")
    mc, me = 2, 2
    s, counts, _ = oracle.analyse_reads(reads, k, mc, me)
    want, want_cut = link_ref(s, s, k)
    assert want_cut > 0 or k < 8                               # all 64 3-mers fork both ways: nothing is left to cut
    for world in (1, 2, 3, 8):
        r = subprocess.run([host_check, str(k), str(max(1024, 2 * reads.size)), str(mc), str(me), str(world), str(tmp_path / "reads.bin")],
                           capture_output=True, check=True)
        body, tail = r.stdout.rsplit(b"\n", 2)[0] + b"\n", r.stdout.rsplit(b"\n", 2)[1]
        got = np.sort(np.frombuffer(body, dtype=f"S{k + 4}"))
        assert (got == lines_of(want, k)).all()
        assert [int(v) for v in tail.split()] == [want_cut, want_cut, want_cut, 1, 1]
    if k >= 8:                                                 # the homopolymer's self-loop survives the check
        pl = (k + 3) // 4
        a = np.flatnonzero(_strs(_codes(want, k)) == b"A" * k)
        assert a.size == 1 and bytes(want[a[0], pl:pl + 2]) == b"AA" and counts[np.flatnonzero(_strs(_codes(s, k)) == b"A" * k)[0], 0] == 255


# ------------------------------------------------------------------------------------------- CPU: CLI and kernel build
def test_kmer_count_cli_unitigs_usage(tmp_path):
    from cs267_hw3_b200 import build
    exe = build.build_count_cli()
    (tmp_path / "reads.txt").write_bytes(b"ACGTACGTAC\n")
    for args in (["19", "reads.txt", "--unitigs"], ["19", "reads.txt", "--histo", "h.txt", "--unitigs"],
                 ["19", "reads.txt", "--unitigs", "--depth", "k.txt"],
                 ["19", "reads.txt", "--unitigs", "--contigs"]):
        r = subprocess.run([exe, *args], cwd=tmp_path, capture_output=True, text=True)
        assert r.returncode == 1 and r.stderr.startswith("Usage: kmer_count K reads_file"), (args, r.stderr)
        assert "[--unitigs]" in r.stderr
    assert sorted(os.listdir(tmp_path)) == ["reads.txt"]


def test_link_kernel_has_no_spills(tmp_path):
    """kc_link_kernel for sm_100a: ptxas reports no stack frame and no spills (both slot widths)."""
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        pytest.skip("nvcc not available")
    from cs267_hw3_b200 import build
    r = subprocess.run([nvcc, *build.NVCC_FLAGS, "-Xptxas", "-v", "-c", os.path.join(build.CSRC, "count.cu"),
                        "-o", str(tmp_path / "count.o")], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    blocks = re.findall(r"Function properties for (\S*kc_link_kernel\S*)\n\s*(.*)", r.stderr)
    assert len(blocks) == 2, r.stderr[-2000:]
    for name, props in blocks:
        assert "0 bytes stack frame, 0 bytes spill stores, 0 bytes spill loads" in props, (name, props)


# --------------------------------------------------------------------------------------------------- GPU
def _dev(a, pad=0):
    import torch
    t = torch.zeros(np.asarray(a).nbytes + pad + 64, dtype=torch.uint8, device="cuda:0")
    t[pad:pad + np.asarray(a).nbytes] = torch.from_numpy(np.ascontiguousarray(a).view(np.uint8).ravel().copy()).to("cuda:0")
    torch.cuda.synchronize()
    return t


@pytest.mark.gpu
@pytest.mark.parametrize("k", KS)
def test_gpu_link_check_matches_the_restatement(k):
    """Host and device entry points against the restatement, records and n_cut: in place and out of place at odd
    offsets, with extract_device's buffer as input, after the table grew, and the world-3 partials; one launch per call."""
    import torch

    import cs267_hw3_b200 as kh
    reads = mixed_reads(k, 60 + k)
    mc, me = 2, 2
    s, _, _ = oracle.analyse_reads(reads, k, mc, me)
    want, want_cut = link_ref(s, s, k)
    pb = kh.pair_bytes(k)
    with kh.KmerCounter(k, 64, 0.5, 0) as kc:
        kc.count_reads(reads)
        assert kc.stats()["n_grows"] > 0
        recs = kc.extract(mc, me)
        n = recs.shape[0]
        assert (np.sort(recs.view(f"S{pb}").ravel()) == np.sort(s.view(f"S{pb}").ravel())).all()
        n0 = kc.stats()["n_launches"]
        got, cut = kc.link_check(recs, mc, me)
        assert kc.stats()["n_launches"] == n0 + 1 and cut == want_cut and (lines_of(got, k) == lines_of(want, k)).all()
        for pad_in, pad_out in ((0, 0), (3, 3), (1, 6)):
            src = _dev(recs, pad_in)
            if pad_in == pad_out:
                dst, off = src, pad_in
            else:
                dst, off = _dev(np.zeros_like(recs), pad_out), pad_out
            cut = kc.link_check_device(src.data_ptr() + pad_in, dst.data_ptr() + off, n, mc, me)
            out = dst.cpu().numpy()
            assert cut == want_cut and (lines_of(out[off:off + n * pb], k) == lines_of(want, k)).all()
            assert not out[:off].any() and not out[off + n * pb:].any()
        ptr, n2 = kc.extract_device(mc, me)
        dst = torch.zeros(n * pb, dtype=torch.uint8, device="cuda:0")
        torch.cuda.synchronize()
        assert kc.link_check_device(ptr, dst.data_ptr(), n2, mc, me) == want_cut
        assert (lines_of(dst.cpu().numpy(), k) == lines_of(want, k)).all()
        assert kc.link_check_device(ptr, ptr, n2, mc, me) == want_cut                 # the extract buffer itself
        part, total = recs, 0
        for o in (2, 0, 1):
            part, c = kc.link_check(part, mc, me, 3, o)
            total += c
        assert total == want_cut and (lines_of(part, k) == lines_of(want, k)).all()


@pytest.mark.gpu
def test_gpu_link_check_errors():
    """KH_ERR_ARG for null pointers, thresholds and world / rank; KH_ERR_BAD_INPUT for an extension byte outside ACGTF;
    KH_ERR_TABLE_FULL after an overflowed count; n = 0 launches nothing."""
    import ctypes as C

    import cs267_hw3_b200 as kh
    k = 31
    reads = mixed_reads(k, 90)
    with kh.KmerCounter(k, reads.size, 0.5, 0) as kc:
        kc.count_reads(reads)
        recs = kc.extract(2, 2)
        n = recs.shape[0]
        L, h = kh.lib(), kc._h
        cut = C.c_uint64(7)
        n0 = kc.stats()["n_launches"]
        assert L.kh_count_link_check(h, None, 0, 2, 2, 1, 0, C.byref(cut)) == kh.KH_OK and cut.value == 0
        assert L.kh_count_link_check_device(h, None, None, 0, 2, 2, 1, 0, C.byref(cut)) == kh.KH_OK
        assert kc.stats()["n_launches"] == n0
        d = _dev(recs)
        p = d.data_ptr()
        rp = recs.ctypes.data
        for args in ((rp, n, 0, 2, 1, 0), (rp, n, 256, 2, 1, 0), (rp, n, 2, 0, 1, 0), (rp, n, 2, 128, 1, 0),
                     (rp, n, 2, 2, 0, 0), (rp, n, 2, 2, 65, 0), (rp, n, 2, 2, 3, 3), (None, n, 2, 2, 1, 0)):
            assert L.kh_count_link_check(h, *args, C.byref(cut)) == kh.KH_ERR_ARG, args
        for a in ((p, p, n, 0, 2, 1, 0), (p, p, n, 2, 2, 2, 5), (None, p, n, 2, 2, 1, 0), (p, None, n, 2, 2, 1, 0),
                  (rp, p, n, 2, 2, 1, 0)):
            assert L.kh_count_link_check_device(h, *a, C.byref(cut)) == kh.KH_ERR_ARG, a
        assert L.kh_count_link_check(h, rp, n, 2, 2, 1, 0, None) == kh.KH_ERR_ARG
        assert L.kh_count_link_check(None, rp, n, 2, 2, 1, 0, C.byref(cut)) == kh.KH_ERR_ARG
        assert kc.stats()["n_launches"] == n0
        bad = recs.copy()
        bad[n // 2, (k + 3) // 4 + 1] = ord("N")
        with pytest.raises(kh.KhError) as e:
            kc.link_check(bad, 2, 2)
        assert e.value.status == kh.KH_ERR_BAD_INPUT
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
            c.link_check(recs, 2, 2)
        assert e.value.status == kh.KH_ERR_TABLE_FULL
        L.kh_device_free(p)


@pytest.mark.gpu
@pytest.mark.parametrize("world", [2, 3, 8])
def test_gpu_sharded_unitigs_equal_one_counter(world):
    """ShardedCounter.extract_unitigs: the union over ranks (a multiset) is the single counter's checked records, and the
    cuts add up; ranks share GPU 0 when there are fewer GPUs."""
    import cs267_hw3_b200 as kh
    from cs267_hw3_b200.sharded_count import ShardedCounter, split_reads
    k = 31
    reads, mc = _case("repeat20_errors")
    with kh.KmerCounter(k, reads.size, 0.5, 0) as one:
        one.count_reads(reads)
        want, want_cut = one.link_check(one.extract(mc, 2), mc, 2)
    s, _, _ = oracle.analyse_reads(reads, k, mc, 2)
    assert (lines_of(want, k) == lines_of(link_ref(s, s, k)[0], k)).all()
    cuts = split_reads(reads, world)
    with ShardedCounter(k, world, reads.size) as sc:
        for r in range(world):
            sc.count(r, reads[cuts[r]:cuts[r + 1]])
        sc.reduce()
        parts = [sc.extract_unitigs(r, mc, 2) for r in range(world)]
    got = np.concatenate([p for p, _ in parts])
    assert sum(c for _, c in parts) == want_cut
    assert (lines_of(got, k) == lines_of(want, k)).all()


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(CASES))
def test_gpu_closed_loop_through_kh_assemble(name):
    """reads -> count -> extract_device -> link_check_device in place -> kh_insert_pairs_device -> kh_assemble: the call
    succeeds, n_nodes = the records minus the k-mers on cycles, and the contigs are the traversal's on the checked file."""
    import cs267_hw3_b200 as kh
    k = 31
    reads, mc = _case(name)
    with kh.KmerCounter(k, reads.size, 0.5, 0) as kc:
        kc.count_reads(reads)
        ptr, n = kc.extract_device(mc, 2)
        kc.link_check_device(ptr, ptr, n, mc, 2)
        recs = kc.extract(mc, 2)
        checked, _ = kc.link_check(recs, mc, 2)
        with kh.KmerHashTable(k, n, 0.5, 0) as tab:
            ptr, n = kc.extract_device(mc, 2)
            kc.link_check_device(ptr, ptr, n, mc, 2)
            tab.insert_pairs_device(ptr, n)
            text, offs, nodes = tab.assemble()
    on_path = paths_of(checked, k)
    assert nodes == int(on_path.sum())
    ref, _, ref_nodes = _assemble_oracle(checked, k)
    assert ref_nodes == nodes and sorted(bytes(text).splitlines()) == sorted(ref.splitlines())


@pytest.mark.gpu
def test_gpu_long_unitigs_take_the_pointer_jumping_path():
    """K = 51, a 1.2 Mb genome with a repeat: unitigs of hundreds of thousands of k-mers (far more than 512 segments)
    assemble without KH_ERR_CONVERGE, every record on a contig, as the traversal on the checked file does."""
    import cs267_hw3_b200 as kh
    k = 51
    reads = reads_of(genome(1_200_000, 5, repeat=700, copies=3), k, 6, coverage=3, read_len=120)
    with kh.KmerCounter(k, reads.size, 0.5, 0) as kc:
        kc.count_reads(reads)
        recs = kc.extract(2, 2)
        checked, cut = kc.link_check(recs, 2, 2)
        assert cut > 0
        with kh.KmerHashTable(k, recs.shape[0], 0.5, 0) as tab:
            tab.insert_pairs(checked)
            text, offs, nodes = tab.assemble()
    assert nodes == checked.shape[0] and paths_of(checked, k).all()
    assert int(np.diff(offs).max()) > 200_000
    ref, _, ref_nodes = _assemble_oracle(checked, k)
    assert ref_nodes == nodes and sorted(bytes(text).splitlines()) == sorted(ref.splitlines())


def _run_cli(tmp_path, args, env=None, timeout=300):
    from cs267_hw3_b200 import build
    exe = build.build_count_cli()
    base = {x: v for x, v in os.environ.items() if x not in ("KH_RANKS", "KH_COUNT_BATCH_BYTES")}
    r = subprocess.run([exe, *args], cwd=tmp_path, capture_output=True, text=True, timeout=timeout, env=dict(base, **(env or {})))
    assert r.returncode == 0, r.stdout + r.stderr
    return r.stdout


@pytest.mark.gpu
@pytest.mark.parametrize("ranks", [1, 2])
def test_gpu_kmer_count_unitigs(tmp_path, ranks):
    """kmer_count --unitigs: the k-mer file is the restatement's checked records; --contigs (with --depth) writes the
    traversal's contigs of that file, every k-mer once; the stdout line reports the cuts.  Without --unitigs the k-mer
    file is the plain extract and stdout has no such line."""
    k, mc = 31, 2
    reads, _ = _case("repeat3_clean")
    (tmp_path / "reads.txt").write_bytes(bytes(reads))
    env = {"KH_RANKS": str(ranks)}
    s, _, _ = oracle.analyse_reads(reads, k, mc, 2)
    want, want_cut = link_ref(s, s, k)
    plain = _run_cli(tmp_path, [str(k), "reads.txt", "plain.txt", str(mc)], env=env)
    assert "Unitig" not in plain
    assert (np.sort(np.frombuffer((tmp_path / "plain.txt").read_bytes(), dtype=f"S{k + 4}")) == lines_of(s, k)).all()
    out = _run_cli(tmp_path, [str(k), "reads.txt", "--unitigs", "uni.txt", str(mc)], env=env)
    assert (np.sort(np.frombuffer((tmp_path / "uni.txt").read_bytes(), dtype=f"S{k + 4}")) == lines_of(want, k)).all()
    line = "Unitig extensions: %d of %d k-mers' extensions set to F" % (want_cut, s.shape[0])
    assert line in out
    strip = lambda x: [re.sub(r"[0-9.]+ s\b", "T s", v).replace("uni.txt", "plain.txt") for v in x.splitlines() if "Unitig" not in v]  # noqa: E731
    assert strip(out) == strip(plain)
    out = _run_cli(tmp_path, [str(k), "reads.txt", "--depth", "--unitigs", "--contigs", "c", str(mc)], env=env)
    assert line in out
    dat = b"".join((tmp_path / f"c_{r}.dat").read_bytes() for r in range(ranks))
    ref, _, ref_nodes = _assemble_oracle(want, k)
    assert sorted(dat.splitlines()) == sorted(ref.splitlines())
    got = contig_kmers(dat, k)
    assert got.size == ref_nodes == int(paths_of(want, k).sum()) and np.unique(got).size == got.size
    depth = sum(len((tmp_path / f"c_{r}.depth").read_text().splitlines()) for r in range(ranks))
    assert depth == dat.count(b"\n")
