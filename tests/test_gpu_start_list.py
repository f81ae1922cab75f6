"""The start list, shared by both tables: every insert call scans its start bitmask, appends its start nodes (backward
extension 'F') to the list in input order, and grows the list to the start count, not to the number of records."""
import ctypes as C

import numpy as np
import pytest

import oracle
import test_gpu_parity as P
from tools import kmergen

pytestmark = pytest.mark.gpu

kh = P.kh


def _start_list_bytes(kh, tab):
    p, b = C.c_void_p(), C.c_uint64()
    tab._check(kh.lib().kh_debug_buffer(tab._h, b"starts", C.byref(p), C.byref(b)))
    return b.value


@pytest.mark.parametrize("ct,k", [("2", 51), ("0", 51), ("0", 19)])
def test_start_list_follows_the_start_count(kh, monkeypatch, ct, k):
    """12 start nodes among 120 000 records in 6 calls: half of them in the first call, the rest in the last, none in
    the calls between.  After every call n_starts is exact and the start list holds about that many slots; the contigs
    match the oracle's.  KH_CT=2 is the single-GPU chunk table, KH_CT=0 the plain table."""
    monkeypatch.setenv("KH_CT", ct)
    n, c, calls = 120_000, 12, 6
    d = kmergen.Dataset(k, n, c, seed=5 + k)
    lines = d.text().reshape(n, k + 4)
    d.close()
    is_start = lines[:, k + 1] == ord("F")
    assert is_start.sum() == c
    starts, others = np.flatnonzero(is_start), np.flatnonzero(~is_start)
    text = lines[np.concatenate([starts[:c // 2], others, starts[c // 2:]])].reshape(-1)
    want = oracle.assemble_text(text, k)[0]
    pairs = oracle.parse_lines(text, k)
    pl, step = kh.packed_bytes(k), -(-n // calls)
    with kh.KmerHashTable(k, n) as tab:
        slot_bytes = tab.stats()["slot_bits"] // 8
        seen = 0
        for lo in range(0, n, step):
            part = pairs[lo:lo + step]
            tab.insert_pairs(part)
            seen += int((part[:, pl] == ord("F")).sum())
            assert tab.stats()["n_starts"] == seen
            assert seen * slot_bytes <= _start_list_bytes(kh, tab) <= max(256, 2 * seen * slot_bytes)
        assert seen == c
        buf, offs, nodes = tab.assemble()
    assert buf.tobytes() == want and nodes == n and len(offs) - 1 == c
