"""Debug aid: run the sharded path with all ranks on one GPU and, if a step fails, dump the segment lists."""
import ctypes as C
import sys

import numpy as np

sys.path.insert(0, ".")
import cs267_hw3_b200 as kh
from cs267_hw3_b200 import sharded as sh
from tools import kmergen

k, n, c, world = int(sys.argv[1]), int(sys.argv[2]), int(sys.argv[3]), int(sys.argv[4])
reps = int(sys.argv[5]) if len(sys.argv) > 5 else 1
d = kmergen.Dataset(k, n, c, seed=world)
pairs = d.pairs()
L = kh.lib()
L.kh_debug_buffer.argtypes = [C.c_void_p, C.c_char_p, C.POINTER(C.c_void_p), C.POINTER(C.c_uint64)]
shards = [sh.Shard(k, r, world, (n + world - 1) // world, n, 0.5, device=0) for r in range(world)]
comm = sh.LocalComm(shards)
comm.connect()


def buf(s, name, dtype, count=None):
    p, b = C.c_void_p(), C.c_uint64()
    s.tab._check(L.kh_debug_buffer(s.tab._h, name.encode(), C.byref(p), C.byref(b)))
    if name == "caps":
        return np.ctypeslib.as_array(C.cast(p, C.POINTER(C.c_uint64)), shape=(8,)).copy()
    nbytes = b.value if count is None else count * np.dtype(dtype).itemsize
    out = np.empty(nbytes, dtype=np.uint8)
    s.tab._check(L.kh_copy_to_host(s.tab._h, out.ctypes.data, p, nbytes))
    return out.view(dtype)


blocks = []
for r, s in enumerate(shards):
    lo, hi = sh.block_of_rank(n, world, r)
    p = C.c_void_p()
    L.kh_device_alloc(C.byref(p), max(1, (hi - lo) * pairs.shape[1]))
    blk = np.ascontiguousarray(pairs[lo:hi])
    s.tab._check(L.kh_copy_device(s.tab._h, p, blk.ctypes.data, blk.nbytes))
    s.tab.sync()
    blocks.append((p.value, hi - lo))
for rep in range(reps):
    comm.begin()
    sh.sharded_insert(comm, blocks)
    comm.assemble()
    bits = [s.finish() for s in shards]
    print("rep", rep, "error bits per rank:", bits)
    if any(bits):
        links = []
        for r, s in enumerate(shards):
            caps = buf(s, "caps", None)
            ctr = buf(s, "counters", np.uint32)
            hcap, seg_cap = int(caps[0]), int(caps[1])
            next_seg = int(ctr[1])
            lk = buf(s, "link", np.uint64, max(next_seg, hcap))
            links.append(lk)
            print(f"rank {r}: hcap {hcap} next_seg {next_seg} n_starts {s.tab.stats()['n_starts']} inbox_cnt {buf(s, 'inbox_cnt', np.uint32, 8)} "
                  f"out_cursor {buf(s, 'out_cursor', np.uint32, 8)} epoch {caps[6]} flags(moved) {ctr[15:15 + 12]}")
        names = {0xFFFFFFFF: "TAIL", 0xFFFFFFFE: "UNUSED", 0xFFFFFFFD: "CLAIMED", 0xFFFFFFFC: "PENDING", 0xFFFFFFFB: "MISSING", 0xFFFFFFFA: "CONVERGE"}
        shown = 0
        for r, s in enumerate(shards):
            ns = s.tab.stats()["n_starts"]
            hi = (links[r] >> np.uint64(32)).astype(np.uint64)
            lo = (links[r] & np.uint64(0xFFFFFFFF)).astype(np.uint64)
            pend = int(((hi == 0xFFFFFFFC)).sum())
            print(f"rank {r}: pending links left {pend}")
            for cidx in range(ns):
                h, l = int(hi[cidx]), int(lo[cidx])
                if h >= 0xFFFFFFFA or not (l & 0x80000000):
                    chain = [f"stub{cidx}@{r}:{names.get(h, hex(h))}/{hex(l)}"]
                    g = h
                    for _ in range(12):
                        if g >= 0xFFFFFFFA:
                            break
                        rr, li = g >> 28, g & 0x0FFFFFFF
                        if li >= len(links[rr]):
                            chain.append(f"OUT-OF-RANGE {hex(g)}")
                            break
                        v = int(links[rr][li])
                        chain.append(f"{li}@{rr}:{names.get(v >> 32, hex(v >> 32))}/{hex(v & 0xFFFFFFFF)}")
                        g = v >> 32
                    print("  " + " -> ".join(chain))
                    shown += 1
                    if shown > 12:
                        break
            if shown > 12:
                break
        break
    else:
        outs = [s.result_host() for s in shards]
        ok = all(outs[r][0].tobytes() == d.expected(world, r)[0] for r in range(world))
        print("outputs equal reference per-rank files:", ok)
        if not ok:
            for r in range(world):
                want, wnc = d.expected(world, r)
                got, nc, nn = outs[r]
                got = got.tobytes()
                gl, wl = got.split(b"\n"), want.split(b"\n")
                bad = [i for i in range(min(len(gl), len(wl))) if gl[i] != wl[i]]
                print(f"rank {r}: bytes {len(got)} vs {len(want)}, contigs {nc} vs {wnc}, nodes {nn}, differing lines {len(bad)} of {len(wl)}, stats {s.tab.stats()['n_segments']}")
                for i in bad[:3]:
                    g_, w_ = gl[i], wl[i]
                    j = next((x for x in range(min(len(g_), len(w_))) if g_[x] != w_[x]), min(len(g_), len(w_)))
                    print(f"   line {i}: len {len(g_)} vs {len(w_)}, first diff at {j}: got {g_[max(0, j - 5):j + 30]!r} want {w_[max(0, j - 5):j + 30]!r}")
