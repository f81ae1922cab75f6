"""Compile the CUDA library (libkh_b200.so) and the kmer_hash_<K> CLIs for sm_100a, in-tree."""
from __future__ import annotations

import os
import shutil
import subprocess

PKG = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(PKG)
CSRC = os.path.join(PKG, "csrc")
LIB = os.path.join(PKG, "libkh_b200.so")
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17"]


def _nvcc() -> str:
    exe = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(exe):
        raise RuntimeError("nvcc not found: libkh_b200.so cannot be built (there is no CPU fallback)")
    return exe


def _run(cmd: list[str]) -> None:
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("build failed: " + " ".join(cmd) + "\n" + r.stdout + r.stderr)


def _stale(target: str, sources: list[str]) -> bool:
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(s) > t for s in sources)


def lib_sources() -> list[str]:
    return [os.path.join(CSRC, f) for f in sorted(os.listdir(CSRC))] + [os.path.join(ROOT, "include", "kh_capi.h")]


def build_lib(force: bool = False) -> str:
    if force or _stale(LIB, lib_sources()):
        # two translation units: capi.cu (tables, traversal, multi-GPU) and count.cu (k-mer analysis)
        _run([_nvcc(), *NVCC_FLAGS, "-Xcompiler", "-fPIC", "-shared", os.path.join(CSRC, "capi.cu"),
              os.path.join(CSRC, "count.cu"), "-o", LIB])
    return LIB


def build_cli(ks=(19, 31, 51), force: bool = False) -> list[str]:
    """kmer_hash_<K>: the reference's CLI (kmer_hash.cpp:84-152) over the C ABI, one binary per K."""
    build_lib()                      # only if stale: `force` is about the binaries
    src = os.path.join(ROOT, "src", "kmer_hash.cpp")
    hdrs = [os.path.join(ROOT, "include", f) for f in os.listdir(os.path.join(ROOT, "include"))]
    outs = []
    for k in ks:
        out = os.path.join(ROOT, f"kmer_hash_{k}")
        if force or _stale(out, [src, LIB, *hdrs]):
            _run(["g++", "-O2", "-std=c++17", "-pthread", f"-DKMER_LEN={k}", "-I" + os.path.join(ROOT, "include"), src,
                  "-L" + PKG, "-lkh_b200", "-Wl,-rpath," + PKG, "-o", out])
        outs.append(out)
    return outs


def build_count_cli(force: bool = False) -> str:
    """kmer_count: reads -> the reference's k-mer file (or straight to contigs); K is a run-time argument."""
    build_lib()
    src = os.path.join(ROOT, "src", "kmer_count.cpp")
    hdrs = [os.path.join(ROOT, "include", "kh_capi.h")] + [os.path.join(ROOT, "include", "kh", f) for f in
                                                            ("kmer_counter.hpp", "sharded_counter.hpp", "sharded_host.hpp")]
    out = os.path.join(ROOT, "kmer_count")
    if force or _stale(out, [src, LIB, *hdrs]):
        _run(["g++", "-O2", "-std=c++17", "-pthread", "-I" + os.path.join(ROOT, "include"), src,
              "-L" + PKG, "-lkh_b200", "-Wl,-rpath," + PKG, "-o", out])
    return out


if __name__ == "__main__":
    print(build_lib(force=True))
    if os.path.exists(os.path.join(ROOT, "src", "kmer_hash.cpp")):
        print("\n".join(build_cli(force=True)))
        print(build_count_cli(force=True))
