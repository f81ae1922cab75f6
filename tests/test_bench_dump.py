"""bench.py --dump-outputs: what the last timed step computed, written as .npy so that two builds can be compared."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import bench
from conftest import ROOT
from tools import kmergen


def _load(d, name):
    return np.load(os.path.join(d, name + ".npy"))


def test_dump_keeps_short_arrays_whole(tmp_path):
    contigs = np.frombuffer(b"ACGTA\nCCGTT\nGG\n", dtype=np.uint8)
    offsets = np.array([0, 6, 12, 15], dtype=np.uint64)
    files = bench.dump_outputs(str(tmp_path), contigs, offsets, 7)
    assert sorted(files) == ["contigs.npy", "counts.npy", "offsets.npy"]
    c, o, n = _load(tmp_path, "contigs"), _load(tmp_path, "offsets"), _load(tmp_path, "counts")
    assert c.dtype == np.float32 and np.array_equal(c, contigs)
    assert o.dtype == np.float64 and np.array_equal(o, offsets)
    assert n.tolist() == [3, 15, 7]


def test_dump_samples_long_arrays_the_same_way_every_time(tmp_path, monkeypatch):
    blk = bench.DUMP_BLOCK
    monkeypatch.setitem(bench.DUMP_CAP, "contigs", 3 * blk)
    contigs = np.random.default_rng(5).integers(0, 256, 10 * blk + 17, dtype=np.uint8)
    offsets = np.arange(0, contigs.size + 1, 100, dtype=np.uint64)
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), contigs, offsets, 1)
    blocks = _load(tmp_path / "a", "contigs_blocks")
    assert blocks.size == 3 and np.all(np.diff(blocks) > 0) and blocks.max() <= 10
    idx = (blocks.astype(np.int64)[:, None] * blk + np.arange(blk)).ravel()
    want = contigs[idx[idx < contigs.size]]
    for run in ("a", "b"):
        assert np.array_equal(_load(tmp_path / run, "contigs"), want)
        assert np.array_equal(_load(tmp_path / run, "contigs_blocks"), blocks)
        assert np.array_equal(_load(tmp_path / run, "offsets"), offsets)       # under its cap: whole
    assert not os.path.exists(tmp_path / "a" / "offsets_blocks.npy")


def test_dump_caps_fit_the_size_limit():
    blocks = sum(cap // bench.DUMP_BLOCK for cap in bench.DUMP_CAP.values())
    worst = 4 * bench.DUMP_CAP["contigs"] + 8 * bench.DUMP_CAP["offsets"] + 8 * blocks + 3 * 8
    assert worst <= bench.DUMP_MAX_BYTES == 64 << 20


@pytest.mark.gpu
def test_bench_dumps_the_last_timed_step(tmp_path):
    """A chunk-table-sized run (>= 2^20 k-mers, the table the default workload uses): the dumped contigs and offsets
    are the generator's expected output, byte for byte in start order, and --steps sets the number of timed steps."""
    n, steps = 1_200_000, 2
    out = tmp_path / "dump"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(steps), "--warmup", "1",
                        "--workload", "chr14_k51", "--kmers", str(n), "--no-cpu-baseline", "--no-e2e",
                        "--dump-outputs", str(out)], cwd=tmp_path, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-4000:] + r.stderr[-4000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["steps"] == steps and line["verified"]
    assert sorted(line["dumped"]["files"]) == ["contigs.npy", "counts.npy", "offsets.npy"]
    k, _, c_full, _ = bench.WORKLOADS["chr14_k51"]
    c = max(1, int(round(n * c_full / bench.WORKLOADS["chr14_k51"][1])))
    want, nc = kmergen.Dataset(k, n, c, seed=bench.SEED).expected_array()
    offs = np.concatenate(([0], np.flatnonzero(want == ord("\n")) + 1))
    assert np.array_equal(_load(out, "contigs"), want)
    assert np.array_equal(_load(out, "offsets"), offs)
    assert _load(out, "counts").tolist() == [nc, want.size, n]
