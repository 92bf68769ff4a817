"""``bench.py --dump-outputs``: the last timed membership step's bitset and count, written as float arrays that two builds
can be compared by (the bitset -> flag conversion runs in torch on whatever device holds the bitset, here the host)."""
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT


@pytest.mark.parametrize("n", [5000, 1_000_003])
def test_dump_outputs_unpacks_the_bitset(n, tmp_path):
    import torch
    import bench
    words = np.random.default_rng(n).integers(-2**31, 2**31, size=(n + 31) // 32, dtype=np.int64).astype(np.int32)
    flags = np.unpackbits(words.view(np.uint8), bitorder="little")[:n]          # bit i & 31 of word i >> 5
    bench.dump_outputs(str(tmp_path), torch.from_numpy(words), int(flags.sum()), n)
    got = {f[:-4]: np.load(os.path.join(str(tmp_path), f)) for f in os.listdir(str(tmp_path))}
    assert sorted(got) == ["flags_sample", "group_members", "members"]
    assert got["members"].dtype == np.float64 and got["members"].tolist() == [flags.sum()]
    groups = np.concatenate([flags, np.zeros(-n % 1024, dtype=np.uint8)]).reshape(-1, 1024).sum(1)
    assert got["group_members"].dtype == np.float64 and np.array_equal(got["group_members"], groups)
    idx = np.unique(np.random.default_rng(0).integers(0, n, bench.DUMP_SAMPLES))
    assert got["flags_sample"].dtype == np.float32 and np.array_equal(got["flags_sample"], flags[idx])
    # the benchmark's 10^8-point grid stays within 64 MB of dumped arrays
    assert 4 * bench.DUMP_SAMPLES + 8 * (10**8 // 1024 + 1) + 8 <= 64 << 20


@pytest.mark.parametrize("argv", [["--steps", "0"], ["--impl", "reference", "--dump-outputs", "out"]])
def test_bench_rejects_arguments_it_cannot_honour(argv, tmp_path):
    proc = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + argv, cwd=str(tmp_path),
                          capture_output=True, text=True)
    assert proc.returncode == 2 and "error:" in proc.stderr
    assert not os.listdir(str(tmp_path))
