"""bench.py --dump-outputs: which entries it writes, in which types, within 64 MB.  No GPU (CPU tensors)."""
import os
import sys

import numpy as np
import pytest
import torch

import bench
from kmerml_b200 import engine


def test_selection_is_fixed_and_covers_every_level():
    ks = list(range(1, 13))
    rows, cols = bench.dump_selection(100, ks)
    rows2, cols2 = bench.dump_selection(100, ks)
    assert np.array_equal(rows, rows2) and np.array_equal(cols, cols2)
    assert np.array_equal(rows, np.arange(100))
    lay, row_len = engine.row_layout(ks)
    assert np.all(np.diff(cols) > 0) and cols[-1] < row_len
    for k, (off, n) in lay.items():
        inside = int(((cols >= off) & (cols < off + n)).sum())
        assert inside == min(n, bench.DUMP_BINS_PER_K), k
    assert rows.size * (cols.size * 12 + len(ks) * 8) <= bench.DUMP_BUDGET_BYTES


def test_many_genomes_are_sampled_within_the_budget():
    ks = list(range(1, 13))
    rows, cols = bench.dump_selection(5000, ks)
    assert 1 <= rows.size < 5000 and np.all(np.diff(rows) > 0) and rows[-1] < 5000
    assert np.array_equal(rows, bench.dump_selection(5000, ks)[0])
    assert rows.size * (cols.size * 12 + len(ks) * 8) <= bench.DUMP_BUDGET_BYTES


def test_written_arrays(tmp_path):
    ks = [2, 7, 11]
    _, row_len = engine.row_layout(ks)
    g = torch.Generator().manual_seed(0)
    counts = torch.randint(-2 ** 31, 2 ** 31 - 1, (6, row_len), dtype=torch.int32, generator=g)
    freq = torch.rand((6, row_len), generator=g)
    totals = torch.randint(0, 2 ** 40, (6, len(ks)), dtype=torch.int64, generator=g)
    bench.write_dump(str(tmp_path / "out"), bench.dump_sample(counts, freq, totals, ks, torch))
    files = sorted(os.listdir(tmp_path / "out"))
    assert files == ["counts.npy", "freq.npy", "totals.npy"]
    assert sum(os.path.getsize(tmp_path / "out" / f) for f in files) <= 64 << 20
    rows, cols = bench.dump_selection(6, ks)
    c = np.load(tmp_path / "out" / "counts.npy")
    f = np.load(tmp_path / "out" / "freq.npy")
    t = np.load(tmp_path / "out" / "totals.npy")
    assert c.dtype == np.float64 and f.dtype == np.float32 and t.dtype == np.float64
    assert np.array_equal(c, counts.numpy().view(np.uint32)[np.ix_(rows, cols)].astype(np.float64))
    assert np.array_equal(f, freq.numpy()[np.ix_(rows, cols)])
    assert np.array_equal(t, totals.numpy()[rows].astype(np.float64))


@pytest.mark.parametrize("argv", [["--steps", "0"], ["--warmup", "-1"], ["--impl", "reference", "--dump-outputs", "d"]])
def test_rejected_arguments(argv, monkeypatch):
    monkeypatch.setattr(sys, "argv", ["bench.py"] + argv)
    with pytest.raises(SystemExit):
        bench.parse_args()
