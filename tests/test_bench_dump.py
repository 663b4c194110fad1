"""bench.py --dump-outputs without a GPU: the seeded sample of a returned array and the files written for it."""
import numpy as np

import bench


def test_sample_rows_is_fixed_and_covers_every_stratum():
    assert np.array_equal(bench.sample_rows(1000, 4096), np.arange(1000))
    n, k = 300_000_123, 1 << 16
    rows = bench.sample_rows(n, k)
    assert np.array_equal(rows, bench.sample_rows(n, k))
    assert np.all(np.diff(rows) > 0) and rows[0] == 0 and rows[-1] == n - 1
    assert np.array_equal(rows[:bench.DUMP_EDGE], np.arange(bench.DUMP_EDGE))
    edges = np.arange(k + 1, dtype=np.int64) * n // k
    assert np.unique(np.searchsorted(edges, rows, side="right") - 1).size == k


def test_dump_writes_exact_float_arrays_within_the_limit(tmp_path):
    """Both tables of the archive workload sampled at bench.py's sizes: the largest dump it writes."""
    rng = np.random.default_rng(1)
    stream = rng.integers(0, 256, 30 << 20, dtype=np.uint8)
    crc = rng.integers(0, 1 << 32, 300_000, dtype=np.uint64)
    offset = np.cumsum(rng.integers(30, 70_000, 300_000)).astype(np.uint64)
    out = bench.dump_outputs(str(tmp_path / "d"), {"archive": (4 << 20, {"bytes": stream}),
                                                   "entries": (256 << 10, {"crc32": crc, "header_offset": offset})})
    files = {p.name: np.load(p) for p in (tmp_path / "d").iterdir()}
    assert sorted(files) == sorted(k + ".npy" for k in out)
    assert all(a.dtype in (np.float32, np.float64) for a in files.values())
    assert sum(a.nbytes for a in files.values()) <= 64_000_000
    assert files["archive_length.npy"].tolist() == [stream.size] and files["entries_length.npy"].tolist() == [crc.size]
    pos = files["archive_positions.npy"].astype(np.int64)
    assert np.array_equal(pos, bench.sample_rows(stream.size, 4 << 20))
    assert files["archive_bytes.npy"].dtype == np.float32 and np.array_equal(files["archive_bytes.npy"], stream[pos])
    rows = files["entries_positions.npy"].astype(np.int64)
    assert np.array_equal(files["entries_crc32.npy"].astype(np.uint64), crc[rows])
    assert np.array_equal(files["entries_header_offset.npy"].astype(np.uint64), offset[rows])
