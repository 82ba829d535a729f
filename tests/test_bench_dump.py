"""bench.py --dump-outputs on the CPU: the seeded sample of an output file (window bounds, the footer window,
determinism) and the 64 MB cap on what is written."""
import numpy as np
import pytest

import bench


def _file(n, seed=3):
    return np.random.default_rng(seed).integers(0, 256, n, dtype=np.uint8)


@pytest.mark.parametrize("n", [0, 100, bench.DUMP_FILE_BYTES])
def test_small_file_is_dumped_whole(n):
    f = _file(n)
    d = {}
    bench.dump_file_sample(d, "x_data", f)
    assert list(d) == ["x_data"] and d["x_data"].dtype == np.float32
    assert np.array_equal(d["x_data"], f.astype(np.float32))


@pytest.mark.parametrize("n", [bench.DUMP_FILE_BYTES + 1, 50_000_000 + 123])
def test_large_file_is_sampled_in_windows(n):
    f = _file(n)
    d = {}
    bench.dump_file_sample(d, "x_data", f)
    off = d["x_data_offsets"].astype(np.int64)
    w = d["x_data"]
    assert w.dtype == np.float32 and w.shape == (len(off), bench.DUMP_WINDOW)
    assert w.nbytes <= 4 * bench.DUMP_FILE_BYTES
    assert np.all(np.diff(off) > 0) and off[0] >= 0 and off[-1] == n - bench.DUMP_WINDOW      # sorted, in bounds, footer last
    for i in (0, len(off) // 2, len(off) - 1):
        assert np.array_equal(w[i], f[off[i]:off[i] + bench.DUMP_WINDOW].astype(np.float32))
    again = {}
    bench.dump_file_sample(again, "x_data", f.copy())
    assert all(np.array_equal(d[k], again[k]) for k in d)                                     # same size, same windows


def test_dump_of_four_large_files_fits_64_mb(tmp_path):
    d = {}
    bench.dump_counters(d, "value", {k: i for i, k in enumerate(bench.DUMP_COUNTERS)})
    for name in ("value_data", "value_meta", "e2e_data", "e2e_meta"):
        bench.dump_file_sample(d, name, _file(40_000_000))
    bench.write_dumps(str(tmp_path / "out"), d)
    files = sorted(p.name for p in (tmp_path / "out").iterdir())
    assert files == sorted(k + ".npy" for k in d)
    assert sum((tmp_path / "out" / f).stat().st_size for f in files) <= 64 << 20
    assert np.array_equal(np.load(tmp_path / "out" / "value_data.npy"), d["value_data"])
    with pytest.raises(ValueError):
        bench.write_dumps(str(tmp_path / "big"), {"x": np.zeros((64 << 20) // 4 + 1, np.float32)})
    with pytest.raises(ValueError):
        bench.write_dumps(str(tmp_path / "int"), {"x": np.zeros(4, np.uint8)})
    assert not (tmp_path / "big").exists() and not (tmp_path / "int").exists()
