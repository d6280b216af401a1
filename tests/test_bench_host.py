"""bench.py's host side: the synthetic table is one table however a run loads it, and --dump-outputs writes exact,
bounded arrays of the last timed step (no GPU needed)."""
import sys

import numpy as np
import pytest

import bench


def test_device_route_blocks_equal_the_host_table(monkeypatch):
    """build_shard (device route, any row range, e.g. one shard) uploads exactly the rows host_table holds for the
    store route, block boundaries and partial blocks included."""
    monkeypatch.setattr(bench, "BLOCK_ROWS", 100)
    full = bench.host_table(1000, 512, threads=3)
    assert np.allclose(np.linalg.norm(full, axis=1), 1.0, atol=1e-6)
    for lo, hi in ((0, 1000), (150, 777), (99, 101), (200, 300), (0, 1)):
        got = np.full((hi - lo, 512), np.nan, dtype=np.float32)
        for start, blk in bench.table_blocks(lo, hi, 512, threads=2):
            got[start - lo:start - lo + len(blk)] = blk
        assert np.array_equal(got, full[lo:hi]), (lo, hi)


def test_dump_outputs_is_exact_and_bounded(tmp_path):
    rng = np.random.default_rng(1)
    scores = rng.standard_normal((50, 10)).astype(np.float32)
    rows = rng.integers(0, 10_000_000, (50, 10))
    bench.dump_outputs(str(tmp_path / "all"), {"scores": scores, "rows": rows})
    s, r = np.load(tmp_path / "all" / "scores.npy"), np.load(tmp_path / "all" / "rows.npy")
    assert s.dtype == np.float32 and r.dtype == np.float64
    assert np.array_equal(s, scores) and np.array_equal(r, rows)
    assert sorted(p.name for p in (tmp_path / "all").iterdir()) == ["rows.npy", "scores.npy"]

    for name in ("cut", "cut2"):
        bench.dump_outputs(str(tmp_path / name), {"scores": scores, "rows": rows}, limit=2000)
    got = {p.stem: np.load(p) for p in (tmp_path / "cut").iterdir()}
    assert sum(a.nbytes for a in got.values()) <= 2000
    keep = got["query_index"].astype(np.int64)
    assert 0 < len(keep) < 50 and np.array_equal(got["scores"], scores[keep]) and np.array_equal(got["rows"], rows[keep])
    for p in (tmp_path / "cut2").iterdir():                  # the sample is seeded: the same queries every run
        assert np.array_equal(np.load(p), got[p.stem])


@pytest.mark.parametrize("argv", [["--steps", "0"], ["--warmup", "-1"], ["--impl", "reference", "--dump-outputs", "d"]])
def test_bench_rejects_arguments_it_cannot_honour(monkeypatch, argv):
    monkeypatch.setattr(sys, "argv", ["bench.py", *argv])
    with pytest.raises(SystemExit):
        bench.parse()
