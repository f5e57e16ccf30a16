"""CPU tests of bench.py's --dump-outputs writer and argument checks (no GPU: the writer takes host arrays)."""
import os
import sys

import numpy as np
import pytest

import bench


def _outs(nq, k, seed=0):
    rng = np.random.default_rng(seed)
    ids = rng.integers(0, 1 << 40, (nq, k)).astype(np.int64)
    ids[:, -1] = -1                                    # an empty slot, as the kernels leave it
    return {"ids": ids, "dist": rng.random((nq, k), dtype=np.float32),
            "counts": np.full(nq, k - 1, np.int32), "evals": rng.integers(0, 5000, nq).astype(np.int32)}


def test_dump_writes_every_array_in_float32_or_float64(tmp_path):
    outs = _outs(300, 10)
    bench.dump_outputs(str(tmp_path), outs)
    assert sorted(os.listdir(tmp_path)) == ["counts.npy", "dist.npy", "evals.npy", "ids.npy"]
    for name, a in outs.items():
        got = np.load(tmp_path / f"{name}.npy")
        assert got.dtype == (np.float32 if a.dtype == np.float32 else np.float64)
        assert np.array_equal(got, a)                  # exact: ids below 2**53, -1 kept


def test_dump_samples_the_same_rows_of_a_large_output_within_the_limit(tmp_path, monkeypatch):
    monkeypatch.setattr(bench, "DUMP_BYTES", 1 << 20)
    outs = _outs(20000, 10)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), outs)
        assert sum(f.stat().st_size for f in (tmp_path / d).iterdir()) <= 1 << 20
    rows = np.load(tmp_path / "a" / "rows.npy").astype(np.int64)
    assert 0 < len(rows) < 20000 and np.all(np.diff(rows) > 0)
    for name, a in outs.items():
        got = np.load(tmp_path / "a" / f"{name}.npy")
        assert np.array_equal(got, a[rows]) and np.array_equal(got, np.load(tmp_path / "b" / f"{name}.npy"))


@pytest.mark.parametrize("argv", [["--steps", "0"], ["--warmup", "-1"], ["--impl", "reference", "--dump-outputs", "x"]])
def test_bench_rejects_arguments_it_cannot_honour(monkeypatch, argv):
    monkeypatch.setattr(sys, "argv", ["bench.py", *argv])
    with pytest.raises(SystemExit):
        bench.parse_args()


def test_bench_steps_and_dump_dir_are_parsed(monkeypatch):
    monkeypatch.setattr(sys, "argv", ["bench.py", "--steps", "7", "--warmup", "0", "--dump-outputs", "out"])
    a = bench.parse_args()
    assert (a.steps, a.warmup, a.dump_outputs) == (7, 0, "out")
