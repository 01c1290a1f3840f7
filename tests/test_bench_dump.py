"""bench.py --dump-outputs writer: float32 .npy files, at most 64 MB in all, and the same seeded row sample on every
run, so two builds can be compared output for output."""
import importlib.util
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _load_bench():
    flag = sys.dont_write_bytecode
    try:
        spec = importlib.util.spec_from_file_location("bench", os.path.join(ROOT, "bench.py"))
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
    finally:
        sys.dont_write_bytecode = flag
    return mod


def test_dump_outputs_small_arrays_are_written_whole(tmp_path):
    bench = _load_bench()
    rng = np.random.default_rng(0)
    y = rng.standard_normal((32, 4096)).astype(np.float32)
    bench.write_dumps(str(tmp_path), {"int4_stack_bs32": y, "int4_stack_bs1": y[:1].astype(np.float64)})
    assert sorted(os.listdir(tmp_path)) == ["int4_stack_bs1.npy", "int4_stack_bs32.npy"]
    a, b = np.load(tmp_path / "int4_stack_bs32.npy"), np.load(tmp_path / "int4_stack_bs1.npy")
    assert a.dtype == b.dtype == np.float32
    assert np.array_equal(a, y) and np.array_equal(b, y[:1])


def test_dump_outputs_above_64mb_keep_a_fixed_row_sample(tmp_path):
    bench = _load_bench()
    rng = np.random.default_rng(1)
    big = rng.standard_normal((8192, 4096), dtype=np.float32)   # 128 MB
    one = rng.standard_normal((1, 4096), dtype=np.float32)
    for run in ("a", "b"):
        bench.write_dumps(str(tmp_path / run), {"int4_stack_bs8192": big, "int4_stack_bs1": one})
    files = sorted(os.listdir(tmp_path / "a"))
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in files) <= 64 << 20
    assert np.array_equal(np.load(tmp_path / "a" / "int4_stack_bs1.npy"), one)
    s = np.load(tmp_path / "a" / "int4_stack_bs8192.npy")
    assert s.dtype == np.float32 and s.shape[1] == 4096 and s.shape[0] >= 4000
    assert np.array_equal(s, np.load(tmp_path / "b" / "int4_stack_bs8192.npy"))
    rows = np.array([np.flatnonzero(big[:, 0] == r[0])[0] for r in s])
    assert np.all(np.diff(rows) > 0) and np.array_equal(big[rows], s)
