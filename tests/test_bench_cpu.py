"""bench.py's host-side pieces that can be checked without a GPU: the C4 instance generator exists twice (numpy for the
CPU / reference arm, torch for the GPU arm) and both arms must differentiate the SAME problem; `config` must be identical
in both arms for the same workload (the driver compares them)."""
import sys
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

torch = pytest.importorskip("torch")
import bench  # noqa: E402


def test_c4_generators_agree_and_are_valid():
    n, K, Cc = 64 * 700, 8, 64
    cols_np, coef_np = bench.c4_instance_numpy(n, K, Cc)
    cols_t, coef_t = bench.c4_instance_torch("cpu", n, K, Cc)
    assert np.array_equal(cols_np, cols_t.numpy()) and np.array_equal(coef_np, coef_t.numpy())
    assert cols_np.min() >= 0 and cols_np.max() < n and -1.0 <= coef_np.min() and coef_np.max() < 1.0
    # every row takes K DISTINCT colours (the cyclic colouring colorvec[j] = j mod 64 + 1 is then valid by construction)
    colours = np.sort(cols_np % Cc, axis=0)
    assert (np.diff(colours, axis=0) > 0).all()
    colptr, rowval = bench.ell_csc_numpy(n, K, cols_np)
    assert colptr[0] == 1 and colptr[-1] == n * K + 1 and (np.diff(colptr) >= 0).all()
    # rows sorted inside every column (SparseMatrixCSC invariant)
    for c in (0, 1, n // 2, n - 1):
        seg = rowval[colptr[c] - 1: colptr[c + 1] - 1]
        assert (np.diff(seg) > 0).all()


def test_tridiagonal_patterns_agree():
    cp_n, rv_n = bench.tridiag_pattern_numpy(1000)
    cp_t, rv_t = bench.tridiag_pattern_torch(1000, "cpu")
    assert np.array_equal(cp_n, cp_t.numpy()) and np.array_equal(rv_n, rv_t.numpy())


def test_config_is_shared_by_both_arms():
    for w in ("c1", "c2", "c3", "c4", "c5"):
        for fd in ("forward", "central"):
            a, b = bench.workload_config(w, fd), bench.workload_config(w, fd)
            assert a == b and set(a) == {"workload", "l2"}


def test_output_dumper_writes_a_fixed_bounded_sample(tmp_path):
    small = torch.arange(1000, dtype=torch.float64)
    big = torch.arange(bench.DUMP_ELEMENTS + 12345, dtype=torch.float64) * 0.5
    for d in ("a", "b"):
        for name, a in (("small", small), ("big", big)):
            bench.output_dumper(tmp_path / d, name, a)()
    for name in ("small", "big"):
        a, b = np.load(tmp_path / "a" / f"{name}.npy"), np.load(tmp_path / "b" / f"{name}.npy")
        assert a.dtype == np.float64 and np.array_equal(a, b)
    assert np.array_equal(np.load(tmp_path / "a" / "small.npy"), small.numpy())
    sample = np.load(tmp_path / "a" / "big.npy")
    # entries of `big` at distinct positions in storage order, no more than the budget
    assert 0 < sample.size <= bench.DUMP_ELEMENTS and (np.diff(sample) > 0).all()
    assert np.isin(sample, big.numpy()).all()
    assert (tmp_path / "a" / "big.npy").stat().st_size <= 64 << 20
    # the values are read when the dumper runs (after the timed steps), not when it is made
    later = small.clone()
    dump = bench.output_dumper(tmp_path / "c", "later", later)
    later.fill_(7.0)
    dump()
    assert (np.load(tmp_path / "c" / "later.npy") == 7.0).all()
