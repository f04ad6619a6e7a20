"""CPU tests of the sparse block path: the reference's LocalMatrixSuite against the sparse oracle, the seeded generator's
properties, the CSC validation the library runs before any upload, and the multSparseDense deviation (DESIGN.md)."""
import ctypes as C

import numpy as np
import pytest

from marlin_b200 import _native as nat
from tests import sparse_oracle as so

# LocalMatrixSuite.scala:9-14 (the same sparse matrix in all four cases) and :23-27 (the dense operand)
SP_COLUMNS = [([1], [1.0]), ([0, 3], [2.0, 1.0]), ([0], [3.0]), ([2], [4.0])]
DENSE = np.array([[0.0, 1.0, 2.0, 3.0], [2.0, 3.0, 4.0, 5.0], [3.0, 2.0, 1.0, 0.0], [1.0, 1.0, 1.0, 1.0]])
EXPECTED_TO_DENSE = np.array([[0.0, 2.0, 3.0, 0.0], [1.0, 0.0, 0.0, 0.0], [0.0, 0.0, 0.0, 4.0], [0.0, 1.0, 0.0, 0.0]])
EXPECTED_DENSE_SPARSE = np.array([[1.0, 3.0, 0.0, 8.0], [3.0, 9.0, 6.0, 16.0], [2.0, 6.0, 9.0, 4.0], [1.0, 3.0, 3.0, 4.0]])
EXPECTED_SPARSE_SPARSE = np.array([[2.0, 0.0, 0.0, 12.0], [0.0, 2.0, 3.0, 0.0], [0.0, 4.0, 0.0, 0.0], [1.0, 0.0, 0.0, 0.0]])
EXPECTED_SPARSE_DENSE = np.array([[13.0, 12.0, 11.0, 10.0], [0.0, 1.0, 2.0, 3.0], [4.0, 4.0, 4.0, 4.0], [2.0, 3.0, 4.0, 5.0]])


def suite_matrix() -> so.Csc:
    return so.Csc.from_columns(4, 4, SP_COLUMNS)


@pytest.fixture(scope="module")
def lib():
    return nat.load()


# ---- LocalMatrixSuite.scala, exact
def test_local_suite_sparse_to_dense():                          # :8-21
    assert np.array_equal(so.to_dense(suite_matrix()), EXPECTED_TO_DENSE)


def test_local_suite_dense_times_sparse():                       # :23-40
    assert np.array_equal(so.mult_dense_sparse(DENSE, suite_matrix()), EXPECTED_DENSE_SPARSE)


def test_local_suite_sparse_times_sparse():                      # :42-53
    assert np.array_equal(so.multiply(suite_matrix(), suite_matrix()), EXPECTED_SPARSE_SPARSE)


def test_local_suite_sparse_times_dense():                       # :55-72
    assert np.array_equal(so.mult_sparse_dense(suite_matrix(), DENSE), EXPECTED_SPARSE_DENSE)
    # K = N = 4 <= 32: the reference's literal loop is right here too
    assert np.array_equal(so.mult_sparse_dense(suite_matrix(), DENSE, literal=True), EXPECTED_SPARSE_DENSE)


# ---- the documented deviation
def test_mult_sparse_dense_reference_loop_is_wrong_beyond_32():
    """LibMatrixMult.scala:60 indexes B with `i * cd + bi` instead of `+ bk`: at K = 40 the second 32-wide k block re-reads
    rows 0..7 of B's column instead of rows 32..39, so the literal loop disagrees with the product it names."""
    rng = np.random.default_rng(7)
    K, m, n = 40, 6, 3
    a_dense = np.where(rng.random((m, K)) < 0.5, rng.integers(1, 9, (m, K)).astype(float), 0.0)
    b = rng.integers(-4, 5, (K, n)).astype(float)
    a = so.Csc.from_dense(a_dense)
    true = a_dense @ b                                       # small integers: exact in any order
    assert np.array_equal(so.mult_sparse_dense(a, b), true)
    literal = so.mult_sparse_dense(a, b, literal=True)
    assert literal is not None                               # in bounds at this shape, just wrong
    assert not np.array_equal(literal, true)
    # what the literal loop computes: column i reads B's column i at rows (k mod 32) for every k
    rows = np.arange(K) % 32
    assert np.array_equal(literal, a_dense @ b[rows, :])


# ---- the seeded generator (SparseMatrix.rand)
@pytest.mark.parametrize("rows,cols,sparsity", [(50, 40, 0.1), (7, 13, 0.5), (1000, 300, 0.01), (5, 5, 1.0), (9, 3, 0.0)])
def test_generator_properties(rows, cols, sparsity):
    s = so.rand(rows, cols, sparsity, seed=12345)
    count = int(cols * sparsity)                             # the count follows numCols (Matrices.scala:240)
    assert np.array_equal(np.diff(s.col_ptr), np.full(cols, count))
    for c in range(cols):
        idx = s.row_idx[s.col_ptr[c]:s.col_ptr[c + 1]]
        assert np.all(np.diff(idx) > 0)                      # sorted and distinct
        assert idx.size == 0 or (idx[0] >= 0 and idx[-1] < rows)
    assert np.all((s.val >= 0.0) & (s.val < 1.0))
    again = so.rand(rows, cols, sparsity, seed=12345)
    assert all(np.array_equal(x, y) for x, y in zip(s[2:], again[2:]))
    if count and count < rows:
        other = so.rand(rows, cols, sparsity, seed=54321)
        assert not np.array_equal(s.row_idx, other.row_idx)


def test_generator_rows_are_spread_uniformly():
    s = so.rand(64, 2000, 0.008, seed=3)                     # 16 rows of 64 per column, 2000 columns
    hist = np.bincount(s.row_idx, minlength=64)
    expect = 2000 * 16 / 64
    assert hist.min() > 0.8 * expect and hist.max() < 1.2 * expect


def test_generator_count_and_rejections(lib):
    out = C.c_int32()
    assert lib.mb_sparse_rand_count(100, 300, 0.01, C.byref(out)) == nat.MB_OK and out.value == 3
    assert lib.mb_sparse_rand_count(10, 30, 1.0 / 3.0, C.byref(out)) == nat.MB_OK and out.value == int(30 * (1.0 / 3.0))
    # more distinct rows per column than rows: the reference loops forever; the library refuses
    assert lib.mb_sparse_rand_count(5, 100, 0.1, C.byref(out)) == nat.MB_ERR_INVALID_ARG
    assert b"distinct rows" in lib.mb_last_error()
    assert lib.mb_sparse_rand_count(5, 5, -0.1, C.byref(out)) == nat.MB_ERR_INVALID_ARG
    assert lib.mb_sparse_rand_count(5, 5, float("nan"), C.byref(out)) == nat.MB_ERR_INVALID_ARG
    assert lib.mb_sparse_rand_count(70000, 70000, 0.5, C.byref(out)) == nat.MB_ERR_INVALID_ARG     # nnz >= 2^31
    with pytest.raises(ValueError):
        so.rand_count(5, 100, 0.1)


# ---- CSC validation (mb_csc_check, run by mb_spblock_upload before anything is uploaded)
def _check(lib, rows, cols, cp, ri):
    cp = np.ascontiguousarray(cp, np.int32)
    ri = np.ascontiguousarray(ri if len(ri) else [0], np.int32)
    return lib.mb_csc_check(rows, cols, cp.ctypes.data_as(C.POINTER(C.c_int32)), ri.ctypes.data_as(C.POINTER(C.c_int32)))


def test_csc_check_accepts_well_formed(lib):
    s = suite_matrix()
    assert _check(lib, 4, 4, s.col_ptr, s.row_idx) == nat.MB_OK
    assert _check(lib, 3, 2, [0, 0, 0], []) == nat.MB_OK                     # nnz = 0, empty columns
    assert _check(lib, 0, 0, [0], []) == nat.MB_OK


@pytest.mark.parametrize("cp,ri,what", [
    ([0, 2, 3], [1, 0, 2], b"not strictly increasing"),     # unsorted
    ([0, 2, 3], [1, 1, 2], b"not strictly increasing"),     # duplicate row
    ([0, 1, 2], [0, 4], b"outside"),                         # row >= rows
    ([0, 1, 2], [-1, 0], b"outside"),                        # negative row
    ([0, 2, 1], [0, 1], b"decreases"),                       # col_ptr not monotone
    ([1, 2, 3], [0, 1, 2], b"col_ptr[0]"),
])
def test_csc_check_rejects_malformed(lib, cp, ri, what):
    assert _check(lib, 4, 2, cp, ri) == nat.MB_ERR_INVALID_ARG
    assert what in lib.mb_last_error()


def test_block_multiply_model_sums_partials_in_k_order():
    """The oracle's BlockMatrix.multiply model on a 1x2x1 grid: P0 + P1 of the sparse products."""
    rng = np.random.default_rng(1)
    a = {(0, 0): so.rand(5, 4, 0.5, 1), (0, 1): so.rand(5, 6, 0.5, 2)}
    b = {(0, 0): rng.random((4, 3)), (1, 0): rng.random((6, 3))}
    got = so.block_multiply(a, b, 1, 2, 1)[(0, 0)]
    want = so.mult_sparse_dense(a[(0, 0)], b[(0, 0)]) + so.mult_sparse_dense(a[(0, 1)], b[(1, 0)])
    assert np.array_equal(got, want)
    dense = np.hstack([so.to_dense(a[(0, 0)]), so.to_dense(a[(0, 1)])]) @ np.vstack([b[(0, 0)], b[(1, 0)]])
    assert np.allclose(got, dense, rtol=1e-13, atol=1e-13)
