"""Sparse blocks on the B200: the three sparse products, toDense and the seeded generator bit-identical to the CPU
restatements in tests/sparse_oracle.c, through Python, the C ABI and the C++ mirror; sparse BlockMatrix.multiply against
the oracle's block model; and the MB_ERR_UNSUPPORTED refusals of the operations the reference cannot run on sparse
blocks."""
import ctypes as C
import shutil
import subprocess
from pathlib import Path

import numpy as np
import pytest

from marlin_b200 import _native as nat
from tests import sparse_oracle as so
from tests.test_sparse_oracle import (DENSE, EXPECTED_DENSE_SPARSE, EXPECTED_SPARSE_DENSE, EXPECTED_SPARSE_SPARSE,
                                      EXPECTED_TO_DENSE, SP_COLUMNS, suite_matrix)

ROOT = Path(__file__).resolve().parents[1]
LMS = ROOT / "scripts" / "bin" / "local_matrix_suite"


def build_local_matrix_suite() -> Path:
    nat.load()
    LMS.parent.mkdir(parents=True, exist_ok=True)
    cmd = [shutil.which("g++") or "g++", "-std=c++17", "-O1", "-Wall", "-Werror", f"-I{ROOT / 'include'}",
           str(ROOT / "tests" / "cpp" / "local_matrix_suite.cpp"), f"-L{ROOT / 'marlin_b200' / 'lib'}", "-lmarlin_b200",
           "-Wl,-rpath,$ORIGIN/../../marlin_b200/lib", "-o", str(LMS)]
    subprocess.run(cmd, check=True, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    return LMS


def bits(a) -> np.ndarray:
    return np.ascontiguousarray(np.asarray(a, dtype=np.float64)).view(np.uint64)


def same_bits(a, b) -> bool:
    return np.asarray(a).shape == np.asarray(b).shape and np.array_equal(bits(a), bits(b))


def test_local_matrix_suite_port_builds_and_fails_loudly_without_gpu():
    import torch
    exe = build_local_matrix_suite()
    if torch.cuda.is_available():
        pytest.skip("GPU present: covered by test_local_matrix_suite_cpp_port")
    out = subprocess.run([str(exe)], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=120)
    assert out.returncode == 3 and "no CPU fallback" in out.stdout


# ------------------------------------------------------------------ helpers
def sp(csc: so.Csc):
    from marlin_b200 import SparseMatrix
    return SparseMatrix.fromCSC(csc.rows, csc.cols, csc.col_ptr, csc.row_idx, csc.val)


def random_csc(rng, rows, cols, density, empty_frac=0.2, ones_frac=0.1, neg_zero=True) -> so.Csc:
    """Random CSC with empty columns, single-1.0 columns and stored -0.0 values."""
    cp, ri, v = [0], [], []
    for c in range(cols):
        u = rng.random()
        if u < empty_frac:
            pass
        elif u < empty_frac + ones_frac and rows:
            ri.append(int(rng.integers(rows))); v.append(1.0)
        else:
            k = min(rows, rng.binomial(rows, density))
            idx = np.sort(rng.choice(rows, size=k, replace=False)) if k else np.zeros(0, int)
            vals = rng.standard_normal(k)
            if neg_zero and k:
                vals[rng.random(k) < 0.05] = -0.0
            ri.extend(int(i) for i in idx); v.extend(vals)
        cp.append(len(ri))
    return so.Csc(rows, cols, np.array(cp, np.int32), np.array(ri, np.int32), np.array(v, np.float64))


def random_dense(rng, rows, cols):
    a = rng.standard_normal((rows, cols))
    a[rng.random((rows, cols)) < 0.05] = -0.0
    return np.asfortranarray(a)


# ------------------------------------------------------------------ LocalMatrixSuite through Python, the C ABI and C++
@pytest.mark.gpu
def test_local_matrix_suite_python():
    from marlin_b200 import LibMatrixMult, SparseMatrix, SubMatrix
    s = SparseMatrix(4, 4, SP_COLUMNS)
    assert np.array_equal(s.toDense().toBreeze(), EXPECTED_TO_DENSE)
    assert np.array_equal(s.toBreeze().toarray(), EXPECTED_TO_DENSE)
    assert np.array_equal(LibMatrixMult.multDenseSparse(DENSE, s).toBreeze(), EXPECTED_DENSE_SPARSE)
    assert np.array_equal(s.multiply(s).toBreeze(), EXPECTED_SPARSE_SPARSE)
    assert np.array_equal(LibMatrixMult.multSparseDense(s, DENSE).toBreeze(), EXPECTED_SPARSE_DENSE)
    # the same four through SubMatrix's dispatch (SubMatrix.scala:87-119)
    ss, dd = SubMatrix(spMatrix=s), SubMatrix(DENSE)
    assert ss.isSparse and not dd.isSparse and ss.denseBlock is None and ss.sparseBlock is s
    assert np.array_equal(dd.multiply(ss).toBreeze(), EXPECTED_DENSE_SPARSE)
    assert np.array_equal(ss.multiply(ss).toBreeze(), EXPECTED_SPARSE_SPARSE)
    assert np.array_equal(ss.multiply(dd).toBreeze(), EXPECTED_SPARSE_DENSE)
    assert np.array_equal(ss.multiply(DENSE).toBreeze(), EXPECTED_SPARSE_DENSE)       # multiply(other: BDM) :112-114


@pytest.mark.gpu
def test_local_matrix_suite_c_abi():
    from marlin_b200.runtime import Runtime
    rt = Runtime.get(); rt.sync_stream()
    lib, ctx = rt.lib, rt.ctx
    s = suite_matrix()
    ip = C.POINTER(C.c_int32)
    h = nat.c_sp()
    nat.check(lib.mb_spblock_upload(ctx, 4, 4, s.col_ptr.ctypes.data_as(ip), s.row_idx.ctypes.data_as(ip),
                                    s.val.ctypes.data_as(nat.c_dp), C.byref(h)))
    d = nat.c_blk()
    dense = np.asfortranarray(DENSE)
    nat.check(lib.mb_block_upload(ctx, dense.ctypes.data_as(nat.c_dp), 0, 4, 4, 4, 0, nat.MB_F64, C.byref(d)))
    out = nat.c_blk()
    nat.check(lib.mb_block_alloc(ctx, 4, 4, nat.MB_F64, C.byref(out)))
    host = np.zeros((4, 4), order="F")

    def got():
        nat.check(lib.mb_block_download(ctx, out, host.ctypes.data_as(nat.c_dp), 4))
        return host.copy()

    try:
        nat.check(lib.mb_spblock_to_dense(ctx, h, out)); assert np.array_equal(got(), EXPECTED_TO_DENSE)
        nat.check(lib.mb_spmm_dense_sparse(ctx, d, h, out, 0)); assert np.array_equal(got(), EXPECTED_DENSE_SPARSE)
        nat.check(lib.mb_spgemm_to_dense(ctx, h, h, out, 0)); assert np.array_equal(got(), EXPECTED_SPARSE_SPARSE)
        nat.check(lib.mb_spmm_sparse_dense(ctx, h, d, out, 0)); assert np.array_equal(got(), EXPECTED_SPARSE_DENSE)
        nat.check(lib.mb_spmm_sparse_dense(ctx, h, d, out, 1)); assert np.array_equal(got(), 2 * EXPECTED_SPARSE_DENSE)
        # round trip and info
        rows, cols, nnz = C.c_int32(), C.c_int32(), C.c_int64()
        nat.check(lib.mb_spblock_info(h, C.byref(rows), C.byref(cols), C.byref(nnz)))
        assert (rows.value, cols.value, nnz.value) == (4, 4, 5)
        cp, ri, v = np.zeros(5, np.int32), np.zeros(5, np.int32), np.zeros(5)
        nat.check(lib.mb_spblock_download(ctx, h, cp.ctypes.data_as(ip), ri.ctypes.data_as(ip), v.ctypes.data_as(nat.c_dp)))
        assert np.array_equal(cp, s.col_ptr) and np.array_equal(ri, s.row_idx) and np.array_equal(v, s.val)
        # dimension mismatch: the reference's message
        wide = nat.c_blk()
        nat.check(lib.mb_block_alloc(ctx, 4, 3, nat.MB_F64, C.byref(wide)))
        assert lib.mb_spmm_dense_sparse(ctx, wide, h, out, 0) == nat.MB_ERR_DIM_MISMATCH
        assert lib.mb_last_error() == b"matrix dimension mismatch: 3 v.s 4"
        lib.mb_block_free(ctx, wide)
        # malformed input is refused before anything is uploaded
        bad_ri = np.array([1, 3, 0, 0, 2], np.int32)
        bad = nat.c_sp()
        assert lib.mb_spblock_upload(ctx, 4, 4, s.col_ptr.ctypes.data_as(ip), bad_ri.ctypes.data_as(ip),
                                     s.val.ctypes.data_as(nat.c_dp), C.byref(bad)) == nat.MB_ERR_INVALID_ARG
    finally:
        lib.mb_block_free(ctx, out); lib.mb_block_free(ctx, d); lib.mb_spblock_free(ctx, h)


@pytest.mark.gpu
def test_local_matrix_suite_cpp_port():
    exe = build_local_matrix_suite()
    out = subprocess.run([str(exe)], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=300)
    assert out.returncode == 0, out.stdout[-3000:]
    assert "0 failed checks" in out.stdout


# ------------------------------------------------------------------ random shapes, bit-identical to the oracle
SHAPES = [  # m, K, n, density
    (1, 1, 1, 1.0), (7, 5, 3, 0.5), (33, 70, 41, 0.1), (300, 257, 129, 0.02), (5, 40, 6, 0.3),
    (3000, 64, 9, 0.05),          # several row tiles in every kernel
    (30000, 24, 5, 0.02),         # more than 27 k rows
    (6, 12, 70000, 0.2),          # more than 65 535 output columns
]


@pytest.mark.gpu
@pytest.mark.parametrize("m,K,n,density", SHAPES)
def test_products_bit_identical(m, K, n, density):
    from marlin_b200 import LibMatrixMult, SubMatrix
    rng = np.random.default_rng(m * 7919 + K * 31 + n)
    a_sp, b_sp = random_csc(rng, m, K, density), random_csc(rng, K, n, density)
    a_de, b_de = random_dense(rng, m, K), random_dense(rng, K, n)
    ga, gb = sp(a_sp), sp(b_sp)
    assert same_bits(LibMatrixMult.multDenseSparse(a_de, gb).toBreeze(), so.mult_dense_sparse(a_de, b_sp))
    assert same_bits(LibMatrixMult.multSparseDense(ga, b_de).toBreeze(), so.mult_sparse_dense(a_sp, b_de))
    assert same_bits(ga.multiply(gb).toBreeze(), so.multiply(a_sp, b_sp))
    assert same_bits(ga.toDense().toBreeze(), so.to_dense(a_sp))
    # accumulate = a separate product added with one rounding
    c0 = random_dense(rng, m, n)
    for prod, ref in ((lambda o: LibMatrixMult.multDenseSparse(a_de, gb, out=o, accumulate=True), so.mult_dense_sparse(a_de, b_sp)),
                      (lambda o: LibMatrixMult.multSparseDense(ga, b_de, out=o, accumulate=True), so.mult_sparse_dense(a_sp, b_de)),
                      (lambda o: ga.multiply(gb, out=o, accumulate=True), so.multiply(a_sp, b_sp))):
        out = SubMatrix(c0)
        prod(out)
        assert same_bits(out.toBreeze(), c0 + ref)


@pytest.mark.gpu
def test_empty_and_special_operands():
    from marlin_b200 import LibMatrixMult
    rng = np.random.default_rng(5)
    zero = so.Csc(9, 6, np.zeros(7, np.int32), np.zeros(0, np.int32), np.zeros(0))       # nnz = 0
    a = random_dense(rng, 4, 9)
    assert same_bits(LibMatrixMult.multDenseSparse(a, sp(zero)).toBreeze(), np.zeros((4, 6)))
    assert same_bits(LibMatrixMult.multSparseDense(sp(zero), random_dense(rng, 6, 3)).toBreeze(), np.zeros((9, 3)))
    # the single-1.0-column shortcut keeps -0.0; a column holding 1.0 and another entry does not copy
    a = np.asfortranarray(np.array([[-0.0, 2.0], [3.0, -0.0]]))
    one = so.Csc.from_columns(2, 3, [([0], [1.0]), ([1], [1.0]), ([0, 1], [1.0, 0.0])])
    got = LibMatrixMult.multDenseSparse(a, sp(one)).toBreeze()
    ref = so.mult_dense_sparse(a, one)
    assert same_bits(got, ref)
    assert np.signbit(got[0, 0]) and np.signbit(got[1, 1]) and not np.signbit(got[0, 2])


@pytest.mark.gpu
def test_strided_sliced_and_transposed_dense_operands():
    from marlin_b200 import LibMatrixMult, SubMatrix
    rng = np.random.default_rng(11)
    m, K, n = 37, 45, 29
    a_sp, b_sp = random_csc(rng, m, K, 0.2), random_csc(rng, K, n, 0.2)
    big = random_dense(rng, 80, 90)
    # slices (majorStride = parent rows, offset != 0)
    a_view = SubMatrix(big).slice(3, 3 + m, 7, 7 + K)
    b_view = SubMatrix(big).slice(10, 10 + K, 2, 2 + n)
    assert same_bits(LibMatrixMult.multDenseSparse(a_view, sp(b_sp)).toBreeze(), so.mult_dense_sparse(big[3:3 + m, 7:7 + K], b_sp))
    assert same_bits(LibMatrixMult.multSparseDense(sp(a_sp), b_view).toBreeze(), so.mult_sparse_dense(a_sp, big[10:10 + K, 2:2 + n]))
    # transposed views (Breeze .t)
    at = random_dense(rng, K, m)
    bt = random_dense(rng, n, K)
    assert same_bits(LibMatrixMult.multDenseSparse(SubMatrix(at).t, sp(b_sp)).toBreeze(), so.mult_dense_sparse(at.T, b_sp))
    assert same_bits(LibMatrixMult.multSparseDense(sp(a_sp), SubMatrix(bt).t).toBreeze(), so.mult_sparse_dense(a_sp, bt.T))
    # a strided output view
    c_big = SubMatrix(np.zeros((m + 5, n + 4)))
    LibMatrixMult.multSparseDense(sp(a_sp), b_view, out=c_big.slice(2, 2 + m, 1, 1 + n))
    assert same_bits(c_big.toBreeze()[2:2 + m, 1:1 + n], so.mult_sparse_dense(a_sp, big[10:10 + K, 2:2 + n]))
    assert not c_big.toBreeze()[0:2, :].any() and not c_big.toBreeze()[:, 0].any()


@pytest.mark.gpu
def test_scalar_ops_map_stored_values_only():
    from marlin_b200 import SubMatrix
    s = SubMatrix(spMatrix=sp(suite_matrix()))
    dense = EXPECTED_TO_DENSE
    mask = dense != 0
    for got, want in ((s.add(1.5), np.where(mask, dense + 1.5, 0.0)), (s.subtract(0.25), np.where(mask, dense - 0.25, 0.0)),
                      (s.multiply(3.0), dense * 3.0), (s.divide(3.0), np.where(mask, dense / 3.0, 0.0))):
        assert got.isSparse
        assert same_bits(got.toBreeze(), want)
    assert same_bits(s.toBreeze(), dense)                      # the source block is unchanged


# ------------------------------------------------------------------ generator, BlockMatrix
@pytest.mark.gpu
def test_random_block_matrix_sparse_equals_cpu_restatement():
    from marlin_b200 import MTUtils
    seed = 20240917
    mat = MTUtils.randomBlockMatrix(None, 1000, 700, 3, 2, (True, 0.01), seed=seed)
    seeds = MTUtils._partition_seeds(seed, 6)
    assert len(mat.blocks) == 6
    for b, blk in mat.blocks:
        assert blk.isSparse
        want = so.rand(blk.rows, blk.cols, 0.01, seeds[b.row * 2 + b.column])
        cp, ri, v = blk.sparseBlock.csc()
        assert np.array_equal(cp, want.col_ptr) and np.array_equal(ri, want.row_idx) and same_bits(v, want.val)
    again = MTUtils.randomBlockMatrix(None, 1000, 700, 3, 2, (True, 0.01), seed=seed)
    assert same_bits(again.toBreeze(), mat.toBreeze())
    with pytest.raises(nat.MarlinArgumentError) as e:           # 100 rows per column from a 34-row block
        MTUtils.randomBlockMatrix(None, 100, 600, 3, 2, (True, 0.5), seed=1)
    assert e.value.code == nat.MB_ERR_INVALID_ARG


def _oracle_blocks(mat):
    return {(b.row, b.column): (so.Csc(blk.rows, blk.cols, *blk.sparseBlock.csc()) if blk.isSparse else blk.toBreeze())
            for b, blk in mat.blocks}


@pytest.mark.gpu
@pytest.mark.parametrize("grid", [(2, 2, 2), (3, 2, 4)])
@pytest.mark.parametrize("kinds", ["sparse-sparse", "dense-sparse", "sparse-dense"])
def test_block_matrix_multiply_against_oracle_model(grid, kinds):
    from marlin_b200 import MTUtils
    m, k, n = grid
    M, K, N = 301, 260, 333
    a_sparse, b_sparse = kinds.split("-")[0] == "sparse", kinds.split("-")[1] == "sparse"
    A = MTUtils.randomBlockMatrix(None, M, K, m, k, (a_sparse, 0.05), seed=3)
    B = MTUtils.randomBlockMatrix(None, K, N, k, n, (b_sparse, 0.05), seed=4)
    C_ = A.multiply(B)
    model = so.block_multiply(_oracle_blocks(A), _oracle_blocks(B), m, k, n)
    got = {(b.row, b.column): blk.toBreeze() for b, blk in C_.blocks}
    assert set(got) == set(model)
    for key in model:
        assert same_bits(got[key], model[key]), key
    # and the product it names
    ref = A.toBreeze() @ B.toBreeze()
    assert np.allclose(C_.toBreeze(), ref, rtol=1e-12, atol=1e-12)


@pytest.mark.gpu
def test_to_dense_blocks_and_multiply_local_matrix():
    from marlin_b200 import MTUtils
    A = MTUtils.randomBlockMatrix(None, 200, 150, 2, 3, (True, 0.05), seed=8)
    D = A.toDenseBlocks()
    assert all(not blk.isSparse for _, blk in D.blocks)
    for (b, s), (_, d) in zip(A.blocks, D.blocks):
        assert same_bits(d.toBreeze(), so.to_dense(so.Csc(s.rows, s.cols, *s.sparseBlock.csc())))
    assert same_bits(D.toBreeze(), A.toBreeze())
    # multiply(B: BDM) (BlockMatrix.scala:280-303): row slices of B against every sparse block, partials summed per row
    rng = np.random.default_rng(2)
    Bl = rng.standard_normal((150, 40))
    got = A.multiply(Bl)
    blocks = _oracle_blocks(A)
    for r in range(2):
        want = None
        for c in range(3):
            p = so.mult_sparse_dense(blocks[(r, c)], Bl[c * 50:(c + 1) * 50, :])
            want = p if want is None else want + p
        blk = dict(((b.row, b.column), s) for b, s in got.blocks)[(r, 0)]
        assert same_bits(blk.toBreeze(), want)


@pytest.mark.gpu
def test_unsupported_operations_on_sparse_blocks():
    from marlin_b200 import MTUtils, SubMatrix
    A = MTUtils.randomBlockMatrix(None, 64, 64, 2, 2, (True, 0.1), seed=1)
    Dn = MTUtils.randomBlockMatrix(None, 64, 64, 2, 2, seed=2)
    odd = MTUtils.randomBlockMatrix(None, 64, 64, 2, 4, (True, 0.1), seed=3)
    calls = {
        "transpose": lambda: A.transpose(),
        "add": lambda: A.add(Dn),
        "subtract": lambda: Dn.subtract(A),
        "dotProduct": lambda: A.dotProduct(Dn),
        "sum": lambda: A.sum(),
        "toDenseVecMatrix": lambda: A.toDenseVecMatrix(),
        "re-grid": lambda: A.toBlockMatrix(4, 4),
        "save": lambda: A.saveToFileSystem("/nonexistent-dir-not-created"),
        "subtractBy": lambda: A.subtractBy(1.0),
        "divideBy": lambda: A.divideBy(1.0),
        "ratio re-split": lambda: odd.multiply(A),
        "vector": lambda: A.multiply(np.ones(64)),
    }
    for name, f in calls.items():
        with pytest.raises(nat.MarlinArgumentError) as e:
            f()
        assert e.value.code == nat.MB_ERR_UNSUPPORTED, name
        assert "toDenseBlocks" in str(e.value), (name, str(e.value))
    s = SubMatrix(spMatrix=A.blocks[0][1].sparseBlock)
    d = SubMatrix(np.ones((32, 32)))
    for f in (lambda: s.add(d), lambda: d.subtract(s), lambda: s.transpose()):
        with pytest.raises(nat.MarlinArgumentError) as e:
            f()
        assert e.value.code == nat.MB_ERR_UNSUPPORTED
