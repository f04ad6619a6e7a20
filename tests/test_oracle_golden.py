"""Pins the CPU oracle against the reference's own golden vectors (DistributedMatrixSuite.scala) — CPU only."""
import hashlib

import numpy as np
import pytest

from tests import marlin_cases as mc


def _dvm(rm):
    return rm.DenseVecMatrix([(i, np.array(v)) for i, v in mc.DATA_ROWS])


def _blk(rm):
    return rm.BlockMatrix([(k, np.array(v)) for k, v in mc.BLKS])


def _blocks_equal(bm, expected):
    got = {k: v for k, v in bm.blocks}
    assert set(got) == set(expected)
    for k, v in expected.items():
        assert np.array_equal(got[k], np.array(v)), (k, got[k])


@pytest.mark.parametrize("gemm", ["f2j", "blas"])
class TestReferenceSuite:
    def test_matrix_size(self, oracle, gemm):            # DMS.scala:42-51
        mat, ma = _dvm(oracle), _blk(oracle)
        assert (mat.num_rows(), mat.num_cols()) == (4, 4)
        assert (ma.num_rows(), ma.num_cols(), ma.num_blks_by_row(), ma.num_blks_by_col()) == (4, 4, 2, 2)

    def test_empty_rows(self, oracle, gemm):             # :53-71
        with pytest.raises(RuntimeError):
            oracle.DenseVecMatrix([]).num_rows()
        with pytest.raises(RuntimeError):
            oracle.DenseVecMatrix([]).num_cols()
        with pytest.raises(RuntimeError):
            oracle.BlockMatrix([]).num_rows()
        with pytest.raises(RuntimeError):
            oracle.BlockMatrix([]).num_cols()

    def test_to_breeze(self, oracle, gemm):              # :73-84
        assert np.array_equal(_dvm(oracle).to_breeze(), mc.EXPECTED_DENSE)
        assert np.array_equal(_blk(oracle).to_breeze(), mc.EXPECTED_DENSE)

    def test_to_block_matrix(self, oracle, gemm):        # :86-105
        mat = _dvm(oracle)
        blk = mat.to_block_matrix(2, 2)
        _blocks_equal(blk, dict(mc.BLKS))
        assert np.array_equal(mat.to_block_matrix(1, 4).to_breeze(), mc.EXPECTED_DENSE)

    def test_to_dense_vec_matrix(self, oracle, gemm):    # :108-119
        rows = dict(_blk(oracle).to_dense_vec_matrix().rows)
        for i in range(4):
            assert np.array_equal(rows[i], mc.EXPECTED_DENSE[i])

    def test_elementwise(self, oracle, gemm):            # :164-205
        mat, ma = _dvm(oracle), _blk(oracle)
        for x in (mat, ma):
            assert np.array_equal(x.scalar("add", 1).to_breeze(), mc.ELE_ADD1)
            assert np.array_equal(x.add(x).to_breeze(), mc.ADD_SELF)
            assert np.array_equal(x.scalar("subtract", 1).to_breeze(), mc.ELE_SUB1)
            assert np.array_equal(x.add(x, subtract=True).to_breeze(), np.zeros((4, 4)))
            assert np.array_equal(x.scalar("multiply", 2).to_breeze(), mc.ADD_SELF)
            assert np.array_equal(x.scalar("divide", 2).to_breeze(), mc.DIVIDE2)
        assert np.array_equal(ma.add(mat).to_breeze(), mc.ADD_SELF)
        assert np.array_equal(ma.add(mat, subtract=True).to_breeze(), np.zeros((4, 4)))

    def test_multiply_broadcast_choice(self, oracle, gemm):     # :225-234
        mat = _dvm(oracle)
        assert np.array_equal(mat.multiply_auto(mat, 2, gemm=gemm).to_breeze(), mc.EXPECTED_PRODUCT)

    @pytest.mark.parametrize("split", [(2, 2, 1), (2, 1, 2), (2, 2, 2)])
    def test_new_matrix_multiplication(self, oracle, gemm, split):   # :236-249
        mat = _dvm(oracle)
        assert np.array_equal(mat.multiply_split(mat, split, gemm=gemm).to_breeze(), mc.EXPECTED_PRODUCT)

    def test_multiply_local_matrix(self, oracle, gemm):         # :251-267
        assert np.array_equal(_dvm(oracle).multiply_local(mc.EXPECTED_DENSE, gemm=gemm).to_breeze(), mc.EXPECTED_PRODUCT)

    def test_multiply_block_matrix(self, oracle, gemm):         # :269-287
        mat, ma = _dvm(oracle), _blk(oracle)
        assert np.array_equal(mat.multiply_auto(ma, 2, gemm=gemm).to_breeze(), mc.EXPECTED_PRODUCT)
        _blocks_equal(ma.multiply(ma, gemm=gemm), mc.EXPECTED_PRODUCT_BLOCKS)

    def test_block_times_densevec_broadcast(self, oracle, gemm):   # :289-299
        assert np.array_equal(_blk(oracle).multiply_auto(_dvm(oracle), 2, gemm=gemm).to_breeze(), mc.EXPECTED_PRODUCT)

    def test_transpose(self, oracle, gemm):                     # :302-316
        _blocks_equal(_dvm(oracle).transpose(), mc.EXPECTED_T_DVM_BLOCKS)
        _blocks_equal(_blk(oracle).transpose(), mc.EXPECTED_T_BLK_BLOCKS)

    def test_sum(self, oracle, gemm):                           # :319-324
        assert _dvm(oracle).sum() == mc.SUM
        assert _blk(oracle).sum() == mc.SUM

    def test_dot_product(self, oracle, gemm):                   # :326-338
        mat, ma = _dvm(oracle), _blk(oracle)
        for a, b in ((mat, mat), (mat, ma), (ma, mat), (ma, ma)):
            assert np.array_equal(a.dot_product(b).to_breeze(), mc.DOT_PRODUCT)

    def test_block_to_block(self, oracle, gemm):                # :411-418
        blk1 = _dvm(oracle).to_block_matrix(2, 2)
        assert np.array_equal(blk1.to_block_matrix(1, 4).to_breeze(), blk1.to_breeze())
        assert np.array_equal(blk1.to_block_matrix(4, 1).to_breeze(), blk1.to_breeze())

    def test_block_multiply_block_regrid(self, oracle, gemm):   # :420-432
        mat = _dvm(oracle)
        m = mat.to_block_matrix(2, 2).to_block_matrix(2, 1)
        assert np.array_equal(m.multiply(mat.to_block_matrix(1, 4), gemm=gemm).to_breeze(), mc.EXPECTED_PRODUCT)

    def test_block_multiply_broadcast(self, oracle, gemm):      # :434-448
        assert np.array_equal(_blk(oracle).multiply_local(mc.EXPECTED_DENSE, gemm=gemm).to_breeze(), mc.EXPECTED_PRODUCT)


def test_ratio_resplit_branches(oracle):
    """BlockMatrix.scala:187-216 (untested by the reference suite): (2x4 grid) x (2x2 grid) and the mirror."""
    rng = np.random.default_rng(5)
    A = rng.integers(-3, 4, size=(8, 8)).astype(float)
    B = rng.integers(-3, 4, size=(8, 8)).astype(float)
    a = oracle.DenseVecMatrix(list(enumerate(A))).to_block_matrix(2, 4)
    b = oracle.DenseVecMatrix(list(enumerate(B))).to_block_matrix(2, 2)
    assert np.array_equal(a.multiply(b).to_breeze(), A @ B)


def test_split_method_and_seq(oracle):
    # SURVEY §8 a7: cfg3 -> (2,2,2); MTUtils.scala:150-175
    assert oracle.split_method(16384, 16384, 16384, 8) == (2, 2, 2)
    assert oracle.split_method(1048576, 1024, 1024, 8) == (8, 1, 1)
    assert oracle.split_method(100, 100, 100, 1) == (1, 1, 1)
    assert oracle.split_method(10, 1000, 10, 4) == (1, 4, 1)
    assert oracle.mult_seq(1, 0, 1, 2, 2, 2) == 5     # i*n*k + j*k + kk


def test_config1_files(oracle, golden_dir):
    """BASELINE config[0]: data/a.100.100 x data/b.100.100 through loadMatrixFile -> multiply (broadcast branch and
    the (2,2,2) shuffle path); known answers from SURVEY §8(c)."""
    for name, sha in mc.SHA256.items():
        assert hashlib.sha256((golden_dir / name).read_bytes()).hexdigest() == sha
    a = oracle.load_matrix_file(str(golden_dir / "a.100.100"))
    b = oracle.load_matrix_file(str(golden_dir / "b.100.100"))
    assert (a.num_rows(), a.num_cols(), b.num_rows(), b.num_cols()) == (100, 100, 100, 100)
    A, B = a.to_breeze(), b.to_breeze()
    assert A.sum() == pytest.approx(mc.CFG1["sumA"], rel=1e-12)
    assert B.sum() == pytest.approx(mc.CFG1["sumB"], rel=1e-12)
    for gemm in ("f2j", "blas"):
        c1 = a.multiply_auto(b, 2, gemm=gemm).to_breeze()
        c2 = a.multiply_split(b, (2, 2, 2), gemm=gemm).to_breeze()
        for c in (c1, c2):
            assert c[0, 0] == pytest.approx(mc.CFG1["C00"], rel=1e-12)
            assert c[0, 1] == pytest.approx(mc.CFG1["C01"], rel=1e-12)
            assert c[99, 99] == pytest.approx(mc.CFG1["C9999"], rel=1e-12)
            assert c.sum() == pytest.approx(mc.CFG1["sumC"], rel=1e-11)
            assert np.trace(c) == pytest.approx(mc.CFG1["traceC"], rel=1e-11)
            assert np.linalg.norm(c) == pytest.approx(mc.CFG1["frobC"], rel=1e-12)
    assert (A + B).sum() == pytest.approx(mc.CFG1["sumAplusB"], rel=1e-12)


def test_f2j_dgemm_matches_exact_rational(oracle):
    """The F2J-order dgemm equals an exactly rounded dot product to within K ulp-level rounding (no FMA)."""
    from fractions import Fraction
    rng = np.random.default_rng(1)
    A = np.asfortranarray(rng.random((7, 9)) - 0.5)
    B = np.asfortranarray(rng.random((9, 5)) - 0.5)
    C = oracle.block_multiply(A, B, "f2j")
    for i in range(7):
        for j in range(5):
            exact = sum(Fraction(A[i, l]) * Fraction(B[l, j]) for l in range(9))
            bound = sum(abs(Fraction(A[i, l]) * Fraction(B[l, j])) for l in range(9)) * Fraction(10, 2 ** 53)
            assert abs(Fraction(C[i, j]) - exact) <= bound
    # transposed views go through the 'T' branches of dgemm.f
    assert np.allclose(oracle.block_multiply(np.ascontiguousarray(A), B, "f2j"), C, rtol=0, atol=1e-15)
    assert np.allclose(oracle.block_multiply(A, np.ascontiguousarray(B), "f2j"), C, rtol=0, atol=1e-15)


def test_rng_properties(oracle):
    """XORShift / hashSeed / java.util.Random restatement: structural checks (the reference has no golden values
    for its generators — parity unpinned, see DESIGN.md)."""
    # java.util.Random(42).nextLong() is a widely published constant of the JDK LCG
    assert oracle.java_random_longs(42, 1)[0] == -5025562857975149833
    v = oracle.uniform_stream(7, 0, 1000)
    assert v.min() >= 0.0 and v.max() < 1.0 and 0.4 < v.mean() < 0.6
    assert np.array_equal(oracle.uniform_stream(7, 10, 5), v[10:15])          # skip-ahead consistency
    m = oracle.random_den_vec_matrix(10, 3, 2, seed=3)
    assert m.to_breeze().shape == (10, 3) and [i for i, _ in m.rows] == list(range(10))
    b = oracle.random_block_matrix(5, 7, 2, 3, seed=3)
    assert b.to_breeze().shape == (5, 7)
    assert sorted(k for k, _ in b.blocks) == [(i, j) for i in range(2) for j in range(3)]
    assert [blk.shape for _, blk in sorted(b.blocks)] == [(3, 3), (3, 3), (3, 1), (2, 3), (2, 3), (2, 1)]


def test_save_load_roundtrip(oracle):
    blk = oracle.BlockMatrix([(k, np.array(v)) for k, v in mc.BLKS])
    again = oracle.load_block_matrix_lines(blk.save_block_lines())
    assert np.array_equal(again.to_breeze(), mc.EXPECTED_DENSE)
    assert blk.save_block_lines()[0] == "0-0-2-2:0.0,2.0,1.0,3.0"


def test_disvec_to_disvec(oracle):                        # DMS.scala:121-143
    v1 = oracle.DistributedVector([(i, np.array(v)) for i, v in mc.DISVEC_PIECES])
    v2 = v1.to_dis_vector(mc.DISVEC_SPLIT_STATUS, 4)
    assert [i for i, _ in v2.vectors] == [0, 1, 2, 3] and all(v.shape[0] == 3 for _, v in v2.vectors)
    assert np.array_equal(v1.to_breeze(), v2.to_breeze())
    assert np.array_equal(v1.to_breeze(), np.arange(12.0))


def test_blas1_distributed_vector(oracle):                # DMS.scala:390-409
    pieces = [(i, np.array(v)) for i, v in mc.BLAS1_PIECES]
    v1, v2 = oracle.DistributedVector(pieces), oracle.DistributedVector(pieces)
    assert np.array_equal(v1.multiply(v2.transpose()).to_breeze(), mc.BLAS1_OUTER)
    assert v1.transpose().multiply(v2) == mc.BLAS1_INNER
    assert v1.transpose().multiply(v2, "local") == mc.BLAS1_INNER
    with pytest.raises(ValueError):
        v1.multiply(v2)                                   # same orientation (DistributedVector.scala:177-179)
    with pytest.raises(ValueError):
        v1.transpose().multiply(v2, "elsewhere")


def test_matrix_vector(oracle):                           # BlockMatrix.scala:240-274, DenseVecMatrix.scala:149-184
    x = np.array(mc.MATVEC_X)
    ma, mat = _blk(oracle), _dvm(oracle)
    dv = oracle.DistributedVector.from_vector(x, 2)
    assert np.array_equal(ma.multiply_dist_vector(dv).to_breeze(), mc.MATVEC_Y)
    assert np.array_equal(mat.multiply_dist_vector(dv, (2, 2)).to_breeze(), mc.MATVEC_Y)
    assert np.array_equal(mat.multiply_vector(x, 2).to_breeze(), mc.MATVEC_Y)
    assert np.array_equal(mat.multiply_vector(x), mc.MATVEC_Y)
    with pytest.raises(ValueError):
        ma.multiply_vector(x)                             # "should not split the matrix by column" (:267)
    with pytest.raises(ValueError):
        ma.multiply_dist_vector(oracle.DistributedVector.from_vector(x, 4))
    rng = np.random.default_rng(5)
    A, xx = np.asfortranarray(rng.standard_normal((37, 23))), rng.standard_normal(23)
    for arr in (A, np.ascontiguousarray(A)):              # plain and isTranspose operands of dgemv
        y = oracle.block_multiply_vector(arr, xx)
        assert np.abs(y - A @ xx).max() <= 1e-13
    assert abs(oracle.vector_dot(xx, xx) - float(xx @ xx)) <= 1e-13


def test_xorshift_jump_equals_stepping(oracle):
    """The oracle's own skip-ahead (GF(2) matrix power) against plain stepping — it checks the device jump tables."""
    for seed, first in ((5, 0), (123456789, 1000), (-42, 123457)):
        assert np.array_equal(oracle.uniform_stream(seed, first, 40), oracle.uniform_stream_far(seed, first, 40))
    s = 0x9E3779B97F4A7C15
    t = s
    for _ in range(777):
        t = oracle._xs_step(t)
    assert oracle.xorshift_jump(s, 777) == t


def _parse_plain(text):
    rows = {}
    for line in text.strip().splitlines():
        head, body = line.split(":")
        rows[int(head)] = [float(t) for t in body.split(",")]
    return np.array([rows[i] for i in sorted(rows)])


def test_reference_tool_output_loads(oracle, golden_dir):
    """Files written by the reference's own tools/generateMatrix.cpp (two stored runs, see tests/golden/make_generated.sh)
    load through the oracle's and the product's loadMatrixFile (utils/MTUtils.scala:286-300) to exactly the values
    printed."""
    import marlin_b200 as mb
    for p in (golden_dir / "generated.9.6", golden_dir / "generated.11.3"):
        want = _parse_plain(p.read_text())
        assert want.shape in ((9, 6), (11, 3)) and (want >= 0).all() and (want <= 5).all()
        assert np.array_equal(oracle.load_matrix_file(str(p)).to_breeze(), want)
        got = mb.MTUtils.loadMatrixFile(None, str(p))            # host-resident rows: no arithmetic involved
        assert (got.numRows(), got.numCols()) == want.shape
        assert np.array_equal(got.toBreeze(), want)


def test_dense_vec_matrix_save_formats(oracle, tmp_path):
    """DenseVecMatrix.saveToFileSystem / saveWithDescription (matrix/DenseVecMatrix.scala:1042-1064) through the product's
    host layer on host-resident rows (no arithmetic): the row text is Breeze's DenseVector.toString, the description
    file has the two tab-separated lines, and the loader here reads the files back."""
    import marlin_b200 as mb
    rows = [(i, np.array(v)) for i, v in mc.DATA_ROWS]
    mat, omat = mb.DenseVecMatrix(rows), oracle.DenseVecMatrix(rows)
    mat.saveWithDescription(str(tmp_path / "out"))
    lines = (tmp_path / "out" / "part-00000").read_text().splitlines()
    assert lines == omat.save_lines()
    assert lines[0] == "0:DenseVector(0.0, 1.0, 2.0, 3.0)" and lines[1].startswith("2:DenseVector(3.0, ")
    assert (tmp_path / "out" / "_description").read_text() == "MatrixName\tN/A\nMatrixSize\t4 4" == omat.description()
    (tmp_path / "out" / "_description").unlink()
    again = mb.MTUtils.loadMatrixFile(None, str(tmp_path / "out"))
    assert np.array_equal(again.toBreeze(), mc.EXPECTED_DENSE)
    mat.saveToFileSystem(str(tmp_path / "plain"))
    assert (tmp_path / "plain" / "part-00000").read_text().splitlines() == lines
    big = mb.DenseVecMatrix([(0, np.array([1e-7, 123456789.125, -0.5, 1e21]))])
    big.saveToFileSystem(str(tmp_path / "sci"))
    assert (tmp_path / "sci" / "part-00000").read_text() == "0:DenseVector(1.0E-7, 1.23456789125E8, -0.5, 1.0E21)\n"


def test_fast_generator_arithmetic_equals_oracle_stream(oracle):
    """The fast fill kernel (csrc/elementwise.cu: xs_step32 / xs_next_double) keeps the XORShift state as two 32-bit
    halves, shifts by multiplying with 2^21 / 2^4, and converts next(26), next(27) with the 2^52 magic number and one FMA.
    The same integer/float steps restated here must reproduce the oracle's UniformGenerator stream bit for bit — the GPU
    test (tests/test_gpu_cabi.py) then only has to show that the kernel executes these steps."""
    import struct
    M32 = 0xFFFFFFFF

    def step32(lo, hi):
        for c, rsh in ((1 << 21, True), (1 << 4, False)):
            w = lo * c
            h = ((hi * c) & M32) + (w >> 32)
            assert h <= M32                                   # disjoint bit ranges: the add never carries
            hi ^= h
            lo ^= w & M32
            if rsh:
                lo ^= hi >> 3
        return lo, hi

    def magic(v):                                             # __hiloint2double(0x43300000, v) - 2^52
        return struct.unpack("<d", struct.pack("<II", v, 0x43300000))[0] - 4503599627370496.0

    for seed in (123456789, 1, -77, 2 ** 40 + 5):
        s = oracle.hash_seed(seed) & ((1 << 64) - 1)
        lo, hi = s & M32, s >> 32
        want = oracle.uniform_stream(seed, 0, 257)
        for i in range(257):
            lo, hi = step32(lo, hi)
            da = magic(lo & 0x3FFFFFF)
            lo, hi = step32(lo, hi)
            db = magic(lo & 0x7FFFFFF)
            x = da * 2.0 ** -26 + db * 2.0 ** -53              # exact: at most 53 significant bits
            assert x == want[i], (seed, i)
        # the 64-bit update and the halves agree
        assert oracle._xs_step(s) == (lambda t: t[0] | (t[1] << 32))(step32(s & M32, s >> 32))
