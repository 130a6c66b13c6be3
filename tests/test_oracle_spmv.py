"""Pins the SpMV oracle (oracle/kk_oracle.c) against the reference's own
known-answer tests and checks its variants against each other (CPU only)."""
import numpy as np
import pytest

from helpers import dense_from_csr, kk_matrix, spmv_tolerance
from ref_digests import Case

EPS_F = np.finfo(np.float32).eps


def _issue101(dtype_mat):
    rp = np.array([0, 2], dtype=np.int32)
    ci = np.array([0, 1], dtype=np.int32)
    if dtype_mat == np.float64:
        v = np.array([1.0, float(EPS_F) / 2.0], dtype=np.float64)
    else:
        v = np.array([1.0, EPS_F / np.float32(2.0)], dtype=np.float32)
    return rp, ci, v


@pytest.mark.parametrize("dtype_mat", [np.float64, np.float32])
def test_issue101_rank1_exact(oracle, dtype_mat):
    """test_github_issue_101 (Test_Sparse_spmv.hpp:822-961): y must EQUAL 1 + eps_f/2 in double,
    also with a float matrix and double vectors."""
    rp, ci, v = _issue101(dtype_mat)
    x = np.ones(2)
    expected = 1.0 + float(EPS_F) / 2.0
    assert expected != 1.0
    y = np.zeros(1)
    oracle.spmv_serial(rp, ci, v, x, y, 1.0, 0.0)
    assert y[0] == expected
    if dtype_mat == np.float64:
        y2 = np.zeros(1)
        oracle.spmv_functor(rp, ci, v, 2, x, y2, 1.0, 0.0)
        assert y2[0] == expected
        y3 = np.zeros(1)
        oracle.spmv_test("N", rp, ci, v, x, y3, 1.0, 0.0)
        assert y3[0] == expected


@pytest.mark.parametrize("dtype_mat", [np.float64, np.float32])
@pytest.mark.parametrize("order", ["F", "C"])
def test_issue101_multivector_exact(oracle, dtype_mat, order):
    rp, ci, v = _issue101(dtype_mat)
    expected = 1.0 + float(EPS_F) / 2.0
    for nv in range(1, 23):  # 1..22 columns exercises every strip length incl. 17
        X = np.ones((2, nv), order=order)
        Y = np.zeros((1, nv), order=order)
        oracle.spmv_mv(rp, ci, v, 2, X, Y, 1.0, 0.0)
        assert np.all(Y == expected), nv


def test_beta_zero_overwrites_nan(oracle):
    """beta == 0 must overwrite NaN in y (Test_Sparse_spmv.hpp:394-408,434-436)."""
    rp, ci, v = kk_matrix(1000, 1000, 1000 * 3, 10, 200)
    x = np.random.default_rng(0).random(1000)
    for alpha in (0.0, 1.0, 2.5):
        for fn in ("serial", "functor", "test"):
            y = np.random.default_rng(1).random(1000)
            y[::19] = np.nan
            if fn == "serial":
                oracle.spmv_serial(rp, ci, v, x, y, alpha, 0.0)
            elif fn == "functor":
                oracle.spmv_functor(rp, ci, v, 1000, x, y, alpha, 0.0)
            else:
                oracle.spmv_test("N", rp, ci, v, x, y, alpha, 0.0)
            assert not np.isnan(y).any(), (alpha, fn)
    yt = np.random.default_rng(2).random(1000)
    yt[::23] = np.nan
    oracle.spmv_transpose(rp, ci, v, 1000, x, yt, 1.0, 0.0)
    assert not np.isnan(yt).any()


SWEEP = [  # (rows, nnz/row, bandwidth, variance, heavy) -- Test_Sparse_spmv.hpp:1060-1068
    (1000, 3, 200, 10, True), (1000, 3, 100, 10, True), (1000, 20, 100, 5, True),
    (50000, 3, 20, 10, False), (50000, 3, 100, 10, False), (10000, 2, 100, 5, False),
]


@pytest.mark.parametrize("rows,per,bw,var,heavy", SWEEP)
def test_oracle_variants_agree_reference_law(oracle, rows, per, bw, var, heavy):
    """O1 (Serial), O2 (functor) and O3 (test oracle) agree within the reference's own acceptance
    law; O3 == dense matmul within the same law."""
    rp, ci, v = kk_matrix(rows, rows, rows * per, var, bw)
    rng = np.random.default_rng(13718)
    x, y0 = rng.random(rows), rng.random(rows)
    coefs = [0.0, 1.0, -1.0, 2.5] if heavy else [0.0, 1.0]
    eps = np.finfo(np.float64).eps
    for alpha in coefs:
        for beta in coefs:
            tol = spmv_tolerance(eps, alpha, beta, per + var) + 1e-300
            y1 = oracle.spmv_serial(rp, ci, v, x, y0.copy(), alpha, beta)
            y2 = oracle.spmv_functor(rp, ci, v, rows, x, y0.copy(), alpha, beta)
            y3 = oracle.spmv_test("N", rp, ci, v, x, y0.copy(), alpha, beta)
            assert np.max(np.abs(y1 - y3)) <= tol and np.max(np.abs(y2 - y3)) <= tol, (alpha, beta)
            t5 = oracle.spmv_transpose(rp, ci, v, rows, x, y0.copy(), alpha, beta)
            t3 = oracle.spmv_test("T", rp, ci, v, x, y0.copy(), alpha, beta)
            assert np.max(np.abs(t5 - t3)) <= tol
    if rows <= 1000:
        A = dense_from_csr(rp, ci, v, rows)
        y3 = oracle.spmv_test("N", rp, ci, v, x, y0.copy(), 2.5, -1.0)
        assert np.max(np.abs(y3 - (2.5 * A @ x - y0))) <= spmv_tolerance(eps, 2.5, 1.0, per + var)


def test_functor_threads_bitwise_invariant(oracle):
    rp, ci, v = kk_matrix(20000, 20000, 20000 * 20, 5, 2000)
    rng = np.random.default_rng(3)
    x, y0 = rng.random(20000), rng.random(20000)
    a = oracle.spmv_functor(rp, ci, v, 20000, x, y0.copy(), 2.5, -1.0, threads=1)
    b = oracle.spmv_functor(rp, ci, v, 20000, x, y0.copy(), 2.5, -1.0, threads=max(2, oracle.num_threads()))
    assert np.array_equal(a, b)


@pytest.mark.parametrize("nv", [1, 5, 10, 16, 17, 30])
@pytest.mark.parametrize("order", ["F", "C"])
def test_mv_oracle_matches_rank1_columns(oracle, nv, order):
    """O4 per column == O2 on that column when alpha in {0,+-1}; within the law otherwise
    (alpha folded per term, spmv_impl.hpp:773-780)."""
    rp, ci, v = kk_matrix(1000, 1000, 1000 * 20, 5, 100)
    rng = np.random.default_rng(11)
    X = np.asarray(rng.random((1000, nv)), order=order)
    Y0 = np.asarray(rng.random((1000, nv)), order=order)
    eps = np.finfo(np.float64).eps
    for alpha in (0.0, 1.0, -1.0, 2.5):
        for beta in (0.0, 1.0, -1.0, 2.5):
            Y = oracle.spmv_mv(rp, ci, v, 1000, X, Y0.copy(order=order), alpha, beta)
            for j in range(nv):
                yj = oracle.spmv_functor(rp, ci, v, 1000, np.ascontiguousarray(X[:, j]), np.ascontiguousarray(Y0[:, j]), alpha, beta)
                tol = spmv_tolerance(eps, alpha, beta, 25) + 1e-300
                assert np.max(np.abs(Y[:, j] - yj)) <= tol
                if alpha == 1.0 and beta in (0.0, 1.0, 2.5):
                    assert np.array_equal(Y[:, j], yj)


def test_mv_transpose_oracle(oracle):
    rp, ci, v = kk_matrix(800, 600, 800 * 10, 5, 100)
    rng = np.random.default_rng(5)
    X, Y0 = rng.random((800, 7)), rng.random((600, 7))
    A = dense_from_csr(rp, ci, v, 600)
    Y = oracle.spmv_mv_transpose(rp, ci, v, 600, X, Y0.copy(), 2.5, -1.0)
    assert np.allclose(Y, 2.5 * A.T @ X - Y0, rtol=1e-12, atol=1e-12)


def test_fma_build_brackets(oracle):
    """The contraction-on build differs from the strict build by at most the law."""
    import oracle_lib

    fma = oracle_lib.Oracle(fma=True)
    rp, ci, v = kk_matrix(5000, 5000, 5000 * 20, 5, 500)
    rng = np.random.default_rng(9)
    x, y0 = rng.random(5000), rng.random(5000)
    a = oracle.spmv_serial(rp, ci, v, x, y0.copy(), 2.5, -1.0)
    b = fma.spmv_serial(rp, ci, v, x, y0.copy(), 2.5, -1.0)
    assert np.max(np.abs(a - b)) <= spmv_tolerance(np.finfo(np.float64).eps, 2.5, 1.0, 25)


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
@pytest.mark.parametrize("rows,per,bw,var", [(1000, 3, 200, 10), (1000, 20, 100, 5), (5000, 3, 100, 10), (300, 61, 250, 40)])
def test_o1_o2_equal_the_reference_code_bit_for_bit(oracle, dtype, rows, per, bw, var):
    """O1 (the Serial loop north_star names as the parity oracle) and O2 (the generic functor) against the reference's OWN code:
    sparse/impl/KokkosSparse_spmv_impl.hpp compiled from the reference tree in place (oracle/_ref, oracle/kkref_spmv.cpp) and
    run through its own dispatch on dobeta.  Every alpha x beta of the reference's sweep (Test_Sparse_spmv.hpp:1060-1068 +
    the dobeta = -1 branch), rows with 0..60+ entries (the 4-way unrolled loop with every remainder), NaN in y for beta = 0.
    Without oracle/_ref the outputs are checked against the reference's recorded ones (tests/ref_digests.py)."""
    live = oracle.ref is not None and hasattr(oracle.ref, "kkref_spmv_serial_f64")
    gold = Case(live, "spmv_o1_o2", np.dtype(dtype).name, rows, per, bw, var)
    rp, ci, v = kk_matrix(rows, rows, rows * per, var, bw, dtype=dtype)
    rng = np.random.default_rng(13718)
    x = rng.random(rows).astype(dtype)
    y0 = rng.random(rows).astype(dtype)
    for alpha in (0.0, 1.0, -1.0, 2.5):
        for beta in (0.0, 1.0, -1.0, 2.5):
            yin = y0.copy()
            if beta == 0.0:
                yin[::19] = np.nan
            a = oracle.spmv_serial(rp, ci, v, x, yin.copy(), alpha, beta)
            c = oracle.spmv_functor(rp, ci, v, rows, x, yin.copy(), alpha, beta)
            gold.add(a, c)
            if live:
                b = oracle.ref_spmv("serial", rp, ci, v, x, yin.copy(), alpha, beta)
                assert np.array_equal(a, b, equal_nan=True), ("O1", alpha, beta)
                d = oracle.ref_spmv("functor", rp, ci, v, x, yin.copy(), alpha, beta)
                assert np.array_equal(c, d, equal_nan=True), ("O2", alpha, beta)
    gold.check()


@pytest.mark.parametrize("rows,cols,per", [(1000, 1000, 7), (800, 300, 21), (300, 2000, 5)])
def test_o5_equals_the_reference_transpose_code(oracle, rows, cols, per):
    """O5 (Serial transpose: y scaled first, then the order-preserving unrolled scatter) against the reference's own
    spmv_beta_transpose compiled in place (sparse/impl/KokkosSparse_spmv_impl.hpp:383-460), bit for bit; without oracle/_ref,
    against its recorded output."""
    live = oracle.ref is not None and hasattr(oracle.ref, "kkref_spmv_transpose_f64")
    gold = Case(live, "spmv_o5", rows, cols, per)
    rp, ci, v = kk_matrix(rows, cols, rows * per, 6, min(cols, 200))
    rng = np.random.default_rng(5)
    x = rng.random(rows)
    y0 = rng.random(cols)
    for alpha in (0.0, 1.0, -1.0, 2.5):
        for beta in (0.0, 1.0, -1.0, 2.5):
            yin = y0.copy()
            if beta == 0.0:
                yin[::23] = np.nan
            a = oracle.spmv_transpose(rp, ci, v, cols, x, yin.copy(), alpha, beta)
            assert not np.isnan(a).any(), (alpha, beta)
            gold.add(a)
            if live:
                b = oracle.ref_spmv("transpose", rp, ci, v, x, yin.copy(), alpha, beta)
                assert np.array_equal(a, b), (alpha, beta)
    gold.check()


@pytest.mark.parametrize("order", ["F", "C"])
@pytest.mark.parametrize("k", [1, 3, 16, 17, 33])
def test_o4_equals_the_reference_multivector_code(oracle, order, k):
    """O4 (CPU multivector strips, alpha folded per term when alpha is not 0 / +-1, dobeta = -1 as -y + sum) and the multivector
    transpose against the reference's own spmv_alpha_mv compiled in place (sparse/impl/KokkosSparse_spmv_impl.hpp:547-1270),
    bit for bit, for every alpha x beta, column counts around the strip widths (16 / 17) and both layouts; without oracle/_ref,
    against its recorded output."""
    live = oracle.ref is not None and hasattr(oracle.ref, "kkref_spmv_mv_f64")
    gold = Case(live, "spmv_o4", order, k)
    rows, cols = 700, 500
    rp, ci, v = kk_matrix(rows, cols, rows * 9, 8, 150)
    rng = np.random.default_rng(k)
    for mode in ("N", "T"):
        nx, ny = (rows, cols) if mode == "T" else (cols, rows)
        X = np.asarray(rng.random((nx, k)), order=order)
        Y0 = np.asarray(rng.random((ny, k)), order=order)
        for alpha in (0.0, 1.0, -1.0, 2.5):
            for beta in (0.0, 1.0, -1.0, 2.5):
                Yin = Y0.copy(order=order)
                if beta == 0.0 and alpha != 0.0:
                    Yin[::19] = np.nan
                if mode == "N":
                    a = oracle.spmv_mv(rp, ci, v, cols, X, Yin.copy(order=order), alpha, beta)
                else:
                    a = oracle.spmv_mv_transpose(rp, ci, v, cols, X, Yin.copy(order=order), alpha, beta)
                assert not np.isnan(a).any(), (mode, alpha, beta)
                gold.add(a)
                if live:
                    b = oracle.ref_spmv_mv(mode, rp, ci, v, cols, X, Yin.copy(order=order), alpha, beta)
                    assert np.array_equal(a, b), (mode, alpha, beta)
    gold.check()


def test_raw_openmp_path_a8(oracle):
    """a8 of SURVEY.md section 8: spmv_raw_openmp_no_transpose (spmv_impl_omp.hpp:20-78).  Folding alpha into every coefficient
    is exact for alpha == 1, so there the path equals the functor (O2, itself pinned on the reference's own code) bit for bit,
    whatever the row blocks; for other alpha it obeys the reference's tolerance law; beta == 0 overwrites NaN."""
    from helpers import kk_matrix, spmv_tolerance
    import sys, os
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "kokkos-kernels_b200"))
    import partition

    rp, ci, v = kk_matrix(5000, 4000, 60000, 12, 300)
    rng = np.random.default_rng(3)
    x = rng.uniform(-1, 1, 4000)
    y0 = rng.uniform(-1, 1, 5000)
    for nblocks in (1, 3, 8):
        bo = partition.balanced_row_blocks(rp, nblocks)
        for alpha, beta in ((1.0, 0.0), (1.0, 0.5), (2.5, -1.0), (-0.75, 0.0)):
            y = y0.copy()
            if beta == 0.0:
                y[::19] = np.nan
            oracle.spmv_raw_openmp(bo, rp, ci, v, x, y, alpha, beta)
            ref = y0.copy()
            oracle.spmv_functor(rp, ci, v, 4000, x, ref, alpha, beta)
            assert not np.isnan(y).any()
            if alpha == 1.0:
                assert np.array_equal(y, ref)
            else:
                tol = spmv_tolerance(np.finfo(np.float64).eps, alpha, beta, int(np.diff(rp).max()))
                assert np.max(np.abs(y - ref)) <= tol
