"""Pins oracle/kk_oracle_bsr.c (BsrMatrix SpMV): the restatement of the reference's mode-N functor must equal
(a) the reference's own functor compiled from the reference tree (oracle/_ref/libkkref.so) and (b) the pinned
CrsMatrix functor order on bsr_to_crs(A), bit for bit; the host functors (all four modes) by the unit test's law
(sparse/unit_test/Test_Sparse_spmv_bsr.hpp:142-213,351-456)."""
import numpy as np
import pytest

from bsr_cases import BLOCK_SIZES, COEFS_ALPHA, COEFS_BETA, PRIME_CASE, SHAPES, bsr_random, op_max_nnz_per_row, tolerance
from ref_digests import Case

CASES = [(bs, mb, nb) for (mb, nb) in SHAPES for bs in BLOCK_SIZES] + [PRIME_CASE]


def vectors(rng, n, k, dtype, order="F"):
    a = rng.uniform(0.0, 10.0, (n, k)).astype(dtype)
    return np.asarray(a, order=order)


@pytest.mark.parametrize("bs,mb,nb", CASES)
@pytest.mark.parametrize("dtype", [np.float64, np.float32])
def test_v42_restatement_equals_reference_functor(oracle, bs, mb, nb, dtype):
    """Without oracle/_ref, against the reference functor's recorded output (tests/ref_digests.py)."""
    live = oracle.ref is not None and hasattr(oracle.ref, "kkref_bsr_spmv_v42_f64")
    gold = Case(live, "bsr_v42", np.dtype(dtype).name, bs, mb, nb)
    rp, ci, v = bsr_random(bs, mb, nb, seed=bs * 100 + mb, dtype=dtype, sort=False)
    rng = np.random.default_rng(5)
    for k, order in ((1, "F"), (3, "F"), (4, "C")):
        X = vectors(rng, nb * bs, k, dtype, order)
        Y0 = vectors(rng, mb * bs, k, dtype, order)
        for alpha in COEFS_ALPHA:
            for beta in COEFS_BETA:
                Y0n = Y0.copy(order=order)
                if beta == 0.0:
                    Y0n[::3] = np.nan
                a = oracle.bsr_spmv_v42(bs, rp, ci, v, X, Y0n.copy(order=order), alpha, beta)
                gold.add(a)
                if live:
                    b = oracle.bsr_spmv_v42(bs, rp, ci, v, X, Y0n.copy(order=order), alpha, beta, ref=True)
                    assert np.array_equal(a, b), (k, order, alpha, beta)
                assert not np.isnan(a).any()
    gold.check()


@pytest.mark.parametrize("bs,mb,nb", CASES)
def test_v42_equals_crs_functor_on_point_matrix(oracle, bs, mb, nb):
    """What the reference's test compares against: spmv on bsr_to_crs(A).  With block rows sorted by block
    column the two accumulate in the same order, so equality is exact."""
    rp, ci, v = bsr_random(bs, mb, nb, seed=7 + bs, sort=True)
    crp, cci, cv = oracle.bsr_to_crs(bs, rp, ci, v)
    assert crp[-1] == len(ci) * bs * bs and np.all(np.diff(crp) == np.repeat(np.diff(rp), bs) * bs)
    rng = np.random.default_rng(1)
    x = rng.uniform(0, 10, nb * bs)
    y0 = rng.uniform(0, 10, mb * bs)
    for alpha, beta in ((1.0, 0.0), (3.7, -1.5), (-1.0, 1.0)):
        got = oracle.bsr_spmv_v42(bs, rp, ci, v, x, y0.copy(), alpha, beta)
        exp = oracle.spmv_functor(crp, cci, cv, nb * bs, x, y0.copy(), alpha, beta)
        assert np.array_equal(got, exp), (alpha, beta)


@pytest.mark.parametrize("bs,mb,nb", CASES)
@pytest.mark.parametrize("mode", ["N", "C", "T", "H"])
@pytest.mark.parametrize("dtype", [np.float64, np.float32])
def test_host_functors_by_the_unit_test_law(oracle, bs, mb, nb, mode, dtype):
    rp, ci, v = bsr_random(bs, mb, nb, seed=11 + bs + mb, dtype=dtype, sort=False)
    crp, cci, cv = oracle.bsr_to_crs(bs, rp, ci, v)
    trans = mode in "TH"
    rng = np.random.default_rng(2)
    nx, ny = (mb * bs, nb * bs) if trans else (nb * bs, mb * bs)
    max_row = op_max_nnz_per_row(bs, rp, ci, nb, trans)
    for k in (1, 7):  # test_spm_mv_combos (:626)
        X = vectors(rng, nx, k, dtype)
        Y0 = vectors(rng, ny, k, dtype)
        for alpha in COEFS_ALPHA:
            for beta in COEFS_BETA:
                Yin = Y0.copy(order="F")
                if beta == 0.0:
                    Yin[::5] = np.nan
                got = oracle.bsr_spmv_v41(mode, bs, nb, rp, ci, v, X, Yin.copy(order="F"), alpha, beta)
                assert not np.isnan(got).any()
                tol = tolerance(dtype, alpha, beta, max_row)
                for j in range(k):
                    exp = oracle.spmv_test(mode, crp, cci, cv, X[:, j].copy(), np.nan_to_num(Yin[:, j].copy()), alpha, beta)
                    assert np.max(np.abs(got[:, j] - exp), initial=0.0) <= tol, (mode, k, alpha, beta)
                if not trans:  # the two mode-N orders agree within the same law
                    g42 = oracle.bsr_spmv_v42(bs, rp, ci, v, X, Yin.copy(order="F"), alpha, beta)
                    assert np.max(np.abs(got - g42), initial=0.0) <= tol


def test_corner_cases(oracle):
    """bsr_corner_case_0_by_0 / 0_by_1 / 1_by_0 (:101-116, :221-278): empty matrices leave beta*y."""
    for bs in BLOCK_SIZES:
        rp0 = np.zeros(1, np.int32)
        e = np.zeros(0, np.int32)
        v = np.zeros(0)
        # 0 x 1 block: y is empty for N, has bs entries for T
        y = np.full(bs, 2.0)
        oracle.bsr_spmv_v41("T", bs, 1, rp0, e, v, np.zeros(0), y, 3.7, -1.5)
        assert np.array_equal(y, np.full(bs, -3.0))
        # 1 x 0 block: one empty block row
        rp1 = np.zeros(2, np.int32)
        y = np.full(bs, np.nan)
        oracle.bsr_spmv_v42(bs, rp1, e, v, np.zeros(0), y, 1.0, 0.0)
        assert np.array_equal(y, np.zeros(bs))
