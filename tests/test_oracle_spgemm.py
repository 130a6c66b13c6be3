"""Pins the SpGEMM oracle: the C restatement must equal, bit for bit, the
REFERENCE's own spgemm_debug_symbolic/numeric compiled from the reference tree
(oracle/_ref/libkkref.so, see oracle/Makefile), plus the reference's fixtures
and degenerate shapes (Test_Sparse_spgemm.hpp:483-511)."""
import os

import numpy as np
import pytest

from helpers import dense_from_csr, kk_matrix
from ref_digests import Case

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "issue402.npz")


def _ab(oracle, m, k, n, nnz, bw, var):
    rpA, ciA, vA = kk_matrix(m, k, nnz, var, bw, lo=1.0, hi=50.0, seed=1, sort=True, oracle=oracle)
    rpB, ciB, vB = kk_matrix(k, n, nnz, var, bw, lo=1.0, hi=50.0, seed=2, sort=True, oracle=oracle)
    return (rpA, ciA, vA), (rpB, ciB, vB)


@pytest.mark.parametrize("m,k,n,nnz", [(1000, 500, 1600, 20000), (2500, 2000, 1500, 40000)])
def test_restatement_equals_reference_build(oracle, m, k, n, nnz):
    """Without oracle/_ref, against the reference build's recorded output (tests/ref_digests.py)."""
    gold = Case(oracle.ref is not None, "spgemm", m, k, n, nnz)
    A, B = _ab(oracle, m, k, n, nnz, 500, 10)
    rpC, ciC, vC = oracle.spgemm(*A, *B, n, sort=False)
    assert not np.isnan(vC).any()
    gold.add(rpC, ciC, vC)
    if gold.live:
        rrp, rci, rv = oracle.ref_spgemm(*A, k, *B, n)
        assert np.array_equal(rpC, rrp) and np.array_equal(ciC, rci)
        assert np.array_equal(vC, rv)  # same operation order -> same bits
    gold.check()


def test_against_dense(oracle):
    A, B = _ab(oracle, 300, 200, 250, 3000, 100, 5)
    rpC, ciC, vC = oracle.spgemm(*A, *B, 250)
    D = dense_from_csr(*A, 200) @ dense_from_csr(*B, 250)
    Cd = dense_from_csr(rpC, ciC, vC, 250)
    assert np.allclose(Cd, D, rtol=1e-12, atol=0)
    # structure is symbolic: every structurally reachable entry is stored, rows sorted, no duplicates
    for i in range(300):
        row = ciC[rpC[i]:rpC[i + 1]]
        assert np.all(np.diff(row) > 0)
    assert rpC[-1] == np.count_nonzero(D)  # values in [1,50]: no cancellation


@pytest.mark.parametrize("m,k,n", [(0, 0, 0), (0, 12, 5), (10, 10, 0), (10, 10, 10)])
def test_degenerate_shapes(oracle, m, k, n):
    """Empty products: zero row_ptr, c_nnz 0 (Test_Sparse_spgemm.hpp:487-499)."""
    rpA = np.zeros(m + 1, dtype=np.int32)
    rpB = np.zeros(k + 1, dtype=np.int32)
    e_i, e_v = np.zeros(0, dtype=np.int32), np.zeros(0)
    rpC, ciC, vC = oracle.spgemm(rpA, e_i, e_v, rpB, e_i, e_v, n)
    assert len(rpC) == m + 1 and not rpC.any() and len(ciC) == 0


def test_issue402_fixture(oracle):
    """C = A*A^T on the circuit matrix of issue 402 (Test_Sparse_spgemm.hpp:372-442): the oracle
    agrees with the reference build (or, without oracle/_ref, its recorded output) and the product is symmetric."""
    gold = Case(oracle.ref is not None, "spgemm_issue402")
    z = np.load(GOLD)
    rp, ci, v = z["rowmap"].copy(), z["entries"].copy(), z["values"].copy()
    n = 1813
    assert len(rp) == n + 1 and rp[-1] == 11156
    trp, tci, tv = oracle.transpose(rp, ci, v, n)
    oracle.sort_crs(rp, ci, v)
    oracle.sort_crs(trp, tci, tv)
    rpC, ciC, vC = oracle.spgemm(rp, ci, v, trp, tci, tv, n)
    gold.add(rpC, ciC, vC)
    if gold.live:
        rrp, rci, rv = oracle.ref_spgemm(rp, ci, v, n, trp, tci, tv, n)
        oracle.sort_crs(rrp, rci, rv)
        assert np.array_equal(rpC, rrp) and np.array_equal(ciC, rci) and np.array_equal(vC, rv)
    gold.check()
    Cd = dense_from_csr(rpC, ciC, vC, n)
    assert np.allclose(Cd, Cd.T, rtol=1e-9, atol=1e-18)
    Ad = dense_from_csr(rp, ci, v, n)
    assert np.allclose(Cd, Ad @ Ad.T, rtol=1e-9, atol=1e-16)


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
def test_row_block_variant_equals_serial(oracle, dtype):
    """okk_spgemm_block (rows dealt to OpenMP threads, used by the full-size GPU parity tests) == the serial restatement,
    bit for bit, for any block and thread count"""
    from spgemm_cases import cases

    for name, A, B, m, n, k in cases(dtype)[3:8]:
        rpC, ciC, vC = oracle.spgemm(*A, *B, k)
        for r0, r1, thr in ((0, m, 3), (m // 3, m // 2 + 1, 1), (m - 5, m, 8), (7, 7, 2)):
            rowlen, ent, val = oracle.spgemm_block(r0, r1, *A, *B, k, threads=thr)
            assert np.array_equal(rowlen, np.diff(rpC)[r0:r1]), name
            assert np.array_equal(ent, ciC[rpC[r0]:rpC[r1]]) and np.array_equal(val, vC[rpC[r0]:rpC[r1]]), name
