"""The oracle's spgemm_jacobi (oracle/kk_oracle_crs.c, restating
sparse/impl/KokkosSparse_spgemm_jacobi_seq_impl.hpp:26-131) against the dense definition
C = (I - omega * diag(dinv) * A) * B on the pattern of A*B, with the reference test's inputs
(diagonally dominant matrix, omega = 3, dinv = 2: sparse/unit_test/Test_Sparse_spgemm_jacobi.hpp:176-221)."""
import numpy as np
import pytest

from helpers import dense_from_csr
from ref_digests import Case


def diag_dominant(n, per, seed):
    """Rows of `per` distinct random off-diagonals plus the diagonal (sorted), diagonal = 10 * sum |row|
    (kk_generate_diagonally_dominant_sparse_matrix, sparse/src/KokkosSparse_IOUtils.hpp:112-183)."""
    rng = np.random.default_rng(seed)
    rp, ci, v = [0], [], []
    for i in range(n):
        cols = set(rng.choice(n, size=min(per, n - 1), replace=False).tolist()) - {i}
        vals = {c: rng.uniform(-1.0, 1.0) for c in cols}
        vals[i] = 10.0 * sum(abs(x) for x in vals.values()) + 1.0
        for c in sorted(vals):
            ci.append(c)
            v.append(vals[c])
        rp.append(len(ci))
    return np.array(rp, np.int32), np.array(ci, np.int32), np.array(v)


@pytest.mark.parametrize("n,per", [(50, 4), (300, 9)])
@pytest.mark.parametrize("dtype,tol", [(np.float64, 1e-12), (np.float32, 1e-4)])
def test_jacobi_matches_dense(oracle, n, per, dtype, tol):
    rp, ci, v = diag_dominant(n, per, n)
    v = v.astype(dtype)
    omega = dtype(3.0)
    dinv = np.full(n, 2.0, dtype=dtype)
    rpC, ciC, vC = oracle.spgemm_jacobi(rp, ci, v, rp, ci, v, n, omega, dinv)
    A = dense_from_csr(rp, ci, v.astype(np.float64), n)
    want = (np.eye(n) - 3.0 * np.diag(np.full(n, 2.0)) @ A) @ A
    got = dense_from_csr(rpC, ciC, vC.astype(np.float64), n)
    pattern = (np.abs(A) @ np.abs(A)) > 0
    assert np.array_equal(dense_from_csr(rpC, ciC, np.ones(len(ciC)), n) > 0, pattern), "structure = structure of A*B"
    assert np.max(np.abs(got - want)) <= tol * np.max(np.abs(want))
    for i in range(n):
        assert np.all(np.diff(ciC[rpC[i]:rpC[i + 1]]) > 0)


@pytest.mark.parametrize("n,per", [(60, 4), (500, 9), (3000, 7)])
def test_jacobi_restatement_equals_reference_seq(oracle, n, per):
    """The restatement equals the reference's own spgemm_jacobi_seq -- sparse/impl/KokkosSparse_spgemm_jacobi_seq_impl.hpp
    compiled from the reference tree in place (oracle/_ref) -- bit for bit: entries in first-touch order, values; without
    oracle/_ref, against its recorded output."""
    live = oracle.ref is not None and hasattr(oracle.ref, "kkref_spgemm_jacobi_f64")
    gold = Case(live, "spgemm_jacobi", n, per)
    rp, ci, v = diag_dominant(n, per, n + 1)
    rng = np.random.default_rng(n)
    vB = rng.uniform(-1, 1, len(ci))
    dinv = rng.uniform(0.5, 1.5, n)
    got = oracle.spgemm_jacobi(rp, ci, v, rp, ci, vB, n, 0.7, dinv, sort=False)
    assert not np.isnan(got[2]).any()
    gold.add(*got)
    if live:
        ref = oracle.ref_spgemm_jacobi(rp, ci, v, rp, ci, vB, n, 0.7, dinv)
        assert np.array_equal(got[0], ref[0]) and np.array_equal(got[1], ref[1]) and np.array_equal(got[2], ref[2])
    gold.check()
