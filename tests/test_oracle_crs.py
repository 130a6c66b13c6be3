"""The oracle's CrsMatrix utilities (oracle/kk_oracle_crs.c) against the reference's own golden
cases and acceptance laws:
  * sort_and_merge: the five hard-coded matrices of sparse/unit_test/Test_Sparse_SortCrs.hpp:195-290;
  * sort_crs_matrix: equals a row-by-row host sort (testSortCRS, :44-139) -- and is stable;
  * spadd: dense row sums to 1 ulp, rows sorted and unique (test_spadd, Test_Sparse_spadd.hpp:96-187),
    with the reference's shapes incl. duplicated entries (maxNNZ > ncols) and test_spadd_known_columns."""
import numpy as np
import pytest

from crs_cases import MERGE_CASES, random_matrix, spadd_dense_check
from helpers import kk_matrix
from ref_digests import Case


@pytest.mark.parametrize("case", sorted(MERGE_CASES))
@pytest.mark.parametrize("graph", [False, True])
def test_sort_and_merge_golden(oracle, case, graph):
    c = MERGE_CASES[case]
    rp, ci, v = c["rowmap"].copy(), c["entries"].copy(), c["values"].copy()
    rpo, cio, vo = oracle.sort_and_merge(rp, ci, None if graph else v)
    assert np.array_equal(rpo, c["gold_rowmap"])
    assert np.array_equal(cio, c["gold_entries"])
    if not graph:
        assert np.array_equal(vo, c["gold_values"])


@pytest.mark.parametrize("m,n,nnz", [(10, 10, 20), (100, 100, 2000), (1000, 1000, 30000), (50, 200, 3000)])
def test_sort_crs_matches_row_sort(oracle, m, n, nnz):
    rp, ci, v = kk_matrix(m, n, nnz, 2, n // 2)
    exp_c, exp_v = ci.copy(), v.copy()
    for i in range(m):
        s, e = rp[i], rp[i + 1]
        o = np.argsort(ci[s:e], kind="stable")
        exp_c[s:e], exp_v[s:e] = ci[s:e][o], v[s:e][o]
    g = ci.copy()
    oracle.sort_crs_stable(rp, ci, v)
    assert np.array_equal(ci, exp_c) and np.array_equal(v, exp_v)
    oracle.sort_crs_stable(rp, g, None)
    assert np.array_equal(g, exp_c)


def test_sort_is_stable_on_duplicates(oracle):
    rng = np.random.default_rng(5)
    m = 200
    lens = rng.integers(0, 40, m)
    rp = np.concatenate([[0], np.cumsum(lens)]).astype(np.int32)
    ci = rng.integers(0, 7, rp[-1]).astype(np.int32)      # few distinct columns -> many ties
    v = np.arange(rp[-1], dtype=np.float64)                 # value = original position
    oracle.sort_crs_stable(rp, ci, v)
    for i in range(m):
        s, e = rp[i], rp[i + 1]
        assert np.all(np.diff(ci[s:e]) >= 0)
        same = np.diff(ci[s:e]) == 0
        assert np.all(np.diff(v[s:e])[same] > 0), "equal columns must keep their original order"


@pytest.mark.parametrize("sort_rows", [True, False])
@pytest.mark.parametrize("m,n,lo,hi", [(10, 10, 0, 0), (10, 10, 0, 2), (100, 100, 50, 100), (50, 50, 75, 100)])
@pytest.mark.parametrize("dtype", [np.float64, np.float32])
def test_spadd_reference_law(oracle, sort_rows, m, n, lo, hi, dtype):
    A = random_matrix(m, n, lo, hi, sort_rows, seed=(m << 1) ^ n, dtype=dtype)
    B = random_matrix(m, n, lo, hi, sort_rows, seed=((m << 1) ^ n) + 1, dtype=dtype)
    rpC, ciC, vC = oracle.spadd(*A, dtype(1), *B, dtype(1), sort_rows)
    spadd_dense_check(A, B, (rpC, ciC, vC), n, 1.0, 1.0)


def test_spadd_known_columns(oracle):
    """A = B = 4x4 identity in the top-left corner of a 6x7 zero matrix (Test_Sparse_spadd.hpp:189-232)."""
    rp = np.array([0, 1, 2, 3, 4, 4, 4], dtype=np.int32)
    ci = np.arange(4, dtype=np.int32)
    v = np.ones(4)
    rpC, ciC, vC = oracle.spadd(rp, ci, v, 1.0, rp, ci, v, 1.0, True)
    assert np.array_equal(rpC, rp) and np.array_equal(ciC, ci) and np.array_equal(vC, 2 * v)


def test_spadd_sorted_equals_unsorted_on_strict_input(oracle):
    A = random_matrix(300, 400, 0, 30, True, seed=1)
    B = random_matrix(300, 400, 0, 30, True, seed=2)
    s = oracle.spadd(*A, 0.5, *B, -2.0, True)
    u = oracle.spadd(*A, 0.5, *B, -2.0, False)
    for a, b in zip(s, u):
        assert np.array_equal(a, b)


@pytest.mark.parametrize("n,kmax", [(0, 10), (1, 10), (2, 3), (17, 4), (1000, 16), (5000, 70000), (3000, 2**31 - 1)])
def test_row_sort_equals_reference_radix_sort(oracle, n, kmax):
    """The restated per-row sort of sort_crs_matrix (host path) equals the reference's own SerialRadixSort2 -- compiled from
    common/src/KokkosKernels_Sorting.hpp in place (oracle/_ref) -- bit for bit, ties included (stability); without oracle/_ref,
    against its recorded output."""
    live = oracle.ref is not None and hasattr(oracle.ref, "kkref_radix_sort2_u32_f64")
    gold = Case(live, "radix_sort2", n, kmax)
    rng = np.random.default_rng(n + kmax % 97)
    ci = rng.integers(0, kmax, n).astype(np.int32)
    v = rng.uniform(-1, 1, n)
    rp = np.array([0, n], dtype=np.int32)
    eci, ev = ci.copy(), v.copy()
    oracle.sort_crs_stable(rp, eci, ev)
    ids = np.arange(n, dtype=np.int32)  # graph sort with a payload that exposes the order of ties
    eci2, eid = ci.copy(), ids.copy()
    oracle.sort_crs_stable(rp, eci2, eid)
    gold.add(eci.astype(np.uint32), ev, eid)
    if live:
        keys, perm = ci.astype(np.uint32), v.copy()
        oracle.ref_radix_sort2(keys, perm)
        assert np.array_equal(eci.astype(np.uint32), keys) and np.array_equal(ev, perm)
        keys2, perm2 = ci.astype(np.uint32), ids.copy()
        oracle.ref_radix_sort2(keys2, perm2)
        assert np.array_equal(eid, perm2)
    gold.check()


@pytest.mark.parametrize("sorted_input", [True, False])
@pytest.mark.parametrize("m,n,lo,hi", [(50, 50, 0, 8), (700, 300, 0, 40), (400, 30, 20, 60)])
def test_spadd_numeric_equals_reference_functors(oracle, sorted_input, m, n, lo, hi):
    """The restated numeric phase of spadd equals the reference's own functors -- sparse/impl/KokkosSparse_spadd_numeric_impl.hpp
    compiled from the reference tree in place (oracle/_ref) -- bit for bit, for sorted / merged and for unsorted input
    (rows longer than the column count repeat columns); without oracle/_ref, against its recorded output."""
    live = oracle.ref is not None and hasattr(oracle.ref, "kkref_spadd_sorted_numeric_f64")
    gold = Case(live, "spadd_numeric", sorted_input, m, n, lo, hi)
    from crs_cases import random_matrix

    hi_eff = min(hi, n) if sorted_input else hi  # sorted + merged input has distinct columns
    A = random_matrix(m, n, min(lo, hi_eff), hi_eff, sorted_input, seed=1)
    B = random_matrix(m, n, min(lo, hi_eff), hi_eff, sorted_input, seed=2)
    got = oracle.spadd(*A, 0.3, *B, -1.7, sorted_input)
    assert not np.isnan(got[2]).any()
    gold.add(*got)
    if live:
        ref = oracle.ref_spadd_numeric(*A, 0.3, *B, -1.7, sorted_input)
        assert np.array_equal(got[0], ref[0]) and np.array_equal(got[1], ref[1]) and np.array_equal(got[2], ref[2])
    gold.check()
