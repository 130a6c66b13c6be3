"""Higher-precision reference of rank-2 SpMV, Y = alpha*op(A)*X + beta*Y0, with a per-element error bound.

The kernels add the products of a row in many orders: storage order, pieces of LMAX entries joined by a tree, lanes of a
shuffle tree, atomics of the transpose and split kernels.  The standard bound of a sum of L products in ANY order,
|fl(s) - s| <= gamma(L) * sum |a_ij||x_jc|, with gamma(n) = n*u / (1 - n*u), covers all of them; the alpha scaling, the
beta*y0 product and the final addition add three roundings.  So one law serves every kernel:

    |Y_ic - Yref_ic| <= C_SAFETY * gamma(L_i + 3) * (|alpha| * sum_j |a_ij||x_jc| + |beta||y0_ic|)

L_i is the number of entries that contribute to output row i (the row length for mode N, the column count of A for
T / H).  C_SAFETY = 2 leaves room for the reference's own rounding and for fused multiply-adds, which only ever lower
the error: the reference is float64 for fp32 kernels (52 more bits than the kernel) and long double for fp64 kernels
(at least 11 more bits), so its error is below u * gamma(L) of the kernel's type for every L used here, well inside the
factor 2.  A short row therefore gets a bound of a few ulps of its own magnitude, and a hub a wide one: a kernel that
drops or repeats a single product, or reads one wrong X element, fails on a short row where one absolute tolerance for
the whole matrix would not notice.  The reference uses numpy only, never the library or the C oracle."""
import numpy as np

C_SAFETY = 2.0


def unit_roundoff(dtype):
    return 2.0 ** -24 if np.dtype(dtype) == np.float32 else 2.0 ** -53


def ref_dtype(dtype):
    """float64 for fp32 kernels, long double for fp64 kernels."""
    return np.float64 if np.dtype(dtype) == np.float32 else np.longdouble


def gamma(n, u):
    n = np.asarray(n, dtype=np.float64)
    return n * u / (1.0 - n * u)


def reference(rp, ci, v, X, Y0, alpha, beta, mode="N", ncols=None):
    """(Yref, bound, L) in the reference precision.  rp, ci, v: CSR of A (m rows, ncols columns; columns may repeat
    and need not be sorted); X, Y0: 2-D numpy arrays in the kernel's dtype.  alpha and beta are rounded to the kernel's
    dtype first, as the C ABI does.  With beta == 0, Y0 is not read (it may hold NaN)."""
    dt = v.dtype
    hp = ref_dtype(dt)
    u = unit_roundoff(dt)
    m = len(rp) - 1
    k = X.shape[1]
    rows = np.repeat(np.arange(m), np.diff(rp))
    if mode in "NnCc":
        orow, irow, nout = rows, ci.astype(np.int64), m
    else:
        assert ncols is not None, "modes T / H need the column count of A"
        orow, irow, nout = ci.astype(np.int64), rows, ncols
    order = np.argsort(orow, kind="stable")
    counts = np.bincount(orow, minlength=nout)
    starts = np.concatenate([[0], np.cumsum(counts)[:-1]])
    nz = counts > 0
    s = np.zeros((nout, k), dtype=hp)
    sa = np.zeros((nout, k), dtype=hp)
    vals = v[order].astype(hp)
    xs = X.astype(hp)
    step = max(1, (1 << 22) // max(len(ci), 1))  # columns per slab: keeps the (nnz x slab) product array small
    for c0 in range(0, k, step):
        prod = vals[:, None] * xs[irow[order], c0:c0 + step]
        if nz.any():
            s[nz, c0:c0 + step] = np.add.reduceat(prod, starts[nz], axis=0)
            sa[nz, c0:c0 + step] = np.add.reduceat(np.abs(prod), starts[nz], axis=0)
    a = hp(dt.type(alpha))
    b = hp(dt.type(beta))
    y = a * s
    scale = abs(a) * sa
    if beta != 0:
        y0 = Y0.astype(hp)
        y = y + b * y0
        scale = scale + abs(b) * np.abs(y0)
    bound = (C_SAFETY * gamma(counts + 3, u))[:, None].astype(hp) * scale
    return y, bound, counts


def check(Y, ref, what=""):
    """Assert every element of Y (numpy, kernel dtype) within the bound of reference(); NaN and Inf always fail."""
    yref, bound, counts = ref
    err = np.abs(Y.astype(yref.dtype) - yref)
    bad = ~(err <= bound)
    if bad.any():
        r, c = np.argwhere(bad)[0]
        raise AssertionError(f"{what}: {int(bad.sum())} elements outside the bound; first at row {r} (length {counts[r]}) column {c}: "
                             f"got {Y[r, c]!r} want {float(yref[r, c])!r} |err| {float(err[r, c]):.3e} bound {float(bound[r, c]):.3e}")
