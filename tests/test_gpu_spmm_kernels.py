"""Every rank-2 SpMV kernel of spmm.cu against a float64 / long-double reference (spmm_ref.py), with the kernel that ran
asserted by name, at the column counts, operand strides and row lengths where the kernels change behaviour.

What the cases reach (W = 16 bytes / sizeof(S): 4 for fp32, 2 for fp64; a strip covers KTL*VW columns):

  item kernel, 16-byte loads (VW = W), contiguous or W-padded row-major operands with k % W == 0:
    fp32  KTL 1,2,4,8,16,32  <- k 4, 8, 16, 32, 64, 128 (one strip); k 200 (2 strips), 260 (3 strips)
    fp64  KTL 1,2,4,8,16,32  <- k 2, 4, 8, 16, 32, 64 (one strip); k 128 (2 strips), 200 (4 strips), 260 (5 strips)
  item kernel, scalar loads (VW = 1): k % W != 0, or an odd leading dimension, or a misaligned operand
    both  KTL 1,2,4,8,16,32  <- k 1, 2, 3, 7, 15, 17 (one strip); k 33, 63, 64 (2 strips), 65, 127, 128, 129, 200, 257, 260 (3+)
  reduce kernels: the dispatch matrix has rows of 2..64 pieces (warp per row) and of more (CTA per row), so both run at
    every k, including the jb loop past 32 columns
  relayout (LayoutLeft X or Y, k >= 4) with k up to 260: the j0 loop over 32-column tiles
  spmm_general (LayoutLeft, k < 4, or no plan), spmm_rowmajor (row-major, no plan), spmm_transpose (modes T, H)
  tile (VW 1) and tilev (VW W) with the default ring, segment kernels scalar and B200SP_SPMM_SEG=vec, rings
    B200SP_SPMM_CFG=1..3, row limit B200SP_SPMM_LMAX=64; split scalar and B200SP_SPMM_VEC=1; row (spmm_rowmajor through
    a plan): test_kernel_switches, k in (1, 2, 3, 4, 8, 16, 32, 33, 64, 128, 200) --
    scalar KTL / KT 1,2,4,8,16,32 <- k 1, 2, 3 and 4, 8, 16, 32 and 33 and up (33, 64, 128, 200: several strips)
    fp32 16-byte KTL 1,2,4,8,16,32 <- k 4, 8, 16, 32, 64, 128; k 200: 2 strips
    fp64 16-byte KTL 1,2,4,8,16,32 <- k 2, 4, 8, 16, 32, 64; k 128, 200: 2 and 4 strips
  item-analysis boundaries (row lengths 0, 1, 3..9, 63..65, 128, 129, 64*64, 64*64+1, a hub): test_item_boundaries
  B200SP_SPMM_ITEM_LMAX 16 / 64 / 256 on one handle, B200SP_SPMM_ITEM_COOP 0 / 4 / 8 bit-identical (one child process each)

Runs on a B200 (-m gpu) and under B200SP_TEST_EMULATED=1 on the CPU emulation of the library."""
import functools
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import spmm_ref

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
EMULATED = os.environ.get("B200SP_TEST_EMULATED") == "1"
DTYPES = [np.float32, np.float64]
TORCH = {np.float32: torch.float32, np.float64: torch.float64}
LAYOUTS = {"RR": (True, True), "LL": (False, False), "RL": (True, False), "LR": (False, True)}
# k order on one handle: grow (16 -> 257), shrink (5), grow again (129), then the rest
K_ORDER = (16, 257, 5, 129, 1, 2, 3, 4, 7, 8, 15, 17, 31, 32, 33, 63, 64, 65, 127, 128, 200, 260)
K_TRANS = (65, 129, 257)  # modes T and H: several strips whichever load width
# (alpha, beta) by position in the k loop; beta == 0 calls get NaN rows in Y, which must not survive
COEFFS = ((1.5, -0.5), (1.0, 0.0), (-1.0, 1.0))
MMI_LMAX, MMI_LONG_PIECES = 64, 64  # spmm.cu: default item length; rows of more pieces are reduced by a CTA
TILE_SEG = 2048  # spmm.cu launch_mm_tile: long rows are cut into segments of this many entries


def _vw(dtype):
    return 16 // np.dtype(dtype).itemsize


def _csr(lens, n, rng, dtype, dup=True):
    """CSR with the given row lengths, columns in random (unsorted) order, a repeated column in some rows."""
    lens = np.asarray(lens, dtype=np.int64)
    rp = np.concatenate([[0], np.cumsum(lens)]).astype(np.int32)
    cols = []
    for L in lens:
        c = rng.choice(n, int(L), replace=L > n).astype(np.int32)
        if dup and L >= 4 and rng.random() < 0.3:
            c[-1] = c[0]  # duplicates are legal for spmv: both products count
        cols.append(c)
    ci = np.concatenate(cols).astype(np.int32) if cols else np.zeros(0, np.int32)
    v = rng.uniform(-1, 1, len(ci)).astype(dtype)
    return rp, ci, v


@functools.lru_cache(maxsize=None)
def dispatch_matrix(dtype):
    """900 x 700: short rows of 0..16 entries, a few of 2..7 pieces and one of 65 pieces (both reduce kernels)."""
    rng = np.random.default_rng(2024)
    m, n = 900, 700
    lens = rng.integers(0, 17, m)
    lens[[0, m - 1]] = 0
    lens[[10, 200, 401, 650, 777]] = [65, 128, 129, 300, 450]
    lens[500] = MMI_LMAX * MMI_LONG_PIECES + 1
    return _csr(lens, n, rng, dtype) + (n,)


@functools.lru_cache(maxsize=None)
def boundary_matrix(dtype):
    """Row lengths pinned at the item analysis' edges: runs of empty rows (first and last row included), 1..9 around
    the batch sizes EB = 4 / 8, 63..65 and 128 / 129 around LMAX = 64, 64*64 and 64*64+1 (warp vs CTA reduce), a hub."""
    rng = np.random.default_rng(77)
    m, n = 400, 6000
    lens = rng.integers(0, 13, m)
    lens[0:3] = 0
    lens[150:160] = 0
    lens[m - 2:] = 0
    pinned = [1, 3, 4, 5, 7, 8, 9, 63, 64, 65, 128, 129, 64 * 64, 64 * 64 + 1, 5500]
    lens[np.linspace(5, m - 5, len(pinned)).astype(int)] = pinned
    return _csr(lens, n, rng, dtype) + (n,)


@functools.lru_cache(maxsize=None)
def inputs(dtype, k, xrows, yrows, seed):
    rng = np.random.default_rng(seed * 1000 + k)
    X = rng.uniform(-1, 1, (xrows, k)).astype(dtype)
    Y0 = rng.uniform(-1, 1, (yrows, k)).astype(dtype)
    return X, Y0


@functools.lru_cache(maxsize=None)
def reference(which, dtype, k, mode, alpha, beta):
    rp, ci, v, n = MATRICES[which](dtype)
    m = len(rp) - 1
    xrows, yrows = (n, m) if mode == "N" else (m, n)
    X, Y0 = inputs(dtype, k, xrows, yrows, 1 if mode == "N" else 2)
    return spmm_ref.reference(rp, ci, v, X, Y0, alpha, beta, mode, ncols=n)


MATRICES = {"dispatch": dispatch_matrix, "boundary": boundary_matrix}


@functools.lru_cache(maxsize=None)
def _device_matrix(which, dtype, dev):
    from kokkos_kernels_b200 import sparse as sp

    rp, ci, v, n = MATRICES[which](dtype)
    return sp.CrsMatrix(torch.from_numpy(rp).to(dev), torch.from_numpy(ci).to(dev), torch.from_numpy(v).to(dev), n)


def operand(dev, a, rowmajor, shape):
    """a (rows x k) on the device as LayoutRight (rowmajor) or LayoutLeft, inside a NaN-filled buffer:
    "c" contiguous, "pad1" / "padw" leading dimension 1 / W elements longer than needed (a [:, :k] subview),
    "off1" contiguous but starting one element into the buffer (misaligned for 16-byte loads)."""
    rows, k = a.shape
    pad = {"c": 0, "pad1": 1, "padw": _vw(a.dtype), "off1": 0}[shape]
    off = 1 if shape == "off1" else 0
    ld = (k if rowmajor else rows) + pad
    stride = (ld, 1) if rowmajor else (1, ld)
    buf = torch.full(((rows if rowmajor else k) * ld + off,), float("nan"), dtype=TORCH[a.dtype.type], device=dev)
    view = torch.as_strided(buf, (rows, k), stride, off)
    view.copy_(torch.from_numpy(a).to(dev))
    return view, buf


def assert_padding_untouched(view, buf):
    mask = torch.ones(buf.numel(), dtype=torch.bool)
    torch.as_strided(mask, view.shape, view.stride(), view.storage_offset()).fill_(False)
    rest = buf.cpu()[mask]
    assert bool(torch.isnan(rest).all()), "the kernel wrote outside the operand's view"


def host(t):
    return np.array(t.cpu().numpy(), copy=True)


def rm_ld(t):
    """(row-major?, leading dimension) as sparse.spmv passes them: a single column counts as LayoutRight."""
    if t.shape[1] == 1 or t.stride(1) == 1:
        return True, max(t.stride(0), 1)
    return False, t.stride(1)


def expected_kernel(k, X, Y, plan=True):
    """The dispatch rule of spmm_impl (spmm.cu) for mode N with the default kernel."""
    xrm, ldx = rm_ld(X)
    yrm, ldy = rm_ld(Y)
    W = 16 // X.element_size()
    if xrm and yrm:
        vec = k % W == 0 and ldx % W == 0 and ldy % W == 0 and (X.data_ptr() | Y.data_ptr()) % 16 == 0
        return "spmm_items_vec" if vec else "spmm_items"
    return "spmm_relayout+items" if k >= 4 else "spmm_general"


def run(h, mode, A, dev, X, Y0, alpha, beta, xrm, yrm, xshape="c", yshape="c"):
    """One call; returns (Y on the host, X view, Y view).  beta == 0: every 7th row of Y starts as NaN."""
    from kokkos_kernels_b200 import sparse as sp

    y_in = Y0.copy()
    if beta == 0.0:
        y_in[::7] = np.nan
    Xv, Xb = operand(dev, X, xrm, xshape)
    Yv, Yb = operand(dev, y_in, yrm, yshape)
    sp.spmv(h, mode, alpha, A, Xv, beta, Yv)
    torch.cuda.synchronize()
    assert_padding_untouched(Xv, Xb)
    assert_padding_untouched(Yv, Yb)
    return host(Yv), Xv, Yv


# ---------------------------------------------------------------------------------------------------------------------
# 2. dispatch matrix: every k on one handle, every layout, contiguous / padded / misaligned operands
# ---------------------------------------------------------------------------------------------------------------------
SHAPES = [("c", "c"), ("pad1", "c"), ("c", "pad1"), ("padw", "padw"), ("off1", "c"), ("c", "off1")]


@pytest.mark.parametrize("shapes", SHAPES, ids=["-".join(s) for s in SHAPES])
@pytest.mark.parametrize("layout", list(LAYOUTS))
@pytest.mark.parametrize("dtype", DTYPES, ids=["f32", "f64"])
def test_dispatch_matrix(cuda, dtype, layout, shapes):
    from kokkos_kernels_b200 import sparse as sp

    xrm, yrm = LAYOUTS[layout]
    xs, ys = shapes
    A = _device_matrix("dispatch", dtype, cuda)
    rp, ci, v, n = dispatch_matrix(dtype)
    m = len(rp) - 1
    h = sp.SPMVHandle()  # one handle for the whole k loop: partial buffer and relayout scratch grow and are reused
    for i, k in enumerate(K_ORDER):
        alpha, beta = COEFFS[i % len(COEFFS)]
        X, Y0 = inputs(dtype, k, n, m, 1)
        Y, Xv, Yv = run(h, "N", A, cuda, X, Y0, alpha, beta, xrm, yrm, xs, ys)
        want = expected_kernel(k, Xv, Yv)
        assert h.last_kernel() == want, (k, h.last_kernel(), want)
        spmm_ref.check(Y, reference("dispatch", dtype, k, "N", alpha, beta), f"N k={k} {layout} {shapes}")
        if k in K_TRANS:
            for mode in ("T", "H"):
                Xt, Yt0 = inputs(dtype, k, m, n, 2)
                Yt, _, _ = run(h, mode, A, cuda, Xt, Yt0, alpha, beta, xrm, yrm, xs, ys)
                assert h.last_kernel() == "spmm_transpose", (k, mode, h.last_kernel())
                spmm_ref.check(Yt, reference("dispatch", dtype, k, "T", alpha, beta), f"{mode} k={k} {layout} {shapes}")


@pytest.mark.parametrize("layout", list(LAYOUTS))
@pytest.mark.parametrize("dtype", DTYPES, ids=["f32", "f64"])
def test_null_plan(cuda, dtype, layout):
    """plan = NULL through the C ABI: row-major operands run spmm_rowmajor_kernel, any LayoutLeft operand
    spmm_general_kernel (there is no last_kernel without a plan; the result is what is checked)."""
    import kokkos_kernels_b200 as kk
    from kokkos_kernels_b200 import sparse as sp

    xrm, yrm = LAYOUTS[layout]
    A = _device_matrix("dispatch", dtype, cuda)
    rp, ci, v, n = dispatch_matrix(dtype)
    m = len(rp) - 1
    lib = kk._lib.sparse()
    fn = lib.b200sp_spmm_f64_i32 if dtype == np.float64 else lib.b200sp_spmm_f32_i32
    for i, k in enumerate((1, 3, 16, 33, 129)):
        alpha, beta = COEFFS[i % len(COEFFS)]
        X, Y0 = inputs(dtype, k, n, m, 1)
        y_in = Y0.copy()
        if beta == 0.0:
            y_in[::7] = np.nan
        Xv, _ = operand(cuda, X, xrm, "c")
        Yv, _ = operand(cuda, y_in, yrm, "c")
        xr, ldx = rm_ld(Xv)
        yr, ldy = rm_ld(Yv)
        rc = fn(None, sp._stream(), b"N", m, n, len(ci), k, alpha, sp._ptr(A.row_map), sp._ptr(A.entries), sp._ptr(A.values),
                sp._ptr(Xv), ldx, int(xr), beta, sp._ptr(Yv), ldy, int(yr))
        assert rc == 0, lib.b200sp_last_error_string().decode()
        torch.cuda.synchronize()
        spmm_ref.check(host(Yv), reference("dispatch", dtype, k, "N", alpha, beta), f"null plan k={k} {layout}")


@pytest.mark.parametrize("layout", list(LAYOUTS))
@pytest.mark.parametrize("dtype", DTYPES, ids=["f32", "f64"])
def test_alpha_zero_beta_one(cuda, dtype, layout):
    """alpha == 0 leaves beta*Y0 exactly (one rounding, as numpy does it); beta == 0 too gives exact zeros over NaN;
    alpha == 0 and beta == 1 leave Y untouched."""
    from kokkos_kernels_b200 import sparse as sp

    xrm, yrm = LAYOUTS[layout]
    A = _device_matrix("dispatch", dtype, cuda)
    rp, ci, v, n = dispatch_matrix(dtype)
    m = len(rp) - 1
    h = sp.SPMVHandle()
    for k in (1, 5, 16, 33):
        X, Y0 = inputs(dtype, k, n, m, 1)
        for beta in (2.5, 1.0, 0.0, -0.75):
            Y, _, _ = run(h, "N", A, cuda, X, Y0, 0.0, beta, xrm, yrm, "pad1", "pad1")
            want = np.zeros_like(Y0) if beta == 0.0 else (dtype(beta) * Y0 if beta != 1.0 else Y0)
            assert np.array_equal(Y, want), (k, beta)


# ---------------------------------------------------------------------------------------------------------------------
# 3. item-analysis boundaries
# ---------------------------------------------------------------------------------------------------------------------
def _pieces(rp, lmax):
    lens = np.diff(rp)
    return np.where(lens <= lmax, 1, (lens + lmax - 1) // lmax)


def test_boundary_matrix_shape():
    """The boundary matrix has what the item analysis must get right: every pinned length, and rows for both reduce
    kernels at the default LMAX (2..64 pieces: a warp per row; more: a CTA per row)."""
    rp, ci, v, n = boundary_matrix(np.float32)
    lens = np.diff(rp)
    for L in (0, 1, 3, 4, 5, 7, 8, 9, 63, 64, 65, 128, 129, 64 * 64, 64 * 64 + 1):
        assert (lens == L).any(), L
    assert lens[0] == 0 and lens[-1] == 0 and lens.max() >= 5000
    p = _pieces(rp, MMI_LMAX)
    assert ((p >= 2) & (p <= MMI_LONG_PIECES)).any() and (p > MMI_LONG_PIECES).any()
    assert p[lens == 64 * 64][0] == MMI_LONG_PIECES and p[lens == 64 * 64 + 1][0] == MMI_LONG_PIECES + 1
    rows = np.repeat(np.arange(len(lens)), lens)
    assert (np.diff(ci)[np.diff(rows) == 0] < 0).any(), "columns must be unsorted somewhere"
    p = _pieces(*dispatch_matrix(np.float32)[:1], MMI_LMAX)
    assert ((p >= 2) & (p <= MMI_LONG_PIECES)).any() and (p > MMI_LONG_PIECES).any()


@pytest.mark.parametrize("dtype", DTYPES, ids=["f32", "f64"])
def test_item_boundaries(cuda, dtype):
    from kokkos_kernels_b200 import sparse as sp

    A = _device_matrix("boundary", dtype, cuda)
    rp, ci, v, n = boundary_matrix(dtype)
    m = len(rp) - 1
    h = sp.SPMVHandle()
    for i, k in enumerate((16, 1, 5, 8, 33, 129, 200)):
        alpha, beta = COEFFS[i % len(COEFFS)]
        X, Y0 = inputs(dtype, k, n, m, 1)
        Y, Xv, Yv = run(h, "N", A, cuda, X, Y0, alpha, beta, True, True)
        assert h.last_kernel() == expected_kernel(k, Xv, Yv), (k, h.last_kernel())
        spmm_ref.check(Y, reference("boundary", dtype, k, "N", alpha, beta), f"k={k}")


# ---------------------------------------------------------------------------------------------------------------------
# 4. every kernel switch
# ---------------------------------------------------------------------------------------------------------------------
# name, environment, deterministic rows: "all", "short" (rows of one tile segment: the tile kernel's rows of more than
# TILE_SEG entries are several segments added with atomics) or "none" (the split kernel adds rows cut by its chunks with
# atomics: no fixed order)
SWITCHES = [
    ("items", {"B200SP_SPMM_KERNEL": "items"}, "all"),
    ("tile", {"B200SP_SPMM_KERNEL": "tile"}, "short"),
    ("tilev", {"B200SP_SPMM_KERNEL": "tilev"}, "short"),
    ("tilev-segvec", {"B200SP_SPMM_KERNEL": "tilev", "B200SP_SPMM_SEG": "vec"}, "short"),
    ("tilev-lmax64", {"B200SP_SPMM_KERNEL": "tilev", "B200SP_SPMM_LMAX": "64"}, "short"),
    ("tilev-cfg1", {"B200SP_SPMM_KERNEL": "tilev", "B200SP_SPMM_CFG": "1"}, "short"),
    ("tilev-cfg2", {"B200SP_SPMM_KERNEL": "tilev", "B200SP_SPMM_CFG": "2"}, "short"),
    ("tilev-cfg3", {"B200SP_SPMM_KERNEL": "tilev", "B200SP_SPMM_CFG": "3"}, "short"),
    ("split", {"B200SP_SPMM_KERNEL": "split"}, "none"),
    ("split-vec", {"B200SP_SPMM_KERNEL": "split", "B200SP_SPMM_VEC": "1"}, "none"),
    ("row", {"B200SP_SPMM_KERNEL": "row"}, "all"),
]
SWITCH_ENV = ("B200SP_SPMM_KERNEL", "B200SP_SPMM_SEG", "B200SP_SPMM_LMAX", "B200SP_SPMM_CFG", "B200SP_SPMM_VEC",
              "B200SP_SPMM_ITEM_LMAX")
# every lane count of the scalar (k 1..33) and 16-byte (k % W == 0) instantiations, one and several strips
K_SWITCH = (16, 1, 2, 3, 4, 8, 32, 33, 64, 128, 200)


def _switch_kernel(name, k, W):
    vec = k % W == 0
    if name == "items":
        return "spmm_items_vec" if vec else "spmm_items"
    if name == "tile":
        return "spmm_tile"
    if name.startswith("tilev"):
        return "spmm_tile_vec" if vec else "spmm_tile"
    if name.startswith("split"):
        return "spmm_split"
    return "spmm_rowmajor"


@pytest.mark.parametrize("name,env,det", SWITCHES, ids=[s[0] for s in SWITCHES])
@pytest.mark.parametrize("dtype", DTYPES, ids=["f32", "f64"])
def test_kernel_switches(cuda, monkeypatch, dtype, name, env, det):
    from kokkos_kernels_b200 import sparse as sp

    for e in SWITCH_ENV:
        monkeypatch.delenv(e, raising=False)
    for e, val in env.items():
        monkeypatch.setenv(e, val)
    A = _device_matrix("boundary", dtype, cuda)
    rp, ci, v, n = boundary_matrix(dtype)
    m = len(rp) - 1
    lens = np.diff(rp)
    h = sp.SPMVHandle()
    for i, k in enumerate(K_SWITCH):
        alpha, beta = COEFFS[i % len(COEFFS)]
        X, Y0 = inputs(dtype, k, n, m, 1)
        ref = reference("boundary", dtype, k, "N", alpha, beta)
        outs = []
        for _ in range(2):
            Y, _, _ = run(h, "N", A, cuda, X, Y0, alpha, beta, True, True)
            assert h.last_kernel() == _switch_kernel(name, k, _vw(dtype)), (name, k, h.last_kernel())
            spmm_ref.check(Y, ref, f"{name} k={k}")
            outs.append(Y)
        rows = {"all": lens >= 0, "short": lens <= TILE_SEG, "none": lens < 0}[det]
        assert np.array_equal(outs[0][rows], outs[1][rows], equal_nan=True), f"{name} k={k}: two calls differ"


@pytest.mark.parametrize("dtype", DTYPES, ids=["f32", "f64"])
def test_item_lmax_reanalyses(cuda, monkeypatch, dtype):
    """B200SP_SPMM_ITEM_LMAX changed between calls on one handle: the plan's item list is rebuilt (two analysis launches,
    mmi_count + mmi_fill, more than a repeated call makes) and the result is right for every value."""
    import kokkos_kernels_b200 as kk
    from kokkos_kernels_b200 import sparse as sp

    for e in SWITCH_ENV:
        monkeypatch.delenv(e, raising=False)
    lib = kk._lib.sparse()
    A = _device_matrix("boundary", dtype, cuda)
    rp, ci, v, n = boundary_matrix(dtype)
    m = len(rp) - 1
    h = sp.SPMVHandle()
    k = 33
    X, Y0 = inputs(dtype, k, n, m, 1)
    ref = reference("boundary", dtype, k, "N", 1.5, -0.5)
    for lmax in (16, 64, 256, 16):
        monkeypatch.setenv("B200SP_SPMM_ITEM_LMAX", str(lmax))
        counts = []
        for _ in range(2):
            c0 = lib.b200sp_launch_count()
            Y, _, _ = run(h, "N", A, cuda, X, Y0, 1.5, -0.5, True, True)
            counts.append(lib.b200sp_launch_count() - c0)
            assert h.last_kernel() == "spmm_items"
            spmm_ref.check(Y, ref, f"ITEM_LMAX={lmax}")
        assert counts[0] == counts[1] + 2, (lmax, counts)


_COOP_CASES = [(dt, k) for dt in ("f32", "f64") for k in (5, 16, 33, 129)]

_COOP_CHILD = r"""
import os, sys
sys.path[:0] = [sys.argv[2], os.path.dirname(sys.argv[2])]
import numpy as np, torch
import test_gpu_spmm_kernels as t
if os.environ.get("B200SP_TEST_EMULATED") == "1":
    import conftest
    dev = conftest._emulated_device()
else:
    dev = torch.device("cuda:0")
np.savez(sys.argv[1], **t.coop_outputs(dev))
"""


def coop_outputs(dev):
    """Y of the item kernel for the cases of test_item_coop_bit_identical (run in a child process: the
    B200SP_SPMM_ITEM_COOP switch is read once per process)."""
    from kokkos_kernels_b200 import sparse as sp

    out = {}
    for name, k in _COOP_CASES:
        dtype = np.float32 if name == "f32" else np.float64
        A = _device_matrix("boundary", dtype, dev)
        rp, ci, v, n = boundary_matrix(dtype)
        X, Y0 = inputs(dtype, k, n, len(rp) - 1, 1)
        h = sp.SPMVHandle()
        Y, _, _ = run(h, "N", A, dev, X, Y0, 1.5, -0.5, True, True)
        out[f"{name}_{k}"] = Y
        out[f"{name}_{k}_kernel"] = np.array(h.last_kernel())
    return out


def test_item_coop_bit_identical(cuda, tmp_path):
    """DESIGN.md 4.2: the cooperative item kernel (batches of 4 or 8) adds in the order of the first item kernel, so
    B200SP_SPMM_ITEM_COOP=0 / 4 / 8 give bit-identical Y.  One short child process per value."""
    outs = {}
    env_base = {key: val for key, val in os.environ.items() if key not in SWITCH_ENV + ("B200SP_SPMM_ITEM_COOP",)}
    flags = [f for f, on in (("-s", sys.flags.no_user_site), ("-E", sys.flags.ignore_environment)) if on]
    for coop in ("0", "4", "8"):
        path = str(tmp_path / f"coop{coop}.npz")
        env = dict(env_base, B200SP_SPMM_ITEM_COOP=coop)
        r = subprocess.run([sys.executable, *flags, "-c", _COOP_CHILD, path, HERE], env=env, cwd=os.path.dirname(HERE),
                           capture_output=True, text=True, timeout=900)
        assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
        with np.load(path) as z:
            outs[coop] = {key: z[key] for key in z.files}
    for name, k in _COOP_CASES:
        dtype = np.float32 if name == "f32" else np.float64
        key = f"{name}_{k}"
        spmm_ref.check(outs["4"][key], reference("boundary", dtype, k, "N", 1.5, -0.5), f"coop {key}")
        for coop in ("0", "8"):
            assert str(outs[coop][key + "_kernel"]) == str(outs["4"][key + "_kernel"])
            assert np.array_equal(outs[coop][key], outs["4"][key]), f"ITEM_COOP={coop} differs from 4 at {key}"
