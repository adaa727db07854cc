"""Transposed product y = alpha*A^T*x + beta*y on the CPU: the transposed layout (gpu_layout.cpp) is executed through
the text of gather_kernel.cuh (gather over the transposed tables, heavy-column segments) on the fibre emulation of the
warp intrinsics (tests/emul/trans_emul.cpp, built by tests/emul/trans.mk), with the instantiation csxb_spmv_t picks.  y within 1e-12 of scipy's
A.T @ x, componentwise against |A|^T |x|; the coordinates the transposed tables gather every value at equal the
forward decode of the emulated engine, bit for bit.  Test infrastructure: the product has no CPU path."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest
import scipy.sparse as sp

from tests.emul.run_emul import emul_spmv
from tests.matrices import _csr_from_coo, poisson2d, random_structured, rmat, stencil27, sym_block_banded

HERE = os.path.join(os.path.dirname(os.path.abspath(__file__)), "emul")
ROOT = os.path.dirname(os.path.dirname(HERE))
TOL = 1e-12
XFORMS = ["none", "h", "v", "d", "ad", "br", "bc", "all", "h,d", "bc,v,ad", "br3{2,3},h{1}", "d{1},ad{2},v{1}"]
_LIB = None


def _lib():
    global _LIB
    if _LIB is None:
        subprocess.check_call(["make", "-s", "-C", os.path.join(ROOT, "sparsex_b200", "csrc"), "encoder.o", "gpu_layout.o", "mmf.o"])
        subprocess.check_call(["make", "-s", "-C", HERE, "-f", "trans.mk"], stderr=subprocess.DEVNULL)
        L = C.CDLL(os.path.join(HERE, "libtrans_emul.so"))
        vp, i64 = C.c_void_p, C.c_int64
        L.emul_spmv_t.restype = C.c_int
        L.emul_spmv_t.argtypes = [vp, vp, vp, i64, i64, C.c_char_p, C.c_double, vp, C.c_double, vp, C.c_int, vp, vp, vp,
                                  C.c_char_p, C.c_size_t]
        _LIB = L
    return _LIB


def emul_spmv_t(rp, ci, va, n, m, opts, alpha, x, beta=0.0, y=None, overwrite=True):
    rp, ci = np.ascontiguousarray(rp, np.int32), np.ascontiguousarray(ci, np.int32)
    va, x = np.ascontiguousarray(va, np.float64), np.ascontiguousarray(x, np.float64)
    y = np.full(m, np.nan) if y is None else np.array(y, np.float64)
    nnz = int(rp[-1])
    dr, dc = np.full(nnz + 1, -2, np.int32), np.full(nnz + 1, -2, np.int32)
    stats = np.zeros(16, np.int64)
    err = C.create_string_buffer(1024)
    o = ";".join("%s=%s" % kv for kv in (opts or {}).items()).encode()
    rc = _lib().emul_spmv_t(rp.ctypes.data, ci.ctypes.data, va.ctypes.data, n, m, o, alpha, x.ctypes.data, beta,
                            y.ctypes.data, int(overwrite), dr.ctypes.data, dc.ctypes.data, stats.ctypes.data, err, 1024)
    if rc != 0:
        raise RuntimeError(err.value.decode())
    return y, dr[:nnz], dc[:nnz], stats


def _check(rp, ci, va, n, m, opts, seed=1):
    rng = np.random.default_rng(seed)
    x = rng.uniform(-1, 1, n)
    A = sp.csr_matrix((va, ci, rp), shape=(n, m))
    ref, bound = A.T @ x, abs(A).T @ np.abs(x)
    y, dr, dc, st = emul_spmv_t(rp, ci, va, n, m, opts, 0.5, x)   # y starts as NaN: every column is written
    assert np.all(np.abs(y - 0.5 * ref) <= TOL * (0.5 * bound + 1e-300)), (opts, st)
    y0 = rng.uniform(-1, 1, m)
    y2, _, _, _ = emul_spmv_t(rp, ci, va, n, m, opts, -1.5, x, beta=0.25, y=y0, overwrite=False)
    assert np.all(np.abs(y2 - (-1.5 * ref + 0.25 * y0)) <= TOL * (1.5 * bound + 0.25 * np.abs(y0) + 1e-300)), opts
    # the transposed tables gather every value at the coordinates the forward decode gives it
    _, fr, fc, _ = emul_spmv(rp, ci, va, n, m, opts, 0.5, rng.uniform(-1, 1, m))
    nnz = int(rp[-1])
    assert np.array_equal(dr, fr[:nnz]) and np.array_equal(dc, fc[:nnz]), opts
    return st


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_transpose_xforms_rectangular(seed):
    """Ragged rectangular matrices with every unit kind, every xform set, 1-4 partitions, full_colind."""
    rng = np.random.default_rng(seed)
    n, m = int(rng.integers(50, 400)), int(rng.integers(50, 400))
    rp, ci, va = random_structured(rng, n, m)
    for xf in XFORMS:
        for fc in ("false", "true"):
            _check(rp, ci, va, n, m, {"spx.preproc.xform": xf, "spx.matrix.full_colind": fc, "spx.preproc.sampling": "none",
                                      "spx.rt.nr_threads": 1 + seed + (fc == "true")})


def test_transpose_option_grid():
    """The option grid of the forward emulation: slices, rows per thread 1 and 4, empty rows and empty columns."""
    rng = np.random.default_rng(7)
    n, m = 300, 500
    rp, ci, va = random_structured(rng, n, m)
    keep = (ci % 7 != 3)                                   # empty columns
    rows = np.repeat(np.arange(n), np.diff(rp))
    keep &= (rows % 11 != 5)                               # empty rows
    rp, ci, va = _csr_from_coo(rows[keep], ci[keep], va[keep], n, m)
    for xf in ("all", "none", "h", "v", "d,ad", "br,bc"):
        for sl in (0, 4, 32):
            for rpt in (1, 4):
                st = _check(rp, ci, va, n, m, {"spx.preproc.xform": xf, "spx.b200.slice": sl, "spx.b200.rows_per_thread": rpt,
                                              "spx.preproc.sampling": "none", "spx.rt.nr_threads": 3})
                assert st[1] == rpt


def test_transpose_stencils_keep_the_diagonal_instantiation():
    """A diagonal stencil transposes to forward diagonal units: no images, the stride-1 diagonal gather."""
    rp, ci, va, n = poisson2d(40)
    for rpt in (1, 4):
        st = _check(rp, ci, va, n, n, {"spx.preproc.xform": "d", "spx.preproc.sampling": "none", "spx.b200.rows_per_thread": rpt})
        assert st[0] == 0 and st[2] == 1, st
    rp, ci, va, n = stencil27(12)
    st = _check(rp, ci, va, n, n, {"spx.preproc.sampling": "none"})
    assert st[0] == 0 and st[2] == 1, st
    for nt in (1, 4):
        st = _check(rp, ci, va, n, n, {"spx.preproc.xform": "br,bc", "spx.preproc.sampling": "none", "spx.rt.nr_threads": nt})
        assert st[4] > 0, st    # block images in the block tables
    rp, ci, va, n = sym_block_banded(600, b=40)
    _check(rp, ci, va, n, n, {"spx.preproc.sampling": "none", "spx.rt.nr_threads": 3})


def test_transpose_heavy_columns():
    """Columns long enough to be cut into warp segments (and R-MAT): exact, and the same bits twice."""
    rng = np.random.default_rng(3)
    n, m = 3000, 400
    r = rng.integers(0, n, 6000)
    c = rng.integers(0, m, 6000)
    dense = np.arange(0, n, 2)                               # column 17: 1500 entries, column 300: 750
    r = np.concatenate([r, dense, dense[::2]])
    c = np.concatenate([c, np.full(dense.size, 17), np.full(dense[::2].size, 300)])
    rc = np.unique(np.stack([r, c], 1), axis=0)
    rp, ci, va = _csr_from_coo(rc[:, 0], rc[:, 1], rng.standard_normal(rc.shape[0]), n, m)
    for nt in (1, 3):
        opts = {"spx.preproc.xform": "none", "spx.preproc.sampling": "none", "spx.rt.nr_threads": nt}
        st = _check(rp, ci, va, n, m, opts)
        assert st[5] >= 2 and st[6] > st[5], st
        x = rng.uniform(-1, 1, n)
        a = emul_spmv_t(rp, ci, va, n, m, opts, 1.0, x)[0]
        b = emul_spmv_t(rp, ci, va, n, m, opts, 1.0, x)[0]
        assert np.array_equal(a, b)
    rp, ci, va, n = rmat(11)
    st = _check(rp, ci, va, n, n, {"spx.preproc.xform": "none", "spx.rt.nr_threads": 2})
    assert st[5] > 0, st


def test_decode_coords_t_through_the_library_without_a_device():
    """csxb_decode_coords_t builds the transposed tables on the host: the CSR coordinates of every value."""
    from sparsex_b200 import CsxMatrix
    rng = np.random.default_rng(11)
    n, m = 200, 260
    rp, ci, va = random_structured(rng, n, m)
    rows = np.repeat(np.arange(n), np.diff(rp))
    for xf in ("all", "none", "br,bc"):
        A = CsxMatrix.tune_csr(rp, ci, va, n, m, {"spx.preproc.xform": xf, "spx.preproc.sampling": "none", "spx.rt.nr_threads": 2})
        r, c = A.decode_coords_t()
        order = np.lexsort((c, r))
        assert np.array_equal(r[order], rows) and np.array_equal(c[order], ci), xf
