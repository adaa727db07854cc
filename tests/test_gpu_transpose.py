"""Transposed product y = alpha*A^T*x (+ beta*y) on the B200 (csxb_spmv_t and everything built on it): against
scipy's A.T @ x within 1e-12 (componentwise against |A|^T |x|), bit-identical across calls and paths."""
import ctypes as C
import os

import numpy as np
import pytest
import scipy.sparse as sp

from tests.conftest import GOLDEN
from tests.matrices import _csr_from_coo, poisson2d, random_structured, rmat, stencil27, sym_block_banded

pytestmark = pytest.mark.gpu
TOL = 1e-12


def _torch():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch


def _ref(rp, ci, va, n, m, x):
    A = sp.csr_matrix((va, ci, rp), shape=(n, m))
    return A.T @ x, abs(A).T @ np.abs(x)


def _close(y, ref, bound):
    return np.all(np.abs(y - ref) <= TOL * (bound + 1e-300))


def check_t(rp, ci, va, n, m, opts, seed=0, free_host=False):
    """Device and host-buffer transposed products, mult and kernel semantics; returns the matrix."""
    torch = _torch()
    from sparsex_b200 import CsxMatrix
    rng = np.random.default_rng(seed)
    x = rng.uniform(-1, 1, n)
    ref, bound = _ref(rp, ci, va, n, m, x)
    A = CsxMatrix.tune_csr(rp, ci, va, n, m, opts).upload(0, free_host=free_host)
    dx = torch.from_numpy(x).cuda()
    dy = torch.full((m,), float("nan"), dtype=torch.float64, device="cuda")
    A.spmv_t(0.5, dx, dy)
    y1 = dy.cpu().numpy()
    assert _close(y1, 0.5 * ref, 0.5 * bound), (opts, A.transpose_info())
    A.spmv_t(0.5, dx, dy)
    assert np.array_equal(dy.cpu().numpy(), y1), "two calls differ"
    yh = np.full(m, np.nan)
    A.spmv_t_host(0.5, x, yh)
    assert np.array_equal(yh, y1), "host-buffer and device products differ"
    y0 = rng.uniform(-1, 1, m)
    dy = torch.from_numpy(y0.copy()).cuda()
    A.spmv_t(-2.0, dx, dy, beta=0.25, overwrite=False)
    assert _close(dy.cpu().numpy(), -2.0 * ref + 0.25 * y0, 2.0 * bound + 0.25 * np.abs(y0)), opts
    yh = y0.copy()
    A.spmv_t_host(-2.0, x, yh, beta=0.25, overwrite=False)
    assert np.array_equal(yh, dy.cpu().numpy())
    return A


def test_transpose_config_kinds():
    """The kinds the benchmark configs encode to, at GPU sizes; stencils keep the forward tables' shape."""
    rp, ci, va, n = poisson2d(1100)            # > 2^20 rows: four rows per thread, diagonal instantiation
    A = check_t(rp, ci, va, n, n, {})
    info = A.transpose_info()
    assert info["launches"] == 1 and info["heavy_cols"] == 0, info
    rp, ci, va, n = stencil27(48)
    check_t(rp, ci, va, n, n, {})
    for nt in (1, 4):
        check_t(rp, ci, va, n, n, {"spx.preproc.xform": "br,bc", "spx.rt.nr_threads": nt})
    rp, ci, va, n = sym_block_banded(20000, b=64)
    check_t(rp, ci, va, n, n, {})
    rp, ci, va, n = rmat(16)
    A = check_t(rp, ci, va, n, n, {"spx.preproc.xform": "none"})
    assert A.transpose_info()["heavy_cols"] > 0


@pytest.mark.parametrize("seed", range(2))
def test_transpose_rectangular_all_xforms(seed):
    from tests.test_gpu_parity import XFORMS
    rng = np.random.default_rng(300 + seed)
    n, m = int(rng.integers(2000, 6000)), int(rng.integers(2000, 6000))
    rp, ci, va = random_structured(rng, n, m)
    for xf in XFORMS:
        for extra in ({}, {"spx.rt.nr_threads": 3}, {"spx.matrix.full_colind": "true"}):
            check_t(rp, ci, va, n, m, dict({"spx.preproc.xform": xf, "spx.preproc.sampling": "none"}, **extra))


@pytest.mark.parametrize("name", ["demopatt", "test", "test2", "test3"])
def test_transpose_reference_fixtures(name):
    from oracle.pyoracle import OracleMatrix
    M = OracleMatrix.from_mmf(os.path.join(GOLDEN, "matrices", name + ".mtx.sorted"))
    rp, ci, va = M.csr()
    for xf in ("none", "all", "h,d", "bc,v,ad"):
        check_t(rp, ci, va, M.nrows, M.ncols, {"spx.preproc.xform": xf})


def test_transpose_decode_matches_forward():
    from sparsex_b200 import CsxMatrix
    _torch()
    rng = np.random.default_rng(5)
    rp, ci, va = random_structured(rng, 3000, 2500)
    for xf in ("all", "none", "br,bc", "v,ad"):
        A = CsxMatrix.tune_csr(rp, ci, va, 3000, 2500, {"spx.preproc.xform": xf, "spx.rt.nr_threads": 3}).upload(0)
        fr = np.concatenate([A.decode_coords(p)[0] for p in range(A.nparts)])
        fc = np.concatenate([A.decode_coords(p)[1] for p in range(A.nparts)])
        r, c = A.decode_coords_t()
        assert np.array_equal(r, fr) and np.array_equal(c, fc), xf
        A.prepare_transpose()
        r2, c2 = A.decode_coords_t()
        assert np.array_equal(r2, r) and np.array_equal(c2, c)


def test_transpose_csx_sym_is_the_forward_product():
    torch = _torch()
    from sparsex_b200 import CsxMatrix
    rp, ci, va, n = sym_block_banded(5000, b=40)
    x = torch.from_numpy(np.random.default_rng(1).uniform(-1, 1, n)).cuda()
    for nt in (1, 3):
        A = CsxMatrix.tune_csr(rp, ci, va, n, n, {"spx.matrix.symmetric": "true", "spx.rt.nr_threads": nt}).upload(0)
        y1 = torch.empty(n, dtype=torch.float64, device="cuda")
        y2 = torch.empty(n, dtype=torch.float64, device="cuda")
        A.spmv(0.5, x, y1)
        A.spmv_t(0.5, x, y2)
        assert torch.equal(y1, y2)


def test_transpose_sees_set_entry_save_restore_free_host(tmp_path):
    torch = _torch()
    from sparsex_b200 import CsxMatrix
    rng = np.random.default_rng(8)
    n, m = 4000, 3000
    rp, ci, va = random_structured(rng, n, m)
    A = check_t(rp, ci, va, n, m, {"spx.preproc.xform": "all"}, free_host=True)
    k = int(rp[1234])
    r = int(np.searchsorted(rp, k, side="right") - 1)
    assert A.set_entry(r, int(ci[k]), 7.5)
    va2 = va.copy()
    va2[k] = 7.5
    x = rng.uniform(-1, 1, n)
    ref, bound = _ref(rp, ci, va2, n, m, x)
    y = np.empty(m)
    A.spmv_t_host(1.0, x, y)
    assert _close(y, ref, bound)
    path = str(tmp_path / "t.csxb")
    A.save(path)
    B = CsxMatrix.load(path).upload(0)
    y2 = torch.empty(m, dtype=torch.float64, device="cuda")
    B.spmv_t(1.0, torch.from_numpy(x).cuda(), y2)
    assert np.array_equal(y2.cpu().numpy(), y)


def test_transpose_partial_handles_sum_to_the_whole():
    torch = _torch()
    from sparsex_b200 import CsxMatrix
    rng = np.random.default_rng(9)
    n, m = 6000, 5000
    rp, ci, va = random_structured(rng, n, m)
    x = rng.uniform(-1, 1, n)
    ref, bound = _ref(rp, ci, va, n, m, x)
    opts = {"spx.preproc.xform": "all", "spx.rt.nr_threads": 4}
    total = np.zeros(m)
    for p in range(4):
        A = CsxMatrix.tune_csr(rp, ci, va, n, m, opts, part_lo=p, part_hi=p + 1).upload(0).prepare_transpose()
        info = A.transpose_info()
        lo, hi = info["col_lo"], info["col_hi"]
        y = torch.full((m,), 123.0, dtype=torch.float64, device="cuda")
        A.spmv_t(1.0, torch.from_numpy(x).cuda(), y)
        yn = y.cpu().numpy()
        assert np.all(yn[:lo] == 123.0) and np.all(yn[hi:] == 123.0)   # columns outside the window untouched
        total[lo:hi] += yn[lo:hi]
    assert _close(total, ref, 4 * bound)


def test_transpose_groups():
    torch = _torch()
    from sparsex_b200 import CsxMatrix, DeviceGroup
    rng = np.random.default_rng(10)
    n, m = 7000, 5000
    rp, ci, va = random_structured(rng, n, m)
    x = rng.uniform(-1, 1, n)
    ref, bound = _ref(rp, ci, va, n, m, x)
    opts = {"spx.preproc.xform": "all", "spx.rt.nr_threads": 3}
    single = np.empty(m)
    CsxMatrix.tune_csr(rp, ci, va, n, m, opts).upload(0).spmv_t_host(1.0, x, single)
    layouts = [[0, 0, 0]]
    if torch.cuda.device_count() > 1:
        layouts.append([0, 1])
    for devs in layouts:
        G = DeviceGroup(CsxMatrix.tune_csr(rp, ci, va, n, m, opts), devs)
        y1, y2 = np.full(m, np.nan), np.full(m, np.nan)
        G.spmv_t(1.0, x, y1)
        G.spmv_t(1.0, x, y2)
        assert np.array_equal(y1, y2) and _close(y1, ref, bound) and _close(y1, single, 2 * bound), devs
        y0 = rng.uniform(-1, 1, m)
        dy = torch.from_numpy(y0.copy()).cuda()
        G.spmv_t(0.5, torch.from_numpy(x).cuda(), dy, beta=-1.0, overwrite=False)
        assert _close(dy.cpu().numpy(), 0.5 * ref - y0, 0.5 * bound + np.abs(y0)), devs
        G.close()
    # CSX-Sym group: the forward product
    rp, ci, va, n = sym_block_banded(3000, b=30)
    xs = rng.uniform(-1, 1, n)
    o = {"spx.matrix.symmetric": "true", "spx.rt.nr_threads": 3}
    G = DeviceGroup(CsxMatrix.tune_csr(rp, ci, va, n, n, o), [0, 0, 0])
    a, b = np.empty(n), np.empty(n)
    G.spmv(1.0, xs, a)
    G.spmv_t(1.0, xs, b)
    assert np.array_equal(a, b)


def test_transpose_heavy_column_rmat():
    """R-MAT with one added dense column: the heavy-column segments are exact and deterministic."""
    torch = _torch()
    from sparsex_b200 import CsxMatrix
    rp, ci, va, n = rmat(15)
    rows = np.repeat(np.arange(n), np.diff(rp))
    extra = np.arange(0, n, 3)
    r = np.concatenate([rows, extra])
    c = np.concatenate([ci, np.full(extra.size, 4321)])
    rc, idx = np.unique(np.stack([r, c], 1), axis=0, return_index=True)
    v = np.concatenate([va, np.random.default_rng(2).standard_normal(extra.size)])[idx]
    rp, ci, va = _csr_from_coo(rc[:, 0], rc[:, 1], v, n, n)
    A = check_t(rp, ci, va, n, n, {"spx.preproc.xform": "none", "spx.rt.nr_threads": 2})
    info = A.transpose_info()
    assert info["heavy_cols"] > 0 and info["segments"] > info["heavy_cols"] and info["launches"] == 3, info
    x = torch.from_numpy(np.random.default_rng(4).uniform(-1, 1, n)).cuda()
    ys = []
    for _ in range(3):
        y = torch.empty(n, dtype=torch.float64, device="cuda")
        A.spmv_t(1.0, x, y)
        ys.append(y)
    assert torch.equal(ys[0], ys[1]) and torch.equal(ys[0], ys[2])


def test_spx_matvec_trans():
    _torch()
    from sparsex_b200 import load_spx_api, SpxApi
    from tests.test_cpu_api_errors import ERR_DIM, Recorder
    from tests.test_cpu_rcm import scrambled_banded, csr
    api = load_spx_api()
    api.spx_init()
    rng = np.random.default_rng(12)
    n, m = 900, 700
    rp, ci, va = random_structured(rng, n, m)
    api.spx_option_set(b"spx.preproc.sampling", b"none")
    api.spx_option_set(b"spx.rt.nr_threads", b"2")
    api.spx_option_set(b"spx.matrix.symmetric", b"false")
    inp = api.spx_input_load_csr(rp.ctypes.data, ci.ctypes.data, va.ctypes.data, n, m)
    M = api.spx_mat_tune(inp)
    assert M
    xs = rng.uniform(-1, 1, n)
    ref, bound = _ref(rp, ci, va, n, m, xs)
    parts = api.spx_mat_get_partition(M)
    x, y = api.spx_vec_create(n, parts), api.spx_vec_create(m, parts)   # library vectors
    SpxApi.as_numpy(x)[:] = xs
    assert api.spx_matvec_mult_trans(0.5, M, x, y) == 0
    api.spx_device_synchronize()
    assert _close(SpxApi.as_numpy(y), 0.5 * ref, 0.5 * bound)
    y0 = SpxApi.as_numpy(y).copy()
    assert api.spx_matvec_kernel_trans(2.0, M, x, 0.5, y) == 0
    api.spx_device_synchronize()
    assert _close(SpxApi.as_numpy(y), 2.0 * ref + 0.5 * y0, 2.0 * bound + 0.5 * np.abs(y0))
    xb, yb = xs.copy(), np.full(m, np.nan)                           # buffer vectors
    tuned = C.c_void_p()
    xv = api.spx_vec_create_from_buff(xb.ctypes.data, C.byref(tuned), n, None, 43)
    yv = api.spx_vec_create_from_buff(yb.ctypes.data, C.byref(tuned), m, None, 43)
    assert api.spx_matvec_mult_trans(0.5, M, xv, yv) == 0
    assert _close(yb, 0.5 * ref, 0.5 * bound)
    rec = Recorder(api)
    try:                                                             # x with ncols entries: wrong for A^T
        assert api.spx_matvec_mult_trans(1.0, M, y, x) != 0
        assert api.spx_matvec_kernel_trans(1.0, M, y, 1.0, x) != 0
        assert [c[0] for c in rec.take()] == [ERR_DIM, ERR_DIM]
    finally:
        rec.close()
    for h in (x, y, xv, yv):
        api.spx_vec_destroy(h)
    api.spx_partition_destroy(parts)
    api.spx_mat_destroy(M)
    api.spx_input_destroy(inp)
    # SPX_MAT_REORDER: the permuted numbering, as spx_matvec_mult
    n = 5000
    a = scrambled_banded(n, 6, 31)
    rp, ci, va = csr(a)
    api.spx_option_set(b"spx.rt.nr_threads", b"2")
    inp = api.spx_input_load_csr(rp.ctypes.data, ci.ctypes.data, va.ctypes.data, n, n)
    M = api.spx_mat_tune(inp, 42)
    pp = api.spx_mat_get_perm(M)
    perm = np.ctypeslib.as_array(pp, shape=(n,)).copy()
    parts = api.spx_mat_get_partition(M)
    x, y = api.spx_vec_create(n, parts), api.spx_vec_create(n, parts)
    xs = rng.uniform(-1, 1, n)
    SpxApi.as_numpy(x)[:] = xs
    api.spx_vec_reorder(x, pp)
    assert api.spx_matvec_mult_trans(1.0, M, x, y) == 0
    api.spx_device_synchronize()
    api.spx_vec_inv_reorder(y, pp)
    ref, bound = _ref(rp, ci, va, n, n, xs)
    assert _close(SpxApi.as_numpy(y), ref, bound)
    for h in (x, y):
        api.spx_vec_destroy(h)
    api.spx_partition_destroy(parts)
    api.spx_mat_destroy(M)
    api.spx_input_destroy(inp)
    api.spx_option_set(b"spx.rt.nr_threads", b"1")
