"""GPU parity tests (run with -m gpu on the B200 box).

Every check goes through the C-ABI of libsparsex_b200.so (csxb_* / spx_*) and
compares against the oracle (oracle/: CPU restatement of the reference) on the
same seeded inputs:
  * CSX encoding (ctl, values, id_map, rows_info) bit-exact,
  * decoded (row, column) per value from the device-side traversal bit-exact,
  * y = alpha*A*x (+ beta*y) within 1e-12 relative (componentwise against
    |A||x|, SURVEY.md section 8d) — the tolerance BASELINE.json's north_star states.
"""
import os

import numpy as np
import pytest

from tests.conftest import GOLDEN
from tests.matrices import (poisson2d, random_structured, rmat, stencil27,
                            sym_block_banded)

pytestmark = pytest.mark.gpu
TOL = 1e-12


def _torch():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch


def _abs_bound(rowptr, colind, values, x, n):
    rows = np.repeat(np.arange(n), np.diff(rowptr))
    b = np.zeros(n)
    np.add.at(b, rows, np.abs(values) * np.abs(x[colind]))
    return b


def _csr_spmv(rowptr, colind, values, x, n):
    rows = np.repeat(np.arange(n), np.diff(rowptr))
    y = np.zeros(n)
    np.add.at(y, rows, values * x[colind])
    return y


def check_matrix(rowptr, colind, values, n, m, opts, seed=0, check_decode=True, oracle_spmv=True):
    """Tune with the engine and the oracle, compare encodings, decoded coordinates and products."""
    torch = _torch()
    from oracle.pyoracle import OracleMatrix
    from sparsex_b200 import CsxMatrix

    rng = np.random.default_rng(seed)
    oopts = {k: v for k, v in opts.items() if not k.startswith("spx.b200.")}
    oopts["oracle.undefined_sampling"] = "break"
    O = OracleMatrix.from_csr(rowptr, colind, values, n, m).tune(oopts)
    A = CsxMatrix.tune_csr(rowptr, colind, values, n, m, opts)
    assert A.nparts == len(O.parts)
    for p in range(A.nparts):
        P, Q = A.partition(p), O.parts[p]
        assert np.array_equal(P.ctl, Q.ctl), "ctl differs (%s | %s)" % (P.log, O.log)
        assert np.array_equal(P.values, Q.values)
        assert np.array_equal(P.id_map, Q.id_map)
        assert np.array_equal(P.rows_info, Q.rows_info.astype(np.int64))
    A.upload(0)
    sym = str(opts.get("spx.matrix.symmetric", "false")) == "true"
    if check_decode and not sym:
        for p in range(A.nparts):
            r, c = A.decode_coords(p)
            ro, co = O.decode(p)
            assert np.array_equal(r, ro) and np.array_equal(c, co), "device-decoded coordinates differ"
    x = rng.uniform(-1, 1, m)
    y0 = rng.uniform(-1, 1, n)
    bound = _abs_bound(rowptr, colind, values, x, n) + 1e-300
    dx = torch.from_numpy(x).cuda()
    # spx_matvec_mult semantics
    dy = torch.from_numpy(y0.copy()).cuda()
    A.spmv(0.5, dx, dy, overwrite=True)
    y = dy.cpu().numpy()
    yref = O.spmv(0.5, x) if oracle_spmv else 0.5 * _csr_spmv(rowptr, colind, values, x, n)
    err = np.max(np.abs(y - yref) / (0.5 * bound + np.abs(yref) * 0 + 1e-300))
    assert err <= TOL, "mult: componentwise relative error %.3e (%s)" % (err, O.log)
    # spx_matvec_kernel semantics
    dy = torch.from_numpy(y0.copy()).cuda()
    A.spmv(0.75, dx, dy, beta=-0.3, overwrite=False)
    y = dy.cpu().numpy()
    yref = O.spmv(0.75, x, beta=-0.3, y=y0) if oracle_spmv else 0.75 * _csr_spmv(rowptr, colind, values, x, n) - 0.3 * y0
    err = np.max(np.abs(y - yref) / (0.75 * bound + 0.3 * np.abs(y0) + 1e-300))
    assert err <= TOL, "kernel: componentwise relative error %.3e (%s)" % (err, O.log)
    # host-buffer path (copies inside the call)
    yh = np.zeros(n)
    A.spmv_host(0.5, x, yh)
    yref = O.spmv(0.5, x) if oracle_spmv else 0.5 * _csr_spmv(rowptr, colind, values, x, n)
    assert np.max(np.abs(yh - yref) / (0.5 * bound)) <= TOL
    A.close()
    return O.log


XFORMS = ["none", "h", "v", "d", "ad", "br", "bc", "all", "h,d", "bc,v,ad", "br3{2,3},h{1}", "d{1},ad{2},v{1}"]


@pytest.mark.parametrize("name", ["demopatt", "test", "test2", "test3"])
def test_reference_fixtures(name):
    """The reference's bundled matrices under the option sets of test/scripts/test-sparsex.sh.in."""
    from oracle.pyoracle import OracleMatrix
    M = OracleMatrix.from_mmf(os.path.join(GOLDEN, "matrices", name + ".mtx.sorted"))
    rp, ci, va = M.csr()
    for xf in XFORMS:
        for extra in ({}, {"spx.preproc.sampling": "none"}, {"spx.rt.nr_threads": 2},
                      {"spx.rt.nr_threads": 2, "spx.preproc.sampling.nr_samples": 1, "spx.preproc.sampling.portion": 0.4},
                      {"spx.matrix.full_colind": "true"}):
            o = {"spx.preproc.xform": xf}
            o.update(extra)
            check_matrix(rp, ci, va, M.nrows, M.ncols, o)


@pytest.mark.parametrize("name", ["symmetric", "symmetric-very-sparse"])
def test_reference_symmetric_fixtures(name):
    from oracle.pyoracle import OracleMatrix
    M = OracleMatrix.from_mmf(os.path.join(GOLDEN, "matrices", name + ".mtx.sorted"))
    rp, ci, va = M.csr()
    for xf in XFORMS:
        for extra in ({}, {"spx.preproc.sampling": "none"}, {"spx.rt.nr_threads": 2},
                      {"spx.preproc.sampling.nr_samples": 2, "spx.preproc.sampling.portion": 0.4}):
            for sym in ("true", "false"):
                o = {"spx.preproc.xform": xf, "spx.matrix.symmetric": sym}
                o.update(extra)
                check_matrix(rp, ci, va, M.nrows, M.ncols, o)


@pytest.mark.parametrize("seed", range(6))
def test_random_structured(seed):
    """Ragged random matrices seeded with every substructure kind, all option families."""
    rng = np.random.default_rng(100 + seed)
    for trial in range(4):
        n = int(rng.integers(5, 700))
        sym = trial % 2 == 0
        m = n if sym else int(rng.integers(5, 700))
        rp, ci, va = random_structured(rng, n, m, symmetric=sym)
        for xf in XFORMS:
            extras = [{}, {"spx.preproc.sampling": "none"}, {"spx.rt.nr_threads": int(rng.integers(2, 6))},
                      {"spx.matrix.split_blocks": "false"},
                      {"spx.matrix.min_unit_size": 2, "spx.matrix.max_unit_size": int(rng.integers(8, 255)),
                       "spx.matrix.min_coverage": 0.01}]
            for extra in extras:
                for s in (("true", "false") if sym else ("false",)):
                    o = {"spx.preproc.xform": xf, "spx.matrix.symmetric": s}
                    o.update(extra)
                    check_matrix(rp, ci, va, n, m, o, seed=seed)


def test_empty_and_degenerate():
    """Empty rows at both ends, an empty matrix, single-element rows, a dense row of maximum unit length."""
    # leading / trailing empty rows
    rp = np.array([0, 0, 0, 2, 2, 5, 5, 5], np.int32)
    ci = np.array([0, 3, 1, 2, 6], np.int32)
    va = np.arange(1.0, 6.0)
    for xf in ("none", "all"):
        check_matrix(rp, ci, va, 7, 7, {"spx.preproc.xform": xf})
        check_matrix(rp, ci, va, 7, 7, {"spx.preproc.xform": xf, "spx.rt.nr_threads": 3})
    # dense rows longer than one unit (255) and longer than one warp pass
    n = 40
    m = 1000
    rng = np.random.default_rng(7)
    rows = []
    for r in range(n):
        k = int(rng.integers(1, m)) if r % 3 else m
        rows.append(np.sort(rng.choice(m, k, replace=False)))
    rp = np.concatenate([[0], np.cumsum([len(r) for r in rows])]).astype(np.int32)
    ci = np.concatenate(rows).astype(np.int32)
    va = rng.standard_normal(ci.size)
    for xf in ("none", "h", "all"):
        check_matrix(rp, ci, va, n, m, {"spx.preproc.xform": xf})
    # wide column jumps: delta16 / delta32 units
    m = 300000
    rows = [np.sort(rng.choice(m, 50, replace=False)) for _ in range(64)]
    rp = np.concatenate([[0], np.cumsum([len(r) for r in rows])]).astype(np.int32)
    ci = np.concatenate(rows).astype(np.int32)
    va = rng.standard_normal(ci.size)
    check_matrix(rp, ci, va, 64, m, {"spx.preproc.xform": "none"})
    check_matrix(rp, ci, va, 64, m, {"spx.preproc.xform": "none", "spx.matrix.full_colind": "true"})


@pytest.mark.parametrize("seed", range(3))
def test_random_structured_four_rows_per_thread(seed):
    """Same inputs with the 1024-row tile shape (4 rows per thread) that large partitions use."""
    rng = np.random.default_rng(300 + seed)
    for trial in range(3):
        n = int(rng.integers(900, 4000))
        sym = trial % 2 == 0
        m = n if sym else int(rng.integers(900, 4000))
        rp, ci, va = random_structured(rng, n, m, symmetric=sym)
        for xf in XFORMS:
            for extra in ({}, {"spx.rt.nr_threads": int(rng.integers(2, 4))}, {"spx.preproc.sampling": "none"}):
                for s in (("true", "false") if sym else ("false",)):
                    o = {"spx.preproc.xform": xf, "spx.matrix.symmetric": s, "spx.b200.rows_per_thread": 4}
                    o.update(extra)
                    check_matrix(rp, ci, va, n, m, o, seed=seed)


def test_large_partition_auto_tile():
    """>= 2^20 rows: the automatic choice of the 4-rows-per-thread tile."""
    rp, ci, va, n = poisson2d(1100)
    check_matrix(rp, ci, va, n, n, {})
    check_matrix(rp, ci, va, n, n, {"spx.matrix.symmetric": "true"}, check_decode=False)


@pytest.mark.parametrize("opts", [{}, {"spx.preproc.xform": "none"}, {"spx.preproc.xform": "br,bc"},
                                  {"spx.rt.nr_threads": 4}, {"spx.matrix.symmetric": "true"},
                                  {"spx.matrix.symmetric": "true", "spx.rt.nr_threads": 3}])
def test_poisson2d(opts):
    rp, ci, va, n = poisson2d(160)
    check_matrix(rp, ci, va, n, n, opts)


@pytest.mark.parametrize("opts", [{}, {"spx.preproc.xform": "br,bc"}, {"spx.preproc.xform": "bc3{3},h{1}"},
                                  {"spx.matrix.symmetric": "true"}])
def test_stencil27(opts):
    rp, ci, va, n = stencil27(24)
    check_matrix(rp, ci, va, n, n, opts)


@pytest.mark.parametrize("opts", [{"spx.matrix.symmetric": "true"}, {"spx.matrix.symmetric": "true", "spx.rt.nr_threads": 2},
                                  {"spx.matrix.symmetric": "true", "spx.preproc.xform": "br3{3},bc3{3}"}, {}])
def test_sym_block_banded(opts):
    rp, ci, va, n = sym_block_banded(4000, b=64)
    check_matrix(rp, ci, va, n, n, opts)


@pytest.mark.parametrize("opts", [{"spx.preproc.xform": "none"}, {"spx.preproc.xform": "none", "spx.rt.nr_threads": 8}, {}])
def test_rmat(opts):
    rp, ci, va, n = rmat(14)
    check_matrix(rp, ci, va, n, n, opts)


@pytest.mark.parametrize("world", [2, 3, 5])
def test_symmetric_partition_per_device(world):
    """CSX-Sym with one partition per device (all on cuda:0 here): every logical rank computes its own rows plus
    its transposed contributions to the halo rows of lower ranks; summing the halos reproduces y = A x."""
    torch = _torch()
    from oracle.pyoracle import OracleMatrix
    from sparsex_b200 import CsxMatrix, lib
    rng = np.random.default_rng(world)
    cases = [sym_block_banded(3000, b=40)[:3] + (9000,), random_structured(rng, 1500, 1500, symmetric=True) + (1500,)]
    for rp, ci, va, n in cases:
        for xf in ("all", "none", "d,v,ad", "br,bc"):
            opts = {"spx.matrix.symmetric": "true", "spx.rt.nr_threads": world, "spx.preproc.xform": xf}
            O = OracleMatrix.from_csr(rp, ci, va, n, n).tune(dict(opts, **{"oracle.undefined_sampling": "break"}))
            x = rng.uniform(-1, 1, n)
            yref = O.spmv(0.5, x)
            dx = torch.from_numpy(x).cuda()
            total = np.zeros(n)
            for r in range(world):
                A = CsxMatrix.tune_csr(rp, ci, va, n, n, opts, part_lo=r, part_hi=r + 1)
                assert np.array_equal(A.partition(0).ctl, O.parts[r].ctl)
                A.upload(0)
                P = A.partition(0)
                lo, cnt = P.row_start, len(P.dvalues)
                hlo, hhi = lib().csxb_info(A._h, 8), lib().csxb_info(A._h, 9)
                assert hhi == lo or hlo == hhi == 0 or r == 0
                dy = torch.full((n,), 7.0, dtype=torch.float64, device="cuda")   # stale content must not leak
                A.spmv(0.5, dx, dy, overwrite=True)
                y = dy.cpu().numpy()
                total[lo:lo + cnt] += y[lo:lo + cnt]
                if hhi > hlo:
                    total[hlo:hhi] += y[hlo:hhi]
                A.close()
            bound = _abs_bound(rp, ci, va, x, n) + 1e-300
            assert np.max(np.abs(total - yref) / (0.5 * bound)) <= TOL, (world, xf, O.log)


@pytest.mark.parametrize("slab_rows", [256, 1024, 5000])
def test_pipelined_host_buffer_path(slab_rows):
    """csxb_spmv_host with many slabs: x uploaded in column order, slabs computed as their windows arrive, y rows
    downloaded as they become final; chunks that straddle slab boundaries; both y semantics."""
    _torch()
    from sparsex_b200 import CsxMatrix
    rng = np.random.default_rng(slab_rows)
    cases = [poisson2d(60)[:3] + (3600, 3600, {}), stencil27(14)[:3] + (2744, 2744, {"spx.preproc.xform": "br,bc", "spx.preproc.sampling": "none"}),
             rmat(12)[:3] + (4096, 4096, {"spx.preproc.xform": "none"}),
             random_structured(rng, 3000, 2500) + (3000, 2500, {"spx.preproc.sampling": "none"})]
    for rp, ci, va, n, m, opts in cases:
        for nt in (1, 3):
            o = dict(opts, **{"spx.b200.slab_rows": slab_rows, "spx.rt.nr_threads": nt})
            A = CsxMatrix.tune_csr(rp, ci, va, n, m, o).upload(0)
            x = rng.uniform(-1, 1, m)
            y0 = rng.uniform(-1, 1, n)
            bound = _abs_bound(rp, ci, va, x, n) + 1e-300
            ref = _csr_spmv(rp, ci, va, x, n)
            y = y0.copy()
            A.spmv_host(0.5, x, y)
            assert np.max(np.abs(y - 0.5 * ref) / (0.5 * bound)) <= TOL
            # spx_matvec_kernel semantics: rows behind the last non-empty row belong to no partition and stay as they are
            # (do_kernel_thread scales the rows of its partition only, CsxSpmv.cpp:52-64) — on every path
            owned = int(np.nonzero(np.diff(rp))[0].max()) + 1
            want = 0.75 * ref - 0.3 * y0
            want[owned:] = y0[owned:]
            y = y0.copy()
            A.spmv_host(0.75, x, y, beta=-0.3, overwrite=False)
            assert np.max(np.abs(y - want) / (0.75 * bound + 0.3 * np.abs(y0) + 1e-300)) <= TOL
            import torch
            dx, dy = torch.from_numpy(x).cuda(), torch.from_numpy(y0.copy()).cuda()
            A.spmv(0.75, dx, dy, beta=-0.3, overwrite=False)
            assert np.max(np.abs(dy.cpu().numpy() - want) / (0.75 * bound + 0.3 * np.abs(y0) + 1e-300)) <= TOL
            A.close()


@pytest.mark.parametrize("world,split_max", [(2, None), (4, None), (3, "0")])
def test_peer_exchange_logical_ranks(world, split_max, monkeypatch):
    """csxb_xchg_*: repeated SpMV with the exchange fused into the kernel.  All logical ranks live on cuda:0 in
    this process (csxb_xchg_connect_ptr), every rank issues its steps on its own stream (a step ends with the
    flag exchange with its neighbours); after every step each rank's next x must hold alpha*A*x on every column
    its partition reads."""
    torch = _torch()
    from sparsex_b200 import CsxMatrix, PeerExchange, lib
    if split_max is not None:   # whole edge tiles instead of four one-row-per-thread CTAs (what many edge tiles get)
        monkeypatch.setenv("CSXB_XCHG_SPLIT_MAX", split_max)
    rng = np.random.default_rng(world)
    cases = [poisson2d(70)[:3] + (4900, {}), stencil27(12)[:3] + (1728, {"spx.preproc.xform": "br,bc", "spx.preproc.sampling": "none"}),
             rmat(11)[:3] + (2048, {"spx.preproc.xform": "none"}),
             # 4 rows per thread: edge tiles are split over four one-row-per-thread CTAs (csx_spmv_xe_kernel)
             poisson2d(150)[:3] + (22500, {"spx.b200.rows_per_thread": 4}),
             stencil27(22)[:3] + (10648, {"spx.b200.rows_per_thread": 4})]
    for rp, ci, va, n, opts in cases:
        o = dict(opts, **{"spx.rt.nr_threads": world})
        mats = [CsxMatrix.tune_csr(rp, ci, va, n, n, o, part_lo=r, part_hi=r + 1).upload(0) for r in range(world)]
        L = lib()
        ranges = [(L.csxb_part_info(A._h, 0, 3), L.csxb_part_info(A._h, 0, 1)) for A in mats]
        windows = [(L.csxb_part_info(A._h, 0, 11), L.csxb_part_info(A._h, 0, 12)) for A in mats]
        ex = [PeerExchange(A, r, world) for r, A in enumerate(mats)]
        bases = [e.base() for e in ex]
        for e in ex:
            e.connect_ptr(bases, ranges, windows)
        x = rng.uniform(-1, 1, n)
        for e in ex:
            e.vector(0).copy_(torch.from_numpy(x))
            e.vector(1).fill_(float("nan"))
        alpha = 0.25
        cur = x
        streams = [torch.cuda.Stream() for _ in ex]
        torch.cuda.synchronize()
        for step in range(5):
            for e, st in zip(ex, streams):
                e.spmv(alpha, stream=st.cuda_stream)
            torch.cuda.synchronize()
            ref = alpha * _csr_spmv(rp, ci, va, cur, n)
            bound = alpha * _abs_bound(rp, ci, va, cur, n) + 1e-300
            for r, e in enumerate(ex):
                assert e.error() == 0 and e.steps() == step + 1
                got = e.vector((step + 1) & 1).cpu().numpy()
                lo, hi = windows[r]
                own_lo, own_n = ranges[r]
                need = np.zeros(n, bool)
                if hi >= lo:
                    need[lo:hi + 1] = True
                need[own_lo:own_lo + own_n] = True
                covered = np.zeros(n, bool)   # rows some rank owns (trailing empty rows belong to nobody)
                for a, b in ranges:
                    covered[a:a + b] = True
                need &= covered
                assert np.all(np.abs(got[need] - ref[need]) / bound[need] <= TOL), (step, r)
            # the next step's reference input is what the engine holds (every rank's own rows are authoritative),
            # so that rounding differences of earlier steps do not count against the tolerance of this one
            nxt = np.zeros(n)
            for r, e in enumerate(ex):
                a, b = ranges[r]
                nxt[a:a + b] = e.vector((step + 1) & 1)[a:a + b].cpu().numpy()
            for e in ex:   # rows nobody owns are zero in every step's result (VecInit(y, 0), CsxKernels.cpp:93)
                assert np.all(e.vector((step + 1) & 1).cpu().numpy()[~covered] == 0.0)
            cur = nxt
        for e in ex:
            e.close()
        for A in mats:
            A.close()


def test_set_entry_and_restore_on_device(tmp_path):
    """SURVEY.md 8f rows 2-3 on the device: csxb_set_entry updates the uploaded values (next SpMV sees it without
    re-tuning, also when the host copy was released), and a matrix restored from the container multiplies like the
    tuned one; then the same through spx_mat_set_entry / spx_mat_save / spx_mat_restore."""
    torch = _torch()
    import ctypes as C
    from sparsex_b200 import CsxMatrix, load_spx_api
    rng = np.random.default_rng(11)
    n = 900
    for sym in (False, True):
        rp, ci, va = random_structured(rng, n, n, symmetric=sym)
        opts = {"spx.preproc.sampling": "none", "spx.rt.nr_threads": 2}
        if sym:
            opts["spx.matrix.symmetric"] = "true"
        A = CsxMatrix.tune_csr(rp, ci, va, n, n, opts).upload(0, free_host=True)
        rows = np.repeat(np.arange(n), np.diff(rp))
        va2 = va.copy()
        for _ in range(40):
            k = int(rng.integers(len(va)))
            r, c = int(rows[k]), int(ci[k])
            nv = float(rng.standard_normal())
            assert A.get_entry(r, c) == va2[k]          # read back from the device copy
            assert A.set_entry(r, c, nv)
            va2[k] = nv
            if sym and r != c:                         # the mirrored entry is the same stored value
                k2 = rp[c] + int(np.searchsorted(ci[rp[c]:rp[c + 1]], r))
                va2[k2] = nv
        x = rng.uniform(-1, 1, n)
        y = np.zeros(n)
        A.spmv_host(1.0, x, y)
        ref = _csr_spmv(rp, ci, va2, x, n)
        bound = _abs_bound(rp, ci, va2, x, n) + 1e-300
        assert np.max(np.abs(y - ref) / bound) <= TOL
        path = os.path.join(str(tmp_path), "a.csxb")
        A.save(path)                                    # values come back from the device for the container
        B = CsxMatrix.load(path).upload(0)
        y2 = np.zeros(n)
        B.spmv_host(1.0, x, y2)
        assert np.max(np.abs(y2 - ref) / bound) <= TOL
        A.close()
        B.close()
    # drop-in API
    api = load_spx_api()
    api.spx_init()
    rp, ci, va = random_structured(rng, 500, 500)
    api.spx_option_set(b"spx.preproc.sampling", b"none")
    api.spx_option_set(b"spx.rt.nr_threads", b"1")
    api.spx_option_set(b"spx.matrix.symmetric", b"false")
    inp = api.spx_input_load_csr(rp.ctypes.data, ci.ctypes.data, va.ctypes.data, 500, 500)
    M = api.spx_mat_tune(inp)
    assert M
    v = C.c_double()
    assert api.spx_mat_get_entry(M, int(0), int(ci[rp[0]]), C.byref(v)) == 0 or rp[1] == rp[0]
    k = int(rp[250])
    r = int(np.searchsorted(rp, k, side="right") - 1)
    api.L.spx_mat_set_entry.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_double]
    assert api.L.spx_mat_set_entry(M, r, int(ci[k]), 9.25) == 0
    path = os.path.join(str(tmp_path), "b.csxb").encode()
    api.L.spx_mat_save.argtypes = [C.c_void_p, C.c_char_p]
    api.L.spx_mat_restore.restype = C.c_void_p
    api.L.spx_mat_restore.argtypes = [C.c_char_p]
    assert api.L.spx_mat_save(M, path) == 0
    R = api.L.spx_mat_restore(path)
    assert R
    assert api.spx_mat_get_entry(R, r, int(ci[k]), C.byref(v)) == 0 and v.value == 9.25
    api.spx_mat_destroy(M)
    api.spx_mat_destroy(R)
    api.spx_input_destroy(inp)


def test_spx_mat_tune_reorder(tmp_path):
    """spx_mat_tune(input, SPX_MAT_REORDER) (matvec.c:262-300, Rcm.hpp): the tuned matrix is P A P^T, the permutation is
    the one csxb_rcm_csr computes, vectors go through spx_vec_reorder / spx_vec_inv_reorder, single entries are
    addressed in the original numbering, the container keeps the permutation; symmetric MatrixMarket input."""
    torch = _torch()
    import ctypes as C
    import scipy.sparse as sp
    from sparsex_b200 import load_spx_api, SpxApi, engine
    from tests.test_cpu_rcm import scrambled_banded, csr
    SPX_MAT_REORDER = 42
    api = load_spx_api()
    api.spx_init()
    api.spx_log_disable_all()
    for sym in (b"false", b"true"):
        n = 6000
        a = scrambled_banded(n, 6, 31)
        a = sp.csr_matrix(a + a.T)          # values symmetric too, so that CSX-Sym applies
        rp, ci, va = csr(a)
        api.spx_option_set(b"spx.rt.nr_threads", b"2")
        api.spx_option_set(b"spx.matrix.symmetric", sym)
        inp = api.spx_input_load_csr(rp.ctypes.data, ci.ctypes.data, va.ctypes.data, n, n)
        M = api.spx_mat_tune(inp, SPX_MAT_REORDER)
        assert M
        pp = api.spx_mat_get_perm(M)
        assert pp
        perm = np.ctypeslib.as_array(pp, shape=(n,)).copy()
        want, bw = engine.rcm_csr(rp, ci, n)
        assert np.array_equal(perm, want) and bw[1] < bw[0]
        parts = api.spx_mat_get_partition(M)
        x = api.spx_vec_create(n, parts)
        y = api.spx_vec_create(n, parts)
        rng = np.random.default_rng(5)
        xs = rng.uniform(-1, 1, n)
        SpxApi.as_numpy(x)[:] = xs
        assert api.spx_vec_reorder(x, pp) == 0
        assert np.array_equal(SpxApi.as_numpy(x)[perm], xs)
        assert api.spx_matvec_mult(0.75, M, x, y) == 0
        api.spx_device_synchronize()
        assert api.spx_vec_inv_reorder(y, pp) == 0
        ref = 0.75 * _csr_spmv(rp, ci, va, xs, n)
        bound = 0.75 * _abs_bound(rp, ci, va, xs, n) + 1e-300
        assert np.max(np.abs(SpxApi.as_numpy(y) - ref) / bound) <= TOL
        # entries in the caller's numbering
        v = C.c_double()
        rows = np.repeat(np.arange(n), np.diff(rp))
        for k in rng.integers(0, len(va), 25):
            assert api.spx_mat_get_entry(M, int(rows[k]), int(ci[k]), C.byref(v)) == 0 and v.value == va[k]
        path = os.path.join(str(tmp_path), "r.csxb").encode()
        assert api.spx_mat_save(M, path) == 0
        R = api.spx_mat_restore(path)
        assert R
        rp2 = api.spx_mat_get_perm(R)
        assert rp2 and np.array_equal(np.ctypeslib.as_array(rp2, shape=(n,)), perm)
        api.spx_mat_destroy(R)
        api.spx_partition_destroy(parts)
        api.spx_mat_destroy(M)
        api.spx_input_destroy(inp)
        api.spx_vec_destroy(x)
        api.spx_vec_destroy(y)
    # MatrixMarket: a symmetric file is held in memory and reordered (Rcm.hpp:155-204)
    api.spx_option_set(b"spx.matrix.symmetric", b"false")
    api.spx_option_set(b"spx.rt.nr_threads", b"1")
    path = os.path.join(GOLDEN, "matrices", "symmetric.mtx.sorted").encode()
    inp = api.spx_input_load_mmf(path)
    M = api.spx_mat_tune(inp, SPX_MAT_REORDER)
    assert M
    pp = api.spx_mat_get_perm(M)
    n = api.spx_mat_get_nrows(M)
    assert pp and sorted(np.ctypeslib.as_array(pp, shape=(n,)).tolist()) == list(range(n))
    from tests.test_cpu_rcm import oracle_rcm
    ent = [l.split() for l in open(path.decode()) if not l.startswith("%")][1:]
    r = np.array([int(e[0]) - 1 for e in ent]); c = np.array([int(e[1]) - 1 for e in ent]); v = np.array([float(e[2]) for e in ent])
    off = r != c
    full = sp.csr_matrix((np.concatenate([v, v[off]]), (np.concatenate([r, c[off]]), np.concatenate([c, r[off]]))), shape=(n, n))
    frp, fci, fva = csr(full)
    mperm = np.ctypeslib.as_array(pp, shape=(n,)).copy()
    assert np.array_equal(mperm, oracle_rcm(frp, fci, n, symmetric=1))   # edges = the upper triangle, row-major
    parts = api.spx_mat_get_partition(M)
    x = api.spx_vec_create(n, parts)
    y = api.spx_vec_create(n, parts)
    xs = np.random.default_rng(6).uniform(-1, 1, n)
    SpxApi.as_numpy(x)[:] = xs
    api.spx_vec_reorder(x, pp)
    assert api.spx_matvec_mult(1.0, M, x, y) == 0
    api.spx_device_synchronize()
    api.spx_vec_inv_reorder(y, pp)
    assert np.max(np.abs(SpxApi.as_numpy(y) - _csr_spmv(frp, fci, fva, xs, n)) / (_abs_bound(frp, fci, fva, xs, n) + 1e-300)) <= TOL
    api.spx_vec_destroy(x)
    api.spx_vec_destroy(y)
    api.spx_partition_destroy(parts)
    api.spx_mat_destroy(M)
    api.spx_input_destroy(inp)
    api.spx_option_set(b"spx.rt.nr_threads", b"1")


def _group_cases():
    rng = np.random.default_rng(77)
    rp, ci, va, n = sym_block_banded(2500, b=30)[:3] + (7500,)
    yield "symbb", rp, ci, va, n, True
    rp, ci, va = random_structured(rng, 3000, 3000, symmetric=True)
    yield "random_sym", rp, ci, va, 3000, True
    rp, ci, va, n = poisson2d(90)
    yield "poisson", rp, ci, va, n, False
    rp, ci, va = random_structured(rng, 2500, 2500)
    # trailing empty rows: they belong to no partition
    rp = np.concatenate([rp, np.full(40, rp[-1], dtype=rp.dtype)])
    yield "random_trailing", rp, ci, va, 2540, False


@pytest.mark.parametrize("devices", [[0, 0], [0, 0, 0, 0, 0]], ids=["2members", "5members"])
def test_device_group_logical_members(devices, tmp_path):
    """csxb_group_* (several GPUs behind one handle, one process) with every member on cuda:0: host buffers (the
    members' slab pipelines on concurrent host threads), device vectors, CSX-Sym with the owner-side reduction, both y
    semantics, trailing rows, entries, container round trip."""
    torch = _torch()
    from sparsex_b200 import CsxMatrix, DeviceGroup
    rng = np.random.default_rng(len(devices))
    for name, rp, ci, va, n, symmetric in _group_cases():
        nc = n   # (the case with trailing empty rows is square too: its last 40 columns are never read)
        for sym in ([False, True] if symmetric else [False]):
            opts = {"spx.rt.nr_threads": 6, "spx.b200.slab_rows": 512}
            if sym:
                opts["spx.matrix.symmetric"] = "true"
            A = CsxMatrix.tune_csr(rp, ci, va, n, nc, opts)
            G = DeviceGroup(A, devices)
            assert G.size == min(len(devices), 6)
            x = rng.uniform(-1, 1, nc)
            y0 = rng.uniform(-1, 1, n)
            ref = _csr_spmv(rp, ci, va, x, n)
            bound = _abs_bound(rp, ci, va, x, n) + 1e-300
            last = int(np.max(np.nonzero(np.diff(rp))[0])) + 1   # rows behind it belong to nobody
            # host buffers, spx_matvec_mult semantics: stale content of y must not survive
            y = np.full(n, 7.0)
            G.spmv(0.5, x, y)
            assert np.max(np.abs(y - 0.5 * ref) / (0.5 * bound)) <= TOL, (name, sym, "host mult")
            assert np.all(y[last:] == 0.0)
            # host buffers, spx_matvec_kernel semantics: rows behind the last partition stay as they are
            y = y0.copy()
            G.spmv(0.75, x, y, beta=-0.3, overwrite=False)
            want = 0.75 * ref - 0.3 * y0
            want[last:] = y0[last:]
            assert np.max(np.abs(y - want) / (0.75 * bound + 0.3 * np.abs(y0) + 1e-300)) <= TOL, (name, sym, "host kernel")
            # device vectors
            dx = torch.from_numpy(x).cuda()
            dy = torch.full((n,), 7.0, dtype=torch.float64, device="cuda")
            G.spmv(0.5, dx, dy)
            y = dy.cpu().numpy()
            assert np.max(np.abs(y - 0.5 * ref) / (0.5 * bound)) <= TOL, (name, sym, "device mult")
            assert np.all(y[last:] == 0.0)
            dy = torch.from_numpy(y0.copy()).cuda()
            G.spmv(0.75, dx, dy, beta=-0.3, overwrite=False)
            assert np.max(np.abs(dy.cpu().numpy() - want) / (0.75 * bound + 0.3 * np.abs(y0) + 1e-300)) <= TOL, (name, sym, "device kernel")
            # repeated calls give the same bits (no atomics anywhere, fixed reduction order)
            dy2 = torch.empty_like(dy)
            G.spmv(0.5, dx, dy2)
            dy3 = torch.empty_like(dy)
            G.spmv(0.5, dx, dy3)
            assert torch.equal(dy2, dy3)
            # entries live in the member that owns the row
            rows = np.repeat(np.arange(n), np.diff(rp))
            for k in rng.integers(0, len(va), 12):
                assert G.get_entry(int(rows[k]), int(ci[k])) == va[k]
            # container round trip: all partitions back in one file
            path = os.path.join(str(tmp_path), "g.csxb")
            G.save(path)
            B = CsxMatrix.load(path).upload(0)
            yb = np.zeros(n)
            B.spmv_host(0.5, x, yb)
            assert np.max(np.abs(yb - 0.5 * ref) / (0.5 * bound)) <= TOL
            B.close()
            G.close()


def test_spx_api_on_several_gpus():
    """The drop-in API with spx.b200.devices / spx.rt.nr_gpus: library (managed) vectors and user buffers; real
    GPUs when the box has more than one, logical members on cuda:0 otherwise."""
    torch = _torch()
    from sparsex_b200 import load_spx_api, SpxApi
    api = load_spx_api()
    api.spx_init()
    ndev = torch.cuda.device_count()
    devs = ",".join(str(i % ndev) for i in range(max(2, min(ndev, 4)))).encode()
    rp, ci, va, n = sym_block_banded(3000, b=40)[:3] + (9000,)
    rng = np.random.default_rng(3)
    xs = rng.uniform(-1, 1, n)
    ref = _csr_spmv(rp, ci, va, xs, n)
    bound = _abs_bound(rp, ci, va, xs, n) + 1e-300
    try:
        for sym in (b"false", b"true"):
            api.spx_option_set(b"spx.b200.devices", devs)
            api.spx_option_set(b"spx.matrix.symmetric", sym)
            api.spx_option_set(b"spx.rt.nr_threads", b"1")    # raised to the number of GPUs
            inp = api.spx_input_load_csr(rp.ctypes.data, ci.ctypes.data, va.ctypes.data, n, n)
            M = api.spx_mat_tune(inp)
            assert M
            parts = api.spx_mat_get_partition(M)
            nparts = devs.count(b",") + 1
            rs = api.spx_partition_get_rs(parts)
            re_ = api.spx_partition_get_re(parts)
            assert rs[0] == 0 and all(rs[i + 1] == re_[i] for i in range(nparts - 1)) and re_[nparts - 1] == n
            x = api.spx_vec_create(n, parts)
            y = api.spx_vec_create(n, parts)
            SpxApi.as_numpy(x)[:] = xs
            assert api.spx_matvec_mult(0.5, M, x, y) == 0
            assert np.max(np.abs(SpxApi.as_numpy(y) - 0.5 * ref) / (0.5 * bound)) <= TOL
            y0 = SpxApi.as_numpy(y).copy()
            assert api.spx_matvec_kernel(2.0, M, x, 0.5, y) == 0
            assert np.max(np.abs(SpxApi.as_numpy(y) - (2.0 * ref + 0.5 * y0)) / (2.0 * bound + 0.5 * np.abs(y0) + 1e-300)) <= TOL
            # user buffers
            import ctypes as C
            xb, yb = xs.copy(), np.zeros(n)
            tuned = C.c_void_p()
            xv = api.spx_vec_create_from_buff(xb.ctypes.data, C.byref(tuned), n, parts, 43)
            yv = api.spx_vec_create_from_buff(yb.ctypes.data, C.byref(tuned), n, parts, 43)
            assert api.spx_matvec_mult(0.5, M, xv, yv) == 0
            assert np.max(np.abs(yb - 0.5 * ref) / (0.5 * bound)) <= TOL
            v = C.c_double()
            assert api.spx_mat_get_entry(M, n - 1, int(ci[rp[n - 1]]), C.byref(v)) == 0 and v.value == va[rp[n - 1]]
            for h in (xv, yv, x, y):
                api.spx_vec_destroy(h)
            api.spx_partition_destroy(parts)
            api.spx_mat_destroy(M)
            api.spx_input_destroy(inp)
    finally:
        api.spx_option_set(b"spx.b200.devices", b"")
        api.spx_option_set(b"spx.matrix.symmetric", b"false")
        api.spx_option_set(b"spx.rt.nr_threads", b"1")


def test_blas1_helpers_on_device_vectors():
    """spx_vec_* on library (managed, HBM-resident) vectors run on the GPU; a conjugate-gradient iteration written
    against the SparseX API (src/examples/ style) converges on an SPD matrix."""
    _torch()
    from sparsex_b200 import load_spx_api, SpxApi
    api = load_spx_api()
    api.spx_init()
    n = 4000
    rp, ci, va, _ = poisson2d(int(np.sqrt(n)) + 1, perturb=False)
    n = len(rp) - 1
    for k, v in ((b"spx.rt.nr_threads", b"1"), (b"spx.matrix.symmetric", b"false"), (b"spx.preproc.sampling", b"portion"),
                 (b"spx.preproc.xform", b"all")):
        api.spx_option_set(k, v)
    inp = api.spx_input_load_csr(rp.ctypes.data, ci.ctypes.data, va.ctypes.data, n, n)
    A = api.spx_mat_tune(inp)
    part = api.spx_mat_get_partition(A)
    rng = np.random.default_rng(5)
    mk = lambda: api.spx_vec_create(n, part)
    a, b, c = mk(), mk(), mk()
    an, bn = rng.standard_normal(n), rng.standard_normal(n)
    SpxApi.as_numpy(a)[:] = an
    SpxApi.as_numpy(b)[:] = bn
    api.spx_vec_scale_add(a, b, c, 0.75)
    assert np.allclose(SpxApi.as_numpy(c), an + 0.75 * bn, rtol=0, atol=1e-15 * 8)
    api.spx_vec_sub(a, b, c)
    assert np.array_equal(SpxApi.as_numpy(c), an - bn)
    api.spx_vec_scale(a, c, -2.0)
    assert np.array_equal(SpxApi.as_numpy(c), -2.0 * an)
    d = api.spx_vec_mul(a, b)
    assert abs(d - float(an @ bn)) <= 1e-12 * float(np.abs(an) @ np.abs(bn))
    # CG on A x = rhs, all vectors resident
    x, r, p, q = mk(), mk(), mk(), mk()
    rhs = rng.standard_normal(n)
    SpxApi.as_numpy(r)[:] = rhs
    SpxApi.as_numpy(p)[:] = rhs
    rr = api.spx_vec_mul(r, r)
    rr0 = rr
    for _ in range(400):
        api.spx_matvec_mult(1.0, A, p, q)
        alpha = rr / api.spx_vec_mul(p, q)
        api.spx_vec_scale_add(x, p, x, alpha)
        api.spx_vec_scale_add(r, q, r, -alpha)
        rr_new = api.spx_vec_mul(r, r)
        if rr_new < 1e-24 * rr0:
            break
        api.spx_vec_scale_add(r, p, p, rr_new / rr)
        rr = rr_new
    xs = SpxApi.as_numpy(x).copy()
    res = _csr_spmv(rp, ci, va, xs, n) - rhs
    assert np.linalg.norm(res) <= 1e-8 * np.linalg.norm(rhs)
    for v in (a, b, c, x, r, p, q):
        api.spx_vec_destroy(v)
    api.spx_partition_destroy(part)
    api.spx_mat_destroy(A)
    api.spx_input_destroy(inp)


def test_bench_dumps_the_timed_product(tmp_path):
    """bench.py --dump-outputs writes y = alpha*A*x of the timed path (the whole vector at this size)."""
    import json
    import subprocess
    import sys
    _torch()
    import bench
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = str(tmp_path / "dump")
    r = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--gpus", "1", "--workload", "small", "--steps", "4",
                        "--warmup", "1", "--e2e-steps", "1", "--no-cpu-baseline", "--dump-outputs", out],
                       capture_output=True, text=True, timeout=900, cwd=root)
    assert r.returncode == 0, r.stderr[-3000:]
    line = json.loads([ln for ln in r.stdout.splitlines() if ln.startswith("{")][0])
    W = bench.workload("small")
    rp, ci, va = W.rows(0, W.n)
    x0 = np.random.default_rng(2).uniform(-1, 1, W.n)   # bench.py's x
    alpha = line["detail"]["alpha"]
    y = np.load(os.path.join(out, "y.npy"))
    assert y.dtype == np.float64 and y.shape == (W.n,)
    bound = _abs_bound(rp, ci, va, x0, W.n) + 1e-300
    assert np.max(np.abs(y - alpha * _csr_spmv(rp, ci, va, x0, W.n)) / (abs(alpha) * bound)) <= TOL
