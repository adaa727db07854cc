"""CPU tests against the reference's own SpMV kernels (oracle/_ref: src/templates/*.c of SparseX assembled like
CsxJit does and compiled by gcc).  Pins the multiply half of the oracle and shows that the CSX streams
the engine emits are consumable by the reference's kernels unchanged.

oracle/_ref is built only where the SparseX sources are present.  Without it the tests still run: the y of every
oracle-stream case is pinned bit for bit to tests/golden/ref_kernel_y.json, digests taken from the oracle's unit
loops, which the first test holds bit-identical to the reference kernels wherever both run (the file names the source it
was generated from); and the engine's streams are checked to be the oracle's byte for byte, so that the reference
kernels read the same data from both."""
import hashlib
import json
import os

import numpy as np
import pytest

from tests.conftest import GOLDEN
from tests.matrices import poisson2d, random_structured, stencil27, sym_block_banded

XFORMS = ["none", "h", "v", "d", "ad", "br", "bc", "all", "bc,v,ad", "br3{2,3},h{1}", "d{1},ad{2},v{1}"]
GOLD_Y = os.path.join(GOLDEN, "ref_kernel_y.json")


def _ref():
    """The compiled reference kernels, or None where oracle/_ref was not built."""
    from oracle import refkernels
    return refkernels if refkernels.available() else None


def _truth(rp, ci, va, x, n):
    rows = np.repeat(np.arange(n), np.diff(rp))
    y = np.zeros(n)
    np.add.at(y, rows, va * x[ci])
    return y


def y_digest(y):
    return hashlib.sha256(np.ascontiguousarray(y, np.float64).tobytes()).hexdigest()


def oracle_stream_cases(name):
    """Yields (key, tuned OracleMatrix, options, x, CSR product) of one bundled matrix (shared with the generator
    tests/golden/make_ref_kernel_golden.py)."""
    from oracle.pyoracle import OracleMatrix
    M = OracleMatrix.from_mmf(os.path.join(GOLDEN, "matrices", name + ".mtx.sorted"))
    rp, ci, va = M.csr()
    x = np.random.default_rng(5).uniform(-1, 1, M.ncols)
    truth = _truth(rp, ci, va, x, M.nrows)
    for xf in XFORMS:
        for extra in ({}, {"spx.rt.nr_threads": 2}, {"spx.preproc.sampling": "none"}, {"spx.matrix.full_colind": "true"}):
            for sym in (("false", "true") if name.startswith("symmetric") else ("false",)):
                o = {"spx.preproc.xform": xf, "spx.matrix.symmetric": sym, "oracle.undefined_sampling": "break"}
                o.update(extra)
                M.tune(o)
                yield name + "|" + ";".join("%s=%s" % kv for kv in sorted(o.items())), M, o, x, truth


def _assert_same_streams(A, oracle_opts, rp, ci, va, n, m):
    """The engine's partitions are the oracle's (which the reference kernels consume) byte for byte."""
    from oracle.pyoracle import OracleMatrix
    O = OracleMatrix.from_csr(rp, ci, va, n, m).tune(dict(oracle_opts, **{"oracle.undefined_sampling": "break"}))
    assert A.nparts == len(O.parts)
    for p in range(A.nparts):
        P, Q = A.partition(p), O.parts[p]
        assert (P.row_start, P.nrows) == (Q.row_start, Q.nrows), (oracle_opts, p)
        assert np.array_equal(P.ctl, Q.ctl) and np.array_equal(P.values, Q.values), (oracle_opts, p)
        assert np.array_equal(P.id_map, Q.id_map), (oracle_opts, p)
        if O.symmetric:
            assert np.array_equal(P.dvalues, Q.dvalues), (oracle_opts, p)
    return O


@pytest.mark.parametrize("name", ["demopatt", "test", "test3", "symmetric", "symmetric-very-sparse"])
def test_oracle_streams_run_on_reference_kernels(name):
    """Oracle-encoded CSX -> reference kernels == CSR product; and the oracle's own unit loops give the
    bit-identical vector (same operation order, no contraction), the one stored for the reference kernels."""
    rk = _ref()
    gold = json.load(open(GOLD_Y))["digests"]
    for key, M, o, x, truth in oracle_stream_cases(name):
        y = M.spmv(0.5, x)
        assert np.abs(y - 0.5 * truth).max() <= 1e-12 * max(1.0, np.abs(truth).max()), (o, M.log)
        assert y_digest(y) == gold[key], (o, M.log)
        if rk is not None:
            R = rk.Runner(M, full_colind=o.get("spx.matrix.full_colind") == "true")
            assert np.array_equal(R.spmv(0.5, x), y), (o, M.log)


@pytest.mark.parametrize("seed", range(3))
def test_engine_streams_run_on_reference_kernels(seed):
    """CSX emitted by the engine's encoder (C-ABI) is fed to the reference's kernels unchanged."""
    from sparsex_b200 import CsxMatrix
    rk = _ref()
    rng = np.random.default_rng(40 + seed)
    for trial in range(3):
        sym = trial == 0
        n = int(rng.integers(20, 500))
        m = n if sym else int(rng.integers(20, 500))
        rp, ci, va = random_structured(rng, n, m, symmetric=sym)
        x = rng.uniform(-1, 1, m)
        truth = _truth(rp, ci, va, x, n)
        for xf in XFORMS:
            for extra in ({}, {"spx.rt.nr_threads": 3}, {"spx.preproc.sampling": "none"}):
                for s in (("true", "false") if sym else ("false",)):
                    o = {"spx.preproc.xform": xf, "spx.matrix.symmetric": s}
                    o.update(extra)
                    A = CsxMatrix.tune_csr(rp, ci, va, n, m, o)
                    parts = [A.partition(p) for p in range(A.nparts)]
                    O = _assert_same_streams(A, o, rp, ci, va, n, m)
                    y = O.spmv(1.0, x)
                    if rk is not None:
                        y = rk.Runner(A, parts=parts, symmetric=(s == "true")).spmv(1.0, x)
                    assert np.abs(y - truth).max() <= 1e-12 * max(1.0, np.abs(truth).max()), (o, parts[0].log)
                    A.close()


@pytest.mark.parametrize("gen,opts", [(lambda: poisson2d(96), {}), (lambda: stencil27(16), {"spx.preproc.xform": "br,bc"}),
                                      (lambda: sym_block_banded(800, b=16), {"spx.matrix.symmetric": "true"})])
def test_config_shapes_on_reference_kernels(gen, opts):
    from sparsex_b200 import CsxMatrix
    rk = _ref()
    rp, ci, va, n = gen()
    x = np.random.default_rng(1).uniform(-1, 1, n)
    truth = _truth(rp, ci, va, x, n)
    A = CsxMatrix.tune_csr(rp, ci, va, n, n, opts)
    O = _assert_same_streams(A, opts, rp, ci, va, n, n)
    y = O.spmv(1.0, x)
    if rk is not None:
        R = rk.Runner(A, parts=[A.partition(p) for p in range(A.nparts)], symmetric=A.symmetric)
        y = R.spmv(1.0, x)
        assert R.bench(1.0, x, 2) > 0
    assert np.abs(y - truth).max() <= 1e-12 * np.abs(truth).max()
