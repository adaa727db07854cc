"""Generates tests/golden/ref_kernel_y.json: SHA-256 digests of y = 0.5*A*x for every oracle-stream case of
tests/test_cpu_refkernels.py, the vector the reference's own SpMV kernels compute from those streams.

Where oracle/_ref is built (it needs the SparseX sources, oracle/build_ref.py) the vectors come from the reference
kernels and must equal the oracle's bit for bit.  Elsewhere they come from the oracle's unit loops, which that test
holds bit-identical to the reference kernels wherever both run; the file records which of the two produced it.
Run:  python tests/golden/make_ref_kernel_golden.py
"""
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import refkernels  # noqa: E402
from tests.test_cpu_refkernels import oracle_stream_cases, y_digest  # noqa: E402

if __name__ == "__main__":
    live = refkernels.available()
    out = {}
    for name in ["demopatt", "test", "test3", "symmetric", "symmetric-very-sparse"]:
        for key, M, o, x, truth in oracle_stream_cases(name):
            y = M.spmv(0.5, x)
            if live:
                yr = refkernels.Runner(M, full_colind=o.get("spx.matrix.full_colind") == "true").spmv(0.5, x)
                assert np.array_equal(yr, y), key
            out[key] = y_digest(y)
    source = ("the reference kernels (oracle/_ref), equal to the oracle's unit loops" if live else
              "the oracle's unit loops (oracle/_ref not built)")
    path = os.path.join(ROOT, "tests", "golden", "ref_kernel_y.json")
    json.dump({"source": source, "digests": out}, open(path, "w"), indent=0, sort_keys=True)
    print("wrote %d digests from %s to %s" % (len(out), source, path))
