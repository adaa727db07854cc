"""Forward and transposed SpMV on one B200, one process: y = A x (csxb_spmv) and y = A^T x (csxb_spmv_t) on the
matrices of bench.workload(), timed alternately in the same run (CUDA events, warm-up, median over repeats), each
product checked against the CSR input on sampled rows / columns.  Records the transposed tables' set-up time and
bytes, algorithmic bytes and rates, the share of measured_peak(), and, where heavy columns exist, the share of the
transposed product spent in the heavy-column kernels (torch.profiler, a separate pass).  --sweep times the heavy-column
threshold and segment length (CSXB_T_HEAVY / CSXB_T_SEG) on one workload.

    python tools/transpose_bench.py --workloads c2,c3,c3b,c4n,c5s --out profiles/r03_transpose_n1.json
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_card():
    try:
        out = subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], text=True)
        return out.strip().splitlines()[0]
    except Exception as ex:
        return "unknown (%r)" % (ex,)


def time_products(torch, fns, iters, warmup, repeats):
    """Median time per product of each fn, the fns run alternately repeat by repeat."""
    for f in fns:
        for _ in range(warmup):
            f()
    torch.cuda.synchronize()
    times = [[] for _ in fns]
    for _ in range(repeats):
        for i, f in enumerate(fns):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(iters):
                f()
            b.record()
            b.synchronize()
            times[i].append(a.elapsed_time(b) / iters * 1e-3)
    return [float(np.median(t)) for t in times], times


def check_cols(rp, ci, va, x, y, alpha, ncols, nsample=20000, seed=3):
    """max over sampled columns of |y - alpha*(A^T x)| / (|alpha| |A|^T |x|)."""
    rng = np.random.default_rng(seed)
    cols = np.unique(rng.integers(0, ncols, min(nsample, ncols)))
    lut = np.full(ncols, -1, np.int64)
    lut[cols] = np.arange(cols.size)
    slot = lut[ci]
    sel = slot >= 0
    rows = np.repeat(np.arange(rp.size - 1, dtype=np.int64), np.diff(rp.astype(np.int64)))[sel]
    prod = va[sel] * x[rows]
    ref = np.bincount(slot[sel], weights=prod, minlength=cols.size)
    bound = np.bincount(slot[sel], weights=np.abs(prod), minlength=cols.size)
    err = np.abs(y[cols] - alpha * ref) / (abs(alpha) * bound + 1e-300)
    err[bound == 0] = np.abs(y[cols][bound == 0])
    return float(err.max()), int(cols.size)


def heavy_share(torch, f, n=20):
    """Kernel time per product by kernel name over n products (torch.profiler, CUDA activities)."""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(n):
            f()
        torch.cuda.synchronize()
    per = {}
    for e in prof.events():
        if e.device_type.name == "CUDA":
            k = "segment" if "csx_t_segment" in e.name else ("fixup" if "fixup" in e.name else "gather")
            per[k] = per.get(k, 0.0) + e.device_time_total * 1e-6 / n
    return per


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", default="c2,c3,c3b,c4n,c5s")
    ap.add_argument("--iters", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--sweep", default="", help="workload whose heavy-column threshold / segment length are swept")
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    import torch
    import bench
    from sparsex_b200 import CsxMatrix
    assert torch.cuda.is_available(), "the measurement needs a GPU"
    peak, peak_src = bench.measured_peak()
    res = {"gpu": gpu_card(), "peak_gbs": peak, "peak_source": peak_src, "iters": a.iters, "warmup": a.warmup,
           "repeats": a.repeats, "note": "inputs: the whole matrix, larger than the 126 MB L2 except where stated by bytes",
           "workloads": {}, "sweep": []}
    for key in [k for k in a.workloads.split(",") if k]:
        W = bench.workload(key)
        rp, ci, va = W.rows(0, W.n)
        n = m = W.n
        opts = dict(W.opts, **{"spx.rt.nr_threads": 1})
        t0 = time.perf_counter()
        A = CsxMatrix.tune_csr(rp, ci, va, n, m, opts).upload(0)
        tune_s = time.perf_counter() - t0
        t0 = time.perf_counter()
        A.prepare_transpose()
        prep_s = time.perf_counter() - t0
        rng = np.random.default_rng(1)
        x = rng.uniform(-1, 1, n)
        dx = torch.from_numpy(x).cuda()
        dy = torch.empty(n, dtype=torch.float64, device="cuda")
        dyt = torch.empty(m, dtype=torch.float64, device="cuda")
        fwd = lambda: A.spmv(1.0, dx, dy)
        trn = lambda: A.spmv_t(1.0, dx, dyt)
        (tf, tt), raw = time_products(torch, [fwd, trn], a.iters, a.warmup, a.repeats)
        fwd()
        trn()
        torch.cuda.synchronize()
        ef, nf = bench.csr_check(rp, ci, va, 0, x, dy.cpu().numpy(), 1.0)
        et, nt = check_cols(rp, ci, va, x, dyt.cpu().numpy(), 1.0, m)
        info = A.transpose_info()
        fbytes = A.traffic()["total"]
        r = {"name": W.name, "nrows": n, "nnz": int(va.size), "tune_s": round(tune_s, 3),
             "transpose_prepare_s": round(prep_s, 3), "transpose_build_host_s": info["build_us"] * 1e-6,
             "transpose_added_device_bytes": info["device_bytes"], "transpose_launches": info["launches"],
             "heavy_cols": info["heavy_cols"], "segments": info["segments"],
             "forward": {"time_ms": tf * 1e3, "alg_bytes": fbytes, "gbs": fbytes / tf * 1e-9, "share_of_peak": fbytes / tf * 1e-9 / peak,
                         "times_ms": [v * 1e3 for v in raw[0]], "max_rel_err": ef, "rows_checked": nf},
             "transpose": {"time_ms": tt * 1e3, "alg_bytes": info["alg_bytes"], "gbs": info["alg_bytes"] / tt * 1e-9,
                           "share_of_peak": info["alg_bytes"] / tt * 1e-9 / peak, "times_ms": [v * 1e3 for v in raw[1]],
                           "max_rel_err": et, "cols_checked": nt},
             "transpose_over_forward": tt / tf}
        assert ef <= 1e-12 and et <= 1e-12, (key, ef, et)
        if info["heavy_cols"] > 0:
            r["transpose_kernel_ms"] = {k: v * 1e3 for k, v in heavy_share(torch, trn).items()}
        print(json.dumps({key: r}), flush=True)
        res["workloads"][key] = r
        if key == a.sweep:
            path = os.path.join(tempfile.mkdtemp(), "m.csxb")
            A.save(path)
            for hv in (32, 128, 512, 2048):
                for sg in (128, 256, 1024):
                    os.environ["CSXB_T_HEAVY"], os.environ["CSXB_T_SEG"] = str(hv), str(sg)
                    B = CsxMatrix.load(path).upload(0).prepare_transpose()
                    trb = lambda: B.spmv_t(1.0, dx, dyt)
                    (tb,), _ = time_products(torch, [trb], a.iters, a.warmup, 3)
                    s = {"heavy_min": hv, "seg_len": sg, "time_ms": tb * 1e3, "heavy_cols": B.transpose_info()["heavy_cols"]}
                    print(json.dumps(s), flush=True)
                    res["sweep"].append(s)
                    B.close()
            del os.environ["CSXB_T_HEAVY"], os.environ["CSXB_T_SEG"]
            os.remove(path)
        A.close()
        del rp, ci, va
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
