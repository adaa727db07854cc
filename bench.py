#!/usr/bin/env python
"""bench.py — CSX SpMV throughput of the B200 engine (and of the CPU reference arm).

    python bench.py --gpus N --steps K --warmup W [--workload c3|c2|c3b|c4|c5|...] [--outer R] [--impl reference]

A *step* is one SpMV  y = alpha*A*x  over the whole matrix (the hot path of
BASELINE.json: spx_matvec_mult after spx_mat_tune).  For N > 1 the rows are the
reference's nnz-balanced partitions with spx.rt.nr_threads = N, one partition
per rank, and every step ends with the exchange of the y pieces into the next
x (NCCL all-gather over NVLink) — strong scaling on a fixed matrix.

Metric: GFLOP/s = 2 * nnz * K / t  (reference convention, src/bench/SparsexModule.cpp:80).
Timing: W untimed steps, then exactly K steps (captured into CUDA graphs: a step is kernel launches
only) between a barrier + synchronize on both sides, CUDA events on the launching stream, max over
ranks; --outer R repeats the timed region R times and reports the median (the reference's protocol
is 5 x 128, src/bench/Bench.cpp:29-30).  The default workload is C3 (3.6 GB of values: 450 MB per
GPU even at N = 8, larger than the 126 MB L2, so consecutive steps cannot be served from cache).
After the timed region the result is checked against the CSR product on 10^5 sampled rows per rank
(componentwise 1e-12): the device path, and for N > 1 the vector the in-kernel exchange produced.
"""
import argparse
import ctypes as C
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

class Workload(object):
    """A synthetic matrix of one of BASELINE.json's configs (SURVEY.md section 8d) that any rank can generate by row
    ranges (tests/matrices.py: values are hashes of the coordinates), plus its tuning options."""

    def __init__(self, key, name, kind, opts, **kw):
        self.key, self.name, self.kind, self.opts, self.kw = key, name, kind, dict(opts), kw
        self.sym = str(opts.get("spx.matrix.symmetric", "false")) == "true"
        from tests import matrices as M
        self.M = M
        if kind in ("p2", "s27"):
            self.n = kw["g"] ** (2 if kind == "p2" else 3)
        elif kind == "symbb":
            self.n = kw["nb"] * 3
        else:
            self.n = 1 << kw["scale"]
        self._counts = None

    def counts(self, device=None):
        """Non-zeros per row (int64)."""
        if self._counts is None:
            M, kw = self.M, self.kw
            if self.kind in ("p2", "s27"):
                self._counts = M.stencil_row_counts(self.kind, kw["g"])
            elif self.kind == "symbb":
                self._counts = M.symbb_row_counts(kw["nb"], kw["b"])
            else:
                self._counts = M.rmat_block_row_counts(kw["scale"], device=device)
        return self._counts

    def lower_counts(self):
        """CSX-Sym: entries left of the diagonal per row (block-banded: the row's entries minus the diagonal, halved
        per block structure is not uniform, so count them)."""
        kw = self.kw
        nb, b = kw["nb"], kw["b"]
        I = np.arange(nb, dtype=np.int64)
        left_blocks = ((I - 1 >= 0).astype(np.int64) + (I - b >= 0).astype(np.int64)) * 3
        return np.repeat(left_blocks, 3) + np.tile(np.arange(3, dtype=np.int64), nb)

    def rows(self, lo, hi, device=None):
        """(rowptr, colind, values) of rows [lo, hi), generated in pieces of 2 M rows (bounded temporaries)."""
        M, kw = self.M, self.kw
        if self.kind == "rmat":
            return M.rmat_block_rows(kw["scale"], lo, hi, device=device)
        rps, cis, vas, base = [np.zeros(1, np.int64)], [], [], 0
        for a in range(lo, hi, 1 << 21):
            b = min(hi, a + (1 << 21))
            rp, ci, va = (M.stencil_rows(self.kind, kw["g"], a, b) if self.kind in ("p2", "s27") else M.symbb_rows(kw["nb"], kw["b"], a, b))
            rps.append(rp[1:].astype(np.int64) + base)
            base += int(rp[-1])
            cis.append(ci)
            vas.append(va)
        if base >= 2 ** 31:
            raise SystemExit("%d non-zeros in one partition: the SparseX API has 32-bit indices (spx_index_t = int)" % base)
        return (np.concatenate(rps).astype(np.int32), np.concatenate(cis) if cis else np.zeros(0, np.int32),
                np.concatenate(vas) if vas else np.zeros(0))

    def split(self, nparts, device=None):
        return self.M.split_rows(self.counts(device), nparts, self.lower_counts() if self.sym else None)


def workload(key):
    W = {
        "c2": ("c2_poisson2d_4096", "p2", {}, dict(g=4096)),
        "c3": ("c3_stencil27_256", "s27", {}, dict(g=256)),
        "c3b": ("c3_stencil27_256_blocks", "s27", {"spx.preproc.xform": "br,bc"}, dict(g=256)),
        "c4": ("c4_sym_block_banded_30M", "symbb", {"spx.matrix.symmetric": "true"}, dict(nb=10_000_000, b=1024)),
        "c4n": ("c4_block_banded_30M_not_symmetric_mode", "symbb", {}, dict(nb=10_000_000, b=1024)),
        "c5": ("c5_rmat_26", "rmat", {"spx.preproc.xform": "none"}, dict(scale=26)),
        # scaled-down versions (development, tests)
        "c5s": ("c5_rmat_22_scaled_down", "rmat", {"spx.preproc.xform": "none"}, dict(scale=22)),
        "c4s": ("c4_sym_block_banded_3M_scaled_down", "symbb", {"spx.matrix.symmetric": "true"}, dict(nb=1_000_000, b=1024)),
        "c4ns": ("c4_block_banded_3M_not_symmetric_mode_scaled_down", "symbb", {}, dict(nb=1_000_000, b=1024)),
        "c3s": ("c3_stencil27_128_scaled_down", "s27", {}, dict(g=128)),
        "c3bs": ("c3_stencil27_128_blocks_scaled_down", "s27", {"spx.preproc.xform": "br,bc"}, dict(g=128)),
        "c2q": ("c2_poisson2d_2048_quarter_size", "p2", {}, dict(g=2048)),
        "small": ("small_poisson2d_512", "p2", {}, dict(g=512)),
    }
    name, kind, opts, kw = W[key]
    return Workload(key, name, kind, opts, **kw)


def l2_policy(nnz, world):
    mb = 8.0 * nnz / world / 1e6
    if mb > 2 * 126:
        return "inputs larger than L2: %.0f MB of matrix values per GPU vs 126 MB L2, no flush between steps" % mb
    return ("per-GPU working set (%.0f MB of matrix values) is not larger than twice the 126 MB L2: consecutive steps can be "
            "served partly from L2 (no flush between steps)" % mb)


def config_of(W, nnz, world):
    """Identical in the GPU arm and in the CPU reference arm."""
    return {"workload": W.name, "rows": W.n, "nnz": int(nnz), "options": {k: str(v) for k, v in W.opts.items()},
            "l2_policy": l2_policy(nnz, world)}


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons of one GPU through NVML while the timed region runs."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.max_mhz = index, [], set(), None
        self._stop_evt = threading.Event()
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if not self.nv:
            return
        nv = self.nv
        names = {nv.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown",
                 nv.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
                 nv.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown",
                 nv.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap",
                 nv.nvmlClocksThrottleReasonHwPowerBrakeSlowdown: "hw_power_brake"}
        while not self._stop_evt.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.002)

    def finish(self):
        self._stop_evt.set()
        self.join(timeout=1)
        med = float(np.median(self.samples)) if self.samples else None
        return {"sm_mhz": med, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(self.samples)}


def pin_to_gpu_numa_node(index):
    """One process per GPU: run (and first-touch the pinned host buffers) on the cores NVML reports as local to the
    GPU, so that host<->device copies of different ranks do not cross the socket interconnect."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        ncpu = os.cpu_count() or 1
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (ncpu + 63) // 64)
        cpus = [w * 64 + b for w, word in enumerate(words) for b in range(64) if (word >> b) & 1 and w * 64 + b < ncpu]
        allowed = sorted(set(cpus) & set(os.sched_getaffinity(0)))
        if allowed:
            os.sched_setaffinity(0, allowed)
            return "cpus %d-%d (%d)" % (allowed[0], allowed[-1], len(allowed))
    except Exception as ex:  # affinity is an optimisation only
        return "not set: %r" % (ex,)
    return "not set"


def measured_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_traffic(name, world):
    """dram bytes per launch of the dominant kernel from a committed ncu --set full capture of this workload at this GPU
    count (profiles/ncu_traffic.json, keys "<workload>@<N>"); None when there is no such capture."""
    path = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if os.path.exists(path):
        try:
            return json.load(open(path)).get("%s@%d" % (name, world))
        except Exception:
            return None
    return None


def csr_check(rp, ci, va, row_lo, x_full, y_rows, alpha, nsample=100000, seed=7):
    """max over sampled rows of |y - alpha*A*x| / (|alpha| * |A| * |x|): rows [row_lo, row_lo + len(rp) - 1) given in CSR,
    x_full the whole input vector (only the columns these rows read need to be valid), y_rows the rows' results."""
    nrows = rp.size - 1
    if nrows == 0:
        return 0.0, 0
    rng = np.random.default_rng(seed)
    rows = np.unique(rng.integers(0, nrows, min(nsample, nrows)))
    starts, ends = rp[rows].astype(np.int64), rp[rows + 1].astype(np.int64)
    lens = ends - starts
    idx = np.repeat(starts - np.concatenate([[0], np.cumsum(lens)[:-1]]), lens) + np.arange(int(lens.sum()))
    seg = np.repeat(np.arange(rows.size), lens)
    prod = va[idx] * x_full[ci[idx]]
    ref = np.bincount(seg, weights=prod, minlength=rows.size)
    bound = np.bincount(seg, weights=np.abs(prod), minlength=rows.size)
    err = np.abs(y_rows[rows] - alpha * ref) / (abs(alpha) * bound + 1e-300)
    err[bound == 0] = np.abs(y_rows[rows][bound == 0])
    return float(err.max()) if err.size else 0.0, int(rows.size)


DUMP_MAX_ENTRIES = 1 << 22   # 32 MiB of float64 per dumped vector


def dump_outputs(directory, vectors):
    """Writes each float64 torch vector as <directory>/<name>.npy.  A vector longer than DUMP_MAX_ENTRIES is sampled: the
    entries at DUMP_MAX_ENTRIES distinct indices drawn by a generator seeded with 0, in increasing order, so that two runs
    of the same workload write the same rows."""
    import torch
    os.makedirs(directory, exist_ok=True)
    for name, v in vectors.items():
        if v.numel() > DUMP_MAX_ENTRIES:
            idx = np.sort(np.random.default_rng(0).choice(v.numel(), DUMP_MAX_ENTRIES, replace=False))
            v = v[torch.from_numpy(idx).to(v.device)]
        np.save(os.path.join(directory, name + ".npy"), v.cpu().numpy())


# ----------------------------------------------------------------- CPU arm --
def cpu_reference_run(W, steps, warmup, threads=None, max_nnz=None):
    """The reference's CPU path on this box's host cores, on the same matrix as the GPU arm: CSX with
    spx.rt.nr_threads = T partitions, one persistent pinned thread per partition running the reference's own kernel
    templates (oracle/_ref: src/templates/*.c compiled per partition by gcc, the barrier protocol of CsxKernels.cpp:82-103);
    falls back to the oracle's port of the same loops.  The CSX arrays come from this repository's host encoder, whose
    output is pinned bit for bit to the reference encoder's (tests/test_cpu_refpin.py) — the reference's own
    preprocessing of a matrix of this size takes minutes.  Matrices that one host cannot hold in reasonable time
    (R-MAT scale 26) are replaced by a bounded sample, which is said in the result."""
    from sparsex_b200.engine import CsxMatrix
    T = threads or (os.cpu_count() or 1)
    sample = "the whole matrix"
    if W.kind == "rmat" and W.kw["scale"] > 22:
        W = Workload(W.key, W.name, W.kind, W.opts, scale=22)
        sample = "R-MAT scale 22 instead of %s (bounded sample)" % W.name
    n = W.n
    t0 = time.time()
    rp, ci, va = W.rows(0, n, device="cpu" if W.kind == "rmat" else None)
    gen_s = time.time() - t0
    nnz = int(rp[-1])
    o = dict(W.opts)
    o["spx.rt.nr_threads"] = T
    o["spx.b200.rows_info"] = "false"
    t0 = time.time()
    A = CsxMatrix.tune_csr(rp, ci, va, n, n, o)
    tune_s = time.time() - t0
    del rp, ci, va
    parts = [A.partition(p) for p in range(A.nparts)]
    log = "; ".join("p%d: %s" % (i, P.log.strip()) for i, P in enumerate(parts))[:120]
    x = np.random.default_rng(2).uniform(-1, 1, n)
    kind = "port"
    runner = None
    try:
        from oracle import refkernels
        if refkernels.available():
            runner = refkernels.Runner(A, parts=parts, symmetric=W.sym).bench
            kind = "reference"
    except Exception:
        runner = None
    if runner is None:
        from oracle.pyoracle import OracleMatrix
        rp, ci, va = W.rows(0, n, device="cpu" if W.kind == "rmat" else None)
        o2 = dict(W.opts)
        o2["spx.rt.nr_threads"] = T
        o2["oracle.undefined_sampling"] = "break"
        runner = OracleMatrix.from_csr(rp, ci, va, n, n).tune(o2).bench
    A.close()
    if warmup:
        runner(0.5, x, warmup)
    secs = runner(0.5, x, steps)
    return {"value": 2.0 * nnz * steps / secs / 1e9, "unit": "GFLOP/s", "cores": T, "kind": kind, "nnz": nnz,
            "sample": "%s: %d rows, %d nnz, %d SpMVs on %d threads, CSX %s (generate %.0f s, tune %.0f s)" % (
                sample, n, nnz, steps, T, log, gen_s, tune_s),
            "ms_per_step": secs / steps * 1e3, "same_matrix": sample == "the whole matrix"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=128)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--outer", type=int, default=1, help="repeat the timed region this often and report the median "
                    "(the reference's protocol is --outer 5 --steps 128, src/bench/Bench.cpp:29-30)")
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--workload", default="c3")
    ap.add_argument("--e2e-steps", type=int, default=8)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-steps", type=int, default=16)
    ap.add_argument("--exchange", default="peer", choices=["peer", "nccl"],
                    help="N > 1: exchange fused into the SpMV kernel over peer memory (default) or NCCL after it")
    ap.add_argument("--graph-steps", type=int, default=16, help="steps per captured CUDA graph")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write y of the last timed step as DIR/y.npy (float64; vectors of more than "
                         "%d entries are sampled on fixed rows), so that two builds can be compared output for output; "
                         "GPU arm in one process only" % DUMP_MAX_ENTRIES)
    args = ap.parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl == "reference" or world > 1):
        ap.error("--dump-outputs is implemented for the GPU arm in one process")
    W = workload(args.workload)

    if args.impl == "reference":
        if rank != 0:
            return
        r = cpu_reference_run(W, max(args.steps, 1), args.warmup)
        nnz_full = int(W.counts("cpu" if W.kind == "rmat" and W.kw["scale"] <= 22 else None).sum()) if r["same_matrix"] else r["nnz"]
        line = {"impl": "reference", "metric": "csx_spmv_gflops", "value": r["value"], "unit": "GFLOP/s",
                "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": r["ms_per_step"],
                "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "config": config_of(W, nnz_full, max(world, args.gpus)),
                "detail": {"cpu_arm": r["sample"], "same_matrix": r["same_matrix"]},
                "cpu_baseline": {"value": r["value"], "unit": "GFLOP/s", "cores": r["cores"], "kind": r["kind"],
                                 "sample": r["sample"]},
                "e2e": {"value": r["value"], "unit": "GFLOP/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0}
        print(json.dumps(line))
        return

    import torch
    import torch.distributed as dist
    import sparsex_b200
    from sparsex_b200.engine import CsxMatrix

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a GPU (no CPU fallback); use --impl reference for the CPU arm")
    torch.cuda.set_device(local_rank)
    numa_note = pin_to_gpu_numa_node(local_rank) if world > 1 else None
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    api = sparsex_b200.load_spx_api()
    api.spx_init()
    L = sparsex_b200.lib()

    # ---- this rank's rows: the reference's nnz-balanced split with spx.rt.nr_threads = world, generated per rank ----
    t0 = time.time()
    n = W.n
    ranges = W.split(world, device="cuda")
    row_lo, row_n = ranges[rank]
    rp, ci, va = W.rows(row_lo, row_lo + row_n, device="cuda")
    nnz = int(W.counts().sum())
    gen_s = time.time() - t0
    all_opts = dict(W.opts)
    all_opts["spx.rt.nr_threads"] = world
    all_opts["spx.b200.rows_info"] = "false"
    for k, v in all_opts.items():
        api.spx_option_set(k.encode(), str(v).encode())
    api.spx_option_set(b"spx.b200.device", str(local_rank).encode())
    api.spx_option_set(b"spx.b200.part_lo", str(rank).encode())
    api.spx_option_set(b"spx.b200.part_hi", str(rank + 1).encode())
    if world > 1:   # the CSR arrays hold this rank's rows only (csxb_tune_csr_slab)
        api.spx_option_set(b"spx.b200.slab_row_start", str(row_lo).encode())
        api.spx_option_set(b"spx.b200.slab_total_rows", str(n).encode())
    t0 = time.time()
    inp = api.spx_input_load_csr(rp.ctypes.data, ci.ctypes.data, va.ctypes.data, rp.size - 1, n)
    A = api.spx_mat_tune(inp)
    if not A:
        raise SystemExit("spx_mat_tune failed")
    tune_s = time.time() - t0
    api.spx_input_destroy(inp)
    eng = CsxMatrix(api.spx_mat_get_engine(A))
    eng._h_owned = False
    enc_log = L.csxb_part_log(eng._h, 0).decode()
    if (L.csxb_part_info(eng._h, 0, 3), L.csxb_part_info(eng._h, 0, 8 if W.sym else 1)) != (row_lo, row_n):
        raise SystemExit("rank %d: the engine's partition rows differ from the split computed from the row lengths" % rank)
    traffic = eng.traffic()
    sym = W.sym

    # ---- device-resident timed region -----------------------------------------
    # alpha keeps the iteration x <- alpha*A*x bounded: 1 / max row sum of |A|
    amax = float(np.max(np.add.reduceat(np.abs(va), rp[:-1].astype(np.int64)[np.diff(rp) > 0]))) if rp[-1] else 1.0
    t = torch.tensor([amax], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    alpha = 1.0 / float(t[0])
    rng = np.random.default_rng(2)
    x0 = torch.from_numpy(rng.uniform(-1, 1, n)).cuda()
    x = x0.clone()
    y = torch.zeros(n, dtype=torch.float64, device="cuda")
    exchange = None
    xbuf = [x, y]   # ping-pong: the SpMV writes the own rows of the other buffer, the exchange fills the halo
    peer = None
    peer_note = None
    symred = None
    if world > 1 and args.exchange == "peer" and not sym:
        # the engine's own exchange: halo rows are stored into the neighbours' vectors by the SpMV kernel itself
        import sparsex_b200.dist as sdist
        peer, ranges_p, windows = sdist.connect_peer_exchange(eng, rank, world, "cuda")
        if peer is None:
            peer_note = "peer-memory exchange unavailable (%s): NCCL exchange used instead" % sdist.last_peer_error
    if peer is not None:
        peer.vector(0).copy_(x)
        exchange_kind = ("fused into the SpMV kernel: rows other ranks read are stored into their vectors over NVLink (peer memory), "
                         "device-side flags order the steps; protocol %d (1: edge tiles first, no sync kernel), %d edge tiles" % peer.protocol())
    if world > 1 and peer is None:
        from sparsex_b200.dist import PieceExchange, WindowExchange
        win = torch.tensor([L.csxb_part_info(eng._h, 0, 11), L.csxb_part_info(eng._h, 0, 12)], dtype=torch.int64, device="cuda")
        allwin = [torch.zeros(2, dtype=torch.int64, device="cuda") for _ in range(world)]
        dist.all_gather(allwin, win)
        windows = [(int(t[0]), int(t[1])) for t in allwin]
        if sym:   # CSX-Sym: transposed contributions to rows of lower ranks are sent to their owners and added
            from sparsex_b200.dist import SymHaloReduce
            hl = torch.tensor([L.csxb_info(eng._h, 8), L.csxb_info(eng._h, 9)], dtype=torch.int64, device="cuda")
            allh = [torch.zeros(2, dtype=torch.int64, device="cuda") for _ in range(world)]
            dist.all_gather(allh, hl)
            symred = SymHaloReduce(ranges, [(int(t[0]), int(t[1])) for t in allh], rank, y)
            windows = [(w[0], max(w[1], r[0] + r[1] - 1)) for w, r in zip(windows, ranges)]
        wx = WindowExchange(ranges, windows, rank)
        frac = torch.tensor([wx.fraction], dtype=torch.float64, device="cuda")
        dist.all_reduce(frac, op=dist.ReduceOp.MAX)
        if float(frac[0]) < 0.5:
            exchange, exchange_kind = wx, "halo exchange (grouped NCCL send/recv of the column windows, %.2g%% of the vector)" % (100 * float(frac[0]))
        else:
            pieces = [PieceExchange(xbuf[0], ranges), PieceExchange(xbuf[1], ranges)]
            exchange_kind = "NCCL all-gather of the y pieces"
        if sym:
            exchange_kind = "CSX-Sym halo reduction to the owners (grouped NCCL send/recv + add), then " + exchange_kind
    state = {"cur": 0}

    def step():
        if peer is not None:
            peer.spmv(alpha)
            return
        if world == 1:
            eng.spmv(alpha, x, y, overwrite=True)
            return
        src, dst = xbuf[state["cur"]], xbuf[1 - state["cur"]]
        eng.spmv(alpha, src, dst, overwrite=True)
        if sym and symred is not None:
            symred(dst)
        if exchange is not None:
            exchange(dst)
        else:  # dst's own rows -> every rank's dst
            pieces[1 - state["cur"]](dst[row_lo:row_lo + row_n])
        state["cur"] = 1 - state["cur"]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # A step is kernel launches only when there is no NCCL call in it (N = 1, or the peer exchange): G steps are captured
    # into one CUDA graph (N > 1: the step counter and the buffer parity live on the device, the graph is replayable)
    graph, G = None, 1
    graphable = world == 1 or peer is not None
    if graphable and args.graph_steps > 1:
        G = min(args.graph_steps, args.steps)
        while G > 1 and (args.steps % G or (peer is not None and G % 2)):
            G -= 1
    for _ in range(max(args.warmup, 3)):
        step()
    barrier()
    if G > 1:
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.stream(side):
            with torch.cuda.graph(graph, stream=side):
                for _ in range(G):
                    step()
        torch.cuda.current_stream().wait_stream(side)
        barrier()
        graph.replay()   # one untimed replay
        barrier()

    def timed_region():
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record()
        if graph is not None:
            for _ in range(args.steps // G):
                graph.replay()
        else:
            for _ in range(args.steps):
                step()
        e1.record()
        barrier()
        t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t[0])

    sampler = ClockSampler(local_rank)
    sampler.start()
    region_ms = [timed_region() for _ in range(max(args.outer, 1))]
    # the timed region can be a few milliseconds: keep the same load running, untimed, until the clock sampler has
    # seen it for at least 100 ms.  The number of extra steps is the same on every rank (a rank that issued more steps than
    # its neighbours would wait for them forever).
    ms_med = float(np.median(region_ms))
    extra = int(np.ceil(100.0 / max(ms_med / args.steps, 1e-3)))
    if graph is not None:
        for _ in range((extra + G - 1) // G):
            graph.replay()
    else:
        for _ in range(extra):
            step()
    torch.cuda.synchronize()
    barrier()
    clocks = sampler.finish()
    if args.dump_outputs:   # one process (checked above): every step, the untimed ones after the timed region too, writes
        dump_outputs(args.dump_outputs, {"y": y})   # the same y = alpha*A*x from the same x
    ms = float(np.median(region_ms))
    value = 2.0 * nnz * args.steps / (ms * 1e-3) / 1e9
    if peer is not None and peer.error():
        raise SystemExit("peer exchange: a wait for a neighbour timed out")

    # this rank's SpMV kernels alone (no exchange, no neighbour), timed the same way: a graph of G launches
    kernel_only_ms = None
    if world > 1:
        xs, ys = x0.clone(), torch.zeros_like(x0)
        for _ in range(3):
            eng.spmv(alpha, xs, ys, overwrite=True)
        torch.cuda.synchronize()
        side2 = torch.cuda.Stream()
        side2.wait_stream(torch.cuda.current_stream())
        g2 = torch.cuda.CUDAGraph()
        with torch.cuda.stream(side2):
            with torch.cuda.graph(g2, stream=side2):
                for _ in range(16):
                    eng.spmv(alpha, xs, ys, overwrite=True)
        torch.cuda.current_stream().wait_stream(side2)
        g2.replay()
        torch.cuda.synchronize()
        ka, kb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ka.record()
        for _ in range(4):
            g2.replay()
        kb.record()
        torch.cuda.synchronize()
        t = torch.tensor([ka.elapsed_time(kb) / 64], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        kernel_only_ms = float(t[0])
        del xs, ys, g2

    # ---- check against the CSR product on sampled rows (componentwise, SURVEY 8d tolerance 1e-12) -----------------------
    # (a) the device path on a fresh x; (b) N > 1: one more step of the exchange from a fresh vector — this rank's rows of
    # the target vector against CSR, and the rows it received from the other ranks against what they computed
    checks = {}
    xs = x0.clone()
    ys = torch.full_like(x0, float("nan"))
    eng.spmv(alpha, xs, ys, overwrite=True)
    torch.cuda.synchronize()
    x0h = x0.cpu().numpy()
    err, nchk = csr_check(rp, ci, va, row_lo, x0h, ys[row_lo:row_lo + row_n].cpu().numpy(), alpha)
    if sym and world > 1:
        err, nchk = None, 0   # own rows also receive the other ranks' transposed contributions: checked through the exchange below
    checks["device_path_max_err"] = err
    checks["rows_sampled_per_rank"] = nchk
    if world > 1:
        if peer is not None:
            cur = peer.steps() & 1
            peer.vector(cur).copy_(x0)
            barrier()
            peer.spmv(alpha)
            torch.cuda.synchronize()
            barrier()
            vnext = peer.vector(cur ^ 1)
        else:
            xbuf[state["cur"]].copy_(x0)
            barrier()
            step()
            torch.cuda.synchronize()
            vnext = xbuf[state["cur"]]
        vh = vnext.cpu().numpy()
        e_own, _ = csr_check(rp, ci, va, row_lo, x0h, vh[row_lo:row_lo + row_n], alpha)
        # halo: the columns this rank reads that other ranks own must equal what their owners hold
        own = torch.zeros(n, dtype=torch.float64, device="cuda")
        own[row_lo:row_lo + row_n] = vnext[row_lo:row_lo + row_n]
        dist.all_reduce(own)   # every row's owner's value
        wlo, whi = L.csxb_part_info(eng._h, 0, 11), L.csxb_part_info(eng._h, 0, 12)
        cov = ranges[-1][0] + ranges[-1][1]
        whi = min(whi, cov - 1)
        e_halo = float((vnext[wlo:whi + 1] - own[wlo:whi + 1]).abs().max()) if whi >= wlo else 0.0
        t = torch.tensor([e_own, e_halo], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        checks["exchange_own_rows_max_err"] = float(t[0])
        checks["exchange_halo_max_abs_diff"] = float(t[1])
        del own
    t = torch.tensor([checks["device_path_max_err"] or 0.0], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    if checks["device_path_max_err"] is not None or world == 1:
        checks["device_path_max_err"] = float(t[0])
    bad = [k for k in ("device_path_max_err", "exchange_own_rows_max_err") if checks.get(k) is not None and not checks[k] <= 1e-12]
    if checks.get("exchange_halo_max_abs_diff", 0.0) != 0.0:
        bad.append("exchange_halo_max_abs_diff")
    if bad:
        raise SystemExit("bench.py: result check failed: %r" % (checks,))

    # ---- end to end through spx_matvec_mult with host buffers ---------------------
    xh = torch.from_numpy(rng.uniform(-1, 1, n)).pin_memory()
    yh = torch.zeros(n, dtype=torch.float64).pin_memory()
    vx = api.spx_vec_create_from_buff(xh.data_ptr(), None, n, None, 43)
    vy = api.spx_vec_create_from_buff(yh.data_ptr(), None, n, None, 43)
    for _ in range(6):   # warm-up; the library's host-buffer path settles its slab-kernel setting in the first five calls
        api.spx_matvec_mult(alpha, A, vx, vy)
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.e2e_steps):
        if api.spx_matvec_mult(alpha, A, vx, vy) != 0:
            raise SystemExit("spx_matvec_mult failed")
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    t = torch.tensor([e2e_s], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_s = float(t[0])
    cw_lo, cw_hi = L.csxb_part_info(eng._h, 0, 11), L.csxb_part_info(eng._h, 0, 12)
    hb = torch.tensor([8.0 * (n if sym else max(0, cw_hi - cw_lo + 1)), 8.0 * row_n], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(hb)
    if not (sym and world > 1):
        e_e2e, _ = csr_check(rp, ci, va, row_lo, xh.numpy(), yh.numpy()[row_lo:row_lo + row_n], alpha)
        t = torch.tensor([e_e2e], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        checks["host_buffer_path_max_err"] = float(t[0])
        if not checks["host_buffer_path_max_err"] <= 1e-12:
            raise SystemExit("bench.py: result check failed: %r" % (checks,))
    e2e = {"value": 2.0 * nnz * args.e2e_steps / e2e_s / 1e9, "unit": "GFLOP/s", "h2d_bytes_per_step": int(hb[0]),
           "d2h_bytes_per_step": int(hb[1]), "steps": args.e2e_steps,
           "host_affinity": numa_note,
           "slab_kernel_cap_bytes": int(L.csxb_info(eng._h, 10)),
           "api": "spx_matvec_mult on spx_vec_create_from_buff vectors (pinned host memory); every rank uploads the "
                  "columns its partition reads and downloads its rows, slab-pipelined (H2D, kernels, D2H overlap)"}
    peer_sync_kernel = peer is not None and peer.protocol()[0] == 0   # protocol 0 ends every step with a sync kernel
    if peer is not None:
        barrier()
        peer.close()

    if rank == 0:
        peak, peak_src = measured_peak()
        step_ms = ms / args.steps
        achieved = traffic["total"] / (step_ms * 1e-3) / 1e9
        line = {"metric": "csx_spmv_gflops", "value": value, "unit": "GFLOP/s", "n_gpus": world, "steps": args.steps,
                "warmup": max(args.warmup, 3), "ms_per_step": step_ms, "higher_is_better": True,
                "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "config": config_of(W, nnz, world),
                "detail": {"options": {k: str(v) for k, v in all_opts.items()}, "encoding_rank0": enc_log.strip(), "alpha": alpha,
                           "step": "y = alpha*A*x (spx_matvec_mult semantics)" + (
                               "; then " + exchange_kind + " into the next x" if world > 1 else ""),
                           "protocol": "%d x %d steps, median of the repeats; CUDA graphs of %d steps" % (max(args.outer, 1), args.steps, G)
                                       if graph is not None else "%d x %d steps, median of the repeats" % (max(args.outer, 1), args.steps),
                           "region_ms": region_ms, "rows_rank0": row_n,
                           "exchange_note": peer_note, "tune_s": round(tune_s, 2), "generate_s": round(gen_s, 2),
                           "checks_vs_csr": checks},
                "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                             "traffic": ncu_traffic(W.name, world), "peak_source": peak_src,
                             "kernel": "rank 0's SpMV kernels (gather kernel csx_spmv_kernel; stream kernel where the partition has "
                                       "stream units)" + ("; N > 1: the step of the captured graph includes the fused exchange" if world > 1 else ""),
                             "kernel_ms": step_ms, "kernel_only_ms": kernel_only_ms,
                             "algorithmic_bytes": traffic["total"],
                             "bytes": {k: traffic[k] for k in ("values", "ctl", "tables", "x", "y")},
                             "frac_of_8TBs_nominal": achieved / 8000.0},
                "e2e": e2e, "gpu_launches": (int(traffic["launches"]) + (1 if peer_sync_kernel else 0)) * args.steps * max(args.outer, 1),
                "clocks": clocks}
        if world == 1 and not args.no_cpu_baseline:
            try:
                r = cpu_reference_run(W, args.cpu_steps, 2)
                line["cpu_baseline"] = {"value": r["value"], "unit": "GFLOP/s", "cores": r["cores"], "kind": r["kind"],
                                        "sample": r["sample"]}
            except Exception as ex:  # the CPU baseline is reported, never required for the GPU number
                line["cpu_baseline"] = {"value": None, "unit": "GFLOP/s", "cores": 0, "kind": "port",
                                        "sample": "failed: %r" % (ex,)}
        print(json.dumps(line))
    api.spx_vec_destroy(vx)
    api.spx_vec_destroy(vy)
    eng._h = None  # owned by the spx matrix handle
    api.spx_mat_destroy(A)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
