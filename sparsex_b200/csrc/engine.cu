// CUDA kernels (sm_100a) and the csxb_* C-ABI of the B200 CSX SpMV engine.
//
// Execution model (see gpu_layout.hpp for the tables), up to three kernels per partition on one stream:
//   1. csx_stream_kernel  (stream_kernel.cuh) one warp per chunk of the ctl stream: unit heads parsed one per lane,
//                        units cut into lane tasks (elements of a delta / horizontal unit, block tasks with register
//                        accumulators), row sums combined with segmented shuffle reductions in a shared-memory window
//                        of y rows and written with plain stores (y = alpha*sum + beta*y).  Instantiated per pattern set.
//   2. csx_stream_fixup_kernel  adds what chunks contributed to rows of other chunks, clears long runs of empty rows.
//   3. csx_spmv_kernel   (gather_kernel.cuh) one CTA per tile of 256 / 1024 rows; every thread owns rows and gathers
//                        the contributions of the table units (vertical, diagonal, anti-diagonal; under CSX-Sym also
//                        the transposed image of every unit) listed for its tile, then adds them to y (or writes y
//                        when the partition has no stream units).  No atomics anywhere: results are bit-reproducible.
// Host-buffer calls are slab-pipelined (csxb_spmv_host); repeated SpMV across GPUs exchanges the halo rows from
// inside kernel 3 over CUDA-IPC peer memory (csxb_xchg_*, csx_spmv_xe_kernel).
// SpMV is HBM-bound fp64 work: no tensor cores; every value and ctl byte is read once.
//
// Reference semantics reproduced: src/templates/csx_spmv_tmpl.c:66-101 and the
// nine unit templates (delta/horiz/vert/diag/rdiag/block_row/block_col), the
// symmetric variants (csx_sym_spmv_tmpl.c:60-106, *_sym_tmpl.c) and the
// y handling of CsxKernels.cpp:35-129 / CsxSpmv.cpp:28-86.
#include <cuda_runtime.h>

#include <chrono>
#include <memory>

#include <climits>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <sstream>
#include <string>
#include <type_traits>
#include <vector>

#include "../../include/csx_b200.h"
#include "csx_host.hpp"
#include "gpu_layout.hpp"
#include "part_dev.cuh"
#include "stream_kernel.cuh"

#include "gather_kernel.cuh"

__device__ __forceinline__ unsigned long long ld_acquire_sys(const unsigned long long *p) {
  unsigned long long v;
  asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_release_sys(unsigned long long *p, unsigned long long v) {
  asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
// Edge CTA of the edge-tiles-first protocol (XchgDev.mode 1): waits for the neighbours' edge tiles of the previous
// step, computes and pushes its tile, and the last edge CTA of the step publishes it.  Kept out of line so that
// the interior path of the kernel keeps the register allocation of the plain kernel.
// x is read with L1-bypassing loads here: the neighbours write the halo rows of this vector while the kernel runs.
template <bool XD, bool SYM, int RPT, int KSET, int VAR, bool BT>
__device__ __noinline__ void spmv_edge_cta(const PartDev &P, const double *x, double *y, double alpha, long long tile,
                                           long long row_block, const XchgDev &X, int ypar) {
  // only the edge CTAs use the device-resident step number (the flags count steps across graph replays)
  const unsigned long long xk = *reinterpret_cast<const volatile unsigned long long *>(X.step);
  if (threadIdx.x == 0 && xk > 0) {   // halo of this step arrived; the neighbours no longer read the buffer pushed into
    for (int i = 0; i < X.nwait; i++) {
      const unsigned long long *f = X.flags + X.wait_rank[i];
      const long long t0 = clock64();
      while (ld_acquire_sys(f) < xk) {
        if (clock64() - t0 > 6000000000ll) { atomicExch(X.error, 1ull); break; }
      }
    }
  }
  __syncthreads();
  // spmv_tile pushes into push_vec[p][(k & 1) ^ 1]: hand it a step number with the parity of the target buffer
  spmv_tile<XD, SYM, RPT, KSET, VAR, true, XchgDev, BT, true>(P, x, y, alpha, 0.0, 1, tile, row_block, X, (unsigned long long)(ypar ^ 1));
  // Every edge CTA orders its stores before its count at device scope; the last one then issues the single
  // system-scope fence (cumulative over everything that happened before it) and the release stores of the flags.
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0 && atomicAdd(X.bdone, 1ull) == (unsigned long long)X.nb - 1) {   // last edge CTA of the step
    *reinterpret_cast<volatile unsigned long long *>(X.bdone) = 0;
    *reinterpret_cast<volatile unsigned long long *>(X.step) = xk + 1;
    __threadfence_system();
    for (int i = 0; i < X.nwait; i++) st_release_sys(X.peer_flags[i] + X.rank, xk + 1);
  }
}

template <bool XD, bool SYM, int RPT, int KSET, int MINB = 8, int VAR = 0, class XP = NoXchg, bool BT = false>
__global__ void __launch_bounds__(CTA_THREADS, MINB) csx_spmv_kernel(const __grid_constant__ PartDev P,
                                                                  const double *__restrict__ x,
                                                                  double *__restrict__ y, double alpha, double beta,
                                                                  int overwrite, const __grid_constant__ XP X) {
  constexpr bool XCHG = !std::is_same<XP, NoXchg>::value;
  const long long tile = (long long)blockIdx.x + P.tile0;
  unsigned long long xk = 0;
  if constexpr (XCHG) {   // vectors by step parity (protocol 0: the sync kernel that ended the previous step saw the halo arrive)
    xk = *reinterpret_cast<const volatile unsigned long long *>(X.step);
    x = X.vec[xk & 1]; y = X.vec[(xk & 1) ^ 1];
  }
  spmv_tile<XD, SYM, RPT, KSET, VAR, XCHG, XP, BT>(P, x, y, alpha, beta, overwrite, tile, tile, X, xk);
}

// Kernel 1 under the edge-tiles-first protocol (XchgDev.mode 1): CTAs [0, nb) take the tiles at both ends of the
// partition (out of line: wait, compute, push, publish), the others the interior tiles, which touch no other rank
// and run exactly the plain tile code.  x / y are the step's source and target vectors (the host alternates them,
// so a captured graph must hold an even number of steps); `ypar` is the index of y among the ping-pong vectors.
template <bool XD, int RPT, int KSET, int MINB = 8, int VAR = 0, bool BT = false>
__global__ void __launch_bounds__(CTA_THREADS, MINB) csx_spmv_xe_kernel(const __grid_constant__ PartDev P,
                                                                     const double *__restrict__ x, double *__restrict__ y,
                                                                     double alpha, int ypar, const __grid_constant__ XchgDev X) {
  const int b = (int)blockIdx.x;
  if (b < X.nb) {
    // Edge CTAs walk their tile with one row per thread (a 4-rows-per-thread tile is split over four CTAs): the sooner
    // the edge rows are out, the more slack the neighbours have before their next step needs them.
    // With many edge tiles (a 3-D stencil: 65 tiles per side) the split costs more than it gains: whole tiles then.
    if (RPT == 4 && X.split == 1) {
      const long long tile = b < X.edge_lo_end ? b : X.edge_hi_begin + (b - X.edge_lo_end);
      spmv_edge_cta<XD, false, RPT, KSET, 0, BT>(P, x, y, alpha, tile, tile, X, ypar);
      return;
    }
    constexpr int SPLIT = RPT == 4 ? 4 : 1;
    const int bt = b / SPLIT, sub = b % SPLIT;
    const long long tile = bt < X.edge_lo_end ? bt : X.edge_hi_begin + (bt - X.edge_lo_end);
    spmv_edge_cta<XD, false, 1, KSET, 0, BT>(P, x, y, alpha, tile, tile * SPLIT + sub, X, ypar);
  } else {
    const long long tile = (long long)X.edge_lo_end + (b - X.nb);
    spmv_tile<XD, false, RPT, KSET, VAR, false, NoXchg, BT>(P, x, y, alpha, 0.0, 1, tile, tile, NoXchg(), 0ull);
  }
}

// Exchange for partitions whose rows are only final after the last kernel of the step (stream units): copies the rows
// the peers read into their vectors.  Every element is loaded once (16 bytes per thread where aligned) and stored to
// every peer that reads it.
__global__ void __launch_bounds__(256) csx_xchg_push_kernel(const __grid_constant__ XchgDev X) {
  const unsigned long long k = *reinterpret_cast<const volatile unsigned long long *>(X.step);
  const int par = (int)((k & 1) ^ 1);
  const double *src = X.vec[par];
  long long lo = LLONG_MAX, hi = 0;
  for (int p = 0; p < X.npush; p++) { lo = min(lo, X.push_lo[p]); hi = max(hi, X.push_hi[p]); }
  lo &= ~1ll;   // pairs of rows: the vectors are 16-byte aligned
  const long long stride = 2ll * gridDim.x * blockDim.x;
  for (long long g = lo + 2ll * ((long long)blockIdx.x * blockDim.x + threadIdx.x); g < hi; g += stride) {
    if (g + 1 < hi && g >= lo) {
      const double2 v = *reinterpret_cast<const double2 *>(src + g);
      for (int p = 0; p < X.npush; p++) {
        double *dst = X.push_vec[p][par];
        if (g >= X.push_lo[p] && g + 1 < X.push_hi[p]) *reinterpret_cast<double2 *>(dst + g) = v;
        else {
          if (g >= X.push_lo[p] && g < X.push_hi[p]) dst[g] = v.x;
          if (g + 1 >= X.push_lo[p] && g + 1 < X.push_hi[p]) dst[g + 1] = v.y;
        }
      }
    } else {
      for (long long q = g; q < g + 2 && q < hi; q++)
        for (int p = 0; p < X.npush; p++)
          if (q >= X.push_lo[p] && q < X.push_hi[p]) X.push_vec[p][par][q] = src[q];
    }
  }
}
// Rows past the last partition's rows belong to nobody: zero in every step's result (VecInit(y, 0), CsxKernels.cpp:93).
__global__ void __launch_bounds__(256) csx_xchg_zero_tail_kernel(const __grid_constant__ XchgDev X, long long lo, long long hi,
                                                                 int ypar) {
  const unsigned long long k = *reinterpret_cast<const volatile unsigned long long *>(X.step);
  double *dst = X.vec[ypar >= 0 ? ypar : (int)((k & 1) ^ 1)];   // protocol 1: the host names the step's target vector
  for (long long g = lo + (long long)blockIdx.x * blockDim.x + threadIdx.x; g < hi; g += (long long)gridDim.x * blockDim.x) dst[g] = 0.0;
}
// End of a step (one warp): publish "rank finished step k" to every neighbour, advance the local step counter,
// then wait until every neighbour has finished step k as well — its halo rows for the next step have arrived
// and it no longer reads the buffer the next step overwrites.  Runs after the step's kernels on the same stream,
// so their stores (local and peer) are complete; the next step's kernels start after it.  The wait is bounded:
// a lost peer sets the error word instead of hanging the device.
__global__ void csx_xchg_sync_kernel(const __grid_constant__ XchgDev X, int dbg) {
  const int lane = threadIdx.x;
  const unsigned long long k = *reinterpret_cast<const volatile unsigned long long *>(X.step);
  if (!(dbg & 2)) __threadfence_system();
  if (lane < X.nwait) st_release_sys(X.peer_flags[lane] + X.rank, k + 1);
  if (lane == 0) *reinterpret_cast<volatile unsigned long long *>(X.step) = k + 1;
  if (lane < X.nwait) {
    const unsigned long long *f = X.flags + X.wait_rank[lane];
    const long long t0 = clock64();
    while (ld_acquire_sys(f) < k + 1) {
      if (clock64() - t0 > 6000000000ll) { atomicExch(X.error, 1ull); break; }
    }
  }
}

struct DecodeGatherOp {
  int *rows, *cols;   // device-wide
  int myrow;
  __device__ __forceinline__ void add(uint32_t vi, int col) { rows[vi] = myrow; cols[vi] = col; }
};
// decoded coordinates of the block-table units (their own rows; images repeat the same values)
__global__ void __launch_bounds__(CTA_THREADS) csx_decode_bt_kernel(const __grid_constant__ PartDev P, int *rows, int *cols) {
  const long long lrow = (long long)blockIdx.x * CTA_THREADS + threadIdx.x;
  if (lrow >= P.nrows) return;
  const long long g = P.row_start + lrow;
  for (int c = 0; c < P.nbt; c++) {
    const BtDev &T = P.bt[c];
    if (T.image) continue;
    const long long J = g / T.G;
    const int f = (int)(g - J * T.G) * T.sf;
    for (uint32_t e = T.ptr[J - T.j0]; e < T.ptr[J - T.j0 + 1]; e++) {
      const uint2 b = T.ent[e];
      if (b.y & BT_IMAGE) continue;
      for (int l = 0; l < T.nloop; l++) { rows[b.x + f + l * T.sl] = (int)g; cols[b.x + f + l * T.sl] = (int)b.y + l; }
    }
  }
}
__global__ void __launch_bounds__(CTA_THREADS) csx_decode_gather_kernel(const __grid_constant__ PartDev P, int *rows, int *cols) {
  const long long tile = blockIdx.x;
  const uint32_t b = __ldg(P.tile_xoff + tile), e = __ldg(P.tile_xoff + tile + 1);
  for (int k = 0; k < P.rpt; k++) {
    const long long lrow = (tile * P.rpt + k) * CTA_THREADS + threadIdx.x;
    if (lrow >= P.nrows) return;
    DecodeGatherOp op{rows, cols, (int)(P.row_start + lrow)};
    for (uint32_t j = b; j < e; j++) {
      const uint4 d = __ldg(P.xdesc + j);
      if (d.w & XD_TRANSPOSED) continue;
      gather_desc<false>(d, P.ktab, op.myrow, op);
    }
  }
}

// ---- kernel 2 of non-symmetric partitions: stream kernel (stream_kernel.cuh), one warp per chunk ----------------
__device__ __forceinline__ int sk_vectors(const SkIO &io, const double *&x, double *&y) {
  x = io.x; y = io.y;
  if (io.step) {   // multi-GPU exchange: vectors by step parity
    const unsigned long long k = *reinterpret_cast<const volatile unsigned long long *>(io.step);
    x = io.vec[k & 1]; y = io.vec[(k & 1) ^ 1];
    return (int)((k & 1) ^ 1);
  }
  return 0;
}
template <int R, uint32_t KM, int BC, int BRC>
__global__ void __launch_bounds__(SK_WARPS * 32, 4) csx_stream_kernel(const __grid_constant__ PartDev P, const __grid_constant__ SkIO io,
                                                                     double alpha, double beta, int overwrite) {
  __shared__ double sacc[SK_WARPS][SK_WIN];
  __shared__ uint4 sid[64];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (threadIdx.x < 64) {
    const IdEntry &ie = P.idtab[threadIdx.x];
    sid[threadIdx.x] = make_uint4(ie.kind_align, ie.delta, ie.sl, ie.recip);
  }
  __syncthreads();
  const uint32_t ch = P.sk_c0 + blockIdx.x * SK_WARPS + warp;
  if (ch >= P.sk_c1) return;
  const double *x; double *y;
  const int ypar = sk_vectors(io, x, y);
  sk_chunk<R, KM, BC, BRC, false>(P, ch, sacc[warp], sid, lane, x, y, alpha, beta, overwrite, nullptr, nullptr, &io, ypar);
}
__global__ void __launch_bounds__(SK_WARPS * 32) csx_stream_decode_kernel(const __grid_constant__ PartDev P, int *rows, int *cols) {
  __shared__ double sacc[SK_WARPS][SK_WIN];
  __shared__ uint4 sid[64];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (threadIdx.x < 64) {
    const IdEntry &ie = P.idtab[threadIdx.x];
    sid[threadIdx.x] = make_uint4(ie.kind_align, ie.delta, ie.sl, ie.recip);
  }
  __syncthreads();
  const uint32_t ch = P.sk_c0 + blockIdx.x * SK_WARPS + warp;
  if (ch >= P.sk_c1) return;
  sk_chunk<8, SKM_ROWLOCAL | SKM_BROW | SKM_BCOL, 0, 0, true>(P, ch, sacc[warp], sid, lane, nullptr, nullptr, 0.0, 0.0, 1,
                                                               rows + P.val_base, cols + P.val_base);
}
// After the stream kernel: adds what chunks contributed to rows of other chunks (in chunk order: deterministic) and
// clears the rows no chunk window covers (long runs of empty rows), clipped to [clip_lo, clip_hi).
__global__ void __launch_bounds__(256) csx_stream_fixup_kernel(const __grid_constant__ PartDev P, const __grid_constant__ SkIO io,
                                                                double alpha, double beta, int overwrite, long long clip_lo,
                                                                long long clip_hi) {
  const double *x; double *y;
  const int ypar = sk_vectors(io, x, y);
  const long long tid = (long long)blockIdx.x * blockDim.x + threadIdx.x, nth = (long long)gridDim.x * blockDim.x;
  for (long long i = P.sk_f0 + tid; i < P.sk_f1; i += nth) {
    double s = 0.0;
    for (uint32_t j = P.sk_fix_ptr[i]; j < P.sk_fix_ptr[i + 1]; j++) s += P.sk_scratch[P.sk_fix_idx[j]];
    const long long g = P.row_start + P.sk_fix_rows[i];
    const double v = y[g] + alpha * s;
    y[g] = v;
    sk_push(io, ypar, g, v);   // (the stream kernel pushed the row without these sums: the final value follows)
  }
  for (uint32_t g = P.sk_g0 + blockIdx.x; g < P.sk_g1; g += gridDim.x) {   // one CTA per gap (most gaps are short)
    const long long lo = max(P.sk_gaps[2 * g], clip_lo), hi = min(P.sk_gaps[2 * g + 1], clip_hi);
    for (long long r = lo + threadIdx.x; r < hi; r += blockDim.x) {
      double *yp = y + P.row_start + r;
      const double v = overwrite ? 0.0 : beta * *yp;
      *yp = v;
      sk_push(io, ypar, P.row_start + r, v);
    }
  }
}

// Heavy columns of the transposed product: one warp per segment (gather_kernel.cuh: t_segment_warp).
__global__ void __launch_bounds__(256) csx_t_segment_kernel(const uint2 *__restrict__ ent, const uint32_t *__restrict__ seg,
                                                            uint32_t nseg, const double *__restrict__ values,
                                                            const double *__restrict__ x, double *__restrict__ scratch) {
  const uint32_t s = blockIdx.x * 8 + (threadIdx.x >> 5);
  if (s >= nseg) return;
  t_segment_warp(ent, seg, values, x, scratch, s, (int)(threadIdx.x & 31));
}

// --------------------------------------------------------------- host side --
static thread_local std::string g_last_error;
static int fail(const std::string &m) { g_last_error = m; return -1; }
#define CUDA_TRY(call)                                                                         \
  do {                                                                                         \
    cudaError_t e_ = (call);                                                                   \
    if (e_ != cudaSuccess)                                                                     \
      return fail(std::string(#call) + ": " + cudaGetErrorString(e_));                         \
  } while (0)

// Tables of the transposed product on the device (csxb_transpose_prepare); they reference the forward values.
struct TransState {
  TransLayout lay;
  PartDev P;                           // row owner = columns of A; heavy-column fix-up in P.sk_fix_*
  const uint2 *hent = nullptr;         // heavy-column segments
  const uint32_t *hseg = nullptr;
  int64_t dev_bytes = 0, alg_bytes = 0, launches = 0, build_us = 0;
  double *d_x = nullptr, *d_y = nullptr;   // staging for csxb_spmv_t_host (nrows / ncols doubles)
};

struct csxb_matrix {
  CsxMatrix host;
  DeviceLayout layout;
  bool uploaded = false;
  int device = -1;
  std::vector<void *> allocs;
  std::vector<PartDev> pdev;
  double *d_values = nullptr;
  double *d_x = nullptr, *d_y = nullptr;   // staging for csxb_spmv_host
  int64_t covered_rows_end = 0;
  int64_t sym_halo_lo = 0, sym_halo_hi = 0;   // CSX-Sym, partial device: rows of other devices this one adds into
  // pipelined host-buffer path (csxb_spmv_host): row slabs with the x columns they need and the y rows that are
  // final once they have run
  struct Slab {
    int part; int64_t tile0, tile1;
    uint32_t chunk0, chunk1, f0, f1, g0, g1;   // stream-kernel chunks, fix rows and gaps that run with this slab
    int64_t x_lo, x_hi, row_lo, row_hi, y_lo, y_hi, yup_hi;
  };
  std::vector<Slab> slabs;
  std::vector<cudaEvent_t> slab_ev;
  cudaStream_t s_h2d = nullptr, s_run = nullptr, s_d2h = nullptr;
  int host_calls = 0;                  // csxb_spmv_host: calls so far (the first five choose host_cap)
  double host_tune_s[2] = {0.0, 0.0};  // best time with the cap [0] and without [1]
  size_t host_cap = 0;                 // dynamic shared memory per CTA of the slab kernels (caps the resident CTAs)
  int64_t bytes[7] = {0, 0, 0, 0, 0, 0, 0};
  std::vector<std::string> logs;
  std::vector<RowIndex> row_index;   // per partition, built on the first csxb_get/set_entry
  std::unique_ptr<TransState> trans;   // csxb_transpose_prepare (its device arrays are in allocs)
  ~csxb_matrix() {
    if (!allocs.empty() || d_x || d_y || s_h2d) {
      int cur = -1;
      cudaGetDevice(&cur);
      if (device >= 0) cudaSetDevice(device);
      for (void *p : allocs) cudaFree(p);
      if (d_x) cudaFree(d_x);
      if (d_y) cudaFree(d_y);
      for (cudaEvent_t e : slab_ev) cudaEventDestroy(e);
      if (s_h2d) { cudaStreamDestroy(s_h2d); cudaStreamDestroy(s_run); cudaStreamDestroy(s_d2h); }
      if (cur >= 0) cudaSetDevice(cur);
    }
  }
};

static std::string parse_options(const char *options, TuneOptions &o) {
  if (!options) return "";
  std::stringstream ss(options);
  std::string kv;
  while (std::getline(ss, kv, ';')) {
    if (kv.empty()) continue;
    size_t eq = kv.find('=');
    if (eq == std::string::npos) return "malformed option \"" + kv + "\"";
    std::string e = o.set(kv.substr(0, eq), kv.substr(eq + 1));
    if (!e.empty()) return e;
  }
  return "";
}
static void put_err(char *err, size_t n, const std::string &m) {
  g_last_error = m;
  if (err && n) { strncpy(err, m.c_str(), n - 1); err[n - 1] = 0; }
}

// C++ entry used by api.cpp for inputs already parsed into memory (spx_input_load_mmf)
csxb_matrix_t *csxb_tune_coo_internal(const CooHost &coo, const char *options, int part_lo, int part_hi, char *err, size_t errlen) {
  TuneOptions o;
  std::string e = parse_options(options, o);
  if (!e.empty()) { put_err(err, errlen, e); return nullptr; }
  if (part_hi < 0) { part_lo = 0; part_hi = o.nr_threads; }
  csxb_matrix *m = new csxb_matrix;
  e = tune_coo(coo, o, part_lo, part_hi, m->host);
  if (!e.empty()) { put_err(err, errlen, e); delete m; return nullptr; }
  return m;
}

extern "C" {

csxb_matrix_t *csxb_tune_csr(const int32_t *rowptr, const int32_t *colind, const double *values, int64_t nrows,
                             int64_t ncols, const char *options, int part_lo, int part_hi, char *err, size_t errlen) {
  TuneOptions o;
  std::string e = parse_options(options, o);
  if (e.empty() && (!rowptr || !colind || !values || nrows < 0 || ncols < 0)) e = "invalid CSR arguments";
  if (e.empty() && rowptr[0] != 0) e = "CSR arrays must be zero-based";
  if (!e.empty()) { put_err(err, errlen, e); return nullptr; }
  if (part_hi < 0) { part_lo = 0; part_hi = o.nr_threads; }
  csxb_matrix *m = new csxb_matrix;
  CsrView v{rowptr, colind, values, nrows, ncols};
  e = tune_csr(v, o, part_lo, part_hi, m->host);
  if (!e.empty()) { put_err(err, errlen, e); delete m; return nullptr; }
  return m;
}

csxb_matrix_t *csxb_tune_csr_slab(const int32_t *rowptr, const int32_t *colind, const double *values, int64_t slab_rows,
                                  int64_t nrows_total, int64_t ncols, int64_t row_start, int part, const char *options, char *err,
                                  size_t errlen) {
  TuneOptions o;
  std::string e = parse_options(options, o);
  if (e.empty() && (!rowptr || !colind || !values || slab_rows < 0 || ncols < 0)) e = "invalid CSR arguments";
  if (e.empty() && rowptr[0] != 0) e = "CSR arrays must be zero-based";
  if (!e.empty()) { put_err(err, errlen, e); return nullptr; }
  csxb_matrix *m = new csxb_matrix;
  CsrView v{rowptr, colind, values, slab_rows, ncols};
  e = tune_csr_slab(v, nrows_total, row_start, part, o, m->host);
  if (!e.empty()) { put_err(err, errlen, e); delete m; return nullptr; }
  return m;
}

csxb_matrix_t *csxb_tune_mmf(const char *path, const char *options, int part_lo, int part_hi, char *err, size_t errlen) {
  TuneOptions o;
  std::string e = parse_options(options, o);
  CooHost coo;
  if (e.empty()) e = path ? read_mmf(path, coo) : "invalid file name";
  if (!e.empty()) { put_err(err, errlen, e); return nullptr; }
  if (part_hi < 0) { part_lo = 0; part_hi = o.nr_threads; }
  csxb_matrix *m = new csxb_matrix;
  e = tune_coo(coo, o, part_lo, part_hi, m->host);
  if (!e.empty()) { put_err(err, errlen, e); delete m; return nullptr; }
  return m;
}

void csxb_destroy(csxb_matrix_t *m) { delete m; }

int64_t csxb_info(const csxb_matrix_t *m, int what) {
  switch (what) {
    case CSXB_NROWS: return m->host.nrows;
    case CSXB_NCOLS: return m->host.ncols;
    case CSXB_NNZ: return m->host.nnz;
    case CSXB_SYMMETRIC: return m->host.symmetric;
    case CSXB_NPARTS: return (int64_t)m->host.parts.size();
    case CSXB_NPARTS_TOTAL: return m->host.nparts_total;
    case CSXB_PART_LO: return m->host.part_lo;
    case CSXB_FULL_COLIND: return m->host.full_colind;
    case CSXB_SYM_HALO_LO: return m->sym_halo_lo;
    case CSXB_SYM_HALO_HI: return m->sym_halo_hi;
    case CSXB_HOST_CAP: return (int64_t)m->host_cap;
    case CSXB_HOST_CALLS: return m->host_calls;
    case CSXB_DEVICE: return m->uploaded ? m->device : -1;
  }
  return -1;
}

int64_t csxb_part_info(const csxb_matrix_t *m, int part, int what) {
  if (part < 0 || (size_t)part >= m->host.parts.size()) return -1;
  const CsxPartition &p = m->host.parts[part];
  switch (what) {
    case CSXB_P_NNZ: return p.nnz;
    case CSXB_P_NROWS: return p.nrows;
    case CSXB_P_NCOLS: return p.ncols;
    case CSXB_P_ROW_START: return p.row_start;
    case CSXB_P_CTL_SIZE: return (int64_t)p.ctl.size();
    case CSXB_P_ROW_JUMPS: return p.row_jumps;
    case CSXB_P_ID_MAP_LEN: return (int64_t)p.id_map.size();
    case CSXB_P_MAP_LEN: return (int64_t)p.map_cpus.size();
    case CSXB_P_DVALUES_LEN: return (int64_t)p.dvalues.size();
    case CSXB_P_ROWS_INFO_LEN: return (int64_t)p.rows_info.size();
    case CSXB_P_SAMPLING_UNDEFINED: return p.sampling_undefined;
    case CSXB_P_COL_MIN: return p.col_min;
    case CSXB_P_COL_MAX: return p.col_max;
  }
  return -1;
}

int csxb_part_copy(const csxb_matrix_t *m, int part, int what, void *dst) {
  if (part < 0 || (size_t)part >= m->host.parts.size() || !dst) return fail("invalid argument");
  const CsxPartition &p = m->host.parts[part];
  switch (what) {
    case CSXB_A_VALUES:
      if (p.values.size() != (size_t)p.nnz) return fail("host values were released at upload");
      memcpy(dst, p.values.data(), p.values.size() * 8); break;
    case CSXB_A_CTL: memcpy(dst, p.ctl.data(), p.ctl.size()); break;
    case CSXB_A_ID_MAP: { int64_t *d = (int64_t *)dst; for (size_t i = 0; i < p.id_map.size(); i++) d[i] = p.id_map[i]; break; }
    case CSXB_A_ROWS_INFO: {
      struct R { int64_t rowptr, valptr; int32_t span, pad; } *d = (R *)dst;
      for (size_t i = 0; i < p.rows_info.size(); i++) d[i] = R{p.rows_info[i].rowptr, p.rows_info[i].valptr, p.rows_info[i].span, 0};
      break;
    }
    case CSXB_A_DVALUES: memcpy(dst, p.dvalues.data(), p.dvalues.size() * 8); break;
    case CSXB_A_MAP_CPUS: memcpy(dst, p.map_cpus.data(), p.map_cpus.size() * 4); break;
    case CSXB_A_MAP_POS: memcpy(dst, p.map_pos.data(), p.map_pos.size() * 4); break;
    default: return fail("unknown array");
  }
  return 0;
}

const char *csxb_part_log(const csxb_matrix_t *m, int part) {
  if (part < 0 || (size_t)part >= m->host.parts.size()) return "";
  return m->host.parts[part].encoding_log.c_str();
}

const char *csxb_last_error(void) { return g_last_error.c_str(); }

// Builds the GPU tables on the host only (no device needed) and reports their sizes: per row owner (local partitions,
// then the CSX-Sym halo pseudo-partition) 12 numbers — rows, tiles, table descriptors, stream chunks, stream units,
// fix-up entries, gaps, entries of block tables 0..4.  Returns the number of row owners, -1 on error (tuning aid, tests).
int csxb_layout_stats(csxb_matrix_t *m, int64_t *out, int max_owners) {
  CsxMatrix &H = m->host;
  std::vector<int64_t> saved;
  for (auto &p : H.parts) { saved.push_back(p.nrows); if (H.symmetric) p.nrows = (int64_t)p.dvalues.size(); }
  DeviceLayout L;
  std::string e = build_layout(H, L);
  for (size_t i = 0; i < H.parts.size(); i++) H.parts[i].nrows = saved[i];
  if (!e.empty()) return fail("layout: " + e);
  for (size_t q = 0; q < L.parts.size() && (int)q < max_owners; q++) {
    const PartLayout &pl = L.parts[q];
    int64_t *o = out + 12 * q;
    o[0] = pl.nrows; o[1] = pl.ntiles; o[2] = (int64_t)pl.xdesc.size(); o[3] = (int64_t)pl.sk_chunks.size();
    o[4] = (int64_t)pl.sk_uoffs.size(); o[5] = (int64_t)pl.sk_fix_idx.size(); o[6] = (int64_t)pl.sk_gaps.size();
    for (int t = 0; t < 5; t++) o[7 + t] = 0;
    for (const BlockTable &T : pl.bt) {
      int t = T.G == 1 && T.nloop == 1 ? 4 : (T.image ? (T.sl == 1 ? 3 : 1) : (T.sl == 1 ? 0 : 2));
      o[7 + t] += (int64_t)T.ent.size();
    }
  }
  return (int)L.parts.size();
}

}  // extern "C"

template <class T>
static int dev_copy(csxb_matrix *m, const T *src, size_t n, T **dst, size_t extra_zero = 0) {
  void *p = nullptr;
  size_t bytes = (n + extra_zero) * sizeof(T);
  CUDA_TRY(cudaMalloc(&p, bytes ? bytes : 16));
  m->allocs.push_back(p);
  if (n) CUDA_TRY(cudaMemcpy(p, src, n * sizeof(T), cudaMemcpyHostToDevice));
  if (extra_zero) CUDA_TRY(cudaMemset((char *)p + n * sizeof(T), 0, extra_zero * sizeof(T)));
  *dst = (T *)p;
  return 0;
}

// Row slabs of the pipelined host-buffer path (non-symmetric matrices): about 4 MB of y per slab.  A stream-kernel
// chunk runs with the first slab whose rows reach its window; the rows of a slab are final once its chunks, its
// fix-ups and its tiles of the gather kernel have run, and travel back then.
static void build_slabs(csxb_matrix *m) {
  m->slabs.clear();
  // spx.b200.slab_rows = 0 (default): an eighth of the device's rows, between 2^19 and 2^21 rows.  Uploads and downloads
  // share the host link (measured on the B200 box: 55 GB/s one way, 43 GB/s per direction when both run back to back);
  // with one upload and one download in flight the link gives 33 GB/s per direction in 4 MiB slabs and 38 GB/s in 8 or
  // 16 MiB slabs (config 2: 4.02 -> 3.50 ms per call); slabs that grow and shrink towards the ends did not help (4.03 ms).
  int64_t SLAB_ROWS = m->host.slab_rows;
  if (SLAB_ROWS <= 0) {
    int64_t total_rows = 0;
    for (const PartLayout &pl : m->layout.parts) if (pl.ntiles) total_rows += pl.nrows;
    SLAB_ROWS = int64_t(1) << 19;
    while (SLAB_ROWS < (int64_t(1) << 21) && SLAB_ROWS * 16 <= total_rows) SLAB_ROWS *= 2;
  }
  for (size_t i = 0; i < m->layout.parts.size(); i++) {
    const PartLayout &pl = m->layout.parts[i];
    if (!pl.ntiles) continue;
    const int64_t tr = pl.tile_rows();
    const int64_t tiles_per = std::max<int64_t>(1, SLAB_ROWS / tr);
    uint32_t c = 0, f = 0;
    const uint32_t nc = (uint32_t)pl.sk_chunks.size(), nf = (uint32_t)pl.sk_fix_rows.size(), ng = (uint32_t)pl.sk_gaps.size();
    int64_t xmax = -1, yup = 0;
    for (int64_t t0 = 0; t0 < pl.ntiles; t0 += tiles_per) {
      csxb_matrix::Slab sl;
      sl.part = (int)i; sl.tile0 = t0; sl.tile1 = std::min(pl.ntiles, t0 + tiles_per);
      const int64_t r0 = t0 * tr, r1 = std::min(pl.nrows, sl.tile1 * tr);   // partition-relative rows
      sl.row_lo = pl.row_start + r0; sl.row_hi = pl.row_start + r1;
      for (int64_t t = sl.tile0; t < sl.tile1; t++)
        if (pl.tile_cmax[t] >= pl.tile_cmin[t]) xmax = std::max<int64_t>(xmax, pl.tile_cmax[t]);
      sl.chunk0 = c;
      while (c < nc && pl.sk_first_row[c] < r1) {
        xmax = std::max<int64_t>(xmax, pl.sk_cmax[c]);
        yup = std::max<int64_t>(yup, (int64_t)pl.sk_last_row[c] + 1);
        c++;
      }
      sl.chunk1 = c;
      sl.f0 = f;
      while (f < nf && pl.sk_fix_rows[f] < r1) f++;
      sl.f1 = f;
      sl.g0 = 0;
      while (sl.g0 < ng && pl.sk_gaps[sl.g0].hi <= r0) sl.g0++;
      sl.g1 = sl.g0;
      while (sl.g1 < ng && pl.sk_gaps[sl.g1].lo < r1) sl.g1++;
      sl.x_lo = 0; sl.x_hi = xmax + 1;
      sl.y_lo = sl.row_lo; sl.y_hi = sl.row_hi;
      sl.yup_hi = pl.row_start + std::max(r1, std::min(yup, pl.nrows));
      m->slabs.push_back(sl);
    }
  }
  // x travels in ascending column order starting at the smallest column any local slab reads
  int64_t lo = INT64_MAX;
  for (size_t i = 0; i < m->layout.parts.size(); i++)
    for (int32_t v : m->layout.parts[i].tile_cmin) if (v != INT32_MAX) lo = std::min<int64_t>(lo, v);
  if (lo == INT64_MAX) lo = 0;
  int64_t run = lo;
  for (auto &sl : m->slabs) { sl.x_lo = lo; run = std::max(run, sl.x_hi); sl.x_hi = run; }
}

extern "C" {

int csxb_upload(csxb_matrix_t *m, int device, int free_host) {
  if (m->uploaded) return fail("matrix already uploaded");
  // CSX-Sym: a partition owns dvalues.size() rows (SparsePartitionSym::GetNrRows, SparsePartition.hpp:420-423)
  CsxMatrix &H = m->host;
  std::vector<int64_t> saved_nrows;
  for (auto &p : H.parts) { saved_nrows.push_back(p.nrows); if (H.symmetric) p.nrows = (int64_t)p.dvalues.size(); }
  std::string e = build_layout(H, m->layout);
  for (size_t i = 0; i < H.parts.size(); i++) H.parts[i].nrows = saved_nrows[i];
  if (!e.empty()) return fail("layout: " + e);
  int ndev = 0;
  CUDA_TRY(cudaGetDeviceCount(&ndev));
  if (device < 0 || device >= ndev) return fail("invalid device");
  CUDA_TRY(cudaSetDevice(device));
  m->device = device;
  DeviceLayout &L = m->layout;
  // device-wide arrays
  void *dv = nullptr, *dc = nullptr;
  CUDA_TRY(cudaMalloc(&dv, std::max<uint64_t>(L.total_values, 1) * 8));
  m->allocs.push_back(dv);
  CUDA_TRY(cudaMalloc(&dc, std::max<uint64_t>(L.total_ctl, 16)));
  m->allocs.push_back(dc);
  CUDA_TRY(cudaMemset(dc, 0, std::max<uint64_t>(L.total_ctl, 16)));
  m->d_values = (double *)dv;
  KindEntry *d_ktab = nullptr;
  if (dev_copy(m, L.ktab.data(), L.ktab.size(), &d_ktab)) return -1;
  int64_t tables = (int64_t)L.ktab.size() * 8, nnz_stored = 0, ctl_bytes = 0, rows_owned = 0, launches = 0;
  m->pdev.resize(L.parts.size());
  for (size_t i = 0; i < L.parts.size(); i++) {
    PartLayout &pl = L.parts[i];
    static CsxPartition no_part;   // the CSX-Sym halo pseudo-partition has tables only
    CsxPartition &hp = pl.is_halo ? no_part : H.parts[i];
    PartDev &P = m->pdev[i];
    memset(&P, 0, sizeof(P));
    if (hp.nnz) CUDA_TRY(cudaMemcpy(m->d_values + pl.val_base, hp.values.data(), (size_t)hp.nnz * 8, cudaMemcpyHostToDevice));
    if (!hp.ctl.empty()) CUDA_TRY(cudaMemcpy((uint8_t *)dc + pl.ctl_base, hp.ctl.data(), hp.ctl.size(), cudaMemcpyHostToDevice));
    P.ctl = (const uint8_t *)dc + pl.ctl_base;
    P.values = m->d_values;
    P.ctl_end = (const uint8_t *)dc + std::max<uint64_t>(L.total_ctl, 16);
    P.values_end = m->d_values + std::max<uint64_t>(L.total_values, 1);
    uint32_t *tx = nullptr; XDesc *xd = nullptr;
    if (dev_copy(m, pl.tile_xoff.data(), pl.tile_xoff.size(), &tx)) return -1;
    if (dev_copy(m, pl.xdesc.data(), pl.xdesc.size(), &xd)) return -1;
    for (size_t t = 0; t < pl.bt.size(); t++) {   // block tables
      const BlockTable &T = pl.bt[t];
      uint32_t *bp = nullptr; BlockImage *bi = nullptr;
      if (dev_copy(m, T.ptr.data(), T.ptr.size(), &bp)) return -1;
      if (dev_copy(m, T.ent.data(), T.ent.size(), &bi)) return -1;
      static_assert(sizeof(BlockImage) == sizeof(uint2), "block table entry layout");
      P.bt[t] = BtDev{bp, (const uint2 *)bi, (long long)T.j0, T.G, T.nloop, T.sf, T.sl, T.image, (uint32_t)((0x100000000ull + T.G - 1) / T.G)};
      tables += (int64_t)T.ptr.size() * 4 + (int64_t)T.ent.size() * 8;
    }
    P.nbt = (int)pl.bt.size();
    if (!pl.sk_chunks.empty()) {   // stream kernel tables
      SkEntry *se = nullptr; uint16_t *so = nullptr; int32_t *fr = nullptr; uint32_t *fp = nullptr, *fi = nullptr; long long *gp = nullptr;
      if (dev_copy(m, pl.sk_chunks.data(), pl.sk_chunks.size(), &se)) return -1;
      if (dev_copy(m, pl.sk_uoffs.data(), pl.sk_uoffs.size(), &so)) return -1;
      if (dev_copy(m, pl.sk_fix_rows.data(), pl.sk_fix_rows.size(), &fr)) return -1;
      if (dev_copy(m, pl.sk_fix_ptr.data(), pl.sk_fix_ptr.size(), &fp)) return -1;
      if (dev_copy(m, pl.sk_fix_idx.data(), pl.sk_fix_idx.size(), &fi)) return -1;
      static_assert(sizeof(SkGap) == 16, "gap layout");
      if (dev_copy(m, reinterpret_cast<const long long *>(pl.sk_gaps.data()), pl.sk_gaps.size() * 2, &gp)) return -1;
      void *sc = nullptr;
      CUDA_TRY(cudaMalloc(&sc, std::max<size_t>(pl.sk_scratch, 2) * 8));
      m->allocs.push_back(sc);
      P.sk_chunks = (const uint4 *)se; P.sk_uoffs = so; P.sk_scratch = (double *)sc;
      P.sk_fix_rows = fr; P.sk_fix_ptr = fp; P.sk_fix_idx = fi; P.sk_gaps = gp;
      P.sk_c0 = 0; P.sk_c1 = (uint32_t)pl.sk_chunks.size();
      P.sk_f0 = 0; P.sk_f1 = (uint32_t)pl.sk_fix_rows.size();
      P.sk_g0 = 0; P.sk_g1 = (uint32_t)pl.sk_gaps.size();
      // chunk table, unit offsets, fix-up lists, and the scratch sums (written once, read once)
      tables += (int64_t)pl.sk_chunks.size() * (int64_t)sizeof(SkEntry) + (int64_t)pl.sk_uoffs.size() * 2 +
                (int64_t)pl.sk_fix_rows.size() * 8 + (int64_t)pl.sk_fix_idx.size() * 4 + (int64_t)pl.sk_scratch * 16;
    }
    P.tile_xoff = tx; P.xdesc = (const uint4 *)xd; P.ktab = d_ktab;
    if (H.symmetric && !pl.is_halo) {
      double *dd = nullptr;
      if (dev_copy(m, hp.dvalues.data(), hp.dvalues.size(), &dd)) return -1;
      P.dvalues = dd;
      tables += (int64_t)hp.dvalues.size() * 8;
    }
    P.nrows = pl.nrows; P.row_start = pl.row_start; P.val_base = (uint32_t)pl.val_base;
    P.full_colind = L.full_colind;
    P.rpt = pl.rpt;
    memcpy(P.idtab, pl.idtab, sizeof(P.idtab));
    nnz_stored += hp.nnz; rows_owned += pl.nrows;   // halo rows are written too
    if (!pl.sk_chunks.empty()) ctl_bytes += (int64_t)hp.ctl.size();   // only the stream kernel reads ctl
    tables += (int64_t)pl.tile_xoff.size() * 4 + (int64_t)pl.xdesc.size() * 16;
    if (pl.nrows) {
      if (!pl.sk_chunks.empty())
        launches += 1 + ((pl.sk_fix_rows.empty() && pl.sk_gaps.empty()) ? 0 : 1) + ((pl.xdesc.empty() && pl.bt.empty() && !H.symmetric) ? 0 : 1);
      else launches += 1;
    }
    if (!pl.is_halo) m->covered_rows_end = std::max<int64_t>(m->covered_rows_end, pl.row_start + pl.nrows);
    if (free_host && !pl.is_halo) std::vector<double>().swap(hp.values);
  }
  // CSX-Sym, partial device: transposed updates of the local lower triangle reach rows of lower ranks (gpu_layout.cpp)
  m->sym_halo_lo = L.halo_lo; m->sym_halo_hi = L.halo_hi;
  if (!H.symmetric) build_slabs(m);
  m->bytes[CSXB_B_VALUES] = nnz_stored * 8;
  m->bytes[CSXB_B_CTL] = ctl_bytes;
  m->bytes[CSXB_B_TABLES] = tables;
  // x: the column window the local partitions read (the whole vector when every partition is local)
  int64_t cmin = H.ncols, cmax = -1;
  for (auto &p : H.parts) if (p.col_max >= p.col_min) { cmin = std::min(cmin, p.col_min); cmax = std::max(cmax, p.col_max); }
  int64_t xcols = (int)H.parts.size() == H.nparts_total ? H.ncols : std::max<int64_t>(0, cmax - cmin + 1);
  if (H.symmetric) xcols = H.ncols;
  m->bytes[CSXB_B_X] = xcols * 8;
  m->bytes[CSXB_B_Y] = rows_owned * 8;
  m->bytes[CSXB_B_TOTAL] = nnz_stored * 8 + ctl_bytes + tables + xcols * 8 + rows_owned * 8;
  m->bytes[CSXB_B_LAUNCHES] = launches;
  m->uploaded = true;
  return 0;
}

int64_t csxb_traffic(const csxb_matrix_t *m, int what) {
  if (what < 0 || what > CSXB_B_LAUNCHES) return -1;
  return m->bytes[what];
}

}  // extern "C"

// The diagonal kernel with L2 cache policies (values: no L1 allocation, first to leave L2; x: last to leave L2) for
// partitions whose values outweigh x by far (27-point stencil: +2 % at full size, +10 % on an eighth of the matrix;
// the 5-point stencil loses 5 % with them).  CSXB_GATHER_POLICY = 0 / 1 forces the choice (tuning aid).
static bool gather_cache_policies(const PartLayout &pl) {
  static const int forced = getenv("CSXB_GATHER_POLICY") ? atoi(getenv("CSXB_GATHER_POLICY")) : -1;
  return forced >= 0 ? forced != 0 : pl.nnz >= 12 * pl.nrows;
}

// Resident CTAs per SM the block-table instantiations are compiled for.  The table walk is a chain of dependent loads
// (group pointer -> entry -> values, x), so it lives on occupancy: one row per thread fits 40 registers without spills
// (6 CTAs), four rows per thread 48 (5 CTAs); measured on the block configs in profiles/r02_bt_variants.txt.
template <int RPT> struct BtMinB { static constexpr int value = RPT == 1 ? 6 : 5; };
// csxb_spmv_host only: dynamic shared memory per CTA of the gather kernels it launches.  The kernels do not use it; it caps
// the CTAs resident per SM, i.e. how hard a slab's kernel pulls on HBM while the copy engines move x and y over PCIe.
static thread_local size_t t_gather_dyn = 0;
constexpr size_t HOST_CAP_SMEM = 40000;   // 5 CTAs per SM
template <class K>
static size_t gather_dyn(K kernel) {
  if (t_gather_dyn > 48 * 1024) cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)t_gather_dyn);
  return t_gather_dyn;
}
// Launches kernel 1 over tiles [t0, t1) of one partition.  XP = XchgDev fuses the multi-GPU exchange into it.
template <bool SYM, int RPT, int KSET, class XP>
static void launch_gather_k(const PartDev &P, const PartLayout &pl, unsigned nt, const double *x, double *y, double alpha,
                            double beta, int overwrite, cudaStream_t s, const XP &X) {
  dim3 grid(nt), block(CTA_THREADS);
  if (!pl.bt.empty()) {   // block tables: the generic instantiation with the table loop (64 registers)
    if (!pl.xdesc.empty()) {
      auto k = csx_spmv_kernel<true, SYM, RPT, KSET_ANY, BtMinB<RPT>::value, 0, XP, true>;
      k<<<grid, block, gather_dyn(k), s>>>(P, x, y, alpha, beta, overwrite, X);
    } else {
      auto k = csx_spmv_kernel<false, SYM, RPT, KSET_ANY, BtMinB<RPT>::value, 0, XP, true>;
      k<<<grid, block, gather_dyn(k), s>>>(P, x, y, alpha, beta, overwrite, X);
    }
    return;
  }
  // descriptors can also come from other partitions (transposed images under CSX-Sym, whose many kinds need registers)
  constexpr int MB = SYM ? 4 : 8;
  const size_t dyn = 0;
  if (!pl.xdesc.empty()) csx_spmv_kernel<true, SYM, RPT, KSET, MB, 0, XP><<<grid, block, dyn, s>>>(P, x, y, alpha, beta, overwrite, X);
  else csx_spmv_kernel<false, SYM, RPT, KSET_ANY, MB, 0, XP><<<grid, block, dyn, s>>>(P, x, y, alpha, beta, overwrite, X);
}
template <bool SYM, class XP>
static void launch_gather(const PartDev &P0, const PartLayout &pl, int64_t t0, int64_t t1, const double *x, double *y,
                          double alpha, double beta, int overwrite, cudaStream_t s, const XP &X) {
  if (t1 <= t0) return;
  PartDev P = P0;
  P.tile0 = (uint32_t)t0;
  const unsigned nt = (unsigned)(t1 - t0);
  // kernels are pre-compiled per (tile shape, unit-kind set) — the counterpart of the per-partition JIT (CsxJit.hpp)
  const bool diag1 = !SYM && pl.xd_diag1_only && !pl.xdesc.empty() && pl.bt.empty();
  if (pl.rpt == 4) {
    if (diag1) {  // the instantiation the stencil configs run: loads of a unit issued as one PTX block
      dim3 grid(nt), block(CTA_THREADS);
      if (gather_cache_policies(pl)) {
        auto k = csx_spmv_kernel<true, false, 4, KSET_DIAG1, 8, 3, XP>;
        k<<<grid, block, gather_dyn(k), s>>>(P, x, y, alpha, beta, overwrite, X);
      } else {
        auto k = csx_spmv_kernel<true, false, 4, KSET_DIAG1, 8, 1, XP>;
        k<<<grid, block, gather_dyn(k), s>>>(P, x, y, alpha, beta, overwrite, X);
      }
    }
    else launch_gather_k<SYM, 4, KSET_ANY>(P, pl, nt, x, y, alpha, beta, overwrite, s, X);
  } else {
    if (diag1) launch_gather_k<SYM, 1, SYM ? KSET_ANY : KSET_DIAG1>(P, pl, nt, x, y, alpha, beta, overwrite, s, X);
    else launch_gather_k<SYM, 1, KSET_ANY>(P, pl, nt, x, y, alpha, beta, overwrite, s, X);
  }
}
// Kernel 1 of a whole partition under the edge-tiles-first exchange protocol.
static void launch_gather_xe(const PartDev &P0, const PartLayout &pl, const double *x, double *y, double alpha, int ypar,
                             cudaStream_t s, const XchgDev &X) {
  if (!pl.ntiles) return;
  PartDev P = P0;
  P.tile0 = 0;
  dim3 grid((unsigned)(X.nb + (X.edge_hi_begin - X.edge_lo_end))), block(CTA_THREADS);   // edge CTAs first, then the interior tiles
  const bool xd = !pl.xdesc.empty(), diag1 = pl.xd_diag1_only && xd && pl.bt.empty();
  if (!pl.bt.empty()) {
    if (pl.rpt == 4) {
      if (xd) csx_spmv_xe_kernel<true, 4, KSET_ANY, BtMinB<4>::value, 0, true><<<grid, block, 0, s>>>(P, x, y, alpha, ypar, X);
      else csx_spmv_xe_kernel<false, 4, KSET_ANY, BtMinB<4>::value, 0, true><<<grid, block, 0, s>>>(P, x, y, alpha, ypar, X);
    } else {
      if (xd) csx_spmv_xe_kernel<true, 1, KSET_ANY, BtMinB<1>::value, 0, true><<<grid, block, 0, s>>>(P, x, y, alpha, ypar, X);
      else csx_spmv_xe_kernel<false, 1, KSET_ANY, BtMinB<1>::value, 0, true><<<grid, block, 0, s>>>(P, x, y, alpha, ypar, X);
    }
    return;
  }
  const size_t dyn = 0;
  if (pl.rpt == 4) {
    if (diag1 && gather_cache_policies(pl)) csx_spmv_xe_kernel<true, 4, KSET_DIAG1, 8, 3><<<grid, block, dyn, s>>>(P, x, y, alpha, ypar, X);
    else if (diag1) csx_spmv_xe_kernel<true, 4, KSET_DIAG1, 8, 1><<<grid, block, dyn, s>>>(P, x, y, alpha, ypar, X);
    else if (xd) csx_spmv_xe_kernel<true, 4, KSET_ANY><<<grid, block, dyn, s>>>(P, x, y, alpha, ypar, X);
    else csx_spmv_xe_kernel<false, 4, KSET_ANY><<<grid, block, dyn, s>>>(P, x, y, alpha, ypar, X);
  } else {
    if (diag1) csx_spmv_xe_kernel<true, 1, KSET_DIAG1><<<grid, block, dyn, s>>>(P, x, y, alpha, ypar, X);
    else if (xd) csx_spmv_xe_kernel<true, 1, KSET_ANY><<<grid, block, dyn, s>>>(P, x, y, alpha, ypar, X);
    else csx_spmv_xe_kernel<false, 1, KSET_ANY><<<grid, block, dyn, s>>>(P, x, y, alpha, ypar, X);
  }
}
// Launches the stream kernel over chunks [c0, c1) of one partition: the instantiation is chosen by the partition's
// pattern set (kinds of units, rows of a block task) — the counterpart of the per-partition JIT (CsxJit.hpp:359-732).
static int launch_stream(const PartDev &P0, const PartLayout &pl, uint32_t c0, uint32_t c1, const SkIO &io, double alpha, double beta,
                         int overwrite, cudaStream_t s) {
  if (c1 <= c0) return 0;
  PartDev P = P0;
  P.sk_c0 = c0; P.sk_c1 = c1;
  const unsigned grid = (unsigned)((c1 - c0 + SK_WARPS - 1) / SK_WARPS);
#define SK_TRY(RR, KK, BCC, BRR)                                                                                         \
  if (sk_instance_serves(RR, (KK), BCC, BRR, pl.sk_kmask, pl.sk_rows, pl.sk_bc, pl.sk_brc)) {                            \
    csx_stream_kernel<RR, (KK), BCC, BRR><<<grid, SK_WARPS * 32, 0, s>>>(P, io, alpha, beta, overwrite);                 \
    return 0;                                                                                                            \
  }
  SK_INSTANCES(SK_TRY)
#undef SK_TRY
  return -1;
}
// Fix-up of rows [r0, r1) (partition relative) after the stream kernel: foreign contributions f0..f1, gaps g0..g1.
static void launch_fixup(const PartDev &P0, uint32_t f0, uint32_t f1, uint32_t g0, uint32_t g1, int64_t r0, int64_t r1, const SkIO &io,
                         double alpha, double beta, int overwrite, cudaStream_t s) {
  if (f1 <= f0 && g1 <= g0) return;
  PartDev P = P0;
  P.sk_f0 = f0; P.sk_f1 = f1; P.sk_g0 = g0; P.sk_g1 = g1;
  const int64_t ctas = std::max<int64_t>(((int64_t)(f1 - f0) + 255) / 256, (int64_t)(g1 - g0));
  const unsigned grid = (unsigned)std::min<int64_t>(148 * 8, ctas);
  csx_stream_fixup_kernel<<<grid, 256, 0, s>>>(P, io, alpha, beta, overwrite, (long long)r0, (long long)r1);
}
// One partition of a non-symmetric matrix, whole: stream kernel (writes y), fix-up, then the gather over the table,
// which adds (beta = 1).  Without stream chunks the gather kernel alone writes y.
// CSX-Sym: the stream kernel and the direct table units are phase 1 (every partition writes its own rows), the
// images of all units — gathered by the owners of the rows they update — and the diagonal are phase 2; both
// phases of a row are the work of the thread that owns it, so there is nothing to reduce on one device.
template <bool SYM, class XP>
static int run_partition(const PartDev &P, const PartLayout &pl, const SkIO &io, double alpha, double beta, int overwrite,
                         cudaStream_t s, const XP &X) {
  if (pl.sk_chunks.empty()) {
    launch_gather<SYM>(P, pl, 0, pl.ntiles, io.x, io.y, alpha, beta, overwrite, s, X);
    return 0;
  }
  if (launch_stream(P, pl, 0, (uint32_t)pl.sk_chunks.size(), io, alpha, beta, overwrite, s)) return -1;
  launch_fixup(P, 0, (uint32_t)pl.sk_fix_rows.size(), 0, (uint32_t)pl.sk_gaps.size(), 0, pl.nrows, io, alpha, beta, overwrite, s);
  // CSX-Sym: the gather kernel always runs (diagonal, images)
  if (SYM || !pl.xdesc.empty() || !pl.bt.empty()) launch_gather<SYM>(P, pl, 0, pl.ntiles, io.x, io.y, alpha, 1.0, 0, s, X);
  return 0;
}

extern "C" {

// kernels of a matrix run on the device it was uploaded to, whatever the caller's current device is
static int on_matrix_device(const csxb_matrix *m) {
  int cur = -1;
  if (cudaGetDevice(&cur) != cudaSuccess) return fail("cudaGetDevice failed");
  if (cur != m->device && cudaSetDevice(m->device) != cudaSuccess) return fail("cudaSetDevice failed");
  return 0;
}

int csxb_spmv(csxb_matrix_t *m, double alpha, const double *d_x, double beta, double *d_y, int overwrite, void *stream) {
  if (!m->uploaded) return fail("matrix not uploaded (csxb_upload)");
  if (on_matrix_device(m)) return -1;
  cudaStream_t s = (cudaStream_t)stream;
  const bool sym = m->host.symmetric;
  SkIO io;
  io.x = d_x; io.y = d_y; io.step = nullptr; io.vec[0] = io.vec[1] = nullptr; io.npush = 0;
  for (size_t i = 0; i < m->pdev.size(); i++) {
    const PartLayout &pl = m->layout.parts[i];
    int rc;
    // CSX-Sym halo rows (owned by other devices): this device's updates of them, for the caller to reduce
    if (pl.is_halo) { launch_gather<true>(m->pdev[i], pl, 0, pl.ntiles, d_x, d_y, alpha, 0.0, 1, s, NoXchg()); rc = 0; }
    else if (sym) rc = run_partition<true>(m->pdev[i], pl, io, alpha, beta, overwrite, s, NoXchg());
    else rc = run_partition<false>(m->pdev[i], pl, io, alpha, beta, overwrite, s, NoXchg());
    if (rc) return fail("no stream kernel for the partition's pattern set");
  }
  // rows after the last partition's last non-empty row belong to nobody; VecInit(y,0) clears them (CsxKernels.cpp:93)
  if (overwrite && m->host.part_lo + (int)m->host.parts.size() == m->host.nparts_total && m->covered_rows_end < m->host.nrows)
    CUDA_TRY(cudaMemsetAsync(d_y + m->covered_rows_end, 0, (size_t)(m->host.nrows - m->covered_rows_end) * 8, s));
  CUDA_TRY(cudaGetLastError());
  return 0;
}

// Host-buffer SpMV, pipelined: the rows are cut into slabs; x travels to the device in ascending column order
// on one stream, a slab's kernels start as soon as the columns its rows read have arrived, and its y rows go
// back on a third stream while the next slabs compute — host-to-device, compute and device-to-host overlap
// (PCIe is full duplex).  Banded matrices overlap all three; a matrix whose first rows read the whole x only
// overlaps compute with the way back.  CSX-Sym scatters into rows of earlier slabs, so it runs unpipelined.
int csxb_spmv_host(csxb_matrix_t *m, double alpha, const double *h_x, double beta, double *h_y, int overwrite) {
  if (!m->uploaded) return fail("matrix not uploaded (csxb_upload)");
  int cur = -1;
  CUDA_TRY(cudaGetDevice(&cur));
  if (cur != m->device) CUDA_TRY(cudaSetDevice(m->device));
  size_t nx = (size_t)std::max<int64_t>(m->host.ncols, 1), ny = (size_t)std::max<int64_t>(m->host.nrows, 1);
  if (!m->d_x) CUDA_TRY(cudaMalloc((void **)&m->d_x, nx * 8));
  if (!m->d_y) CUDA_TRY(cudaMalloc((void **)&m->d_y, ny * 8));
  if (!m->s_h2d) {
    CUDA_TRY(cudaStreamCreateWithFlags(&m->s_h2d, cudaStreamNonBlocking));
    CUDA_TRY(cudaStreamCreateWithFlags(&m->s_run, cudaStreamNonBlocking));
    CUDA_TRY(cudaStreamCreateWithFlags(&m->s_d2h, cudaStreamNonBlocking));
  }
  const bool last_local = m->host.part_lo + (int)m->host.parts.size() == m->host.nparts_total;
  if (m->slabs.empty()) {   // CSX-Sym or nothing to pipeline: upload, run, download
    CUDA_TRY(cudaMemcpyAsync(m->d_x, h_x, (size_t)m->host.ncols * 8, cudaMemcpyHostToDevice, m->s_run));
    if (!overwrite) CUDA_TRY(cudaMemcpyAsync(m->d_y, h_y, (size_t)m->host.nrows * 8, cudaMemcpyHostToDevice, m->s_run));
    if (csxb_spmv(m, alpha, m->d_x, beta, m->d_y, overwrite, m->s_run)) return -1;
    // only the rows this handle computes travel back (one process per GPU owns one row range)
    int64_t lo = m->layout.parts.empty() ? 0 : m->layout.parts.front().row_start;
    int64_t hi = last_local ? m->host.nrows : m->covered_rows_end;
    if (!overwrite) { lo = 0; hi = m->host.nrows; }
    if (hi > lo) CUDA_TRY(cudaMemcpyAsync(h_y + lo, m->d_y + lo, (size_t)(hi - lo) * 8, cudaMemcpyDeviceToHost, m->s_run));
    CUDA_TRY(cudaStreamSynchronize(m->s_run));
  } else {
    if (m->slab_ev.size() < 2 * m->slabs.size()) {
      size_t old = m->slab_ev.size();
      m->slab_ev.resize(2 * m->slabs.size());
      for (size_t i = old; i < m->slab_ev.size(); i++) CUDA_TRY(cudaEventCreateWithFlags(&m->slab_ev[i], cudaEventDisableTiming));
    }
    // CSXB_HOST_TRACE=1 (tuning aid): device time stamps of every slab's upload, kernels and download
    static const bool trace = getenv("CSXB_HOST_TRACE") != nullptr;
    std::vector<cudaEvent_t> tev;
    if (trace) {
      tev.resize(3 * m->slabs.size() + 1);
      for (auto &e : tev) CUDA_TRY(cudaEventCreate(&e));
      CUDA_TRY(cudaEventRecord(tev.back(), m->s_h2d));
    }
    // (downloads that trail the uploads by one or two slabs, CSXB_D2H_LAG in an earlier build, were no faster: config 2
    // 3.47 ms per call with none, 3.65 - 3.96 ms with a lag of one slab, at slabs of 2^20 - 2^21 rows)
    auto issue_download = [&](size_t k) -> int {
      const csxb_matrix::Slab &sl = m->slabs[k];
      if (sl.y_hi > sl.y_lo) {
        CUDA_TRY(cudaStreamWaitEvent(m->s_d2h, m->slab_ev[2 * k + 1], 0));
        CUDA_TRY(cudaMemcpyAsync(h_y + sl.y_lo, m->d_y + sl.y_lo, (size_t)(sl.y_hi - sl.y_lo) * 8, cudaMemcpyDeviceToHost, m->s_d2h));
      }
      if (trace) CUDA_TRY(cudaEventRecord(tev[3 * k + 2], m->s_d2h));
      return 0;
    };
    // A slab's kernel at full tilt takes HBM bandwidth from the copy engines that move the other slabs' x and y
    // (27-point stencil, 8 M rows: 1.92 - 1.97 ms per call as is, 1.75 ms with the kernels capped at 5 CTAs per SM, 1.87 - 1.90
    // ms at 3 or 2); whether a cap pays depends on how long the kernels are next to the copies, so the first calls time
    // both settings (calls 1, 3: no cap; 2, 4: cap) and the faster one stays.  CSXB_HOST_SMEM = bytes forces a setting.
    const auto call_t0 = std::chrono::steady_clock::now();
    const int tune_call = m->host_calls < 5 ? m->host_calls : -1;
    {
      const char *v = getenv("CSXB_HOST_SMEM");
      if (v) t_gather_dyn = (size_t)atol(v);
      else if (tune_call > 0) t_gather_dyn = (tune_call % 2 == 0) ? HOST_CAP_SMEM : 0;
      else t_gather_dyn = m->host_cap;
    }
    struct DynReset { ~DynReset() { t_gather_dyn = 0; } } dyn_reset;
    int64_t x_done = m->slabs.front().x_lo;   // columns [x_lo of the first slab, x_done) are on the device
    int64_t y_up = 0;                         // y rows below this one are on the device (spx_matvec_kernel semantics)
    for (size_t k = 0; k < m->slabs.size(); k++) {
      const csxb_matrix::Slab &sl = m->slabs[k];
      const PartLayout &pl = m->layout.parts[sl.part];
      if (sl.x_hi > x_done) {
        CUDA_TRY(cudaMemcpyAsync(m->d_x + x_done, h_x + x_done, (size_t)(sl.x_hi - x_done) * 8, cudaMemcpyHostToDevice, m->s_h2d));
        x_done = sl.x_hi;
      }
      if (!overwrite) {   // y rows the slab's kernels read: its own rows and the rows its chunks own behind them
        if (k == 0 || m->slabs[k - 1].part != sl.part) y_up = sl.row_lo;
        if (sl.yup_hi > y_up) {
          CUDA_TRY(cudaMemcpyAsync(m->d_y + y_up, h_y + y_up, (size_t)(sl.yup_hi - y_up) * 8, cudaMemcpyHostToDevice, m->s_h2d));
          y_up = sl.yup_hi;
        }
      }
      CUDA_TRY(cudaEventRecord(m->slab_ev[2 * k], m->s_h2d));
      if (trace) CUDA_TRY(cudaEventRecord(tev[3 * k], m->s_h2d));
      CUDA_TRY(cudaStreamWaitEvent(m->s_run, m->slab_ev[2 * k], 0));
      if (pl.sk_chunks.empty()) {
        launch_gather<false>(m->pdev[sl.part], pl, sl.tile0, sl.tile1, m->d_x, m->d_y, alpha, beta, overwrite, m->s_run, NoXchg());
      } else {   // stream kernel writes y, fix-up, then the gather over the table adds
        SkIO io;
        io.x = m->d_x; io.y = m->d_y; io.step = nullptr; io.vec[0] = io.vec[1] = nullptr; io.npush = 0;
        if (launch_stream(m->pdev[sl.part], pl, sl.chunk0, sl.chunk1, io, alpha, beta, overwrite, m->s_run)) return fail("no stream kernel for the partition's pattern set");
        launch_fixup(m->pdev[sl.part], sl.f0, sl.f1, sl.g0, sl.g1, sl.row_lo - pl.row_start, sl.row_hi - pl.row_start, io, alpha, beta, overwrite, m->s_run);
        if (!pl.xdesc.empty() || !pl.bt.empty()) launch_gather<false>(m->pdev[sl.part], pl, sl.tile0, sl.tile1, m->d_x, m->d_y, alpha, 1.0, 0, m->s_run, NoXchg());
      }
      CUDA_TRY(cudaEventRecord(m->slab_ev[2 * k + 1], m->s_run));
      if (trace) CUDA_TRY(cudaEventRecord(tev[3 * k + 1], m->s_run));
      if (issue_download(k)) return -1;
    }
    if (trace) {
      CUDA_TRY(cudaStreamSynchronize(m->s_run));
      CUDA_TRY(cudaStreamSynchronize(m->s_d2h));
      for (size_t k = 0; k < m->slabs.size(); k++) {
        float a = 0, b = 0, c = 0;
        cudaEventElapsedTime(&a, tev.back(), tev[3 * k]);
        cudaEventElapsedTime(&b, tev.back(), tev[3 * k + 1]);
        cudaEventElapsedTime(&c, tev.back(), tev[3 * k + 2]);
        const csxb_matrix::Slab &sl = m->slabs[k];
        fprintf(stderr, "[host-trace] slab %3zu rows [%lld, %lld) x to %lld: up %.3f ms, run %.3f ms, down %.3f ms\n", k,
                (long long)sl.row_lo, (long long)sl.row_hi, (long long)sl.x_hi, a, b, c);
      }
      for (auto &e : tev) cudaEventDestroy(e);
    }
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaStreamSynchronize(m->s_run));
    CUDA_TRY(cudaStreamSynchronize(m->s_d2h));
    // rows after the last partition's last non-empty row belong to nobody: zero under spx_matvec_mult
    // semantics (CsxKernels.cpp:93)
    // (spx_matvec_kernel semantics leave them as they are: do_kernel_thread only scales the rows of its partition,
    // CsxSpmv.cpp:52-64 — the same as csxb_spmv on device vectors)
    if (overwrite && last_local && m->covered_rows_end < m->host.nrows)
      for (int64_t r = m->covered_rows_end; r < m->host.nrows; r++) h_y[r] = 0.0;
    if (tune_call >= 0) {
      const double dt = std::chrono::duration<double>(std::chrono::steady_clock::now() - call_t0).count();
      if (tune_call > 0) { double &best = m->host_tune_s[tune_call % 2]; best = best == 0.0 ? dt : std::min(best, dt); }
      if (tune_call == 4) m->host_cap = m->host_tune_s[0] < m->host_tune_s[1] ? HOST_CAP_SMEM : 0;
      m->host_calls++;
    }
  }
  if (cur != m->device && cur >= 0) CUDA_TRY(cudaSetDevice(cur));
  return 0;
}

// ---- transposed product y = alpha*A^T*x + beta*y (gpu_layout.hpp: TransLayout) ---------------------------------------
// Runs on the device's current value array, so csxb_set_entry updates reach it with no extra work.  Launches: the heavy
// column segments (if any), the gather over the transposed tables (writes every column of the window once), the fix-up
// that adds the segment sums (if any).
struct DeviceGuard {   // restores the caller's device
  int d = -1;
  DeviceGuard() { cudaGetDevice(&d); }
  ~DeviceGuard() { if (d >= 0) cudaSetDevice(d); }
};

int csxb_transpose_prepare(csxb_matrix_t *m) {
  if (!m) return fail("invalid argument");
  if (m->host.symmetric || m->trans) return 0;
  if (!m->uploaded) return fail("matrix not uploaded (csxb_upload)");
  DeviceGuard guard;
  const auto t0 = std::chrono::steady_clock::now();
  std::unique_ptr<TransState> T(new TransState);
  // CSX-Sym is excluded above: partitions own nrows rows, the layout the upload built
  std::string e = build_transpose_layout(m->host, m->layout, T->lay);
  if (!e.empty()) return fail("transposed layout: " + e);
  CUDA_TRY(cudaSetDevice(m->device));
  const TransLayout &TL = T->lay;
  const PartLayout &pl = TL.part;
  PartDev &P = T->P;
  memset(&P, 0, sizeof(P));
  KindEntry *kt = nullptr; uint32_t *tx = nullptr; XDesc *xd = nullptr;
  if (dev_copy(m, TL.ktab.data(), TL.ktab.size(), &kt) || dev_copy(m, pl.tile_xoff.data(), pl.tile_xoff.size(), &tx) ||
      dev_copy(m, pl.xdesc.data(), pl.xdesc.size(), &xd))
    return -1;
  int64_t tables = (int64_t)TL.ktab.size() * 8 + (int64_t)pl.tile_xoff.size() * 4 + (int64_t)pl.xdesc.size() * 16;
  for (size_t t = 0; t < pl.bt.size(); t++) {
    const BlockTable &B = pl.bt[t];
    uint32_t *bp = nullptr; BlockImage *bi = nullptr;
    if (dev_copy(m, B.ptr.data(), B.ptr.size(), &bp) || dev_copy(m, B.ent.data(), B.ent.size(), &bi)) return -1;
    P.bt[t] = BtDev{bp, (const uint2 *)bi, (long long)B.j0, B.G, B.nloop, B.sf, B.sl, B.image, (uint32_t)((0x100000000ull + B.G - 1) / B.G)};
    tables += (int64_t)B.ptr.size() * 4 + (int64_t)B.ent.size() * 8;
  }
  P.nbt = (int)pl.bt.size();
  int launches = pl.nrows ? 1 : 0;
  if (!pl.sk_fix_rows.empty()) {   // heavy columns: segments, fix-up lists, scratch sums (written once, read once)
    BlockImage *he = nullptr; uint32_t *hs = nullptr, *fp = nullptr, *fi = nullptr; int32_t *fr = nullptr;
    if (dev_copy(m, TL.hent.data(), TL.hent.size(), &he) || dev_copy(m, TL.hseg.data(), TL.hseg.size(), &hs) ||
        dev_copy(m, pl.sk_fix_rows.data(), pl.sk_fix_rows.size(), &fr) || dev_copy(m, pl.sk_fix_ptr.data(), pl.sk_fix_ptr.size(), &fp) ||
        dev_copy(m, pl.sk_fix_idx.data(), pl.sk_fix_idx.size(), &fi))
      return -1;
    void *sc = nullptr;
    CUDA_TRY(cudaMalloc(&sc, std::max<size_t>(pl.sk_scratch, 2) * 8));
    m->allocs.push_back(sc);
    T->hent = (const uint2 *)he; T->hseg = hs;
    P.sk_scratch = (double *)sc; P.sk_fix_rows = fr; P.sk_fix_ptr = fp; P.sk_fix_idx = fi;
    P.sk_f0 = 0; P.sk_f1 = (uint32_t)pl.sk_fix_rows.size();
    tables += (int64_t)TL.hent.size() * 8 + (int64_t)TL.hseg.size() * 4 + (int64_t)pl.sk_fix_rows.size() * 8 +
              (int64_t)pl.sk_fix_idx.size() * 4 + (int64_t)pl.sk_scratch * 16;
    launches += 2;
  }
  P.values = m->d_values; P.tile_xoff = tx; P.xdesc = (const uint4 *)xd; P.ktab = kt;
  P.nrows = pl.nrows; P.row_start = pl.row_start; P.rpt = pl.rpt;
  P.values_end = m->d_values + std::max<uint64_t>(m->layout.total_values, 1);
  // device bytes of the transposed tables (no values: they are the forward ones)
  T->dev_bytes = (int64_t)TL.ktab.size() * 8 + (int64_t)pl.tile_xoff.size() * 4 + (int64_t)pl.xdesc.size() * 16 +
                 (int64_t)TL.hent.size() * 8 + (int64_t)TL.hseg.size() * 4 + (int64_t)pl.sk_fix_rows.size() * 4 +
                 (int64_t)pl.sk_fix_ptr.size() * 4 + (int64_t)pl.sk_fix_idx.size() * 4 + (int64_t)pl.sk_scratch * 8;
  for (const BlockTable &B : pl.bt) T->dev_bytes += (int64_t)B.ptr.size() * 4 + (int64_t)B.ent.size() * 8;
  int64_t xrows = 0;
  for (const CsxPartition &p : m->host.parts) xrows += p.nrows;
  T->alg_bytes = m->bytes[CSXB_B_VALUES] + tables + 8 * xrows + 8 * pl.nrows;
  T->launches = launches;
  T->build_us = (int64_t)(std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count() * 1e6);
  m->trans = std::move(T);
  return 0;
}

int csxb_spmv_t(csxb_matrix_t *m, double alpha, const double *d_x, double beta, double *d_y, int overwrite, void *stream) {
  if (m->host.symmetric) return csxb_spmv(m, alpha, d_x, beta, d_y, overwrite, stream);   // A^T = A
  if (!m->trans && csxb_transpose_prepare(m)) return -1;
  if (on_matrix_device(m)) return -1;
  cudaStream_t s = (cudaStream_t)stream;
  const TransState &T = *m->trans;
  const PartLayout &pl = T.lay.part;
  if (!pl.nrows) return 0;
  const uint32_t nseg = (uint32_t)(T.lay.hseg.size() - 1);
  if (nseg) csx_t_segment_kernel<<<(nseg + 7) / 8, 256, 0, s>>>(T.hent, T.hseg, nseg, m->d_values, d_x, T.P.sk_scratch);
  if (T.lay.images) launch_gather<true>(T.P, pl, 0, pl.ntiles, d_x, d_y, alpha, beta, overwrite, s, NoXchg());
  else launch_gather<false>(T.P, pl, 0, pl.ntiles, d_x, d_y, alpha, beta, overwrite, s, NoXchg());
  if (nseg) {
    SkIO io;
    io.x = d_x; io.y = d_y; io.step = nullptr; io.vec[0] = io.vec[1] = nullptr; io.npush = 0;
    launch_fixup(T.P, 0, (uint32_t)pl.sk_fix_rows.size(), 0, 0, 0, pl.nrows, io, alpha, beta, overwrite, s);
  }
  CUDA_TRY(cudaGetLastError());
  return 0;
}

// Host buffers, unpipelined: x (nrows) in, the product, the column window of y (ncols) out.
int csxb_spmv_t_host(csxb_matrix_t *m, double alpha, const double *h_x, double beta, double *h_y, int overwrite) {
  if (m->host.symmetric) return csxb_spmv_host(m, alpha, h_x, beta, h_y, overwrite);
  if (!m->trans && csxb_transpose_prepare(m)) return -1;
  DeviceGuard guard;
  CUDA_TRY(cudaSetDevice(m->device));
  TransState &T = *m->trans;
  const int64_t nr = m->host.nrows, lo = T.lay.part.row_start, n = T.lay.part.nrows;
  if (!T.d_x) {
    CUDA_TRY(cudaMalloc((void **)&T.d_x, (size_t)std::max<int64_t>(nr, 1) * 8));
    m->allocs.push_back(T.d_x);
    CUDA_TRY(cudaMalloc((void **)&T.d_y, (size_t)std::max<int64_t>(m->host.ncols, 1) * 8));
    m->allocs.push_back(T.d_y);
  }
  if (!m->s_run) {
    CUDA_TRY(cudaStreamCreateWithFlags(&m->s_h2d, cudaStreamNonBlocking));
    CUDA_TRY(cudaStreamCreateWithFlags(&m->s_run, cudaStreamNonBlocking));
    CUDA_TRY(cudaStreamCreateWithFlags(&m->s_d2h, cudaStreamNonBlocking));
  }
  CUDA_TRY(cudaMemcpyAsync(T.d_x, h_x, (size_t)nr * 8, cudaMemcpyDefault, m->s_run));
  if (!overwrite && n > 0) CUDA_TRY(cudaMemcpyAsync(T.d_y + lo, h_y + lo, (size_t)n * 8, cudaMemcpyDefault, m->s_run));
  if (csxb_spmv_t(m, alpha, T.d_x, beta, T.d_y, overwrite, m->s_run)) { cudaStreamSynchronize(m->s_run); return -1; }
  if (n > 0) CUDA_TRY(cudaMemcpyAsync(h_y + lo, T.d_y + lo, (size_t)n * 8, cudaMemcpyDefault, m->s_run));
  CUDA_TRY(cudaStreamSynchronize(m->s_run));
  return 0;
}

int64_t csxb_transpose_info(const csxb_matrix_t *m, int what) {
  if (!m || !m->trans) return -1;
  const TransState &T = *m->trans;
  switch (what) {
    case CSXB_T_COL_LO: return T.lay.part.row_start;
    case CSXB_T_COL_HI: return T.lay.part.row_start + T.lay.part.nrows;
    case CSXB_T_DEVICE_BYTES: return T.dev_bytes;
    case CSXB_T_ALG_BYTES: return T.alg_bytes;
    case CSXB_T_LAUNCHES: return T.launches;
    case CSXB_T_HEAVY_COLS: return T.lay.heavy_cols;
    case CSXB_T_SEGMENTS: return (int64_t)T.lay.hseg.size() - 1;
    case CSXB_T_BUILD_US: return T.build_us;
  }
  return -1;
}

// Host walk of the host copy of the transposed tables; builds them on the host when the matrix has none (no device
// needed).  rows / cols: one entry per device-wide value index.
int csxb_decode_coords_t(const csxb_matrix_t *mc, int32_t *rows, int32_t *cols) {
  csxb_matrix *m = const_cast<csxb_matrix *>(mc);
  if (!m || !rows || !cols) return fail("invalid argument");
  if (m->host.symmetric) return fail("CSX-Sym has no transposed tables (A^T = A)");
  TransLayout local;
  const TransLayout *TL = m->trans ? &m->trans->lay : nullptr;
  DeviceLayout fl;
  if (!TL) {
    std::string e = build_layout(m->host, fl);
    if (e.empty()) e = build_transpose_layout(m->host, fl, local);
    if (!e.empty()) return fail("transposed layout: " + e);
    TL = &local;
  }
  int64_t n = 0;
  for (const CsxPartition &p : m->host.parts) n += p.nnz;
  std::fill(rows, rows + n, -1);
  std::fill(cols, cols + n, -1);
  decode_transpose_coords(*TL, rows, cols);
  return 0;
}

// ---- csxb_xchg_*: exchange over peer memory (see XchgDev) ------------------------------------------------
struct csxb_xchg {
  csxb_matrix *m = nullptr;
  int rank = 0, world = 1;
  void *base = nullptr;              // [vec0 | vec1 | ctrl] on m's device
  size_t n = 0;
  std::vector<void *> peer_base;     // other ranks' blocks (CUDA IPC mappings; own slot = base)
  XchgDev dev;
  bool connected = false;
  int64_t tail_lo = 0, tail_hi = 0;   // rows no rank owns (after the last partition's rows)
  int parity = 0;                     // protocol 1: index of the vector the next step reads (host side)
  int64_t issued = 0;                 // steps issued so far
};
static size_t xchg_vec_bytes(size_t n) { return ((n * 8 + 255) / 256) * 256; }
static void xchg_choose_mode(csxb_xchg *h, int64_t own_lo, int64_t own_hi);

csxb_xchg_t *csxb_xchg_create(csxb_matrix_t *m, int rank, int world) {
  if (!m || !m->uploaded) { fail("matrix not uploaded (csxb_upload)"); return nullptr; }
  if (m->host.symmetric) { fail("the peer-memory exchange covers non-symmetric CSX (CSX-Sym: SymHaloReduce)"); return nullptr; }
  if (world < 1 || rank < 0 || rank >= world || world - 1 > XCHG_MAX_PEERS) { fail("invalid rank / world size"); return nullptr; }
  if (m->host.nrows != m->host.ncols) { fail("repeated SpMV with exchange needs a square matrix"); return nullptr; }
  if (cudaSetDevice(m->device) != cudaSuccess) { fail("cudaSetDevice failed"); return nullptr; }
  csxb_xchg *h = new csxb_xchg;
  h->m = m; h->rank = rank; h->world = world; h->n = (size_t)m->host.nrows;
  const size_t vb = xchg_vec_bytes(h->n), total = 2 * vb + 4096;
  if (cudaMalloc(&h->base, total) != cudaSuccess || cudaMemset(h->base, 0, total) != cudaSuccess) {
    fail("device allocation for the exchange vectors failed");
    delete h;
    return nullptr;
  }
  memset(&h->dev, 0, sizeof(h->dev));
  h->dev.vec[0] = (double *)h->base;
  h->dev.vec[1] = (double *)((char *)h->base + vb);
  unsigned long long *ctrl = (unsigned long long *)((char *)h->base + 2 * vb);
  h->dev.step = ctrl; h->dev.error = ctrl + 1; h->dev.started = ctrl + 2; h->dev.bdone = ctrl + 3; h->dev.flags = ctrl + 16;
  h->dev.rank = rank;
  if (world == 1) {
    xchg_choose_mode(h, 0, (int64_t)h->n);
    h->connected = true;
    if (m->host.part_lo + (int)m->host.parts.size() == m->host.nparts_total) { h->tail_lo = m->covered_rows_end; h->tail_hi = (int64_t)h->n; }
  }
  return h;
}

int csxb_xchg_handle(csxb_xchg_t *h, void *handle64) {
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
  cudaIpcMemHandle_t ih;
  CUDA_TRY(cudaSetDevice(h->m->device));
  CUDA_TRY(cudaIpcGetMemHandle(&ih, h->base));
  memcpy(handle64, &ih, 64);
  return 0;
}

// Edge-tiles-first protocol (XchgDev.mode 1) when the rank has one partition whose rows are final after kernel 1
// and the tiles that touch other ranks (they read rows outside [own_lo, own_hi), or their rows are pushed) sit
// at the two ends of the partition.
static void xchg_choose_mode(csxb_xchg *h, int64_t own_lo, int64_t own_hi) {
  XchgDev &D = h->dev;
  D.mode = 0; D.nb = 0; D.edge_lo_end = 0; D.edge_hi_begin = 0;
  static const int dbg = getenv("CSXB_XCHG_DEBUG") ? atoi(getenv("CSXB_XCHG_DEBUG")) : 0;
  if (h->m->layout.parts.size() != 1 || !h->m->layout.parts[0].sk_chunks.empty() || (dbg & 8)) return;   // stream units: protocol 0
  const PartLayout &pl = h->m->layout.parts[0];
  if (!pl.ntiles || pl.ntiles > (int64_t(1) << 30)) return;
  const int64_t tr = pl.tile_rows();
  auto is_edge = [&](int64_t t) {
    if (pl.tile_cmax[t] >= pl.tile_cmin[t] && (pl.tile_cmin[t] < own_lo || pl.tile_cmax[t] >= own_hi)) return true;
    const int64_t r0 = pl.row_start + t * tr, r1 = std::min(pl.row_start + pl.nrows, r0 + tr);
    for (int p = 0; p < D.npush; p++) if (r0 < D.push_hi[p] && r1 > D.push_lo[p]) return true;
    return false;
  };
  int64_t a = 0, b = pl.ntiles;
  while (a < pl.ntiles && is_edge(a)) a++;
  while (b > a && is_edge(b - 1)) b--;
  for (int64_t t = a; t < b; t++) if (is_edge(t)) return;   // an interior tile touches another rank: keep the sync kernel
  // edge CTAs per edge tile (csx_spmv_xe_kernel): a few edge tiles are split so that their rows are out early
  const char *smax = getenv("CSXB_XCHG_SPLIT_MAX");   // tests: 0 forces whole edge tiles
  const int split = (pl.rpt == 4 && a + (pl.ntiles - b) <= (smax ? atoi(smax) : 16)) ? 4 : 1;
  D.mode = 1; D.edge_lo_end = (int)a; D.edge_hi_begin = (int)b; D.nb = (int)(a + (pl.ntiles - b)) * split; D.split = split;
}

// bases[q] = rank q's block as seen from this device (IPC mapping, or the pointer itself inside one process)
static int xchg_plan(csxb_xchg *h, const std::vector<void *> &bases, const int64_t *row_lo, const int64_t *row_n,
                     const int64_t *win_lo, const int64_t *win_hi) {
  const size_t vb = xchg_vec_bytes(h->n);
  XchgDev &D = h->dev;
  D.nwait = 0; D.npush = 0;
  auto overlap = [&](int owner, int reader, int64_t &lo, int64_t &hi) {   // rows of `owner` that `reader` reads
    lo = std::max(row_lo[owner], win_lo[reader]);
    hi = std::min(row_lo[owner] + row_n[owner], win_hi[reader] + 1);
    return hi > lo;
  };
  for (int q = 0; q < h->world; q++) {
    if (q == h->rank) continue;
    int64_t lo, hi, lo2, hi2;
    const bool i_push = overlap(h->rank, q, lo, hi), q_pushes = overlap(q, h->rank, lo2, hi2);
    if (!i_push && !q_pushes) continue;
    void *pb = bases[q];
    if (!pb) return fail("missing peer block");
    D.wait_rank[D.nwait] = q;
    D.peer_flags[D.nwait] = (unsigned long long *)((char *)pb + 2 * vb) + 16;
    D.nwait++;
    if (i_push) {
      D.push_lo[D.npush] = lo; D.push_hi[D.npush] = hi;
      D.push_vec[D.npush][0] = (double *)pb;
      D.push_vec[D.npush][1] = (double *)((char *)pb + vb);
      D.npush++;
    }
  }
  int64_t cov = 0;
  for (int q = 0; q < h->world; q++) cov = std::max(cov, row_lo[q] + row_n[q]);
  h->tail_lo = cov; h->tail_hi = (int64_t)h->n;
  xchg_choose_mode(h, row_lo[h->rank], row_lo[h->rank] + row_n[h->rank]);
  h->connected = true;
  return 0;
}

int csxb_xchg_connect(csxb_xchg_t *h, const void *handles, const int64_t *row_lo, const int64_t *row_n,
                      const int64_t *win_lo, const int64_t *win_hi) {
  if (h->connected) return fail("exchange already connected");
  CUDA_TRY(cudaSetDevice(h->m->device));
  h->peer_base.assign(h->world, nullptr);
  for (int q = 0; q < h->world; q++) {
    if (q == h->rank) continue;
    cudaIpcMemHandle_t ih;
    memcpy(&ih, (const char *)handles + (size_t)q * 64, 64);
    CUDA_TRY(cudaIpcOpenMemHandle(&h->peer_base[q], ih, cudaIpcMemLazyEnablePeerAccess));
  }
  std::vector<void *> bases = h->peer_base;
  bases[h->rank] = h->base;
  return xchg_plan(h, bases, row_lo, row_n, win_lo, win_hi);
}

int csxb_xchg_connect_ptr(csxb_xchg_t *h, void *const *bases, const int64_t *row_lo, const int64_t *row_n,
                          const int64_t *win_lo, const int64_t *win_hi) {
  if (h->connected) return fail("exchange already connected");
  std::vector<void *> b(bases, bases + h->world);
  return xchg_plan(h, b, row_lo, row_n, win_lo, win_hi);
}

void *csxb_xchg_base(csxb_xchg_t *h) { return h->base; }

double *csxb_xchg_vector(csxb_xchg_t *h, int which) { return h->dev.vec[which & 1]; }

int csxb_xchg_spmv(csxb_xchg_t *h, double alpha, void *stream) {
  if (!h->connected) return fail("exchange not connected (csxb_xchg_connect)");
  csxb_matrix *m = h->m;
  if (on_matrix_device(m)) return -1;
  cudaStream_t s = (cudaStream_t)stream;
  static const int dbg = getenv("CSXB_XCHG_DEBUG") ? atoi(getenv("CSXB_XCHG_DEBUG")) : 0;   // tuning aid
  XchgDev X = h->dev;
  const bool copy_push = (dbg & 4) != 0;   // tuning aid: rows pushed by a copy kernel after the step's kernels
  SkIO io;
  io.x = nullptr; io.y = nullptr; io.step = h->dev.step; io.vec[0] = h->dev.vec[0]; io.vec[1] = h->dev.vec[1];
  for (size_t i = 0; i < m->pdev.size(); i++) {
    const PartLayout &pl = m->layout.parts[i];
    if (X.mode == 1) { launch_gather_xe(m->pdev[i], pl, X.vec[h->parity], X.vec[h->parity ^ 1], alpha, h->parity ^ 1, s, X); continue; }
    // The exchange is part of whichever kernel writes the final value of a row: the gather kernel when the partition
    // has a gather pass (it runs last), else the stream kernel and its fix-up.
    const bool gather_last = pl.sk_chunks.empty() || !pl.xdesc.empty() || !pl.bt.empty();
    XchgDev Xp = X;
    io.npush = 0;
    if (copy_push) Xp.npush = 0;
    else if (!gather_last) {
      Xp.npush = 0;
      io.npush = X.npush;
      for (int p = 0; p < X.npush; p++) {
        io.push_lo[p] = X.push_lo[p]; io.push_hi[p] = X.push_hi[p];
        io.push_vec[p][0] = X.push_vec[p][0]; io.push_vec[p][1] = X.push_vec[p][1];
      }
    }
    if (run_partition<false>(m->pdev[i], pl, io, alpha, 0.0, 1, s, Xp)) return fail("no stream kernel for the partition's pattern set");
  }
  if (copy_push && h->dev.npush) csx_xchg_push_kernel<<<148 * 8, 256, 0, s>>>(h->dev);
  if (h->tail_hi > h->tail_lo)
    csx_xchg_zero_tail_kernel<<<(unsigned)std::min<int64_t>(148, (h->tail_hi - h->tail_lo + 255) / 256), 256, 0, s>>>(h->dev, h->tail_lo, h->tail_hi, h->dev.mode == 1 ? (h->parity ^ 1) : -1);
  if (!(dbg & 1) && h->dev.mode == 0) csx_xchg_sync_kernel<<<1, 32, 0, s>>>(h->dev, dbg);
  CUDA_TRY(cudaGetLastError());
  h->parity ^= 1;
  h->issued++;
  return 0;
}

int64_t csxb_xchg_status(csxb_xchg_t *h, int what) {
  unsigned long long v[2] = {0, 0};
  if (cudaSetDevice(h->m->device) != cudaSuccess) return -1;
  if (cudaMemcpy(v, h->dev.step, 16, cudaMemcpyDeviceToHost) != cudaSuccess) return -1;
  if (what == 0 && h->dev.mode == 1) { cudaDeviceSynchronize(); return h->issued; }
  if (what == 2) return h->dev.mode;
  if (what == 3) return h->dev.nb;
  return what == 0 ? (int64_t)v[0] : (int64_t)v[1];
}

void csxb_xchg_destroy(csxb_xchg_t *h) {
  if (!h) return;
  cudaSetDevice(h->m->device);
  cudaDeviceSynchronize();
  for (int q = 0; q < (int)h->peer_base.size(); q++)
    if (q != h->rank && h->peer_base[q]) cudaIpcCloseMemHandle(h->peer_base[q]);
  if (h->base) cudaFree(h->base);
  delete h;
}

// ---- BLAS-1 on device-resident vectors (SURVEY.md section 8f row 4; Vector.cpp:259-377) ------------------
// out = alpha*a + beta*b over [0, n); out may alias a or b.  One pass, 16-byte accesses where aligned.
__global__ void __launch_bounds__(256) csx_vec_axpby_kernel(double *__restrict__ out, const double *a, const double *b, double alpha,
                                                            double beta, long long n) {
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    const double bv = b ? b[i] : 0.0;
    out[i] = alpha * a[i] + beta * bv;
  }
}
// partial dot products: one double per CTA (fixed grid, fixed order: deterministic for a given n)
__global__ void __launch_bounds__(256) csx_vec_dot_kernel(const double *__restrict__ a, const double *__restrict__ b, long long n,
                                                          double *__restrict__ partial) {
  __shared__ double warp_part[8];
  double s = 0.0;
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) s = fma(a[i], b[i], s);
  s = warp_sum(s);
  if ((threadIdx.x & 31) == 0) warp_part[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
    for (int w = 0; w < 8; w++) t += warp_part[w];
    partial[blockIdx.x] = t;
  }
}

int csxb_vec_axpby(double *d_out, const double *d_a, const double *d_b, double alpha, double beta, int64_t n, void *stream) {
  if (n <= 0) return 0;
  const unsigned grid = (unsigned)std::min<int64_t>((n + 255) / 256, 148 * 8);
  csx_vec_axpby_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(d_out, d_a, d_b, alpha, beta, (long long)n);
  CUDA_TRY(cudaGetLastError());
  return 0;
}

int csxb_vec_dot(const double *d_a, const double *d_b, int64_t n, double *result, void *stream) {
  *result = 0.0;
  if (n <= 0) return 0;
  const unsigned grid = (unsigned)std::min<int64_t>((n + 255) / 256, 148 * 4);
  // scratch per device (the vectors decide where the kernel runs: the caller's current device)
  static thread_local double *d_part[64] = {nullptr};
  static thread_local double *h_part[64] = {nullptr};
  int dev = 0;
  CUDA_TRY(cudaGetDevice(&dev));
  if (dev < 0 || dev >= 64) return fail("device index out of range");
  if (!d_part[dev]) {
    CUDA_TRY(cudaMalloc((void **)&d_part[dev], 148 * 4 * sizeof(double)));
    CUDA_TRY(cudaMallocHost((void **)&h_part[dev], 148 * 4 * sizeof(double)));
  }
  double *d_partial = d_part[dev], *h_partial = h_part[dev];
  cudaStream_t s = (cudaStream_t)stream;
  csx_vec_dot_kernel<<<grid, 256, 0, s>>>(d_a, d_b, (long long)n, d_partial);
  CUDA_TRY(cudaMemcpyAsync(h_partial, d_partial, grid * sizeof(double), cudaMemcpyDeviceToHost, s));
  CUDA_TRY(cudaStreamSynchronize(s));
  double t = 0.0;
  for (unsigned i = 0; i < grid; i++) t += h_partial[i];
  *result = t;
  return 0;
}

// ---- tuned-matrix container and single-entry access (SURVEY.md section 8f rows 2 and 3) ------------------
int csxb_save(csxb_matrix_t *m, const char *path) {
  if (!m || !path) return fail("invalid argument");
  CsxMatrix &H = m->host;
  for (size_t i = 0; i < H.parts.size(); i++) {   // values released at upload come back from the device
    CsxPartition &p = H.parts[i];
    if ((int64_t)p.values.size() == p.nnz) continue;
    if (!m->uploaded) return fail("partition values are neither on the host nor on a device");
    CUDA_TRY(cudaSetDevice(m->device));
    p.values.resize((size_t)p.nnz);
    CUDA_TRY(cudaMemcpy(p.values.data(), m->d_values + m->layout.parts[i].val_base, (size_t)p.nnz * 8, cudaMemcpyDeviceToHost));
  }
  std::string e = save_matrix(H, path);
  return e.empty() ? 0 : fail(e);
}

csxb_matrix_t *csxb_load(const char *path, char *err, size_t errlen) {
  if (!path) { put_err(err, errlen, "invalid file name"); return nullptr; }
  csxb_matrix *m = new csxb_matrix;
  std::string e;
  try { e = load_matrix(path, m->host); } catch (std::exception &ex) { e = std::string("cannot load the container: ") + ex.what(); }
  if (!e.empty()) { put_err(err, errlen, e); delete m; return nullptr; }
  return m;
}

// The RCM permutation travels with the matrix (matvec.c:298, 422, 445): perm[old] = new, n = 0 clears it.
int csxb_set_perm(csxb_matrix_t *m, const int32_t *perm, int64_t n) {
  if (!m || n < 0 || (n && (!perm || n != m->host.nrows))) return fail("invalid permutation");
  m->host.permutation.assign(perm, perm + n);
  return 0;
}
int64_t csxb_get_perm(const csxb_matrix_t *m, int32_t *perm) {
  if (!m) return -1;
  if (perm) std::copy(m->host.permutation.begin(), m->host.permutation.end(), perm);
  return (int64_t)m->host.permutation.size();
}

// Locates A(row, col) (zero-based): partition, index into its values (or into dvalues when diag is set).
static int locate_entry(csxb_matrix *m, int64_t row, int64_t col, size_t &part, int64_t &idx, bool &diag) {
  CsxMatrix &H = m->host;
  if (row < 0 || row >= H.nrows || col < 0 || col >= H.ncols) return fail("index out of bounds");
  diag = false;
  if (H.symmetric) {
    if (col > row) std::swap(row, col);   // the lower triangle is what is stored (CsxGetSet.hpp:84-135)
    diag = row == col;
  }
  if (m->row_index.size() != H.parts.size()) m->row_index.assign(H.parts.size(), RowIndex());
  for (size_t i = 0; i < H.parts.size(); i++) {
    CsxPartition &p = H.parts[i];
    const int64_t owned = H.symmetric ? (int64_t)p.dvalues.size() : p.nrows;
    if (row < p.row_start || row >= p.row_start + owned) continue;
    part = i;
    if (diag) { idx = row - p.row_start; return 0; }
    RowIndex &ri = m->row_index[i];
    if (ri.ctl_off.empty()) {
      std::string e = build_row_index(p, H.full_colind, ri);
      if (!e.empty()) return fail(e);
    }
    idx = find_entry(p, H.full_colind, ri, row - p.row_start, col);
    return idx < 0 ? 1 : 0;
  }
  return 1;   // the row belongs to no local partition
}

int csxb_get_entry(csxb_matrix_t *m, int64_t row, int64_t col, double *value) {
  size_t part; int64_t idx; bool diag;
  const int rc = locate_entry(m, row, col, part, idx, diag);
  if (rc) return rc;
  CsxPartition &p = m->host.parts[part];
  if (diag) { *value = p.dvalues[(size_t)idx]; return 0; }
  if ((int64_t)p.values.size() == p.nnz) { *value = p.values[(size_t)idx]; return 0; }
  if (!m->uploaded) return fail("partition values are neither on the host nor on a device");
  CUDA_TRY(cudaSetDevice(m->device));
  CUDA_TRY(cudaMemcpy(value, m->d_values + m->layout.parts[part].val_base + idx, 8, cudaMemcpyDeviceToHost));
  return 0;
}

int csxb_set_entry(csxb_matrix_t *m, int64_t row, int64_t col, double value) {
  size_t part; int64_t idx; bool diag;
  const int rc = locate_entry(m, row, col, part, idx, diag);
  if (rc) return rc;
  CsxPartition &p = m->host.parts[part];
  if (diag) p.dvalues[(size_t)idx] = value;
  else if ((int64_t)p.values.size() == p.nnz) p.values[(size_t)idx] = value;
  if (m->uploaded) {   // the device copy is what the kernels read
    CUDA_TRY(cudaSetDevice(m->device));
    double *dst = diag ? const_cast<double *>(m->pdev[part].dvalues) + idx : m->d_values + m->layout.parts[part].val_base + idx;
    CUDA_TRY(cudaMemcpy(dst, &value, 8, cudaMemcpyHostToDevice));
  }
  return 0;
}

int csxb_decode_coords(const csxb_matrix_t *mc, int part, int32_t *rows, int32_t *cols) {
  csxb_matrix *m = const_cast<csxb_matrix *>(mc);
  if (!m->uploaded) return fail("matrix not uploaded (csxb_upload)");
  if (part < 0 || (size_t)part >= m->pdev.size()) return fail("invalid partition");
  CUDA_TRY(cudaSetDevice(m->device));
  const PartLayout &pl = m->layout.parts[part];
  size_t n = (size_t)m->layout.total_values;
  int *dr = nullptr, *dcl = nullptr;
  CUDA_TRY(cudaMalloc((void **)&dr, std::max<size_t>(n, 1) * 4));
  CUDA_TRY(cudaMalloc((void **)&dcl, std::max<size_t>(n, 1) * 4));
  CUDA_TRY(cudaMemset(dr, 0xff, std::max<size_t>(n, 1) * 4));
  CUDA_TRY(cudaMemset(dcl, 0xff, std::max<size_t>(n, 1) * 4));
  if (pl.ntiles && !pl.xdesc.empty()) csx_decode_gather_kernel<<<(unsigned)pl.ntiles, CTA_THREADS>>>(m->pdev[part], dr, dcl);
  if (!pl.bt.empty()) csx_decode_bt_kernel<<<(unsigned)((pl.nrows + CTA_THREADS - 1) / CTA_THREADS), CTA_THREADS>>>(m->pdev[part], dr, dcl);
  if (!pl.sk_chunks.empty())
    csx_stream_decode_kernel<<<(unsigned)((pl.sk_chunks.size() + SK_WARPS - 1) / SK_WARPS), SK_WARPS * 32>>>(m->pdev[part], dr, dcl);
  CUDA_TRY(cudaGetLastError());
  CUDA_TRY(cudaMemcpy(rows, dr + pl.val_base, (size_t)pl.nnz * 4, cudaMemcpyDeviceToHost));
  CUDA_TRY(cudaMemcpy(cols, dcl + pl.val_base, (size_t)pl.nnz * 4, cudaMemcpyDeviceToHost));
  cudaFree(dr); cudaFree(dcl);
  return 0;
}

}  // extern "C"

#include "device_group.inl"
