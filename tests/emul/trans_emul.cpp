// Host emulation of the transposed product (test infrastructure): tunes a CSR matrix with the product encoder, builds
// the forward layout and the transposed layout of sparsex_b200/csrc/gpu_layout.cpp, and executes the gather of
// gather_kernel.cuh over the transposed tables with the instantiation csxb_spmv_t picks, the heavy-column segments
// (t_segment_warp) and the fix-up of their sums, warp by warp on the fibre emulation of warp_emul.hpp.
#include "warp_emul.hpp"

#include <cmath>
#include <sstream>
#include <string>
#include <vector>

#define CSXB_EMUL 1
#include "../../sparsex_b200/csrc/csx_host.hpp"
#include <type_traits>
#include "../../sparsex_b200/csrc/gather_kernel.cuh"

namespace {
void put_err(char *err, size_t n, const std::string &m) {
  if (err && n) { strncpy(err, m.c_str(), n - 1); err[n - 1] = 0; }
}
template <bool XD, bool SYM, int RPT, int KSET, bool BT>
void run_tiles(const PartDev &P, int64_t ntiles, const double *x, double *y, double alpha, double beta, int ow) {
  for (int64_t t = 0; t < ntiles; t++)
    for (int w = 0; w < CTA_THREADS / 32; w++) {
      warp_emul::warp_in_cta() = w;
      warp_emul::run_warp([&](int) { spmv_tile<XD, SYM, RPT, KSET, 0, false, NoXchg, BT>(P, x, y, alpha, beta, ow, t, t, NoXchg(), 0); });
    }
  warp_emul::warp_in_cta() = 0;
}
template <bool SYM, int RPT>
int dispatch(const PartDev &P, const PartLayout &pl, const double *x, double *y, double alpha, double beta, int ow) {
  const bool xd = !pl.xdesc.empty(), bt = !pl.bt.empty(), diag1 = !SYM && pl.xd_diag1_only && xd && !bt;   // launch_gather
  if (bt) { if (xd) run_tiles<true, SYM, RPT, KSET_ANY, true>(P, pl.ntiles, x, y, alpha, beta, ow); else run_tiles<false, SYM, RPT, KSET_ANY, true>(P, pl.ntiles, x, y, alpha, beta, ow); return 3; }
  if (diag1) { run_tiles<true, SYM, RPT, KSET_DIAG1, false>(P, pl.ntiles, x, y, alpha, beta, ow); return 1; }
  if (xd) { run_tiles<true, SYM, RPT, KSET_ANY, false>(P, pl.ntiles, x, y, alpha, beta, ow); return 2; }
  run_tiles<false, SYM, RPT, KSET_ANY, false>(P, pl.ntiles, x, y, alpha, beta, ow);
  return 0;
}
}  // namespace

// y (ncols) = alpha * A^T x (+ beta * y unless overwrite); dec_rows / dec_cols (total values): csxb_decode_coords_t.
// stats: [0] images, [1] rows per thread, [2] instantiation (0 no table, 1 diagonal, 2 generic, 3 block tables),
// [3] descriptors, [4] block tables, [5] heavy columns, [6] segments, [7] column window lo, [8] hi
extern "C" int emul_spmv_t(const int32_t *rowptr, const int32_t *colind, const double *values, int64_t nrows, int64_t ncols,
                           const char *options, double alpha, const double *x, double beta, double *y, int overwrite,
                           int32_t *dec_rows, int32_t *dec_cols, int64_t *stats, char *err, size_t errlen) {
  TuneOptions o;
  if (options) {
    std::stringstream ss(options);
    std::string kv;
    while (std::getline(ss, kv, ';')) {
      if (kv.empty()) continue;
      size_t eq = kv.find('=');
      std::string e = eq == std::string::npos ? "malformed option" : o.set(kv.substr(0, eq), kv.substr(eq + 1));
      if (!e.empty()) { put_err(err, errlen, e); return -1; }
    }
  }
  CsxMatrix M;
  CsrView v{rowptr, colind, values, nrows, ncols};
  std::string e = tune_csr(v, o, 0, o.nr_threads, M);
  if (!e.empty()) { put_err(err, errlen, e); return -1; }
  DeviceLayout L;
  e = build_layout(M, L);
  TransLayout T;
  if (e.empty()) e = build_transpose_layout(M, L, T);
  if (!e.empty()) { put_err(err, errlen, "layout: " + e); return -1; }
  std::vector<double> vals((size_t)L.total_values + 2, 0.0);
  for (size_t i = 0; i < L.parts.size(); i++) memcpy(vals.data() + L.parts[i].val_base, M.parts[i].values.data(), M.parts[i].values.size() * 8);
  for (uint64_t i = 0; i < L.total_values; i++) { dec_rows[i] = -1; dec_cols[i] = -1; }
  decode_transpose_coords(T, dec_rows, dec_cols);
  const PartLayout &pl = T.part;
  PartDev P;
  memset(&P, 0, sizeof(P));
  P.values = vals.data();
  P.tile_xoff = pl.tile_xoff.data();
  P.xdesc = reinterpret_cast<const uint4 *>(pl.xdesc.data());
  P.ktab = T.ktab.data();
  P.nrows = pl.nrows; P.row_start = pl.row_start; P.rpt = pl.rpt;
  for (size_t t = 0; t < pl.bt.size(); t++) {
    const BlockTable &B = pl.bt[t];
    P.bt[t] = BtDev{B.ptr.data(), reinterpret_cast<const uint2 *>(B.ent.data()), (long long)B.j0, B.G, B.nloop, B.sf, B.sl, B.image, (uint32_t)((0x100000000ull + B.G - 1) / B.G)};
  }
  P.nbt = (int)pl.bt.size();
  const uint32_t nseg = (uint32_t)T.hseg.size() - 1;
  std::vector<double> scratch(nseg + 1, std::nan(""));
  for (uint32_t s = 0; s < nseg; s++)   // csx_t_segment_kernel
    warp_emul::run_warp([&](int lane) {
      t_segment_warp(reinterpret_cast<const uint2 *>(T.hent.data()), T.hseg.data(), vals.data(), x, scratch.data(), s, lane);
    });
  int inst = 0;
  if (pl.nrows) {
    if (T.images) inst = pl.rpt == 4 ? dispatch<true, 4>(P, pl, x, y, alpha, beta, overwrite) : dispatch<true, 1>(P, pl, x, y, alpha, beta, overwrite);
    else inst = pl.rpt == 4 ? dispatch<false, 4>(P, pl, x, y, alpha, beta, overwrite) : dispatch<false, 1>(P, pl, x, y, alpha, beta, overwrite);
  }
  for (size_t f = 0; f < pl.sk_fix_rows.size(); f++) {   // csx_stream_fixup_kernel
    double sum = 0.0;
    for (uint32_t j = pl.sk_fix_ptr[f]; j < pl.sk_fix_ptr[f + 1]; j++) sum += scratch[pl.sk_fix_idx[j]];
    double *yp = y + pl.row_start + pl.sk_fix_rows[f];
    *yp = *yp + alpha * sum;
  }
  if (stats) {
    stats[0] = T.images; stats[1] = pl.rpt; stats[2] = inst; stats[3] = (int64_t)pl.xdesc.size(); stats[4] = (int64_t)pl.bt.size();
    stats[5] = T.heavy_cols; stats[6] = nseg; stats[7] = pl.row_start; stats[8] = pl.row_start + pl.nrows;
  }
  return 0;
}
