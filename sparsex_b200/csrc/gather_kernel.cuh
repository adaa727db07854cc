// Device code of kernel 1 (gather over the cross-row unit table + y initialisation) and the exchange descriptor it
// can push through.  Included by engine.cu (nvcc, sm_100a); tests/emul/ compiles the same text for the host on the
// fibre emulation of the warp intrinsics (CSXB_EMUL; generic instantiations only — the PTX block of the
// 4-rows-per-thread diagonal variant is device-only).  Test infrastructure never ships in the product library.
#pragma once
#include "part_dev.cuh"

// Table units are vertical / diagonal / anti-diagonal runs (gpu_layout.hpp: goes_to_xdt); under CSX-Sym the table
// also lists the transposed image of every unit, stream units included (horizontal runs, blocks, single elements).
// Op::add(device-wide value index, x index) for every element of descriptor d that contributes to `myrow`.
template <bool SYM, class Op>
__device__ __forceinline__ void gather_desc(const uint4 d, const KindEntry *__restrict__ ktab, int myrow, Op &op) {
  const uint32_t meta = d.w, kind = (meta >> 24) & 0xf, size = (meta >> 16) & 0xff;
  const int r = (int)d.y, c = (int)d.z;
  const uint32_t voff = d.x;
  const uint32_t delta = (meta & XD_DELTA1) ? 1u : __ldg(&ktab[meta & 0xffff].delta);
  if (!SYM || !(meta & XD_TRANSPOSED)) {  // vert_tmpl.c, diag_tmpl.c, rdiag_tmpl.c
    const int t = myrow - r;
    if (t < 0) return;
    const uint32_t k = (uint32_t)t / delta;
    if (k * delta != (uint32_t)t || k >= size) return;
    op.add(voff + k, kind == K_VERT ? c : (kind == K_DIAG ? c + t : c - t));
  } else if (kind == K_VERT) {
    // transposed image (CSX-Sym): element (r+a, c+b, v) adds v * x[r+a] to y[c+b];
    // vert_sym_tmpl.c: cur[x_indx] += sum v_k x[y_indx + k*delta]
    if (myrow != c) return;
    for (uint32_t k = 0; k < size; k++) op.add(voff + k, r + (int)(k * delta));
  } else if (kind == K_HORIZ) {   // horiz_sym_tmpl.c: element k at (r, c + k*delta) adds v_k * x[r] to y[c + k*delta]
    const int u = myrow - c;
    if (u < 0) return;
    const uint32_t k = (uint32_t)u / delta;
    if (k * delta != (uint32_t)u || k >= size) return;
    op.add(voff + k, r);
  } else if (kind == K_BCOL) {    // block_col_sym_tmpl.c: rows x align block, row-major; y[c + j] += sum_a v[a][j] * x[r + a]
    const uint32_t align = (__ldg(&ktab[meta & 0xffff].kind_align) >> 8) & 0xff;
    const uint32_t j = (uint32_t)(myrow - c);
    if (myrow < c || j >= align) return;
    for (uint32_t a = 0; a * align < size; a++) op.add(voff + a * align + j, r + (int)a);
  } else if (kind == K_BROW) {    // block_row_sym_tmpl.c: align x cols block, column-major; y[c + j] += sum_a v[j][a] * x[r + a]
    const uint32_t align = (__ldg(&ktab[meta & 0xffff].kind_align) >> 8) & 0xff;
    const uint32_t j = (uint32_t)(myrow - c);
    if (myrow < c || j * align >= size) return;
    for (uint32_t a = 0; a < align; a++) op.add(voff + j * align + a, r + (int)a);
  } else {  // diag_sym_tmpl.c, rdiag_sym_tmpl.c
    const int u = kind == K_DIAG ? myrow - c : c - myrow;
    if (u < 0) return;
    const uint32_t k = (uint32_t)u / delta;
    if (k * delta != (uint32_t)u || k >= size) return;
    op.add(voff + k, r + u);
  }
}

// rows a descriptor can contribute to: [lo, hi] (global rows; columns for a transposed image)
template <bool SYM>
__device__ __forceinline__ bool desc_touches(const uint4 d, const KindEntry *__restrict__ ktab, int row_lo, int row_hi) {
  const uint32_t meta = d.w, kind = (meta >> 24) & 0xf, size = (meta >> 16) & 0xff;
  const int r = (int)d.y, c = (int)d.z;
  const uint32_t delta = (meta & XD_DELTA1) ? 1u : __ldg(&ktab[meta & 0xffff].delta);
  const int span = (int)((size - 1) * delta);
  int lo, hi;
  if (!SYM || !(meta & XD_TRANSPOSED)) { lo = r; hi = r + span; }
  else if (kind == K_VERT) { lo = hi = c; }
  else if (kind == K_DIAG || kind == K_HORIZ) { lo = c; hi = c + span; }
  else if (kind == K_ADIAG) { lo = c - span; hi = c; }
  else {   // block image: its columns
    const uint32_t align = (__ldg(&ktab[meta & 0xffff].kind_align) >> 8) & 0xff;
    lo = c; hi = c + (int)(kind == K_BCOL ? align : size / align) - 1;
  }
  return lo <= row_hi && hi >= row_lo;
}

// Linear kinds contribute at most one element per row: returns its value index and x index.
template <bool SYM>
__device__ __forceinline__ bool linear_probe(const uint4 d, const KindEntry *__restrict__ ktab, int myrow, uint32_t &vi, int &xi) {
  const uint32_t meta = d.w, kind = (meta >> 24) & 0xf, size = (meta >> 16) & 0xff;
  const int r = (int)d.y, c = (int)d.z;
  const bool tr = SYM && (meta & XD_TRANSPOSED);
  int t = !tr ? myrow - r : (kind == K_ADIAG ? c - myrow : myrow - c);
  if (t < 0) return false;
  uint32_t k = (uint32_t)t;
  if (!(meta & XD_DELTA1)) {
    uint32_t delta = __ldg(&ktab[meta & 0xffff].delta);
    k = (uint32_t)t / delta;
    if (k * delta != (uint32_t)t) return false;
  }
  if (k >= size) return false;
  vi = d.x + k;
  xi = !tr ? (kind == K_VERT ? c : (kind == K_DIAG ? c + t : c - t)) : (kind == K_HORIZ ? r : r + t);
  return true;
}

// x loads.  COH: the vector is being written by other GPUs while this kernel runs (edge CTAs of the edge-tiles-first
// exchange): ld.global.nc promises read-only data for the whole kernel and goes through L1, where a line fetched by an
// interior CTA of the same SM before the neighbour's halo rows landed would be stale — such loads bypass L1 (ld.global.cg).
template <bool COH>
__device__ __forceinline__ double ldx(const double *p) {
#ifndef CSXB_EMUL
  if (COH) return __ldcg(p);
#endif
  return __ldg(p);
}
template <bool COH>
struct SpmvGatherOp {
  const double *__restrict__ values;  // device-wide
  const double *x;
  double acc;
  __device__ __forceinline__ void add(uint32_t vi, int xi) { acc += __ldg(values + vi) * ldx<COH>(x + xi); }
};

// Entries [e0, e1) of one group of a block table for the row whose values start at `vals` inside every sub-block:
// sum over entries of sum over l < nloop of vals[voff + l * sl] * x[other + l].  NL = nloop at compile time (0: any);
// two entries at a time, all their loads issued before the first FMA.
template <int NL, bool COH>
__device__ __forceinline__ double bt_row(const BtDev &T, const double *__restrict__ vals, const double *__restrict__ x, uint32_t e0,
                                         uint32_t e1) {
  constexpr int N = NL > 0 ? NL : 1;
  const int sl = T.sl;
  double a0 = 0.0, a1 = 0.0;
  uint32_t e = e0;
  if (NL > 0) {
    // the entries of the next pair are requested before the values of this pair are used: the chain entry -> values
    // of one iteration overlaps the next one's entry loads
    uint2 n0{0u, 0u}, n1{0u, 0u};
    if (e + 1 < e1) { n0 = __ldg(T.ent + e); n1 = __ldg(T.ent + e + 1); }
    for (; e + 1 < e1; e += 2) {
      const uint2 b0 = n0, b1 = n1;
      if (e + 3 < e1) { n0 = __ldg(T.ent + e + 2); n1 = __ldg(T.ent + e + 3); }
      const double *v0 = vals + b0.x, *v1 = vals + b1.x, *x0 = x + (b0.y & ~BT_IMAGE), *x1 = x + (b1.y & ~BT_IMAGE);
      double va[N], xa[N], vb[N], xb[N];
#pragma unroll
      for (int l = 0; l < N; l++) { va[l] = __ldg(v0 + l * sl); xa[l] = ldx<COH>(x0 + l); vb[l] = __ldg(v1 + l * sl); xb[l] = ldx<COH>(x1 + l); }
#pragma unroll
      for (int l = 0; l < N; l++) { a0 += va[l] * xa[l]; a1 += vb[l] * xb[l]; }
    }
  }
  for (; e < e1; e++) {
    const uint2 b = __ldg(T.ent + e);
    const double *vp = vals + b.x, *xp = x + (b.y & ~BT_IMAGE);
    if (NL > 0) {
      double va[N], xa[N];
#pragma unroll
      for (int l = 0; l < N; l++) { va[l] = __ldg(vp + l * sl); xa[l] = ldx<COH>(xp + l); }
#pragma unroll
      for (int l = 0; l < N; l++) a0 += va[l] * xa[l];
    } else {
      for (int l = 0; l < T.nloop; l++) a0 += __ldg(vp + l * sl) * ldx<COH>(xp + l);
    }
  }
  return a0 + a1;
}

// ---- multi-GPU exchange over peer memory ---------------------------------------------------------------
// One process per GPU.  Every rank holds two full-length vectors (ping-pong) in one cudaMalloc'ed block that
// the other ranks map through CUDA IPC.  Step k reads vec[k & 1] and writes vec[(k + 1) & 1]: the SpMV kernel
// stores the rows it owns locally and, where another rank's partition reads them (its column window), also
// straight into that rank's copy over NVLink — the exchange is part of the kernel's epilogue, there is no
// separate collective.  Flags in the same block order the steps: after its own kernels of step k a rank
// stores k + 1 into its slot of every neighbour's flag array and then waits (one warp, csx_xchg_sync_kernel)
// until every neighbour has done the same — the halo of the next step has arrived, and no neighbour still
// reads the buffer that the next step overwrites.  The step counter lives on the device, so a captured CUDA
// graph can be replayed.
constexpr int XCHG_MAX_PEERS = 15;
struct XchgDev {
  double *vec[2];                          // local ping-pong vectors
  unsigned long long *step;                // local: number of steps this rank has finished
  unsigned long long *flags;               // local: flags[q] = number of steps rank q has finished
  unsigned long long *error;               // local: set when a wait timed out
  int rank, nwait, npush;
  int wait_rank[XCHG_MAX_PEERS];
  unsigned long long *peer_flags[XCHG_MAX_PEERS];   // neighbours' flag arrays (peer memory), same order as wait_rank
  long long push_lo[XCHG_MAX_PEERS], push_hi[XCHG_MAX_PEERS];   // global rows [lo, hi) of mine that peer p reads
  double *push_vec[XCHG_MAX_PEERS][2];     // that peer's ping-pong vectors (peer memory)
  // "edge tiles first" protocol (mode 1; partitions whose rows are final after kernel 1): the tiles that read rows
  // of other ranks or whose rows other ranks read are the first `nb` CTAs of the step's kernel.  They wait for the
  // neighbours' edge tiles of the previous step, and the last of them to finish publishes this step to the
  // neighbours — a whole step before anybody needs it.  The other tiles touch no remote data and never wait.
  int mode;                                // 0: sync kernel at the end of every step, 1: edge tiles first
  int nb;                                  // number of edge CTAs
  int split;                               // edge CTAs per edge tile: 4 (one row per thread) when there are few edge tiles, else 1
  int edge_lo_end, edge_hi_begin;          // edge tiles are [0, edge_lo_end) and [edge_hi_begin, ntiles)
  unsigned long long *started, *bdone;     // local counters: CTAs that have read the step number / edge CTAs finished
};
struct NoXchg {};

// ---- kernel 1: gather over the cross-row unit table + y initialisation --------------------------
// One CTA = one tile of CTA_THREADS * RPT rows; warp w owns RPT consecutive 32-row groups and lane L owns
// rows  tile0 + (w*RPT + k)*32 + L,  k < RPT  (RPT independent accumulators per thread).  Warps never
// synchronise with each other.  Every owned row of y is written exactly once here
// (y = alpha*acc + beta*y); the chunk kernel adds the remaining units afterwards.
// KSET specialises the gather for the set of unit kinds the partition's table holds:
//   KSET_ANY    vertical / diagonal / anti-diagonal units of any stride, CSX-Sym images included
//   KSET_DIAG1  only diagonal units of stride 1 (what the stencil matrices of the baseline configs encode to)
// The kernel is bandwidth-bound and latency-sensitive: compiled for 8 resident CTAs per SM (32 registers).
// BT: the partition has block tables (block units; gpu_layout.hpp: BlockTable).
// VAR = 1 (4-rows-per-thread diagonal instantiation) issues the eight loads of a unit as one inline-PTX block so
// that all of them are in flight before the first FMA; ptxas otherwise interleaves loads and FMAs at 32 registers.
enum { KSET_ANY = 0, KSET_DIAG1 = 1 };
// The work of one warp of one CTA: rows [row_block * CTA_THREADS * RPT, +CTA_THREADS * RPT) with the descriptor list of
// layout tile `tile` (the same number, unless an edge CTA of the exchange walks a quarter of a 4-rows-per-thread tile
// with one row per thread).  PUSH: rows that other ranks read are also stored into their vectors (exchange).
template <bool XD, bool SYM, int RPT, int KSET, int VAR, bool PUSH, class XP, bool BT = false, bool COH = false>
__device__ __forceinline__ void spmv_tile(const PartDev &P, const double *__restrict__ x, double *__restrict__ y, double alpha,
                                          double beta, int overwrite, const long long tile, const long long row_block, const XP &X,
                                          const unsigned long long xk) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const long long lrow0 = ((row_block * (CTA_THREADS / 32) + warp) * RPT) * 32;   // first row of this warp (partition relative)
  if (lrow0 >= P.nrows) return;
  double acc[RPT];
#pragma unroll
  for (int k = 0; k < RPT; k++) acc[k] = 0.0;

  unsigned long long pol_stream = 0, pol_keep = 0;   // L2 cache policies of VAR 3
#ifndef CSXB_EMUL
  if (VAR == 3) {
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol_stream));
    asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol_keep));
  }
#endif
  if (XD) {
    const uint32_t b = __ldg(P.tile_xoff + tile), e = __ldg(P.tile_xoff + tile + 1);
    const int grow0 = (int)(P.row_start + lrow0);       // global rows of this warp: [grow0, grow0 + 32*RPT)
    const double *__restrict__ values = P.values;
    // each lane inspects one descriptor of the tile; the ones that reach this warp's rows are
    // then visited by the whole warp (warp-uniform loop over the ballot mask)
    for (uint32_t base = b; base < e; base += 32) {
      const uint32_t j = base + lane;
      bool hit = false;
      if (j < e) {
        const uint4 d = __ldg(P.xdesc + j);
        if (KSET == KSET_DIAG1) hit = (int)d.y <= grow0 + 32 * RPT - 1 && (int)d.y + (int)((d.w >> 16) & 0xff) > grow0;
        else hit = desc_touches<SYM>(d, P.ktab, grow0, grow0 + 32 * RPT - 1);
      }
      uint32_t mask = __ballot_sync(FULL, hit);
      while (mask) {
        const uint4 d = __ldg(P.xdesc + base + __ffs(mask) - 1);
        mask &= mask - 1;
        if (KSET == KSET_DIAG1) {  // diag_tmpl.c with delta 1: y[r+k] += x[c+k] * v[k]
          const int t0 = grow0 + lane - (int)d.y;
          const uint32_t size = (d.w >> 16) & 0xff;
          // one base pointer per stream; the RPT rows of this lane sit at fixed 256-byte strides from it
          const double *__restrict__ vp = values + ((long long)d.x + t0);
          const double *__restrict__ xp = x + ((long long)(int)d.z + t0);
#ifndef CSXB_EMUL
          if (VAR == 3 && RPT == 4) {
            // as VAR 1, with cache policies: the values are read once (no L1 allocation, first to leave L2), x is re-read
            // by the other diagonals and by neighbouring tiles (last to leave L2)
            double v0, v1, v2, v3, x0, x1, x2, x3;
            asm volatile(
                "{\n\t.reg .pred p0, p1, p2, p3;\n\t"
                "setp.lt.u32 p0, %8, %12;\n\tsetp.lt.u32 p1, %9, %12;\n\tsetp.lt.u32 p2, %10, %12;\n\tsetp.lt.u32 p3, %11, %12;\n\t"
                "mov.f64 %0, 0d0000000000000000;\n\tmov.f64 %1, 0d0000000000000000;\n\t"
                "mov.f64 %2, 0d0000000000000000;\n\tmov.f64 %3, 0d0000000000000000;\n\t"
                "mov.f64 %4, 0d0000000000000000;\n\tmov.f64 %5, 0d0000000000000000;\n\t"
                "mov.f64 %6, 0d0000000000000000;\n\tmov.f64 %7, 0d0000000000000000;\n\t"
                "@p0 ld.global.nc.L1::no_allocate.L2::cache_hint.f64 %0, [%13], %15;\n\t@p0 ld.global.nc.L2::cache_hint.f64 %4, [%14], %16;\n\t"
                "@p1 ld.global.nc.L1::no_allocate.L2::cache_hint.f64 %1, [%13+256], %15;\n\t@p1 ld.global.nc.L2::cache_hint.f64 %5, [%14+256], %16;\n\t"
                "@p2 ld.global.nc.L1::no_allocate.L2::cache_hint.f64 %2, [%13+512], %15;\n\t@p2 ld.global.nc.L2::cache_hint.f64 %6, [%14+512], %16;\n\t"
                "@p3 ld.global.nc.L1::no_allocate.L2::cache_hint.f64 %3, [%13+768], %15;\n\t@p3 ld.global.nc.L2::cache_hint.f64 %7, [%14+768], %16;\n\t}"
                : "=d"(v0), "=d"(v1), "=d"(v2), "=d"(v3), "=d"(x0), "=d"(x1), "=d"(x2), "=d"(x3)
                : "r"((uint32_t)t0), "r"((uint32_t)(t0 + 32)), "r"((uint32_t)(t0 + 64)), "r"((uint32_t)(t0 + 96)), "r"(size),
                  "l"(vp), "l"(xp), "l"(pol_stream), "l"(pol_keep));
            acc[0] += v0 * x0; acc[1 % RPT] += v1 * x1; acc[2 % RPT] += v2 * x2; acc[3 % RPT] += v3 * x3;
            continue;
          }
          if (VAR == 1 && RPT == 4) {
            // the eight loads of a unit as one block, so that all of them are in flight before the first FMA
            double v0, v1, v2, v3, x0, x1, x2, x3;
            asm volatile(
                "{\n\t.reg .pred p0, p1, p2, p3;\n\t"
                "setp.lt.u32 p0, %8, %12;\n\tsetp.lt.u32 p1, %9, %12;\n\tsetp.lt.u32 p2, %10, %12;\n\tsetp.lt.u32 p3, %11, %12;\n\t"
                "mov.f64 %0, 0d0000000000000000;\n\tmov.f64 %1, 0d0000000000000000;\n\t"
                "mov.f64 %2, 0d0000000000000000;\n\tmov.f64 %3, 0d0000000000000000;\n\t"
                "mov.f64 %4, 0d0000000000000000;\n\tmov.f64 %5, 0d0000000000000000;\n\t"
                "mov.f64 %6, 0d0000000000000000;\n\tmov.f64 %7, 0d0000000000000000;\n\t"
                "@p0 ld.global.nc.f64 %0, [%13];\n\t@p0 ld.global.nc.f64 %4, [%14];\n\t"
                "@p1 ld.global.nc.f64 %1, [%13+256];\n\t@p1 ld.global.nc.f64 %5, [%14+256];\n\t"
                "@p2 ld.global.nc.f64 %2, [%13+512];\n\t@p2 ld.global.nc.f64 %6, [%14+512];\n\t"
                "@p3 ld.global.nc.f64 %3, [%13+768];\n\t@p3 ld.global.nc.f64 %7, [%14+768];\n\t}"
                : "=d"(v0), "=d"(v1), "=d"(v2), "=d"(v3), "=d"(x0), "=d"(x1), "=d"(x2), "=d"(x3)
                : "r"((uint32_t)t0), "r"((uint32_t)(t0 + 32)), "r"((uint32_t)(t0 + 64)), "r"((uint32_t)(t0 + 96)), "r"(size),
                  "l"(vp), "l"(xp));
            acc[0] += v0 * x0; acc[1 % RPT] += v1 * x1; acc[2 % RPT] += v2 * x2; acc[3 % RPT] += v3 * x3;
            continue;
          }
#endif
          double v[RPT], xv[RPT];
#pragma unroll
          for (int k = 0; k < RPT; k++) {
            v[k] = 0.0; xv[k] = 0.0;
            if ((uint32_t)(t0 + k * 32) < size) { v[k] = __ldg(vp + k * 32); xv[k] = ldx<COH>(xp + k * 32); }
          }
#pragma unroll
          for (int k = 0; k < RPT; k++) acc[k] += v[k] * xv[k];
          continue;
        }
        // one element per row, except the transposed images of vertical and block units, which fold several
        // elements into one row
        if (!(SYM && (d.w & XD_TRANSPOSED) && (((d.w >> 24) & 0xf) == K_VERT || ((d.w >> 24) & 0xf) >= K_BROW))) {
          double v[RPT], xv[RPT];  // issue all RPT value / x loads of this unit before using them
#pragma unroll
          for (int k = 0; k < RPT; k++) {
            uint32_t vi; int xi;
            v[k] = 0.0; xv[k] = 0.0;
            if (linear_probe<SYM>(d, P.ktab, grow0 + k * 32 + lane, vi, xi)) { v[k] = __ldg(values + vi); xv[k] = ldx<COH>(x + xi); }
          }
#pragma unroll
          for (int k = 0; k < RPT; k++) acc[k] += v[k] * xv[k];
        } else {
#pragma unroll
          for (int k = 0; k < RPT; k++) {
            SpmvGatherOp<COH> op{values, x, 0.0};
            gather_desc<SYM>(d, P.ktab, grow0 + k * 32 + lane, op);
            acc[k] += op.acc;
          }
        }
      }
    }
  }

  // block tables: every row finds the sub-blocks that add to it through its aligned group of rows (gpu_layout.hpp:
  // BlockTable; block_row_tmpl.c, block_col_tmpl.c, block_*_sym_tmpl.c); entries in source order
  for (int c = 0; BT && c < P.nbt; c++) {
    const BtDev &T = P.bt[c];
#pragma unroll 1
    for (int k = 0; k < RPT; k++) {
      const long long lrow = lrow0 + k * 32 + lane;
      if (lrow < P.nrows) {
        const uint32_t g = (uint32_t)(P.row_start + lrow);
        uint32_t J = g;
        if (T.G != 1) { J = __umulhi(g, T.magic); if (J * (uint32_t)T.G > g) J--; }   // g / G
        const int f = (int)(g - J * (uint32_t)T.G) * T.sf;
        const uint32_t *pp = T.ptr + ((long long)J - T.j0);
        const uint32_t e0 = __ldg(pp), e1 = __ldg(pp + 1);
        switch (T.nloop) {
          case 1: acc[k] += bt_row<1, COH>(T, P.values + f, x, e0, e1); break;
          case 2: acc[k] += bt_row<2, COH>(T, P.values + f, x, e0, e1); break;
          case 3: acc[k] += bt_row<3, COH>(T, P.values + f, x, e0, e1); break;
          case 4: acc[k] += bt_row<4, COH>(T, P.values + f, x, e0, e1); break;
          default: acc[k] += bt_row<0, COH>(T, P.values + f, x, e0, e1);
        }
      }
    }
  }

#pragma unroll
  for (int k = 0; k < RPT; k++) {
    const long long lrow = lrow0 + k * 32 + lane;
    if (lrow < P.nrows) {
      const long long g = P.row_start + lrow;
      double a = acc[k];
      if (SYM && P.dvalues) a += __ldg(P.dvalues + lrow) * ldx<COH>(x + g);   // diagonal (CsxJit.hpp:373-394 new-row hook)
      const double r = overwrite ? alpha * a : alpha * a + beta * y[g];
      y[g] = r;
      if constexpr (PUSH) {   // the exchange: rows another rank's partition reads go straight into its next x.
        // No fence per store (a system fence would wait for every NVLink acknowledgement in turn): the step is
        // published to the neighbours only after a system-scope fence (edge CTAs below, or the sync kernel).
        for (int p = 0; p < X.npush; p++)
          if (g >= X.push_lo[p] && g < X.push_hi[p]) X.push_vec[p][(xk & 1) ^ 1][g] = r;
      }
    }
  }
}


// ---- heavy columns of the transposed product (gpu_layout.hpp: TransLayout) -------------------------------------------
// One warp sums segment s of table-4 entries: the lanes stride the entries (two accumulators, loads of both in flight),
// the fixed butterfly of warp_sum combines the lanes, so the sum does not depend on timing.  Lane 0 stores it in
// scratch[s]; csx_stream_fixup_kernel adds the segments of a column to y in segment order.
__device__ __forceinline__ void t_segment_warp(const uint2 *__restrict__ ent, const uint32_t *__restrict__ seg,
                                               const double *__restrict__ values, const double *__restrict__ x,
                                               double *__restrict__ scratch, uint32_t s, int lane) {
  const uint32_t e0 = __ldg(seg + s), e1 = __ldg(seg + s + 1);
  double a0 = 0.0, a1 = 0.0;
  uint32_t e = e0 + (uint32_t)lane;
  for (; e + 32 < e1; e += 64) {
    const uint2 b0 = __ldg(ent + e), b1 = __ldg(ent + e + 32);
    const double v0 = __ldg(values + b0.x), x0 = __ldg(x + (b0.y & ~BT_IMAGE));
    const double v1 = __ldg(values + b1.x), x1 = __ldg(x + (b1.y & ~BT_IMAGE));
    a0 += v0 * x0;
    a1 += v1 * x1;
  }
  if (e < e1) {
    const uint2 b = __ldg(ent + e);
    a0 += __ldg(values + b.x) * __ldg(x + (b.y & ~BT_IMAGE));
  }
  const double a = warp_sum(a0 + a1);
  if (lane == 0) scratch[s] = a;
}
