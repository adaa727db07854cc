// GPU-side layout derived from the CSX byte stream (product code).
//
// The ctl stream and the values array go to HBM verbatim.  What the reference
// gets from sequential execution on one core per partition
// (src/templates/csx_spmv_tmpl.c:66-101) the GPU gets from side tables built
// once at tune time by decoding ctl on the host:
//
//   * stream-kernel chunk table ("warp-segmented ctl chunks", see below) for
//     delta, horizontal and block units;
//   * cross-row unit table (XDT) — vertical / diagonal / anti-diagonal units
//     are better served by a gather: each gets a 16-byte descriptor (value
//     offset, start row, start column, kind/size) listed under every row tile
//     (256 or 1024 rows) it touches, including tiles after the one it starts
//     in ("carry-in").  The thread that owns a row gathers its contributions
//     from the descriptors of its tile: conflict free, no atomics;
//   * CSX-Sym: the transposed update y[col] += v * x[row] of every stored
//     element is a gather as well — the transposed image of every unit is
//     listed under the tiles of its *columns* (a descriptor with the
//     XD_TRANSPOSED flag, or an entry of a block table).  Phase 1
//     (stream kernel + direct table units) computes the lower triangle's own
//     rows, phase 2 (gather kernel) adds the images: no write conflicts, no
//     atomics, bit-reproducible — the counterpart of the reference's
//     per-thread local vectors and map reduction (CsxSpmv.cpp:37-50).
#pragma once
#include <cstdint>
#include <string>
#include <vector>

#include "csx_host.hpp"

#ifdef __CUDACC__
#define SPXB_HD __host__ __device__
#else
#define SPXB_HD
#endif

namespace spxb {

constexpr int CTA_THREADS = 256;      // gather kernel: threads per CTA; a tile has CTA_THREADS * rpt rows
constexpr int CTL_PAD = 32;           // readable bytes past the end of ctl

// unit kinds as the kernels see them
enum Kind : uint32_t {
  K_DELTA8 = 0, K_DELTA16 = 1, K_DELTA32 = 2, K_DELTA64 = 3, K_HORIZ = 4,   // row-local
  K_VERT = 5, K_DIAG = 6, K_ADIAG = 7, K_BROW = 8, K_BCOL = 9                // cross-row
};
inline bool kind_row_local(uint32_t k) { return k <= K_HORIZ; }
inline bool goes_to_xdt(uint32_t kind) { return kind >= K_VERT && kind <= K_ADIAG; }   // table units

// 16-byte cross-row unit descriptor (device layout: uint4)
struct XDesc {
  uint32_t voff;   // index of the unit's first value in the device-wide values array
  int32_t row;     // global 0-based row of the unit's first element
  int32_t col;     // global 0-based column of the unit's first element
  uint32_t meta;   // [0:16) kind-table index  [16:24) size  [24:28) kind  [28] transposed  [29] stride == 1
};
constexpr uint32_t XD_TRANSPOSED = 1u << 28;
constexpr uint32_t XD_DELTA1 = 1u << 29;

struct KindEntry { uint32_t kind_align; uint32_t delta; };  // kind | align << 8 ; stride or free block dim
// ctl unit id -> kind as the stream kernel sees it.  `sl` is the task parameter of this kind: elements per task for
// row-local units, columns per task for block-row units, rows per task for block-column units; `recip` = ceil(2^16 / sl),
// so that n / sl == (n * recip) >> 16 for n < 256.
struct IdEntry { uint32_t kind_align; uint32_t delta; uint32_t sl; uint32_t recip; };

// ---- stream kernel (stream_kernel.cuh) ---------------------------------
// The ctl stream is cut at unit boundaries into chunks of up to SK_MAX_ROUNDS rounds of at most 32 units (a round
// holds at most SK_MAX_TASKS lane tasks and SK_MAX_ELEMS non-zeros; bit 15 of a unit's entry in the offset table
// marks the last unit of a round), at most SK_MAX_BYTES ctl bytes, whose rows fit a window of SK_WROWS rows.  A warp parses one
// unit head per lane, cuts the units into tasks (at most SK_RL_E consecutive elements of a delta / horizontal
// unit; a column range of a block-row unit or a row range of a block-column unit with all its rows in register
// accumulators) and walks 32 tasks at a time.  Row sums are combined across lanes with a segmented shuffle
// reduction and collected in a per-warp shared-memory window of y rows; at the end of the chunk the warp writes
// the rows the chunk owns with plain coalesced stores (y = alpha*sum + beta*y): no atomics, bit-reproducible.
// Rows are owned by the chunk in which their first unit starts; what a chunk contributes to rows of other chunks
// (a row cut by a chunk boundary, block units reaching below the next chunk's first row) goes to a scratch array
// and is added by a small fix-up kernel in chunk order.  Long runs of empty rows are listed as gaps and cleared
// by the same fix-up kernel.  Vertical / diagonal / anti-diagonal units live in the cross-row unit table; the
// stream kernel only parses their heads (they move the column cursor) and gives them an empty task.
constexpr int SK_ROUND_UNITS = 32;
constexpr int SK_MAX_ROUNDS = 4;
constexpr int SK_MAX_UNITS = SK_ROUND_UNITS * SK_MAX_ROUNDS;
constexpr int SK_MAX_TASKS = 224;      // per round (8-bit task offsets)
constexpr int SK_MAX_ELEMS = 1023;
constexpr int SK_MAX_BYTES = 8191;     // 13-bit offsets of unit bodies inside a chunk
constexpr int SK_WROWS = 256;        // rows of the per-warp y window
constexpr int SK_RL_E = 4;           // elements per task of a row-local unit
constexpr int SK_BLK_E = 12;         // element budget of a block task
constexpr int SK_BLK_LINES = 4;      // at most this many columns (block-row) / rows (block-column) per block task
// 32-byte chunk entry (device layout: 2 x uint4)
//   w0 ctl offset (low 32 bits)      w1 index of the first value (partition relative)
//   w2 column cursor before the first unit   w3 window base row (partition relative)
//   w4 first entry in the unit-offset table  w5 first scratch slot of the chunk's foreign rows
//   w6 [0:8) units-1  [8:16) first unit's row - window base  [16:24) first flushed window row
//      [24:30) ctl offset bits 32..37  [30] head row is foreign  [31] a block-column unit has several tasks
//   w7 [0:9) end of the flushed window rows  [9:18) end of the foreign tail rows
struct SkEntry { uint32_t w[8]; };
struct SkGap { int64_t lo, hi; };    // partition-relative rows [lo, hi) no chunk window covers

// Tasks of a unit (same arithmetic on host and device).  ie.sl = elements (row-local), columns (block-row) or
// rows (block-column) per task, ie.recip = ceil(2^16 / sl).
SPXB_HD inline uint32_t sk_unit_tasks(uint32_t kind, uint32_t size, uint32_t delta, uint32_t sl, uint32_t recip) {
  if (kind <= 4u) return (size + SK_RL_E - 1) / SK_RL_E;          // K_DELTA8..K_HORIZ
  if (kind >= 8u) return ((delta + sl - 1) * recip) >> 16;        // K_BROW, K_BCOL: delta = free dimension
  return 1;                                                       // table units: one empty task
}

// Block tables: block-row and block-column units whose shape and alignment allow it are cut into sub-blocks of one
// shape per table, and every sub-block gets an 8-byte entry in the list of the aligned group of G rows it adds to.
// The thread that owns global row g (gather kernel) walks the entries of group g / G and adds
//   sum over l < nloop of  values[voff + (g % G) * sf + l * sl] * x[other + l].
//   0 block-column unit, own rows (rows x A, row-major):     G = sub-block rows, nloop = A, sf = A, sl = 1, other = first column
//   1 block-column unit, CSX-Sym image (y[col] += v*x[row]): G = A, nloop = sub-block rows, sf = 1, sl = A, other = first row
//   2 block-row unit, own rows (A x cols, column-major):     G = A, nloop = sub-block columns, sf = 1, sl = A, other = first column
//   3 block-row unit, CSX-Sym image, one entry per aligned group of g columns (g = 1 if the columns are not aligned):
//                                                           G = g, nloop = A, sf = A, sl = 1, other = first row
//   4 single elements (own row: other = column; CSX-Sym image: other = row): G = 1, nloop = 1
// Table 4 takes the elements of the delta / horizontal / unaligned block units of a partition in which such units are
// a minority (at most 40 % of the non-zeros): the partition then needs no stream kernel at all.
// No ctl decoding, no write conflicts; under CSX-Sym both uses of a value happen in the same kernel, close in time, so
// the second one is an L2 hit.
struct BlockImage { uint32_t voff; uint32_t other; };   // first value of the sub-block (device wide); first column / row,
                                                        // bit 31: the entry is a CSX-Sym image (table 4 holds both sorts)
constexpr uint32_t BT_IMAGE = 0x80000000u;
struct BlockTable {
  int G = 1, nloop = 0, sf = 0, sl = 0;
  int image = 0;                         // CSX-Sym images (y[col] += v*x[row]) rather than the units' own rows
  int64_t j0 = 0;                        // global index of the partition's first group
  std::vector<uint32_t> ptr;             // groups + 1
  std::vector<BlockImage> ent;
};
constexpr int BT_MAX = 5;                // tables per partition

struct PartLayout {
  int64_t nrows = 0, row_start = 0, nnz = 0, ctl_size = 0;
  // stream kernel tables (non-symmetric partitions)
  std::vector<SkEntry> sk_chunks;
  std::vector<uint16_t> sk_uoffs;        // offset of every unit head inside its chunk
  std::vector<int32_t> sk_fix_rows;      // rows that receive foreign contributions ...
  std::vector<uint32_t> sk_fix_ptr;      // ... their scratch slots sk_fix_idx[ptr[i] .. ptr[i+1]) in chunk order
  std::vector<uint32_t> sk_fix_idx;
  std::vector<SkGap> sk_gaps;
  uint32_t sk_scratch = 0;               // scratch doubles
  uint32_t sk_kmask = 0;                 // unit kinds the stream kernel meets: bit k = Kind k
  int sk_rows = 1;                       // register accumulators a task needs (rows of a block task)
  int sk_bc = 0;                         // > 0: every block-column task is exactly sk_rows rows x sk_bc columns
  int sk_brc = 0;                        // > 0: every block-row task is exactly sk_rows rows x sk_brc columns
  int64_t sk_stat[4] = {0, 0, 0, 0};     // rounds, windows of 32 tasks, tasks, elements (layout statistics)
  // host side only (slabs of the pipelined host-buffer SpMV): per chunk the window base row, the last row it
  // touches and the columns it reads
  std::vector<int32_t> sk_first_row, sk_last_row, sk_cmin, sk_cmax;
  uint64_t val_base = 0, ctl_base = 0;   // offsets into the device-wide arrays
  bool has_flat = false;                 // some unit is handled by the stream kernel
  bool is_halo = false;                  // CSX-Sym pseudo-partition: rows of other devices that local units update
  bool xd_diag1_only = true;             // every descriptor of this partition's table is a direct diagonal unit of stride 1
  int64_t ntiles = 0;
  int rpt = 1;                           // rows per thread (1 or 4): tile_rows = CTA_THREADS * rpt
  int64_t tile_rows() const { return (int64_t)CTA_THREADS * rpt; }
  IdEntry idtab[64];                     // ctl unit id -> kind and task parameter
  // host-side only (pipelined host-buffer SpMV, csxb_spmv_host): per tile the global column window its units read
  // (CSX-Sym: the rows themselves included, x[row] is read too)
  std::vector<int32_t> tile_cmin, tile_cmax;
  std::vector<uint32_t> tile_xoff;       // ntiles + 1
  std::vector<XDesc> xdesc;
  int64_t flat_elems = 0;                // non-zeros handled by the stream kernel
  std::vector<BlockTable> bt;            // block tables (see BlockTable)
};

struct DeviceLayout {
  std::vector<KindEntry> ktab;           // device-wide kind table referenced by XDesc.meta
  std::vector<PartLayout> parts;
  uint64_t total_values = 0, total_ctl = 0;
  bool symmetric = false, full_colind = false;
  // block units that live in the block tables: block-column units of width bc_align cut into sub-blocks of bc_rows rows
  // (0: none), block-row units of height br_align cut into sub-blocks of br_cols columns (0: none)
  int bc_align = 0, bc_rows = 0, br_align = 0, br_cols = 0;
  int br_img_cols = 0;   // CSX-Sym images of block-row units: aligned groups of this many columns per entry (1: per column)
  // CSX-Sym with only some partitions on this device: rows [halo_lo, halo_hi) of lower ranks that local units
  // update; parts.back() is their pseudo-partition (is_halo)
  int64_t halo_lo = 0, halo_hi = 0;
};

// Decodes every local partition's ctl stream and fills the tables.
std::string build_layout(const CsxMatrix &m, DeviceLayout &out);

// ---- transposed product y = alpha*A^T*x + beta*y (non-symmetric matrices) ------------------------------------------
// One row owner whose "rows" are the columns [row_start, row_start + nrows) of A that the local partitions read.  It holds
// only images y[col] += v * x[row] of the units and references the device-wide values of the forward layout (no values
// of its own).  A unit whose transpose is itself a table unit gets a forward descriptor with row and column swapped
// (diagonal (r, c) -> diagonal (c, r); horizontal run in row r -> vertical unit in column r), so a diagonal stencil runs
// the same gather instantiation both ways.  Vertical and anti-diagonal units get XD_TRANSPOSED descriptors, block units
// entries of block tables 1 / 3 (the CSX-Sym images), everything else single entries of table 4 (BT_IMAGE, other = row)
// — or, when such elements are a tiny minority of their partition, one-element diagonal descriptors.
// Columns with more than heavy_min entries in table 4 are taken out of it: their entries are cut into segments of
// seg_len entries, each summed by one warp (csx_t_segment_kernel), and the segment sums are added to y in segment order
// by the stream kernel's fix-up (part.sk_fix_rows / sk_fix_ptr / sk_fix_idx, scratch slot = segment).
constexpr int T_HEAVY_MIN = 128;         // chosen on R-MAT scale 22 on the B200 (DESIGN.md section 3b)
constexpr int T_SEG_LEN = 256;
struct TransLayout {
  PartLayout part;
  std::vector<KindEntry> ktab;           // the forward kind table, plus kinds only the transposed units use
  bool images = false;                   // some descriptor is an XD_TRANSPOSED image (the gather's CSX-Sym form runs)
  std::vector<BlockImage> hent;          // table-4 entries of the heavy columns, column by column, in source order
  std::vector<uint32_t> hseg;            // segments + 1: segment s sums hent[hseg[s] .. hseg[s+1])
  int64_t heavy_cols = 0;
  int heavy_min = T_HEAVY_MIN, seg_len = T_SEG_LEN;
};
// fwd: the forward layout of the same matrix (value offsets, kind table, block-table shapes).
std::string build_transpose_layout(const CsxMatrix &m, const DeviceLayout &fwd, TransLayout &out);
// (row, col) of A for every device-wide value index the transposed tables gather (-1 where none does)
void decode_transpose_coords(const TransLayout &t, int32_t *rows, int32_t *cols);
// pattern id (CsxUtil.hpp:58-74, CsxUtil.cpp:27-33) -> kernel kind
bool classify(long pid, KindEntry &ke);

// csx_tools.cpp ------------------------------------------------------------------------------------------------
// Per-row entry points into the ctl stream (built lazily for spx_mat_get/set_entry).
struct RowIndex {
  std::vector<uint64_t> ctl_off;   // offset of the row's first unit head (UINT64_MAX: the row has no unit)
  std::vector<uint64_t> val_off;   // index of its first value
  std::vector<int32_t> span;       // rows below this one that its units reach
  int32_t max_span = 0;
};
std::string build_row_index(const CsxPartition &cp, bool full_colind, RowIndex &ri);
// index (partition relative) of the value stored for (partition-relative row, zero-based column), or -1
int64_t find_entry(const CsxPartition &cp, bool full_colind, const RowIndex &ri, int64_t prow, int64_t col);
// tuned matrix <-> file (Boost-free container; the GPU tables are rebuilt from ctl at upload)
std::string save_matrix(const CsxMatrix &m, const char *path);
std::string load_matrix(const char *path, CsxMatrix &m);

}  // namespace spxb
