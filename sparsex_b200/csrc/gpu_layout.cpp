// Builds the GPU side tables (segment table, cross-row unit table) by walking
// the CSX ctl stream on the host.  The walk follows the unit grammar of
// CtlBuilder.cpp:62-81 / CtlUtil.hpp:46-133 and the cursor rules of the kernel
// templates (csx_spmv_tmpl.c:83-98; Element.hpp:657-666 for where a unit
// leaves the column cursor).
#include <algorithm>
#include <climits>
#include <cstring>
#include <map>

#include "gpu_layout.hpp"

namespace spxb {
namespace {

inline uint64_t get_varint(const uint8_t *ctl, uint64_t &p) {
  uint64_t v = 0;
  unsigned shift = 0;
  for (;;) {
    uint8_t b = ctl[p++];
    v |= (uint64_t)(b & 0x7f) << shift;
    if (!(b & 0x80)) break;
    shift += 7;
  }
  return v;
}

}  // namespace

// pattern id (CsxUtil.hpp:58-74, CsxUtil.cpp:27-33) -> kernel kind
bool classify(long pid, KindEntry &ke) {
  int type = (int)(pid / PATTERN_ID_OFFSET);
  uint32_t d = (uint32_t)(pid % PATTERN_ID_OFFSET);
  uint32_t kind, align = 0, delta = d;
  if (type == T_NONE) {
    if (d == 8) kind = K_DELTA8; else if (d == 16) kind = K_DELTA16; else if (d == 32) kind = K_DELTA32;
    else if (d == 64) kind = K_DELTA64; else return false;
    delta = d / 8;
  } else if (type == T_HORIZ) kind = K_HORIZ;
  else if (type == T_VERT) kind = K_VERT;
  else if (type == T_DIAG) kind = K_DIAG;
  else if (type == T_ADIAG) kind = K_ADIAG;
  else if (is_brow(type)) {
    align = blk_align(type);
    if (align == 1) { kind = K_HORIZ; delta = 1; align = 0; }   // 1 x c block == horizontal run
    else kind = K_BROW;                                          // delta = number of columns
  } else if (is_bcol(type)) {
    align = blk_align(type);
    if (align == 1) { kind = K_VERT; delta = 1; align = 0; }     // r x 1 block == vertical run
    else kind = K_BCOL;                                          // delta = number of rows
  } else return false;
  if (delta == 0) return false;
  ke.kind_align = kind | (align << 8);
  ke.delta = delta;
  return true;
}

namespace {

struct Pending { int64_t part; int64_t tile; XDesc d; };

// rows per thread of a partition's tiles (a later partition's value is needed while an earlier one is decoded)
// Rows per thread of the gather kernel: 4 for big partitions (more loads in flight per thread, fewer carry-in descriptors)
// unless the matrix has block tables — their walk is serial per row, so one row per thread and more resident warps is
// faster there (27-point stencil with bc2{2}: 220 -> 150 us at 128^3; 3x3 block-banded: 100 -> 93 us).
inline int tile_rpt(int64_t nrows, int forced, bool block_tables) {
  return forced ? forced : ((nrows >= (int64_t(1) << 20) && !block_tables) ? 4 : 1);
}

// ---- stream kernel chunking (see gpu_layout.hpp) -----------------------------------------------------------
struct SkUnit {
  uint64_t off, end;        // ctl offsets of the unit head and of the byte behind the unit
  uint32_t size, ntasks;
  int64_t row, reach;       // partition-relative start row, rows below it the unit touches
  int64_t cmin, cmax;       // columns it reads
  int64_t val;              // partition-relative index of its first value
  int64_t cursor_before;    // column cursor before the unit (0 when it starts a row)
  bool multi_bcol;          // block-column unit cut into several tasks
  bool round_end;           // last unit of its round (set by SkBuilder)
};

class SkBuilder {
 public:
  SkBuilder(PartLayout &L, int64_t nrows) : L_(L), nrows_(nrows) {}
  void add(const SkUnit &u0) {
    SkUnit u = u0;
    u.round_end = false;
    while (!open_.empty() && !fits(u)) {
      std::vector<SkUnit> rest = split(u);   // units behind the cut: their rounds change, so they are added again
      for (const SkUnit &w : rest) add(w);
    }
    if (open_.empty()) { wrow_ = (first_ && u.row + u.reach <= 64) ? 0 : u.row; rounds_ = 1; round_start_ = 0; }
    else if (round_closes(u)) { open_.back().round_end = true; rounds_++; round_start_ = open_.size(); }
    open_.push_back(u);
  }
  void finish() {
    if (!open_.empty()) close(open_.size(), 0, false);
    open_.clear();
    std::stable_sort(fixes_.begin(), fixes_.end(),
                     [](const std::pair<int32_t, uint32_t> &a, const std::pair<int32_t, uint32_t> &b) { return a.first < b.first; });
    for (size_t i = 0; i < fixes_.size(); i++) {
      if (i == 0 || fixes_[i].first != fixes_[i - 1].first) { L_.sk_fix_rows.push_back(fixes_[i].first); L_.sk_fix_ptr.push_back((uint32_t)i); }
      L_.sk_fix_idx.push_back(fixes_[i].second);
    }
    L_.sk_fix_ptr.push_back((uint32_t)fixes_.size());
  }
  void discard() {   // the partition's stream units were folded into the table
    open_.clear(); fixes_.clear();
    L_.sk_chunks.clear(); L_.sk_uoffs.clear(); L_.sk_gaps.clear(); L_.sk_scratch = 0;
    L_.sk_first_row.clear(); L_.sk_last_row.clear(); L_.sk_cmin.clear(); L_.sk_cmax.clear();
    L_.sk_fix_rows.clear(); L_.sk_fix_ptr.clear(); L_.sk_fix_idx.clear();
  }

 private:
  // The current round ends before `u`: it is full, or its last window of 32 tasks is well filled, `u` would open
  // another window and the units still missing to 32 would fill less than a quarter of that one (rounds of small units
  // then walk one full window instead of one full and one nearly empty one).
  bool round_closes(const SkUnit &u) const {
    const size_t units = open_.size() - round_start_;
    uint32_t tasks = 0, elems = 0;
    for (size_t i = round_start_; i < open_.size(); i++) { tasks += open_[i].ntasks; elems += open_[i].size; }
    if (units == (size_t)SK_ROUND_UNITS || tasks + u.ntasks > (uint32_t)SK_MAX_TASKS || elems + u.size > (uint32_t)SK_MAX_ELEMS) return true;
    if (units < 16 || tasks == 0) return false;
    const uint32_t fill = tasks - 32 * ((tasks - 1) / 32);   // tasks in the round's last window
    return fill >= 24 && fill + u.ntasks > 32 && (SK_ROUND_UNITS - units) * tasks < 8 * units;
  }
  bool fits(const SkUnit &u) const {
    if (rounds_ == SK_MAX_ROUNDS && round_closes(u)) return false;
    return u.end - open_.front().off <= (uint64_t)SK_MAX_BYTES && u.row + u.reach - wrow_ <= SK_WROWS - 1 &&
           u.row - wrow_ <= SK_WROWS - 2;
  }
  // The open chunk cannot take `next`: close it, preferably at the start of its last row when `next` continues
  // that row and the cut keeps the chunk at least three quarters full (a chunk that ends with its row needs no
  // fix-up).  Returns the units behind the cut.
  std::vector<SkUnit> split(const SkUnit &next) {
    size_t b = open_.size();
    if (next.row == open_.back().row) {
      for (size_t i = open_.size() - 1; i > 0; i--)
        if (open_[i].row != open_[i - 1].row) { if (4 * i >= 3 * open_.size()) b = i; break; }
    }
    close(b, b < open_.size() ? open_[b].row : next.row, true);
    std::vector<SkUnit> rest(open_.begin() + (long)b, open_.end());
    open_.clear();
    return rest;
  }
  void close(size_t b, int64_t next_row, bool has_next) {
    const int64_t ra = open_[0].row, rl = open_[b - 1].row;
    int64_t touch_hi = 0, cmin = INT64_MAX, cmax = -1;
    bool multib = false;
    for (size_t i = 0; i < b; i++) {
      touch_hi = std::max(touch_hi, open_[i].row + open_[i].reach);
      cmin = std::min(cmin, open_[i].cmin); cmax = std::max(cmax, open_[i].cmax);
      multib |= open_[i].multi_bcol;
    }
    int64_t own_lo = first_ ? 0 : prev_own_hi_;
    if (first_ && wrow_ != 0) { L_.sk_gaps.push_back(SkGap{0, ra}); own_lo = ra; }
    const int64_t own_hi = has_next ? (next_row > rl ? next_row : rl + 1) : nrows_;
    const bool head = !first_ && own_lo > ra;
    const int64_t f_lo = own_lo - wrow_, f_hi = std::min(own_hi, wrow_ + SK_WROWS) - wrow_;
    if (own_hi > wrow_ + SK_WROWS) L_.sk_gaps.push_back(SkGap{wrow_ + SK_WROWS, own_hi});
    const int64_t t_hi = touch_hi >= own_hi ? touch_hi - wrow_ + 1 : f_hi;
    const uint32_t slot = L_.sk_scratch;
    L_.sk_scratch += (uint32_t)(head ? 1 : 0) + (uint32_t)(t_hi - f_hi);
    if (head) fixes_.push_back(std::make_pair((int32_t)ra, slot));
    for (int64_t i = 0; i < t_hi - f_hi; i++) fixes_.push_back(std::make_pair((int32_t)(own_hi + i), slot + (head ? 1u : 0u) + (uint32_t)i));
    SkEntry e;
    const uint64_t off0 = open_[0].off;
    e.w[0] = (uint32_t)off0; e.w[1] = (uint32_t)open_[0].val; e.w[2] = (uint32_t)open_[0].cursor_before;
    e.w[3] = (uint32_t)(int32_t)wrow_; e.w[4] = (uint32_t)L_.sk_uoffs.size(); e.w[5] = slot;
    e.w[6] = (uint32_t)(b - 1) | ((uint32_t)(ra - wrow_) << 8) | ((uint32_t)f_lo << 16) | ((uint32_t)((off0 >> 32) & 0x3f) << 24) |
             ((uint32_t)head << 30) | ((uint32_t)multib << 31);
    e.w[7] = (uint32_t)f_hi | ((uint32_t)t_hi << 9);
    L_.sk_chunks.push_back(e);
    {   // layout statistics
      uint32_t rt = 0;
      for (size_t i = 0; i < b; i++) {
        rt += open_[i].ntasks;
        L_.sk_stat[2] += open_[i].ntasks; L_.sk_stat[3] += open_[i].size;
        if (open_[i].round_end || i + 1 == b) { L_.sk_stat[0]++; L_.sk_stat[1] += (rt + 31) / 32; rt = 0; }
      }
    }
    for (size_t i = 0; i < b; i++)   // bit 15: last unit of its round
      L_.sk_uoffs.push_back((uint16_t)((open_[i].off - off0) | ((open_[i].round_end || i + 1 == b) ? 0x8000u : 0u)));
    L_.sk_first_row.push_back((int32_t)wrow_);
    L_.sk_last_row.push_back((int32_t)std::max(touch_hi, wrow_ + f_hi - 1));
    L_.sk_cmin.push_back(cmin == INT64_MAX ? INT32_MAX : (int32_t)cmin);
    L_.sk_cmax.push_back((int32_t)cmax);
    prev_own_hi_ = own_hi;
    first_ = false;
  }
  PartLayout &L_;
  int64_t nrows_;
  std::vector<SkUnit> open_;
  std::vector<std::pair<int32_t, uint32_t>> fixes_;   // (row, scratch slot), in chunk order
  int64_t wrow_ = 0, prev_own_hi_ = 0;
  int rounds_ = 1;
  size_t round_start_ = 0;   // first unit of the open round
  bool first_ = true;
};

struct BtEnt { int64_t q; int tab; int64_t grp; BlockImage b; };
// Block-table shapes (G, nloop, sf, sl, image) of table t (gpu_layout.hpp: BlockTable); false when the table is unused.
bool block_table_shape(const DeviceLayout &L, int t, BlockTable &T) {
  if (t == 0) { T.G = L.bc_rows; T.nloop = L.bc_align; T.sf = L.bc_align; T.sl = 1; }
  else if (t == 1) { T.G = L.bc_align; T.nloop = L.bc_rows; T.sf = 1; T.sl = L.bc_align; T.image = 1; }
  else if (t == 2) { T.G = L.br_align; T.nloop = L.br_cols; T.sf = 1; T.sl = L.br_align; }
  else if (t == 3) { T.G = L.br_align ? std::max(L.br_img_cols, 1) : 0; T.nloop = L.br_align; T.sf = L.br_align; T.sl = 1; T.image = 1; }
  else { T.G = 1; T.nloop = 1; T.sf = 0; T.sl = 0; }
  if (T.G <= 0) { T.G = 1; return false; }
  return true;
}
// Block tables: counting sort of the entries by (owner, table, group); source order inside a group (deterministic sums).
void sort_block_tables(const DeviceLayout &shape, std::vector<PartLayout> &parts, const std::vector<BtEnt> &btents) {
  for (size_t q = 0; q < parts.size(); q++) {
    PartLayout &L = parts[q];
    if (!L.nrows) continue;
    L.bt.resize(BT_MAX);
    for (int t = 0; t < BT_MAX; t++) {
      BlockTable &T = L.bt[t];
      if (!block_table_shape(shape, t, T)) continue;
      T.j0 = L.row_start / T.G;
      T.ptr.assign((size_t)((L.row_start + L.nrows - 1) / T.G - T.j0 + 1) + 1, 0);
    }
  }
  for (const BtEnt &e : btents) {
    BlockTable &T = parts[e.q].bt[e.tab];
    T.ptr[(size_t)(e.grp - T.j0) + 1]++;
  }
  std::vector<std::vector<uint32_t>> at(parts.size() * BT_MAX);
  for (size_t q = 0; q < parts.size(); q++)
    for (int t = 0; t < BT_MAX && !parts[q].bt.empty(); t++) {
      BlockTable &T = parts[q].bt[t];
      for (size_t j = 1; j < T.ptr.size(); j++) T.ptr[j] += T.ptr[j - 1];
      if (!T.ptr.empty()) T.ent.resize(T.ptr.back());
      at[q * BT_MAX + t].assign(T.ptr.begin(), T.ptr.end());
    }
  for (const BtEnt &e : btents) {
    BlockTable &T = parts[e.q].bt[e.tab];
    T.ent[at[(size_t)e.q * BT_MAX + e.tab][(size_t)(e.grp - T.j0)]++] = e.b;
  }
  for (size_t q = 0; q < parts.size(); q++) {   // keep the tables that have entries
    std::vector<BlockTable> keep;
    for (BlockTable &T : parts[q].bt) if (!T.ent.empty()) keep.push_back(std::move(T));
    parts[q].bt.swap(keep);
  }
}
// Descriptors: stable counting sort by (owner, tile).
std::string distribute_descs(std::vector<PartLayout> &parts, const std::vector<Pending> &pend) {
  std::vector<std::vector<uint32_t>> cnt(parts.size());
  for (size_t q = 0; q < parts.size(); q++) cnt[q].assign((size_t)parts[q].ntiles + 1, 0);
  for (const Pending &e : pend) cnt[e.part][e.tile + 1]++;
  for (size_t q = 0; q < parts.size(); q++) {
    PartLayout &L = parts[q];
    for (int64_t t = 0; t < L.ntiles; t++) cnt[q][t + 1] += cnt[q][t];
    if (cnt[q][L.ntiles] >= 0x80000000u) return "cross-row unit table too large";
    L.xdesc.resize(cnt[q][L.ntiles]);
    for (int64_t t = 0; t <= L.ntiles; t++) L.tile_xoff[t] = cnt[q][t];
  }
  std::vector<std::vector<uint32_t>> fill(cnt);
  for (const Pending &e : pend) {
    parts[e.part].xdesc[fill[e.part][e.tile]++] = e.d;
    if (((e.d.meta >> 24) & 0xf) != K_DIAG || !(e.d.meta & XD_DELTA1) || (e.d.meta & XD_TRANSPOSED))
      parts[e.part].xd_diag1_only = false;
  }
  return "";
}

// ---- images y[col] += v * x[row] of block units in block tables 1 and 3 (CSX-Sym and the transposed product) ---------
// A block unit of the tables (its shape matches bc_align / br_align) whose image can be listed there: sub-blocks of
// bc_rows rows starting on the sub-block grid and columns aligned to the group width.
bool block_image_fits(const DeviceLayout &L, uint32_t kind, int64_t delta, int64_t grow, int64_t start_col) {
  if (kind == K_BCOL) return delta % L.bc_rows == 0 && grow % L.bc_rows == 0 && start_col % L.bc_align == 0;
  return delta % L.br_cols == 0 && grow % L.br_align == 0 && (L.br_img_cols <= 1 || start_col % L.br_img_cols == 0);
}
// Table 1 takes a block-column unit (one entry per sub-block of bc_rows rows), table 3 a block-row unit (one entry per
// aligned group of br_img_cols columns), each once per row owner of its columns.  owner_end(g, hi): end of the run of
// columns [g, hi) that the owner of column g holds, -1 when g has none; put(table, group, entry, first column).
template <class OwnerEnd, class Put>
bool block_images(const DeviceLayout &L, uint32_t kind, uint32_t voff, int64_t grow, int64_t start_col, int64_t delta,
                  OwnerEnd owner_end, Put put) {
  if (kind == K_BCOL) {
    const int64_t A = L.bc_align, R0 = L.bc_rows;
    for (int64_t k = 0; k * R0 < delta; k++)
      for (int64_t g = start_col; g < start_col + A;) {
        const int64_t e = owner_end(g, start_col + A);
        if (e < 0) return false;
        put(1, g / A, BlockImage{voff + (uint32_t)(k * R0 * A), (uint32_t)(grow + k * R0) | BT_IMAGE}, g);
        g = e;
      }
    return true;
  }
  const int64_t A = L.br_align, G = std::max(L.br_img_cols, 1);
  for (int64_t j = 0; j < delta; j += G)
    for (int64_t g = start_col + j; g < start_col + j + G;) {   // a group can be cut by an owner boundary
      const int64_t e = owner_end(g, start_col + j + G);
      if (e < 0) return false;
      put(3, g / G, BlockImage{voff + (uint32_t)(j * A), (uint32_t)grow | BT_IMAGE}, g);
      g = e;
    }
  return true;
}

}  // namespace

std::string build_layout(const CsxMatrix &m, DeviceLayout &out) {
  out = DeviceLayout();
  out.symmetric = m.symmetric;
  out.full_colind = m.full_colind;
  const size_t np = m.parts.size();
  // CSX-Sym with only some partitions on this device: the transposed updates of the local lower triangle reach rows
  // [col_min, first local row) of lower ranks.  Those rows get a pseudo-partition of their own, so that their updates
  // are gathered like every other row's; the caller reduces them across devices (the cross-device form of the
  // reference's local vectors + map reduction, CsxSpmv.cpp:37-50).
  if (m.symmetric && np && (int)np != m.nparts_total) {
    const int64_t first_row = m.parts.front().row_start;
    int64_t lo = first_row;
    for (auto &p : m.parts) if (p.col_max >= p.col_min) lo = std::min(lo, p.col_min);
    out.halo_lo = lo; out.halo_hi = first_row;
  }
  const bool has_halo = out.halo_hi > out.halo_lo;
  const size_t nq = np + (has_halo ? 1 : 0);   // row owners on this device
  out.parts.resize(nq);
  auto q_start = [&](size_t q) { return q < np ? m.parts[q].row_start : out.halo_lo; };
  auto q_rows = [&](size_t q) { return q < np ? m.parts[q].nrows : out.halo_hi - out.halo_lo; };
  auto q_tile = [&](size_t q) { return (int64_t)CTA_THREADS * tile_rpt(q_rows(q), m.rows_per_thread, out.bc_align || out.br_align); };
  // global row -> owner on this device; partitions are contiguous and ordered
  auto owner_of = [&](int64_t grow) -> int64_t {
    for (size_t q = 0; q < nq; q++)
      if (grow >= q_start(q) && grow < q_start(q) + q_rows(q)) return (int64_t)q;
    return -1;
  };
  std::map<std::pair<uint32_t, uint32_t>, uint32_t> kindex;
  auto kind_index = [&](const KindEntry &ke) -> int64_t {
    auto key = std::make_pair(ke.kind_align, ke.delta);
    auto it = kindex.find(key);
    if (it == kindex.end()) {
      if (out.ktab.size() >= 65535) return -1;
      it = kindex.insert(std::make_pair(key, (uint32_t)out.ktab.size())).first;
      out.ktab.push_back(ke);
    }
    return it->second;
  };
  std::vector<Pending> pend;
  // descriptor `d` under every tile of the owners of global rows [lo, hi]
  auto list_rows = [&](const XDesc &d, int64_t lo, int64_t hi, std::vector<Pending> &to) -> bool {
    int64_t g = lo;
    while (g <= hi) {
      const int64_t q = owner_of(g);
      if (q < 0) return false;
      const int64_t rel = g - q_start((size_t)q), qt = q_tile((size_t)q);
      to.push_back(Pending{q, rel / qt, d});
      g = std::min(q_start((size_t)q) + (rel / qt + 1) * qt, q_start((size_t)q) + q_rows((size_t)q));   // next tile or next owner
    }
    return true;
  };
  // ---- which block units go to the block tables (gpu_layout.hpp: BlockTable) -------------------------------------
  // One pass over the unit heads: per block kind and width / height, the sub-block size (2..16 lines) that covers the
  // most elements — a unit is covered when the sub-block divides its free dimension and (block-column units) its start
  // row.  Units of the chosen kind that are not covered (a block cut by a partition boundary) go to the table of single
  // elements.
  {
    constexpr int CAND = 17;
    std::map<uint32_t, std::vector<int64_t>> bc_cov, br_cov, bri_cov;   // align -> elements covered by sub-block size r
    auto cov = [&](std::map<uint32_t, std::vector<int64_t>> &mp, uint32_t a) -> std::vector<int64_t> & {
      std::vector<int64_t> &v = mp[a];
      if (v.empty()) v.assign(CAND, 0);
      return v;
    };
    for (size_t pi = 0; pi < np; pi++) {
      const CsxPartition &cp = m.parts[pi];
      KindEntry tab[64];
      size_t nid = 0;
      bool any = false;
      for (; nid < cp.id_map.size() && cp.id_map[nid] != -1 && nid < 64; nid++) {
        if (!classify(cp.id_map[nid], tab[nid])) return "unsupported pattern id " + std::to_string(cp.id_map[nid]);
        any |= (tab[nid].kind_align & 0xff) >= K_BROW;
      }
      if (!any) continue;
      const uint8_t *ctl = cp.ctl.data();
      uint64_t p = 0, end = cp.ctl.size();
      int64_t row = 0, col = 0;
      while (p + 2 <= end) {
        const uint8_t flags = ctl[p++], size = ctl[p++];
        if (flags & 0x80) { row += (flags & 0x40) ? (int64_t)get_varint(ctl, p) : 1; col = 0; }
        if (m.full_colind) { uint32_t c; memcpy(&c, ctl + p, 4); p += 4; col = c; }
        else col = (int64_t)((uint64_t)col + get_varint(ctl, p));
        const uint32_t id = flags & 0x3f;
        if (id >= nid || size == 0) return "ctl stream uses an unmapped unit id";
        const uint32_t kind = tab[id].kind_align & 0xff, align = (tab[id].kind_align >> 8) & 0xff, delta = tab[id].delta;
        const int64_t grow = cp.row_start + row;
        if (kind <= K_DELTA64) {
          for (int k = 1; k < size; k++) { uint64_t d = 0; memcpy(&d, ctl + p, delta); p += delta; col += (int64_t)d; }
        } else if (kind == K_HORIZ) col += (int64_t)(size - 1) * delta;
        else if (kind == K_BCOL) {
          std::vector<int64_t> &v = cov(bc_cov, align);
          if (!m.symmetric || col % align == 0)
            for (int r = 2; r < CAND; r++) if (delta % r == 0 && grow % r == 0) v[r] += size;
        } else if (kind == K_BROW) {
          if (grow % align == 0) {
            std::vector<int64_t> &v = cov(br_cov, align), &vi = cov(bri_cov, align);
            for (int r = 1; r < CAND; r++) {
              if (delta % r == 0) v[r] += size;
              if (delta % r == 0 && col % r == 0) vi[r] += size;
            }
          }
        }
      }
    }
    auto pick = [&](std::map<uint32_t, std::vector<int64_t>> &mp, int rmin, int &A, int &R0) {
      int64_t best = 0;
      for (auto &kv : mp)
        for (int r = CAND - 1; r >= rmin; r--)   // the largest sub-block among (nearly) equal coverages
          if ((int64_t)r * kv.first >= 4 && kv.second[r] > best + best / 64) { best = kv.second[r]; A = (int)kv.first; R0 = r; }
    };
    pick(bc_cov, 2, out.bc_align, out.bc_rows);
    pick(br_cov, 1, out.br_align, out.br_cols);
    if (out.br_align) {   // CSX-Sym images of the block-row units: aligned groups of columns that divide the sub-block
      const std::vector<int64_t> &vi = bri_cov[(uint32_t)out.br_align];
      out.br_img_cols = 1;
      for (int r = CAND - 1; r >= 2; r--)
        if (out.br_cols % r == 0 && vi[r] >= br_cov[(uint32_t)out.br_align][out.br_cols] - br_cov[(uint32_t)out.br_align][out.br_cols] / 64) { out.br_img_cols = r; break; }
    }
    if (getenv("CSXB_NO_BLOCK_TABLES")) out.bc_align = out.bc_rows = out.br_align = out.br_cols = out.br_img_cols = 0;   // tuning aid
  }
  // entries of the block tables (table numbers: gpu_layout.hpp)
  std::vector<BtEnt> btents;
  // CSX-Sym: images of the block units that stay with the stream kernel get descriptors
  struct BlockTmp { XDesc d; uint32_t kind, align, other; int64_t cmin, cmax; };
  std::vector<BlockTmp> blocks;

  uint64_t vbase = 0, cbase = 0;
  for (size_t pi = 0; pi < nq; pi++) {
    PartLayout &L = out.parts[pi];
    L.nrows = q_rows(pi); L.row_start = q_start(pi);
    L.val_base = vbase; L.ctl_base = cbase;
    L.rpt = tile_rpt(L.nrows, m.rows_per_thread, out.bc_align || out.br_align);
    const int64_t TILE_ROWS = L.tile_rows();
    L.ntiles = (L.nrows + TILE_ROWS - 1) / TILE_ROWS;
    L.tile_xoff.assign((size_t)L.ntiles + 1, 0);
    L.tile_cmin.assign((size_t)L.ntiles, INT32_MAX);
    L.tile_cmax.assign((size_t)L.ntiles, -1);
    memset(L.idtab, 0, sizeof(L.idtab));
    if (pi >= np) { L.is_halo = true; continue; }
    const CsxPartition &cp = m.parts[pi];
    L.nnz = cp.nnz; L.ctl_size = (int64_t)cp.ctl.size();
    vbase += (uint64_t)cp.nnz;
    cbase += ((uint64_t)cp.ctl.size() + CTL_PAD + 15) & ~uint64_t(15);
    if (m.symmetric)   // the diagonal term reads x at the row itself
      for (int64_t t = 0; t < L.ntiles; t++) {
        L.tile_cmin[t] = (int32_t)(cp.row_start + t * TILE_ROWS);
        L.tile_cmax[t] = (int32_t)(cp.row_start + std::min<int64_t>(cp.nrows, (t + 1) * TILE_ROWS) - 1);
      }
    uint32_t id2k[64];
    KindEntry truetab[64];     // what the units are; L.idtab is what the stream kernel treats them as
    bool in_table[64];         // block units that live in the block tables
    size_t nid = 0;
    for (; nid < cp.id_map.size() && cp.id_map[nid] != -1; nid++) {
      if (nid >= 64) return "too many unit kinds";
      KindEntry ke;
      if (!classify(cp.id_map[nid], ke)) return "unsupported pattern id " + std::to_string(cp.id_map[nid]);
      truetab[nid] = ke;
      const uint32_t kd = ke.kind_align & 0xff, al = (ke.kind_align >> 8) & 0xff;
      in_table[nid] = (kd == K_BCOL && (int)al == out.bc_align) || (kd == K_BROW && (int)al == out.br_align);
      // to the stream kernel a unit of the block tables is a table unit: it only moves the column cursor
      L.idtab[nid] = in_table[nid] ? IdEntry{K_VERT, 1, 1, 65536} : IdEntry{ke.kind_align, ke.delta, 1, 65536};
      const int64_t ki = kind_index(ke);
      if (ki < 0) return "too many distinct unit kinds on one device";
      id2k[nid] = (uint32_t)ki;
    }
    // task shapes of the stream kernel (sk_unit_tasks)
    for (size_t id = 0; id < nid; id++) {
      IdEntry &ie = L.idtab[id];
      const uint32_t kind = ie.kind_align & 0xff, align = (ie.kind_align >> 8) & 0xff;
      uint32_t sl = 1;
      if (kind <= K_HORIZ) sl = SK_RL_E;
      else if (kind == K_BROW) { sl = std::min<uint32_t>(SK_BLK_LINES, std::max<uint32_t>(1, SK_BLK_E / align)); L.sk_rows = std::max<int>(L.sk_rows, (int)align); }
      else if (kind == K_BCOL) {   // rows of the unit spread evenly over its tasks
        const uint32_t tmax = std::min<uint32_t>(SK_BLK_LINES, std::max<uint32_t>(1, SK_BLK_E / align));
        const uint32_t nt = (ie.delta + tmax - 1) / tmax;
        sl = (ie.delta + nt - 1) / nt;
        L.sk_rows = std::max<int>(L.sk_rows, (int)sl);
      }
      ie.sl = sl;
      ie.recip = (65536 + sl - 1) / sl;
      if (kind <= K_HORIZ || kind >= K_BROW) L.sk_kmask |= 1u << kind;
    }
    {   // block tasks of one compile-time shape (the kernel is instantiated for the common ones)
      int bc = -1, brc = -1;
      for (size_t id = 0; id < nid; id++) {
        const IdEntry &ie = L.idtab[id];
        const uint32_t kind = ie.kind_align & 0xff, align = (ie.kind_align >> 8) & 0xff;
        if (kind == K_BCOL) {
          const bool full = (int)ie.sl == L.sk_rows && ie.delta % ie.sl == 0;
          bc = (full && (bc == -1 || bc == (int)align)) ? (int)align : 0;
        } else if (kind == K_BROW) {
          const bool full = (int)align == L.sk_rows && ie.delta % ie.sl == 0;
          brc = (full && (brc == -1 || brc == (int)ie.sl)) ? (int)ie.sl : 0;
        }
      }
      L.sk_bc = std::max(bc, 0); L.sk_brc = std::max(brc, 0);
    }

    const uint8_t *ctl = cp.ctl.data();
    uint64_t p = 0, end = cp.ctl.size();
    int64_t row = 0, col = 0, v = 0;
    bool first = true;
    SkBuilder sk(L, cp.nrows);
    // A partition whose stream-kernel share is tiny (stencil matrices: a few boundary elements next to
    // millions of diagonal units) gets those elements as one-element table units instead; that saves the
    // second kernel launch.  Coordinates are collected while the share stays under the cap.
    // A larger minority (up to 40 % of the non-zeros; block stencils, the diagonal-block leftovers of a block-banded
    // matrix) goes to the table of single elements instead (gpu_layout.hpp: BlockTable 4): 8 bytes per element, again
    // no stream kernel.
    struct Single { int32_t row, col; uint32_t v; };
    std::vector<Single> singles;
    const size_t single_cap = (size_t)(cp.nnz / 256), element_cap = getenv("CSXB_NO_BLOCK_TABLES") ? single_cap : (size_t)(cp.nnz / 5 * 2);
    bool singles_ok = true;
    // CSX-Sym: images of this partition's stream units (dropped again if the units are folded into the table)
    std::vector<Pending> simg;
    const size_t blocks_before = blocks.size();
    KindEntry ke_single{K_DIAG, 1};
    const int64_t k_single = kind_index(ke_single);
    if (k_single < 0) return "too many distinct unit kinds on one device";
    int64_t ecols[256];
    while (p < end) {
      if (p + 2 > end) return "ctl stream truncated";
      uint64_t unit_off = p;
      uint8_t flags = ctl[p++], size = ctl[p++];
      bool nr = (flags & 0x80) != 0;
      if (nr) {
        row += (flags & 0x40) ? (int64_t)get_varint(ctl, p) : 1;
        col = 0;
      }
      const int64_t cursor_before = (nr || first) ? 0 : col;
      if (m.full_colind) { uint32_t c; memcpy(&c, ctl + p, 4); p += 4; col = c; }
      else col = (int64_t)((uint64_t)col + get_varint(ctl, p));   // modulo 2^64 (SURVEY App. A: negative ucol)
      if (row >= cp.nrows) return "ctl stream leaves the partition (row " + std::to_string(row) + ")";
      first = false;
      uint32_t id = flags & 0x3f;
      if (id >= nid) return "ctl stream uses an unmapped unit id";
      uint32_t kind = truetab[id].kind_align & 0xff, align = (truetab[id].kind_align >> 8) & 0xff;
      uint32_t delta = truetab[id].delta;
      if (size == 0) return "ctl unit of size 0";
      const int64_t start_col = col;
      uint64_t body = kind <= K_DELTA64 ? (uint64_t)(size - 1) * delta : 0;
      if (p + body > end) return "ctl stream truncated";
      // geometry: rows spanned below the first one, column range
      int64_t span = 0, cmin = start_col, cmax = start_col;
      if (kind <= K_DELTA64) {
        ecols[0] = col;
        for (int k = 1; k < size; k++) {
          uint64_t d = 0;
          memcpy(&d, ctl + p, delta);   // little-endian fixed-width deltas
          p += delta;
          col += (int64_t)d;
          ecols[k] = col;
        }
        cmax = col;
      } else if (kind == K_HORIZ) { col += (int64_t)(size - 1) * delta; cmax = col; }
      else if (kind == K_VERT) span = (int64_t)(size - 1) * delta;
      else if (kind == K_DIAG) { span = (int64_t)(size - 1) * delta; cmax = start_col + span; }
      else if (kind == K_ADIAG) { span = (int64_t)(size - 1) * delta; cmin = start_col - span; }
      else if (kind == K_BROW) {
        if (size % align || size / align != delta) return "inconsistent block-row unit";
        span = align - 1; cmax = start_col + delta - 1;
      } else {
        if (size % align || size / align != delta) return "inconsistent block-col unit";
        span = delta - 1; cmax = start_col + align - 1;
      }
      if (row + span >= cp.nrows) return "cross-row unit leaves its partition";
      if (cmin < 0 || cmax >= cp.ncols) return "unit leaves the column range";
      {
        int64_t wlo = cmin, whi = cmax;
        if (m.symmetric) { wlo = std::min(wlo, cp.row_start + row); whi = std::max(whi, cp.row_start + row + span); }
        for (int64_t t = row / TILE_ROWS; t <= (row + span) / TILE_ROWS; t++) {
          L.tile_cmin[t] = std::min<int32_t>(L.tile_cmin[t], (int32_t)wlo);
          L.tile_cmax[t] = std::max<int32_t>(L.tile_cmax[t], (int32_t)whi);
        }
      }

      // Vertical / diagonal / anti-diagonal units are table units; everything else belongs to the stream kernel,
      // which also parses the heads of the table units (they move the column cursor).
      const bool to_table = goes_to_xdt(kind) || in_table[id];
      {
        const IdEntry &ie = L.idtab[id];
        SkUnit su;
        su.off = unit_off; su.end = p; su.size = size;
        su.ntasks = sk_unit_tasks(ie.kind_align & 0xff, size, ie.delta, ie.sl, ie.recip);
        su.row = row; su.reach = to_table ? 0 : span;   // the stream kernel adds nothing for a table unit
        su.cmin = cmin; su.cmax = cmax; su.val = v; su.cursor_before = cursor_before;
        su.multi_bcol = kind == K_BCOL && su.ntasks > 1;
        su.round_end = false;
        if (L.sk_uoffs.size() >= 0xfffffff0ull) return "unit-offset table too large";
        sk.add(su);
      }
      XDesc d;
      d.voff = (uint32_t)(L.val_base + (uint64_t)v);
      d.row = (int32_t)(cp.row_start + row);
      d.col = (int32_t)start_col;
      d.meta = id2k[id] | ((uint32_t)size << 16) | (kind << 24);
      if (delta == 1) d.meta |= XD_DELTA1;
      if (!to_table) {
        L.has_flat = true;
        L.flat_elems += size;
        if (singles_ok && singles.size() + size <= element_cap) {
          // element coordinates of this unit (same geometry as the stream kernel)
          for (int k = 0; k < size; k++) {
            int64_t er = row, ec = start_col;
            if (kind <= K_DELTA64) ec = ecols[k];
            else if (kind == K_HORIZ) ec = start_col + (int64_t)k * delta;
            else if (kind == K_BROW) { er = row + k % (int)align; ec = start_col + k / (int)align; }
            else { er = row + k / (int)align; ec = start_col + k % (int)align; }
            singles.push_back(Single{(int32_t)er, (int32_t)ec, (uint32_t)(v + k)});
          }
        } else {
          singles_ok = false;
        }
        if (m.symmetric) {   // transposed image of a stream unit: y[col] += v * x[row], gathered by the owners of its columns
          XDesc td = d;
          td.meta |= XD_TRANSPOSED;
          if (kind <= K_DELTA64) {   // irregular columns: one single-element image per element
            for (int k = 0; k < size; k++) {
              XDesc e;
              e.voff = d.voff + (uint32_t)k; e.row = d.row; e.col = (int32_t)ecols[k];
              e.meta = (uint32_t)k_single | (1u << 16) | ((uint32_t)K_DIAG << 24) | XD_DELTA1 | XD_TRANSPOSED;
              if (!list_rows(e, ecols[k], ecols[k], simg)) return "symmetric update targets a row that is not on this device";
            }
          } else if (kind == K_HORIZ) {
            if (!list_rows(td, cmin, cmax, simg)) return "symmetric update targets a row that is not on this device";
          } else {
            blocks.push_back(BlockTmp{td, kind, align, delta, cmin, cmax});
          }
        }
      } else if (in_table[id]) {
        // block tables: one entry per sub-block under the group of rows it adds to (own rows here, images at the owners
        // of its columns)
        const int64_t grow = cp.row_start + row;
        const bool fits = kind == K_BCOL ? (m.symmetric ? block_image_fits(out, kind, delta, grow, start_col)
                                                        : ((int64_t)delta % out.bc_rows == 0 && grow % out.bc_rows == 0))
                                         : ((int64_t)delta % out.br_cols == 0 && grow % out.br_align == 0);
        if (!fits) {   // (a block cut by a partition boundary ...): its elements one by one
          for (int k = 0; k < size; k++) {
            const int64_t er = grow + (kind == K_BROW ? k % (int)align : k / (int)align);
            const int64_t ec = start_col + (kind == K_BROW ? k / (int)align : k % (int)align);
            btents.push_back(BtEnt{(int64_t)pi, 4, er, BlockImage{d.voff + (uint32_t)k, (uint32_t)ec}});
            if (m.symmetric) {
              const int64_t q = owner_of(ec);
              if (q < 0) return "symmetric update targets a row that is not on this device";
              btents.push_back(BtEnt{q, 4, ec, BlockImage{d.voff + (uint32_t)k, (uint32_t)er | BT_IMAGE}});
            }
          }
        } else {
          if (kind == K_BCOL) {
            const int64_t A = out.bc_align, R0 = out.bc_rows;
            for (int64_t k = 0; k * R0 < (int64_t)delta; k++)
              btents.push_back(BtEnt{(int64_t)pi, 0, (grow + k * R0) / R0, BlockImage{d.voff + (uint32_t)(k * R0 * A), (uint32_t)start_col}});
          } else {
            const int64_t A = out.br_align, C0 = out.br_cols;
            for (int64_t k = 0; k * C0 < (int64_t)delta; k++)
              btents.push_back(BtEnt{(int64_t)pi, 2, grow / A, BlockImage{d.voff + (uint32_t)(k * C0 * A), (uint32_t)(start_col + k * C0)}});
          }
          if (m.symmetric && kind == K_BROW && !block_image_fits(out, kind, delta, grow, start_col)) {   // columns off the grid: a descriptor
            XDesc td = d;
            td.meta |= XD_TRANSPOSED;
            if (!list_rows(td, cmin, cmax, pend)) return "symmetric update targets a row that is not on this device";
          } else if (m.symmetric) {   // columns owned by one partition, or cut by a partition boundary
            auto owner_end = [&](int64_t g, int64_t hi) -> int64_t {
              const int64_t q = owner_of(g);
              return q < 0 ? -1 : std::min(hi, q_start((size_t)q) + q_rows((size_t)q));
            };
            auto put = [&](int tab, int64_t grp, BlockImage b, int64_t g) { btents.push_back(BtEnt{owner_of(g), tab, grp, b}); };
            if (!block_images(out, kind, d.voff, grow, start_col, delta, owner_end, put))
              return "symmetric update targets a row that is not on this device";
          }
        }
      } else {
        for (int64_t t = row / TILE_ROWS; t <= (row + span) / TILE_ROWS; t++) pend.push_back(Pending{(int64_t)pi, t, d});
        if (m.symmetric) {  // transposed image, listed under the tiles of its columns
          XDesc td = d;
          td.meta |= XD_TRANSPOSED;
          if (!list_rows(td, cmin, cmax, pend)) return "symmetric update targets a row that is not on this device";
        }
      }
      v += size;
    }
    if (v != cp.nnz) return "ctl stream covers " + std::to_string(v) + " values, expected " + std::to_string(cp.nnz);
    if (L.has_flat) sk.finish(); else sk.discard();
    if (L.has_flat && singles_ok && (int64_t)singles.size() == L.flat_elems && singles.size() > single_cap) {
      // the stream units are a minority: their elements go to the table of single elements
      for (const Single &sg : singles) {
        const uint32_t vo = (uint32_t)(L.val_base + (uint64_t)sg.v);
        const int64_t grow = cp.row_start + sg.row;
        btents.push_back(BtEnt{(int64_t)pi, 4, grow, BlockImage{vo, (uint32_t)sg.col}});
        if (m.symmetric) {
          const int64_t q = owner_of(sg.col);
          if (q < 0) return "symmetric update targets a row that is not on this device";
          btents.push_back(BtEnt{q, 4, sg.col, BlockImage{vo, (uint32_t)grow | BT_IMAGE}});
        }
      }
      sk.discard();
      simg.clear();
      blocks.resize(blocks_before);
      L.has_flat = false;
      L.flat_elems = 0;
    } else if (L.has_flat && singles_ok && (int64_t)singles.size() == L.flat_elems) {
      // fold the few stream-kernel elements into the table as diagonal units of one element
      for (const Single &sg : singles) {
        XDesc d;
        d.voff = (uint32_t)(L.val_base + (uint64_t)sg.v);
        d.row = (int32_t)(cp.row_start + sg.row);
        d.col = (int32_t)sg.col;
        d.meta = (uint32_t)k_single | (1u << 16) | ((uint32_t)K_DIAG << 24) | XD_DELTA1;
        pend.push_back(Pending{(int64_t)pi, sg.row / TILE_ROWS, d});
        if (m.symmetric) {
          XDesc td = d;
          td.meta |= XD_TRANSPOSED;
          if (!list_rows(td, sg.col, sg.col, pend)) return "symmetric update targets a row that is not on this device";
        }
      }
      sk.discard();
      simg.clear();
      blocks.resize(blocks_before);
      L.has_flat = false;
      L.flat_elems = 0;
    }
    pend.insert(pend.end(), simg.begin(), simg.end());
  }
  out.total_values = vbase;
  out.total_ctl = cbase;
  if (vbase >= (uint64_t(1) << 32)) return "more than 2^32 values on one device";

  // CSX-Sym: images of the block units that stayed with the stream kernel
  for (const BlockTmp &b : blocks)
    if (!list_rows(b.d, b.cmin, b.cmax, pend)) return "symmetric update targets a row that is not on this device";
  // block tables, then the descriptors
  if (!btents.empty()) sort_block_tables(out, out.parts, btents);
  return distribute_descs(out.parts, pend);
}

// ---- transposed product (gpu_layout.hpp: TransLayout) -------------------------------------------------------------
std::string build_transpose_layout(const CsxMatrix &m, const DeviceLayout &fwd, TransLayout &out) {
  out = TransLayout();
  if (m.symmetric) return "CSX-Sym needs no transposed tables (A^T = A)";
  const size_t np = m.parts.size();
  if (fwd.parts.size() != np) return "the forward layout does not belong to this matrix";
  if (const char *v = getenv("CSXB_T_HEAVY")) out.heavy_min = std::max(1, atoi(v));   // tuning aids (DESIGN.md section 3b)
  if (const char *v = getenv("CSXB_T_SEG")) out.seg_len = std::max(32, atoi(v));
  // columns the local partitions read (all of them when every partition is local)
  int64_t clo = INT64_MAX, chi = -1;
  for (const CsxPartition &p : m.parts) if (p.col_max >= p.col_min) { clo = std::min(clo, p.col_min); chi = std::max(chi, p.col_max); }
  if ((int)np == m.nparts_total) { clo = 0; chi = m.ncols - 1; }
  if (chi < clo) { clo = 0; chi = -1; }
  out.ktab = fwd.ktab;
  std::map<std::pair<uint32_t, uint32_t>, uint32_t> kindex;
  for (size_t i = 0; i < out.ktab.size(); i++) kindex.insert(std::make_pair(std::make_pair(out.ktab[i].kind_align, out.ktab[i].delta), (uint32_t)i));
  auto kind_index = [&](uint32_t kind_align, uint32_t delta) -> int64_t {
    auto it = kindex.find(std::make_pair(kind_align, delta));
    if (it == kindex.end()) {
      if (out.ktab.size() >= 65535) return -1;
      it = kindex.insert(std::make_pair(std::make_pair(kind_align, delta), (uint32_t)out.ktab.size())).first;
      out.ktab.push_back(KindEntry{kind_align, delta});
    }
    return it->second;
  };
  const int64_t k_single = kind_index(K_DIAG, 1);
  if (k_single < 0) return "too many distinct unit kinds on one device";
  struct Emit { XDesc d; int64_t lo, hi; };   // a descriptor for the columns [lo, hi]
  std::vector<Emit> em;
  std::vector<BtEnt> btents;
  struct Single { int64_t row, col; uint32_t voff; };
  std::vector<Single> singles;
  for (size_t pi = 0; pi < np; pi++) {
    const CsxPartition &cp = m.parts[pi];
    KindEntry truetab[64];
    uint32_t id2k[64];
    size_t nid = 0;
    for (; nid < cp.id_map.size() && cp.id_map[nid] != -1; nid++) {
      if (nid >= 64) return "too many unit kinds";
      if (!classify(cp.id_map[nid], truetab[nid])) return "unsupported pattern id " + std::to_string(cp.id_map[nid]);
      const int64_t ki = kind_index(truetab[nid].kind_align, truetab[nid].delta);
      if (ki < 0) return "too many distinct unit kinds on one device";
      id2k[nid] = (uint32_t)ki;
    }
    const uint64_t vbase = fwd.parts[pi].val_base;
    const uint8_t *ctl = cp.ctl.data();
    uint64_t p = 0;
    const uint64_t end = cp.ctl.size();
    int64_t row = 0, col = 0, v = 0;
    singles.clear();
    while (p < end) {   // the unit grammar of build_layout
      if (p + 2 > end) return "ctl stream truncated";
      const uint8_t flags = ctl[p++], size = ctl[p++];
      if (flags & 0x80) { row += (flags & 0x40) ? (int64_t)get_varint(ctl, p) : 1; col = 0; }
      if (m.full_colind) { uint32_t c; memcpy(&c, ctl + p, 4); p += 4; col = c; }
      else col = (int64_t)((uint64_t)col + get_varint(ctl, p));
      if (row >= cp.nrows) return "ctl stream leaves the partition (row " + std::to_string(row) + ")";
      const uint32_t id = flags & 0x3f;
      if (id >= nid) return "ctl stream uses an unmapped unit id";
      if (size == 0) return "ctl unit of size 0";
      const uint32_t kind = truetab[id].kind_align & 0xff, align = (truetab[id].kind_align >> 8) & 0xff, delta = truetab[id].delta;
      const int64_t start_col = col, grow = cp.row_start + row, span = (int64_t)(size - 1) * delta;
      const uint32_t voff = (uint32_t)(vbase + (uint64_t)v);
      XDesc d;
      d.voff = voff;
      d.meta = id2k[id] | ((uint32_t)size << 16) | (kind << 24) | (delta == 1 ? XD_DELTA1 : 0u);
      if (kind <= K_DELTA64) {
        if (p + (uint64_t)(size - 1) * delta > end) return "ctl stream truncated";
        singles.push_back(Single{grow, col, voff});
        for (int k = 1; k < size; k++) {
          uint64_t dd = 0;
          memcpy(&dd, ctl + p, delta);
          p += delta;
          col += (int64_t)dd;
          singles.push_back(Single{grow, col, voff + (uint32_t)k});
        }
      } else if (kind == K_HORIZ) {   // row r, columns c + k*delta -> vertical unit of A^T in column r
        const int64_t ki = kind_index(K_VERT, delta);
        if (ki < 0) return "too many distinct unit kinds on one device";
        d.row = (int32_t)start_col; d.col = (int32_t)grow;
        d.meta = (uint32_t)ki | ((uint32_t)size << 16) | ((uint32_t)K_VERT << 24) | (delta == 1 ? XD_DELTA1 : 0u);
        em.push_back(Emit{d, start_col, start_col + span});
        col += span;
      } else if (kind == K_DIAG) {    // diagonal (r, c) -> diagonal (c, r), same value order
        d.row = (int32_t)start_col; d.col = (int32_t)grow;
        em.push_back(Emit{d, start_col, start_col + span});
      } else if (kind == K_VERT || kind == K_ADIAG) {   // CSX-Sym image descriptors
        d.row = (int32_t)grow; d.col = (int32_t)start_col;
        d.meta |= XD_TRANSPOSED;
        em.push_back(kind == K_VERT ? Emit{d, start_col, start_col} : Emit{d, start_col - span, start_col});
      } else {
        if (size % align || size / align != delta) return "inconsistent block unit";
        const bool in_table = (kind == K_BCOL && (int)align == fwd.bc_align) || (kind == K_BROW && (int)align == fwd.br_align);
        if (in_table && block_image_fits(fwd, kind, delta, grow, start_col)) {
          auto owner_end = [](int64_t, int64_t hi) -> int64_t { return hi; };
          auto put = [&](int tab, int64_t grp, BlockImage b, int64_t) { btents.push_back(BtEnt{0, tab, grp, b}); };
          block_images(fwd, kind, voff, grow, start_col, delta, owner_end, put);
        } else {
          for (int k = 0; k < size; k++) {
            const int64_t er = grow + (kind == K_BROW ? k % (int)align : k / (int)align);
            const int64_t ec = start_col + (kind == K_BROW ? k / (int)align : k % (int)align);
            singles.push_back(Single{er, ec, voff + (uint32_t)k});
          }
        }
      }
      v += size;
    }
    if (v != cp.nnz) return "ctl stream covers " + std::to_string(v) + " values, expected " + std::to_string(cp.nnz);
    // single elements: one-element diagonal descriptors when they are a tiny minority of the partition (the rule of
    // build_layout: a stencil's boundary elements keep the diagonal instantiation), else entries of table 4
    const bool as_desc = singles.size() <= (size_t)(cp.nnz / 256);
    for (const Single &sg : singles) {
      if (sg.col < clo || sg.col > chi) return "unit leaves the column range";
      if (as_desc) {
        XDesc e;
        e.voff = sg.voff; e.row = (int32_t)sg.col; e.col = (int32_t)sg.row;
        e.meta = (uint32_t)k_single | (1u << 16) | ((uint32_t)K_DIAG << 24) | XD_DELTA1;
        em.push_back(Emit{e, sg.col, sg.col});
      } else {
        btents.push_back(BtEnt{0, 4, sg.col, BlockImage{sg.voff, (uint32_t)sg.row | BT_IMAGE}});
      }
    }
  }
  std::vector<PartLayout> parts(1);
  PartLayout &L = parts[0];
  L.row_start = clo; L.nrows = chi - clo + 1;
  L.rpt = tile_rpt(L.nrows, m.rows_per_thread, !btents.empty());
  const int64_t TILE_ROWS = L.tile_rows();
  L.ntiles = (L.nrows + TILE_ROWS - 1) / TILE_ROWS;
  L.tile_xoff.assign((size_t)L.ntiles + 1, 0);
  memset(L.idtab, 0, sizeof(L.idtab));
  std::vector<Pending> pend;
  for (const Emit &e : em) {
    if (e.lo < clo || e.hi > chi) return "unit leaves the column range";
    for (int64_t t = (e.lo - clo) / TILE_ROWS; t <= (e.hi - clo) / TILE_ROWS; t++) pend.push_back(Pending{0, t, e.d});
    out.images |= (e.d.meta & XD_TRANSPOSED) != 0;
  }
  if (!btents.empty()) sort_block_tables(fwd, parts, btents);
  std::string err = distribute_descs(parts, pend);
  if (!err.empty()) return err;
  // heavy columns of table 4: their entries go to warp-sized segments
  for (size_t ti = 0; ti < L.bt.size(); ti++) {
    BlockTable &T = L.bt[ti];
    if (T.G != 1 || T.nloop != 1) continue;
    std::vector<uint32_t> ptr(1, 0);
    std::vector<BlockImage> ent;
    L.sk_fix_ptr.assign(1, 0);
    for (size_t j = 0; j + 1 < T.ptr.size(); j++) {
      const uint32_t e0 = T.ptr[j], e1 = T.ptr[j + 1];
      if (e1 - e0 > (uint32_t)out.heavy_min) {
        L.sk_fix_rows.push_back((int32_t)(T.j0 + (int64_t)j - L.row_start));
        for (uint32_t e = e0; e < e1; e += (uint32_t)out.seg_len) {
          L.sk_fix_idx.push_back((uint32_t)out.hseg.size());
          out.hseg.push_back((uint32_t)out.hent.size());
          out.hent.insert(out.hent.end(), T.ent.begin() + e, T.ent.begin() + std::min(e1, e + (uint32_t)out.seg_len));
        }
        L.sk_fix_ptr.push_back((uint32_t)L.sk_fix_idx.size());
      } else {
        ent.insert(ent.end(), T.ent.begin() + e0, T.ent.begin() + e1);
      }
      ptr.push_back((uint32_t)ent.size());
    }
    out.hseg.push_back((uint32_t)out.hent.size());
    out.heavy_cols = (int64_t)L.sk_fix_rows.size();
    L.sk_scratch = (uint32_t)(out.hseg.size() - 1);
    T.ptr.swap(ptr);
    T.ent.swap(ent);
    if (T.ent.empty()) L.bt.erase(L.bt.begin() + (long)ti);
    break;
  }
  if (out.hseg.empty()) out.hseg.push_back(0);
  out.part = std::move(L);
  return "";
}

void decode_transpose_coords(const TransLayout &t, int32_t *rows, int32_t *cols) {
  const PartLayout &L = t.part;
  auto put = [&](uint64_t vi, int64_t r, int64_t c) { rows[vi] = (int32_t)r; cols[vi] = (int32_t)c; };
  for (const XDesc &d : L.xdesc) {   // (a descriptor listed under several tiles is decoded once per tile)
    const uint32_t kind = (d.meta >> 24) & 0xf, size = (d.meta >> 16) & 0xff;
    const int64_t delta = (d.meta & XD_DELTA1) ? 1 : t.ktab[d.meta & 0xffff].delta;
    for (uint32_t k = 0; k < size; k++) {
      const int64_t s = (int64_t)k * delta;
      if (!(d.meta & XD_TRANSPOSED))   // unit of A^T: element (row + s, x index) is A(x index, row + s)
        put(d.voff + k, kind == K_VERT ? d.col : (kind == K_DIAG ? d.col + s : d.col - s), d.row + s);
      else                             // image of a vertical / anti-diagonal unit of A at (row, col)
        put(d.voff + k, d.row + s, kind == K_ADIAG ? d.col - s : d.col);
    }
  }
  for (const BlockTable &T : L.bt)
    for (size_t j = 0; j + 1 < T.ptr.size(); j++)
      for (uint32_t e = T.ptr[j]; e < T.ptr[j + 1]; e++)
        for (int64_t i = 0; i < T.G; i++) {   // the columns of the group
          const int64_t g = (T.j0 + (int64_t)j) * T.G + i;
          if (g < L.row_start || g >= L.row_start + L.nrows) continue;
          for (int l = 0; l < T.nloop; l++)
            put((uint64_t)T.ent[e].voff + (uint64_t)(i * T.sf + l * T.sl), (int64_t)(T.ent[e].other & ~BT_IMAGE) + l, g);
        }
  for (size_t i = 0; i < L.sk_fix_rows.size(); i++)
    for (uint32_t j = L.sk_fix_ptr[i]; j < L.sk_fix_ptr[i + 1]; j++)
      for (uint32_t e = t.hseg[L.sk_fix_idx[j]]; e < t.hseg[L.sk_fix_idx[j] + 1]; e++)
        put(t.hent[e].voff, (int64_t)(t.hent[e].other & ~BT_IMAGE), L.row_start + L.sk_fix_rows[i]);
}

}  // namespace spxb
