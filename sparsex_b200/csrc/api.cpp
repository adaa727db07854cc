// SparseX C API (spx_*) on top of the csxb_* engine ABI — the drop-in surface.
// Mirrors src/api/matvec.c, src/api/common.c and src/api/error.c of SparseX:
// same names, argument checks, return values and error-handler calls.  The
// runtime behind it is different: no thread pool, no JIT; spx_mat_tune encodes
// CSX on the host and uploads it to the GPU, spx_matvec_* launch CUDA kernels.
#include <cuda_runtime.h>

#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <sstream>
#include <string>
#include <vector>
#include <unistd.h>

#include <csx_b200.h>
#include <sparsex/sparsex.h>

#include "csx_host.hpp"

// defined in engine.cu (C++ linkage): tune from an in-memory COO input
csxb_matrix_t *csxb_tune_coo_internal(const spxb::CooHost &coo, const char *options, int part_lo, int part_hi, char *err, size_t errlen);

namespace {

// ---- global runtime configuration (RtConfig singleton, Runtime.hpp:74-134) ----
std::map<std::string, std::string> &props() {
  static std::map<std::string, std::string> p;
  return p;
}
int g_device = 0;
std::vector<int> g_devices;   // spx.rt.nr_gpus / spx.b200.devices: the GPUs one matrix is spread over (one process)
bool g_async = false;
bool g_gpu_ok = false;   // a managed vector was allocated successfully: a usable GPU is present
int g_part_lo = 0, g_part_hi = -1;   // one process per GPU: encode and own only partitions [lo, hi)
long long g_slab_row_start = -1, g_slab_total_rows = 0;   // the input holds only the rows of partition g_part_lo (csxb_tune_csr_slab)
int g_log_level = 2;  // 0 none, 1 error, 2 warning, 3 info, 4 verbose, 5 debug
FILE *g_log_file = nullptr;

enum { ALLOC_STD = 0, ALLOC_OTHER = 3, ALLOC_MANAGED = 5 };   // Vector.cpp:35-41 + engine addition
enum { VEC_MODE_AS_IS = 43, VEC_MODE_TUNED = 44, VEC_MODE_INVALID = 45 };

spx_errhandler_t g_handler = err_handle;

std::string options_string() {
  std::string s;
  for (auto &kv : props()) {
    if (kv.first == "spx.b200.device" || kv.first == "spx.b200.async") continue;
    s += kv.first + "=" + kv.second + ";";
  }
  return s;
}

bool is_managed(const spx_vector_t *v) { return v->alloc_type == ALLOC_MANAGED; }

}  // namespace

struct matrix {   // src/api/matvec.c:30-38
  spx_index_t nrows, ncols, nnz;
  int symmetric;
  spx_perm_t *permutation;
  csxb_matrix_t *csx;          // one GPU: the tuned matrix; several GPUs: member 0 of `group`
  csxb_group_t *group;         // several GPUs in this process (spx.rt.nr_gpus > 1), else NULL
  double *stage_x, *stage_y;   // device staging for vectors that live in plain host memory
};
struct input {    // src/api/matvec.c:43-48
  spx_index_t nrows, ncols, nnz;
  char type;      // 'C' CSR wrapper, 'M' MatrixMarket
  const spx_index_t *rowptr, *colind;
  const spx_value_t *values;
  spxb::CooHost *coo;
  spx_index_t *own_rowptr, *own_colind;   // SPX_MAT_REORDER: the reordered copy the input now stands for (Rcm.hpp:289-316)
  spx_value_t *own_values;
};
struct partition {  // src/api/matvec.c:53-60
  size_t nr_partitions;
  size_t *parts;
  int *nodes;
  int *affinity;
  spx_index_t *row_start;
  spx_index_t *row_end;
};

extern "C" {

// ---------------------------------------------------------------- errors --
static const char *err_text(spx_error_t c) {  // src/api/error.c message tables
  switch (c) {
    case SPX_ERR_ARG_INVALID: return "invalid argument";
    case SPX_ERR_FILE: return "file doesn't exist or can't be read";
    case SPX_ERR_INPUT_MAT: return "input matrix wasn't properly created";
    case SPX_ERR_TUNED_MAT: return "tuned matrix wasn't properly created";
    case SPX_ERR_VEC: return "vector creation failed";
    case SPX_ERR_PART: return "partitioning object wasn't properly created";
    case SPX_ERR_PERM: return "error in permutation";
    case SPX_ERR_DIM: return "incompatible matrix and vector dimensions";
    case SPX_ERR_VEC_DIM: return "incompatible vector dimension";
    case SPX_ERR_ENTRY_NOT_FOUND: return "matrix entry doesn't exist";
    case SPX_OUT_OF_BOUNDS: return "index out of bounds";
    case SPX_ERR_FILE_OPEN: return "unable to open file";
    case SPX_ERR_FILE_READ: return "unable to read from file";
    case SPX_ERR_FILE_WRITE: return "unable to write to file";
    case SPX_ERR_MEM_ALLOC: return "memory allocation failed";
    case SPX_ERR_MEM_FREE: return "memory deallocation failed";
    case SPX_WARN_CSXFILE: return "no specific file given to save CSX, using default: \"csx_file\"";
    case SPX_WARN_TUNING_OPT: return "invalid tuning option";
    case SPX_WARN_RUNTIME_OPT: return "invalid runtime option";
    case SPX_WARN_REORDER: return "reordering failed";
    case SPX_WARN_ENTRY_NOT_SET: return "entry not set";
  }
  return "unknown error";
}

void err_handle(spx_error_t code, const char *sourcefile, unsigned long lineno, const char *function, const char *fmt, ...) {
  (void)sourcefile; (void)lineno;
  bool warning = code > SPX_ERR_MAX_VALUE && code < SPX_WARN_MAX_VALUE;
  bool valid = (code > SPX_ERR_MIN_VALUE && code < SPX_ERR_MAX_VALUE) || warning;
  if (g_log_level >= (warning ? 2 : 1)) {
    FILE *out = g_log_file ? g_log_file : stderr;
    char msg[512] = "";
    if (fmt) { va_list ap; va_start(ap, fmt); vsnprintf(msg, sizeof(msg), fmt, ap); va_end(ap); }
    fprintf(out, "[%s]: %s() -> %s%s%s\n", warning ? "WARNING" : "ERROR", function ? function : "?",
            valid ? err_text(code) : "unknown error code", fmt ? ": " : "", msg);
    fflush(out);
  }
  if (code > SPX_ERR_SYSTEM && code < SPX_ERR_MAX_VALUE) exit(1);  // src/api/error.c:86
}
spx_errhandler_t spx_err_get_handler(void) { return g_handler; }
void spx_err_set_handler(spx_errhandler_t h) { g_handler = h ? h : err_handle; }

// --------------------------------------------------------------- logging --
void spx_log_disable_all(void) { g_log_level = 0; }
void spx_log_error_console(void) { g_log_level = 1; g_log_file = nullptr; }
void spx_log_warning_console(void) { g_log_level = 2; g_log_file = nullptr; }
void spx_log_info_console(void) { g_log_level = 3; g_log_file = nullptr; }
void spx_log_verbose_console(void) { g_log_level = 4; g_log_file = nullptr; }
void spx_log_debug_console(void) { g_log_level = 5; g_log_file = nullptr; }
void spx_log_set_file(const char *file) {
  if (g_log_file) fclose(g_log_file);
  g_log_file = file ? fopen(file, "a") : nullptr;
}
static void ensure_log_file() { if (!g_log_file) spx_log_set_file("sparsex.log"); }
void spx_log_error_file(void) { g_log_level = 1; ensure_log_file(); }
void spx_log_warning_file(void) { g_log_level = 2; ensure_log_file(); }
void spx_log_info_file(void) { g_log_level = 3; ensure_log_file(); }
void spx_log_verbose_file(void) { g_log_level = 4; ensure_log_file(); }
void spx_log_debug_file(void) { g_log_level = 5; ensure_log_file(); }
void spx_log_all_console(void) { g_log_level = 5; g_log_file = nullptr; }
void spx_log_all_file(const char *file) { g_log_level = 5; spx_log_set_file(file); }

void spx_init(void) { spx_log_warning_console(); }
void spx_finalize(void) {}

void *malloc_internal(size_t x, const char *sourcefile, unsigned long lineno, const char *function) {
  void *ret = malloc(x);
  if (!ret) { err_handle(SPX_ERR_MEM_ALLOC, sourcefile, lineno, function, NULL); exit(1); }
  return ret;
}
void free_internal(void *ptr, const char *sourcefile, unsigned long lineno, const char *function) {
  if (!ptr) { err_handle(SPX_ERR_MEM_FREE, sourcefile, lineno, function, NULL); exit(1); }
  free(ptr);
}

// --------------------------------------------------------------- options --
void spx_option_set(const char *option, const char *value) {  // matvec.c:753-756
  if (!option || !value) { SETWARNING(SPX_WARN_TUNING_OPT); return; }
  std::string k(option), v(value);
  if (k == "spx.b200.device") { g_device = atoi(value); return; }
  if (k == "spx.rt.nr_gpus" || k == "spx.b200.nr_gpus") {   // GPUs 0 .. n-1
    g_devices.clear();
    for (int i = 0; i < atoi(value); i++) g_devices.push_back(i);
    return;
  }
  if (k == "spx.b200.devices") {   // explicit list, e.g. "2,3" (an index may repeat: logical members on one GPU)
    g_devices.clear();
    std::stringstream ss(v);
    std::string t;
    while (std::getline(ss, t, ',')) if (!t.empty()) g_devices.push_back(atoi(t.c_str()));
    return;
  }
  if (k == "spx.b200.async") { g_async = (v == "true" || v == "1"); return; }
  if (k == "spx.b200.part_lo") { g_part_lo = atoi(value); return; }
  if (k == "spx.b200.part_hi") { g_part_hi = atoi(value); return; }
  if (k == "spx.b200.slab_row_start") { g_slab_row_start = atoll(value); return; }
  if (k == "spx.b200.slab_total_rows") { g_slab_total_rows = atoll(value); return; }
  spxb::TuneOptions probe;
  std::string e = probe.set(k, v);
  if (!e.empty()) {
    spx_err_get_handler()(k.rfind("spx.rt.", 0) == 0 ? SPX_WARN_RUNTIME_OPT : SPX_WARN_TUNING_OPT, __FILE__, __LINE__,
                          __func__, "%s", e.c_str());
    return;
  }
  props()[k] = v;
}
void spx_options_set_from_env(void) {  // Runtime.cpp:97-149
  const char *s;
  if ((s = getenv("SYMMETRIC"))) spx_option_set("spx.matrix.symmetric", s);
  if ((s = getenv("CPU_AFFINITY"))) spx_option_set("spx.rt.cpu_affinity", s);
  if ((s = getenv("NUM_THREADS"))) spx_option_set("spx.rt.nr_threads", s);
  if ((s = getenv("XFORM_CONF"))) spx_option_set("spx.preproc.xform", s);
  if ((s = getenv("WINDOW_SIZE"))) { spx_option_set("spx.preproc.sampling", "window"); spx_option_set("spx.preproc.sampling.window_size", s); }
  if ((s = getenv("SAMPLES"))) spx_option_set("spx.preproc.sampling.nr_samples", s);
  if ((s = getenv("SAMPLING_PORTION"))) { spx_option_set("spx.preproc.sampling", "portion"); spx_option_set("spx.preproc.sampling.portion", s); }
  if ((s = getenv("SAMPLING"))) spx_option_set("spx.preproc.sampling", s);
}

// ----------------------------------------------------------------- input --
spx_input_t *spx_input_load_csr(const spx_index_t *rowptr, const spx_index_t *colind, const spx_value_t *values,
                                spx_index_t nrows, spx_index_t ncols, ...) {
  // the optional indexing argument is read and discarded: the reference's check
  // (matvec.c:171-177) always falls back to zero-based
  if (!check_mat_dim(nrows) || !check_mat_dim(ncols)) { SETERROR_1(SPX_ERR_ARG_INVALID, "invalid matrix dimensions"); return SPX_INVALID_INPUT; }
  if (!rowptr) { SETERROR_1(SPX_ERR_ARG_INVALID, "invalid rowptr argument"); return SPX_INVALID_INPUT; }
  if (!colind) { SETERROR_1(SPX_ERR_ARG_INVALID, "invalid colind argument"); return SPX_INVALID_INPUT; }
  if (!values) { SETERROR_1(SPX_ERR_ARG_INVALID, "invalid values argument"); return SPX_INVALID_INPUT; }
  spx_input_t *A = spx_malloc(spx_input_t, sizeof(spx_input_t));
  A->type = 'C';
  A->nrows = nrows; A->ncols = ncols; A->nnz = rowptr[nrows];
  A->rowptr = rowptr; A->colind = colind; A->values = values;
  A->coo = nullptr;
  A->own_rowptr = A->own_colind = nullptr; A->own_values = nullptr;
  return A;
}

spx_input_t *spx_input_load_mmf(const char *filename) {
  if (!filename) { SETERROR_0(SPX_ERR_FILE); return SPX_INVALID_INPUT; }
  if (access(filename, F_OK | R_OK) == -1) { SETERROR_0(SPX_ERR_FILE); return SPX_INVALID_INPUT; }
  spxb::CooHost *coo = new spxb::CooHost;
  std::string e = spxb::read_mmf(filename, *coo);
  if (!e.empty()) {
    delete coo;
    spx_err_get_handler()(SPX_ERR_INPUT_MAT, __FILE__, __LINE__, __func__, "%s", e.c_str());
    return SPX_INVALID_INPUT;
  }
  spx_input_t *A = spx_malloc(spx_input_t, sizeof(spx_input_t));
  A->type = 'M';
  A->nrows = (spx_index_t)coo->nrows; A->ncols = (spx_index_t)coo->ncols; A->nnz = (spx_index_t)coo->row.size();
  A->rowptr = A->colind = nullptr; A->values = nullptr;
  A->coo = coo;
  A->own_rowptr = A->own_colind = nullptr; A->own_values = nullptr;
  return A;
}

spx_error_t spx_input_destroy(spx_input_t *A) {
  if (!A) { SETERROR_1(SPX_ERR_ARG_INVALID, "invalid input handle"); return SPX_FAILURE; }
  delete A->coo;
  free(A->own_rowptr); free(A->own_colind); free(A->own_values);
  spx_free(A);
  return SPX_SUCCESS;
}

// ---------------------------------------------------------------- tuning --
static void log_line(int level, const char *msg) {   // the reference's LOG_INFO / LOG_WARNING lines of Rcm.hpp
  if (g_log_level >= level) fprintf(g_log_file ? g_log_file : stderr, "%s\n", msg);
}

// ReorderCSR / ReorderMMF (src/internals/Facade.cpp:56-84 -> Rcm.hpp DoReorder_RCM): on success the input stands for
// P A P^T from here on and *permutation holds perm[old] = new; on failure ("no reordering available", "reordering
// failed") the input is left as it is and no permutation exists — the tune goes on either way, as in the reference.
static void reorder_input(spx_input_t *in, spx_perm_t **permutation) {
  log_line(3, "Reordering input matrix...");
  if (in->nrows != in->ncols || in->nrows <= 0 || g_slab_row_start >= 0) { log_line(2, "reordering failed"); return; }
  std::vector<int32_t> eu, ev, perm, inv;
  int64_t bw[2] = {0, 0};
  if (in->type == 'C') spxb::rcm_edges_csr(in->rowptr, in->colind, in->nrows, false, eu, ev);
  else if (in->coo->buffered) spxb::rcm_edges_coo(*in->coo, eu, ev);
  if (!spxb::rcm_find_perm(in->nrows, eu, ev, perm, inv, bw)) {
    log_line(2, "no reordering available for this matrix");
    log_line(2, "reordering failed");
    return;
  }
  char line[96];
  snprintf(line, sizeof(line), "Original Bandwidth: %lld", (long long)bw[0]); log_line(3, line);
  snprintf(line, sizeof(line), "Final Bandwidth: %lld", (long long)bw[1]); log_line(3, line);
  if (in->type == 'C') {
    spx_index_t *rp = (spx_index_t *)malloc(sizeof(spx_index_t) * ((size_t)in->nrows + 1));
    spx_index_t *ci = (spx_index_t *)malloc(sizeof(spx_index_t) * (size_t)(in->nnz ? in->nnz : 1));
    spx_value_t *va = (spx_value_t *)malloc(sizeof(spx_value_t) * (size_t)(in->nnz ? in->nnz : 1));
    if (!rp || !ci || !va || csxb_permute_csr(in->rowptr, in->colind, in->values, in->nrows, perm.data(), rp, ci, va) != 0) {
      free(rp); free(ci); free(va);
      log_line(2, "reordering failed");
      return;
    }
    free(in->own_rowptr); free(in->own_colind); free(in->own_values);
    in->rowptr = in->own_rowptr = rp; in->colind = in->own_colind = ci; in->values = in->own_values = va;
  } else {
    spxb::rcm_apply_coo(*in->coo, perm);
  }
  *permutation = (spx_perm_t *)malloc(sizeof(spx_perm_t) * (size_t)in->nrows);   // Facade.cpp:63-66
  for (spx_index_t i = 0; i < in->nrows; i++) (*permutation)[i] = perm[i];
  log_line(3, "Reordering complete");
}

// One GPU: upload.  Several (spx.rt.nr_gpus / spx.b200.devices, all partitions local): the partitions are dealt out
// to the GPUs (csxb_group_create consumes m).  On failure m is destroyed and the error handler has been called.
static bool place_on_devices(csxb_matrix_t *m, csxb_group_t **group) {
  *group = nullptr;
  const bool whole = csxb_info(m, CSXB_PART_LO) == 0 && csxb_info(m, CSXB_NPARTS) == csxb_info(m, CSXB_NPARTS_TOTAL);
  if (g_devices.size() > 1 && whole && csxb_info(m, CSXB_NPARTS) > 1) {
    char err[512] = "";
    *group = csxb_group_create(m, g_devices.data(), (int)g_devices.size(), 0, err, sizeof(err));
    if (*group) return true;
    spx_err_get_handler()(SPX_ERR_TUNED_MAT, __FILE__, __LINE__, __func__, "%s", err);
    csxb_destroy(m);
    return false;
  }
  if (csxb_upload(m, g_devices.size() == 1 ? g_devices[0] : g_device, 0) != 0) {
    spx_err_get_handler()(SPX_ERR_TUNED_MAT, __FILE__, __LINE__, __func__, "%s", csxb_last_error());
    csxb_destroy(m);
    return false;
  }
  return true;
}

spx_matrix_t *spx_mat_tune(spx_input_t *in, ...) {
  if (!in) { SETERROR_1(SPX_ERR_ARG_INVALID, "invalid input matrix"); return SPX_INVALID_MAT; }
  // matvec.c:268-272 reads the optional argument unconditionally; so does this (a caller that passes nothing leaves
  // whatever the register holds, in the reference as here)
  va_list ap;
  va_start(ap, in);
  spx_option_t option = va_arg(ap, spx_option_t);
  va_end(ap);
  spx_perm_t *permutation = SPX_INVALID_PERM;
  if (option == SPX_MAT_REORDER) reorder_input(in, &permutation);
  char err[512] = "";
  std::string opts = options_string();
  if (g_devices.size() > 1 && g_part_hi < 0 && g_slab_row_start < 0) {
    // at least one partition per GPU: the partition count is the reference's spx.rt.nr_threads
    auto it = props().find("spx.rt.nr_threads");
    if (it == props().end() || atoi(it->second.c_str()) < (int)g_devices.size()) {
      opts += "spx.rt.nr_threads=" + std::to_string(g_devices.size()) + ";";
      log_line(3, "spx.rt.nr_threads raised to the number of GPUs");
    }
  }
  csxb_matrix_t *m = nullptr;
  if (in->type == 'C' && g_slab_row_start >= 0)   // the arrays hold the rows of partition g_part_lo only
    m = csxb_tune_csr_slab(in->rowptr, in->colind, in->values, in->nrows, g_slab_total_rows, in->ncols, g_slab_row_start, g_part_lo,
                           opts.c_str(), err, sizeof(err));
  else if (in->type == 'C')
    m = csxb_tune_csr(in->rowptr, in->colind, in->values, in->nrows, in->ncols, opts.c_str(), g_part_lo, g_part_hi, err,
                      sizeof(err));
  else if (in->type == 'M')
    m = csxb_tune_coo_internal(*in->coo, opts.c_str(), g_part_lo, g_part_hi, err, sizeof(err));
  if (!m) { free(permutation); spx_err_get_handler()(SPX_ERR_TUNED_MAT, __FILE__, __LINE__, __func__, "%s", err); return SPX_INVALID_MAT; }
  if (permutation) csxb_set_perm(m, permutation, in->nrows);   // stored with the matrix by spx_mat_save (matvec.c:422)
  const int nrows_tuned = (int)csxb_info(m, CSXB_NROWS), symmetric = (int)csxb_info(m, CSXB_SYMMETRIC);
  csxb_group_t *group = nullptr;
  if (!place_on_devices(m, &group)) { free(permutation); return SPX_INVALID_MAT; }
  spx_matrix_t *A = spx_malloc(spx_matrix_t, sizeof(spx_matrix_t));
  A->nrows = nrows_tuned; A->ncols = in->ncols; A->nnz = in->nnz;
  A->symmetric = symmetric;
  A->permutation = permutation;
  A->group = group;
  A->csx = group ? csxb_group_member(group, 0) : m;
  A->stage_x = A->stage_y = nullptr;
  return A;
}

spx_error_t spx_mat_destroy(spx_matrix_t *A) {
  if (!A) { SETERROR_1(SPX_ERR_ARG_INVALID, "invalid matrix handle"); return SPX_FAILURE; }
  cudaDeviceSynchronize();
  if (A->stage_x) cudaFree(A->stage_x);
  if (A->stage_y) cudaFree(A->stage_y);
  if (A->group) csxb_group_destroy(A->group);
  else csxb_destroy(A->csx);
  free(A->permutation);
  spx_free(A);
  return SPX_SUCCESS;
}

struct csxb_matrix *spx_mat_get_engine(const spx_matrix_t *A) { return A ? A->csx : nullptr; }
void spx_device_synchronize(void) { cudaDeviceSynchronize(); }

spx_index_t spx_mat_get_nrows(const spx_matrix_t *A) {
  if (!A) { SETERROR_1(SPX_ERR_ARG_INVALID, "invalid matrix handle"); return SPX_FAILURE; }
  return A->nrows;
}
spx_index_t spx_mat_get_ncols(const spx_matrix_t *A) {
  if (!A) { SETERROR_1(SPX_ERR_ARG_INVALID, "invalid matrix handle"); return SPX_FAILURE; }
  return A->ncols;
}
spx_index_t spx_mat_get_nnz(const spx_matrix_t *A) {
  if (!A) { SETERROR_1(SPX_ERR_ARG_INVALID, "invalid matrix handle"); return SPX_FAILURE; }
  return A->nnz;
}

// Single entries (matvec.c:322-403): the optional argument selects the indexing; anything else means zero-based.
static int entry_indexing(va_list ap) {
  int indexing = va_arg(ap, int) - SPX_INDEX_ZERO_BASED;
  return (indexing == 0 || indexing == 1) ? indexing : 0;
}
spx_error_t spx_mat_get_entry(const spx_matrix_t *A, spx_index_t row, spx_index_t column, spx_value_t *value, ...) {
  va_list ap;
  va_start(ap, value);
  const int indexing = entry_indexing(ap);
  va_end(ap);
  if (!A) { SETERROR_1(SPX_ERR_ARG_INVALID, "invalid matrix handle"); return SPX_FAILURE; }
  if (row - indexing < 0 || row - indexing >= A->nrows || column - indexing < 0 || column - indexing >= A->ncols) {
    SETERROR_0(SPX_OUT_OF_BOUNDS);
    return SPX_FAILURE;
  }
  if (A->permutation != SPX_INVALID_PERM) {   // matvec.c:351-354 (and only meaningful for the square matrices RCM accepts)
    row = A->permutation[row - indexing] + indexing;
    column = A->permutation[column - indexing] + indexing;
  }
  if (!value || (A->group ? csxb_group_get_entry(A->group, row - indexing, column - indexing, value)
                          : csxb_get_entry(A->csx, row - indexing, column - indexing, value)) != 0) {
    SETERROR_0(SPX_ERR_ENTRY_NOT_FOUND);
    return SPX_FAILURE;
  }
  return SPX_SUCCESS;
}
spx_error_t spx_mat_set_entry(spx_matrix_t *A, spx_index_t row, spx_index_t column, spx_value_t value, ...) {
  va_list ap;
  va_start(ap, value);
  const int indexing = entry_indexing(ap);
  va_end(ap);
  if (!A) { SETERROR_1(SPX_ERR_ARG_INVALID, "invalid matrix handle"); return SPX_FAILURE; }
  if (row - indexing < 0 || row - indexing >= A->nrows || column - indexing < 0 || column - indexing >= A->ncols) {
    SETERROR_0(SPX_OUT_OF_BOUNDS);
    return SPX_FAILURE;
  }
  if (A->permutation != SPX_INVALID_PERM) {   // matvec.c:394-397
    row = A->permutation[row - indexing] + indexing;
    column = A->permutation[column - indexing] + indexing;
  }
  if ((A->group ? csxb_group_set_entry(A->group, row - indexing, column - indexing, value)
                : csxb_set_entry(A->csx, row - indexing, column - indexing, value)) != 0) {
    SETERROR_0(SPX_ERR_ENTRY_NOT_FOUND);
    return SPX_FAILURE;
  }
  return SPX_SUCCESS;
}
// Tuned-matrix container (matvec.c:405-445; the file format is this engine's own, not the reference's boost::archive)
spx_error_t spx_mat_save(const spx_matrix_t *A, const char *filename) {
  if (!A) { SETERROR_1(SPX_ERR_ARG_INVALID, "invalid matrix handle"); return SPX_FAILURE; }
  if (!filename) { SETWARNING(SPX_WARN_CSXFILE); filename = "csx_file"; }
  if ((A->group ? csxb_group_save(A->group, filename) : csxb_save(A->csx, filename)) != 0) {
    spx_err_get_handler()(SPX_ERR_FILE, __FILE__, __LINE__, __func__, "%s", csxb_last_error());
    return SPX_FAILURE;
  }
  return SPX_SUCCESS;
}
spx_matrix_t *spx_mat_restore(const char *filename) {
  if (!filename || access(filename, F_OK | R_OK) == -1) { SETERROR_0(SPX_ERR_FILE); return SPX_INVALID_MAT; }
  char err[512] = "";
  csxb_matrix_t *m = csxb_load(filename, err, sizeof(err));
  if (!m) { spx_err_get_handler()(SPX_ERR_FILE, __FILE__, __LINE__, __func__, "%s", err); return SPX_INVALID_MAT; }
  spx_matrix_t *A = spx_malloc(spx_matrix_t, sizeof(spx_matrix_t));
  A->nrows = (spx_index_t)csxb_info(m, CSXB_NROWS); A->ncols = (spx_index_t)csxb_info(m, CSXB_NCOLS);
  A->nnz = (spx_index_t)csxb_info(m, CSXB_NNZ);
  A->symmetric = (int)csxb_info(m, CSXB_SYMMETRIC);
  A->permutation = SPX_INVALID_PERM;
  const int64_t np = csxb_get_perm(m, nullptr);   // LoadTuned hands the stored permutation back (matvec.c:444-445)
  if (np > 0) {
    A->permutation = (spx_perm_t *)malloc(sizeof(spx_perm_t) * (size_t)np);
    csxb_get_perm(m, A->permutation);
  }
  csxb_group_t *group = nullptr;
  if (!place_on_devices(m, &group)) { free(A->permutation); spx_free(A); return SPX_INVALID_MAT; }
  A->group = group;
  A->csx = group ? csxb_group_member(group, 0) : m;
  A->stage_x = A->stage_y = nullptr;
  return A;
}
spx_perm_t *spx_mat_get_perm(const spx_matrix_t *A) {   // matvec.c:536-549
  if (!A) { SETERROR_1(SPX_ERR_ARG_INVALID, "invalid matrix handle"); return SPX_INVALID_PERM; }
  if (!A->permutation) { SETERROR_1(SPX_ERR_ARG_INVALID, "a permutation is not available"); return SPX_INVALID_PERM; }
  return A->permutation;
}

// ------------------------------------------------------------- partitions --
static spx_partition_t *part_alloc(size_t n) {
  spx_partition_t *p = spx_malloc(spx_partition_t, sizeof(spx_partition_t));
  p->nr_partitions = n;
  p->parts = nullptr; p->nodes = nullptr; p->affinity = nullptr;
  p->row_start = (spx_index_t *)malloc(sizeof(spx_index_t) * (n ? n : 1));
  p->row_end = (spx_index_t *)malloc(sizeof(spx_index_t) * (n ? n : 1));
  return p;
}
spx_partition_t *spx_mat_get_partition(const spx_matrix_t *A) {  // matvec.c:485-514: a new object, caller destroys
  if (!A) { SETERROR_1(SPX_ERR_ARG_INVALID, "invalid matrix handle"); return SPX_INVALID_PART; }
  const int nh = A->group ? csxb_group_size(A->group) : 1;
  int np = 0;
  for (int h = 0; h < nh; h++) np += (int)csxb_info(A->group ? csxb_group_member(A->group, h) : A->csx, CSXB_NPARTS);
  spx_partition_t *p = part_alloc(np);
  for (int h = 0, k = 0; h < nh; h++) {
    const csxb_matrix_t *m = A->group ? csxb_group_member(A->group, h) : A->csx;
    for (int i = 0; i < (int)csxb_info(m, CSXB_NPARTS); i++, k++) {
      p->row_start[k] = (spx_index_t)csxb_part_info(m, i, CSXB_P_ROW_START);
      p->row_end[k] = p->row_start[k] + (spx_index_t)csxb_part_info(m, i, CSXB_P_NROWS);
    }
  }
  return p;
}
spx_partition_t *spx_partition_csr(const spx_index_t *rowptr, spx_index_t nr_rows, size_t nr_threads) {  // matvec.c:687-735
  if (!rowptr || nr_threads == 0) { SETERROR_1(SPX_ERR_ARG_INVALID, "invalid partition arguments"); return SPX_INVALID_PART; }
  spx_partition_t *ret = part_alloc(nr_threads);
  size_t per = (size_t)(rowptr[nr_rows] - 1) / nr_threads, cur = 0, start = 0, cnt = 0;
  for (size_t k = 0; k < nr_threads; k++) { ret->row_start[k] = 0; ret->row_end[k] = 0; }
  ret->row_start[0] = 0;
  spx_index_t i;
  for (i = 0; i < nr_rows; i++) {
    cur += (size_t)(rowptr[i + 1] - rowptr[i]);
    if (cur >= per && cnt < nr_threads) {
      ret->row_end[cnt] = i + 1;
      start = (size_t)i + 1; cur = 0; ++cnt;
      if (cnt < nr_threads) ret->row_start[cnt] = (spx_index_t)start;
    }
  }
  if (cur < per && cnt < nr_threads) ret->row_end[cnt] = i + 1;
  return ret;
}
spx_index_t *spx_partition_get_rs(const spx_partition_t *p) {
  if (!p) { SETERROR_1(SPX_ERR_ARG_INVALID, "invalid partition handle"); return NULL; }
  return p->row_start;
}
spx_index_t *spx_partition_get_re(const spx_partition_t *p) {
  if (!p) { SETERROR_1(SPX_ERR_ARG_INVALID, "invalid partition handle"); return NULL; }
  return p->row_end;
}
spx_error_t spx_partition_destroy(spx_partition_t *p) {
  if (!p) { SETERROR_1(SPX_ERR_ARG_INVALID, "invalid partition handle"); return SPX_FAILURE; }
  free(p->parts); free(p->nodes); free(p->affinity); free(p->row_start); free(p->row_end);
  spx_free(p);
  return SPX_SUCCESS;
}

// ------------------------------------------------------------------ SpMV --
// x and y may live in managed memory (library vectors: used in place, resident
// in HBM) or in plain host memory (spx_vec_create_from_buff: staged through
// device buffers, copies inside the call).
static spx_error_t run_spmv(const spx_matrix_t *Ac, spx_value_t alpha, const spx_vector_t *x, spx_value_t beta,
                            spx_vector_t *y, int overwrite) {
  spx_matrix_t *A = const_cast<spx_matrix_t *>(Ac);
  if (A->group) {   // several GPUs: columns out, kernels, (CSX-Sym: reduction,) rows back; synchronous
    if (csxb_group_spmv(A->group, alpha, x->elements, beta, y->elements, overwrite) != 0) {
      spx_err_get_handler()(SPX_ERR_TUNED_MAT, __FILE__, __LINE__, __func__, "%s", csxb_last_error());
      return SPX_FAILURE;
    }
    return SPX_SUCCESS;
  }
  // the device the matrix lives on, not the current value of spx.b200.device (it may have changed since spx_mat_tune)
  const int device = (int)csxb_info(A->csx, CSXB_DEVICE);
  cudaSetDevice(device);
  const double *dx = x->elements;
  double *dy = y->elements;
  bool x_host = !is_managed(x), y_host = !is_managed(y);
  if (x_host && y_host) {   // user buffers on both sides: the pipelined host-buffer path of the engine
    if (csxb_spmv_host(A->csx, alpha, x->elements, beta, y->elements, overwrite) != 0) {
      spx_err_get_handler()(SPX_ERR_TUNED_MAT, __FILE__, __LINE__, __func__, "%s", csxb_last_error());
      return SPX_FAILURE;
    }
    return SPX_SUCCESS;
  }
  if (x_host) {
    if (!A->stage_x && cudaMalloc((void **)&A->stage_x, (size_t)(A->ncols ? A->ncols : 1) * 8) != cudaSuccess) {
      SETERROR_1(SPX_ERR_VEC, "device allocation failed");
      return SPX_FAILURE;
    }
    if (cudaMemcpyAsync(A->stage_x, x->elements, (size_t)A->ncols * 8, cudaMemcpyHostToDevice, 0) != cudaSuccess) {
      SETERROR_1(SPX_ERR_VEC, "host to device copy of x failed (no usable GPU?)");
      return SPX_FAILURE;
    }
    dx = A->stage_x;
  } else {
    cudaMemPrefetchAsync(x->elements, x->size * 8, device, 0);
  }
  if (y_host) {
    if (!A->stage_y && cudaMalloc((void **)&A->stage_y, (size_t)(A->nrows ? A->nrows : 1) * 8) != cudaSuccess) {
      SETERROR_1(SPX_ERR_VEC, "device allocation failed");
      return SPX_FAILURE;
    }
    if (!overwrite) cudaMemcpyAsync(A->stage_y, y->elements, (size_t)A->nrows * 8, cudaMemcpyHostToDevice, 0);
    dy = A->stage_y;
  } else {
    cudaMemPrefetchAsync(y->elements, y->size * 8, device, 0);
  }
  if (csxb_spmv(A->csx, alpha, dx, beta, dy, overwrite, nullptr) != 0) {
    spx_err_get_handler()(SPX_ERR_TUNED_MAT, __FILE__, __LINE__, __func__, "%s", csxb_last_error());
    return SPX_FAILURE;
  }
  if (y_host) {  // only the rows this handle owns travel back (all of y when every partition is local)
    int np = (int)csxb_info(A->csx, CSXB_NPARTS);
    bool all = np == (int)csxb_info(A->csx, CSXB_NPARTS_TOTAL);
    long lo = 0, hi = A->nrows;
    if (!all && np > 0) {
      lo = (long)csxb_part_info(A->csx, 0, CSXB_P_ROW_START);
      hi = (long)csxb_part_info(A->csx, np - 1, CSXB_P_ROW_START) + (long)csxb_part_info(A->csx, np - 1, CSXB_P_NROWS);
      if ((int)csxb_info(A->csx, CSXB_PART_LO) + np == (int)csxb_info(A->csx, CSXB_NPARTS_TOTAL)) hi = A->nrows;
    }
    if (hi > lo) cudaMemcpyAsync(y->elements + lo, A->stage_y + lo, (size_t)(hi - lo) * 8, cudaMemcpyDeviceToHost, 0);
  }
  if (y_host || !g_async) {
    cudaError_t e = cudaStreamSynchronize(0);
    if (e != cudaSuccess) {
      spx_err_get_handler()(SPX_ERR_TUNED_MAT, __FILE__, __LINE__, __func__, "%s", cudaGetErrorString(e));
      return SPX_FAILURE;
    }
  }
  return SPX_SUCCESS;
}

static spx_error_t check_spmv_args(const spx_matrix_t *A, const spx_vector_t *x, const spx_vector_t *y) {
  if (!A) { SETERROR_1(SPX_ERR_ARG_INVALID, "invalid matrix handle"); return SPX_FAILURE; }
  if (!x) { SETERROR_1(SPX_ERR_ARG_INVALID, "invalid vector x"); return SPX_FAILURE; }
  if (!y) { SETERROR_1(SPX_ERR_ARG_INVALID, "invalid vector y"); return SPX_FAILURE; }
  // The reference rejects only when BOTH sizes mismatch (matvec.c:571); a single
  // mismatch would make the kernels read or write out of bounds, so either one
  // is an error here.
  if (!check_vec_dim(x, (unsigned long)A->ncols) || !check_vec_dim(y, (unsigned long)A->nrows)) { SETERROR_0(SPX_ERR_DIM); return SPX_FAILURE; }
  return SPX_SUCCESS;
}

spx_error_t spx_matvec_mult(spx_value_t alpha, const spx_matrix_t *A, const spx_vector_t *x, spx_vector_t *y) {
  if (check_spmv_args(A, x, y) != SPX_SUCCESS) return SPX_FAILURE;
  return run_spmv(A, alpha, x, 0.0, y, 1);   // VecInit(y, 0) semantics, CsxKernels.cpp:93
}
spx_error_t spx_matvec_kernel(spx_value_t alpha, const spx_matrix_t *A, const spx_vector_t *x, spx_value_t beta,
                              spx_vector_t *y) {
  if (check_spmv_args(A, x, y) != SPX_SUCCESS) return SPX_FAILURE;
  return run_spmv(A, alpha, x, beta, y, 0);
}
// y = alpha*A^T*x (+ beta*y): x has nrows, y ncols entries.  Library (managed) vectors on both sides run on the device in
// place; a plain host buffer on either side goes through the host-buffer path (copies inside the call).
static spx_error_t run_spmv_t(const spx_matrix_t *Ac, spx_value_t alpha, const spx_vector_t *x, spx_value_t beta,
                              spx_vector_t *y, int overwrite) {
  spx_matrix_t *A = const_cast<spx_matrix_t *>(Ac);
  int rc;
  if (A->group) {
    rc = csxb_group_spmv_t(A->group, alpha, x->elements, beta, y->elements, overwrite);
  } else if (is_managed(x) && is_managed(y)) {
    const int device = (int)csxb_info(A->csx, CSXB_DEVICE);
    cudaSetDevice(device);
    cudaMemPrefetchAsync(x->elements, x->size * 8, device, 0);
    cudaMemPrefetchAsync(y->elements, y->size * 8, device, 0);
    rc = csxb_spmv_t(A->csx, alpha, x->elements, beta, y->elements, overwrite, nullptr);
    if (rc == 0 && !g_async && cudaStreamSynchronize(0) != cudaSuccess) rc = -1;
  } else {
    rc = csxb_spmv_t_host(A->csx, alpha, x->elements, beta, y->elements, overwrite);
  }
  if (rc != 0) {
    spx_err_get_handler()(SPX_ERR_TUNED_MAT, __FILE__, __LINE__, __func__, "%s", csxb_last_error());
    return SPX_FAILURE;
  }
  return SPX_SUCCESS;
}
static spx_error_t check_spmv_t_args(const spx_matrix_t *A, const spx_vector_t *x, const spx_vector_t *y) {
  if (!A) { SETERROR_1(SPX_ERR_ARG_INVALID, "invalid matrix handle"); return SPX_FAILURE; }
  if (!x) { SETERROR_1(SPX_ERR_ARG_INVALID, "invalid vector x"); return SPX_FAILURE; }
  if (!y) { SETERROR_1(SPX_ERR_ARG_INVALID, "invalid vector y"); return SPX_FAILURE; }
  if (!check_vec_dim(x, (unsigned long)A->nrows) || !check_vec_dim(y, (unsigned long)A->ncols)) { SETERROR_0(SPX_ERR_DIM); return SPX_FAILURE; }
  return SPX_SUCCESS;
}
spx_error_t spx_matvec_mult_trans(spx_value_t alpha, const spx_matrix_t *A, const spx_vector_t *x, spx_vector_t *y) {
  if (check_spmv_t_args(A, x, y) != SPX_SUCCESS) return SPX_FAILURE;
  return run_spmv_t(A, alpha, x, 0.0, y, 1);
}
spx_error_t spx_matvec_kernel_trans(spx_value_t alpha, const spx_matrix_t *A, const spx_vector_t *x, spx_value_t beta,
                                    spx_vector_t *y) {
  if (check_spmv_t_args(A, x, y) != SPX_SUCCESS) return SPX_FAILURE;
  return run_spmv_t(A, alpha, x, beta, y, 0);
}
spx_error_t spx_matvec_kernel_csr(spx_matrix_t **A, spx_index_t nrows, spx_index_t ncols, const spx_index_t *rowptr,
                                  const spx_index_t *colind, const spx_value_t *values, spx_value_t alpha,
                                  const spx_vector_t *x, spx_value_t beta, spx_vector_t *y) {  // matvec.c:622-673
  if (!A) { SETERROR_1(SPX_ERR_ARG_INVALID, "invalid matrix handle"); return SPX_FAILURE; }
  if (!x) { SETERROR_1(SPX_ERR_ARG_INVALID, "invalid vector x"); return SPX_FAILURE; }
  if (!y) { SETERROR_1(SPX_ERR_ARG_INVALID, "invalid vector y"); return SPX_FAILURE; }
  if (!*A) {
    spx_input_t *in = spx_input_load_csr(rowptr, colind, values, nrows, ncols, SPX_INDEX_ZERO_BASED);
    if (!in) return SPX_FAILURE;
    *A = spx_mat_tune(in);
    spx_input_destroy(in);
    if (!*A) return SPX_FAILURE;
  }
  return spx_matvec_kernel(alpha, *A, x, beta, y);
}

// --------------------------------------------------------------- vectors --
static spx_vector_t *vec_alloc(size_t size, bool zero) {
  spx_vector_t *v = (spx_vector_t *)malloc(sizeof(spx_vector_t));
  if (!v) { SETERROR_0(SPX_ERR_MEM_ALLOC); return SPX_INVALID_VEC; }
  void *p = nullptr;
  size_t bytes = (size ? size : 1) * sizeof(spx_value_t);
  if (cudaMallocManaged(&p, bytes, cudaMemAttachGlobal) == cudaSuccess) {
    v->alloc_type = ALLOC_MANAGED;
    g_gpu_ok = true;
    if (zero) memset(p, 0, bytes);
  } else {
    cudaGetLastError();  // no usable GPU: a plain host vector still works for the BLAS-1 helpers
    p = zero ? calloc(size ? size : 1, sizeof(spx_value_t)) : malloc(bytes);
    if (!p) { free(v); SETERROR_0(SPX_ERR_MEM_ALLOC); return SPX_INVALID_VEC; }
    v->alloc_type = ALLOC_STD;
  }
  v->elements = (spx_value_t *)p;
  v->size = size;
  v->vec_mode = VEC_MODE_INVALID;
  return v;
}
spx_vector_t *spx_vec_create(size_t size, const spx_partition_t *p) {  // matvec.c:763-779
  if (p == SPX_INVALID_PART) { SETERROR_1(SPX_ERR_ARG_INVALID, "invalid partition handle"); return SPX_INVALID_VEC; }
  return vec_alloc(size, true);
}
spx_vector_t *spx_vec_create_from_buff(spx_value_t *buff, spx_value_t **tuned, size_t size, const spx_partition_t *p,
                                       spx_vecmode_t mode) {  // matvec.c:781-818, Vector.cpp:113-159 (non-NUMA)
  if (!buff) { SETERROR_1(SPX_ERR_ARG_INVALID, "invalid buffer"); return SPX_INVALID_VEC; }
  if (!check_vecmode(mode)) { SETERROR_1(SPX_ERR_ARG_INVALID, "invalid vector mode"); return SPX_INVALID_VEC; }
  if (p == SPX_INVALID_PART && mode == SPX_VEC_TUNE) { SETERROR_1(SPX_ERR_ARG_INVALID, "invalid partition handle"); return SPX_INVALID_VEC; }
  spx_vector_t *v = (spx_vector_t *)malloc(sizeof(spx_vector_t));
  if (!v) { SETERROR_0(SPX_ERR_MEM_ALLOC); return SPX_INVALID_VEC; }
  v->elements = buff;
  v->size = size;
  v->alloc_type = ALLOC_OTHER;
  v->vec_mode = (int)mode;
  if (tuned) *tuned = buff;
  return v;
}
void spx_vec_init_rand_range(spx_vector_t *v, spx_value_t max, spx_value_t min) {  // Vector.cpp:228-236
  for (size_t i = 0; i < v->size; i++) {
    spx_value_t val = ((spx_value_t)(rand() + i) / ((spx_value_t)RAND_MAX + 1));
    v->elements[i] = min + val * (max - min);
  }
}
spx_vector_t *spx_vec_create_random(size_t size, const spx_partition_t *p) {  // Vector.cpp:161-167
  if (p == SPX_INVALID_PART) { SETERROR_1(SPX_ERR_ARG_INVALID, "invalid partition handle"); return SPX_INVALID_VEC; }
  spx_vector_t *v = vec_alloc(size, true);
  if (v) spx_vec_init_rand_range(v, (spx_value_t)-0.1, (spx_value_t)0.1);
  return v;
}
void spx_vec_destroy(spx_vector_t *v) {  // Vector.cpp:187-204
  if (!v) return;
  if (v->alloc_type == ALLOC_MANAGED) { cudaDeviceSynchronize(); cudaFree(v->elements); }
  else if (v->alloc_type == ALLOC_STD) free(v->elements);
  free(v);
}
void spx_vec_init(spx_vector_t *v, spx_value_t val) { for (size_t i = 0; i < v->size; i++) v->elements[i] = val; }
void spx_vec_init_part(spx_vector_t *v, spx_value_t val, spx_index_t start, spx_index_t end) {
  for (spx_index_t i = start; i < end; i++) v->elements[i] = val;
}
spx_error_t spx_vec_set_entry(spx_vector_t *v, spx_index_t idx, spx_value_t val, ...) {  // matvec.c:838-862
  // one-based like the reference (its indexing argument always degrades to one-based + !0)
  if (idx <= 0 || (size_t)idx > v->size) { SETERROR_0(SPX_OUT_OF_BOUNDS); SETWARNING(SPX_WARN_ENTRY_NOT_SET); return SPX_FAILURE; }
  v->elements[idx - 1] = val;
  return SPX_SUCCESS;
}
// BLAS-1 helpers (Vector.cpp:259-377).  Vectors the library allocated live in managed memory and are resident in
// HBM between SpMVs: for those the operation runs on the GPU (csxb_vec_*), so that a solver iteration does not
// migrate them back to the host; user buffers take the host loop.
static bool on_device(const spx_vector_t *a, const spx_vector_t *b, const spx_vector_t *c) {
  return g_gpu_ok && a && is_managed(a) && (!b || is_managed(b)) && (!c || is_managed(c));
}
static void device_done() { if (!g_async) cudaStreamSynchronize(0); }
// out[s:e) = alpha*a[s:e) + beta*b[s:e)
static void axpby(spx_vector_t *out, const spx_vector_t *a, const spx_vector_t *b, double alpha, double beta, size_t s, size_t e) {
  if (e <= s) return;
  if (on_device(out, a, b) && csxb_vec_axpby(out->elements + s, a->elements + s, b ? b->elements + s : nullptr, alpha, beta,
                                             (int64_t)(e - s), nullptr) == 0) {
    device_done();
    return;
  }
  cudaDeviceSynchronize();   // pending device work on managed vectors must finish before the host touches them
  if (b) for (size_t i = s; i < e; i++) out->elements[i] = alpha * a->elements[i] + beta * b->elements[i];
  else for (size_t i = s; i < e; i++) out->elements[i] = alpha * a->elements[i];
}
static double dot(const spx_vector_t *a, const spx_vector_t *b, size_t s, size_t e) {
  double r = 0;
  if (e <= s) return r;
  if (on_device(a, b, nullptr) && csxb_vec_dot(a->elements + s, b->elements + s, (int64_t)(e - s), &r, nullptr) == 0) return r;
  cudaDeviceSynchronize();
  r = 0;
  for (size_t i = s; i < e; i++) r += a->elements[i] * b->elements[i];
  return r;
}
void spx_vec_scale(spx_vector_t *v1, spx_vector_t *v2, spx_value_t num) { axpby(v2, v1, nullptr, num, 0.0, 0, v1->size); }
void spx_vec_scale_add(spx_vector_t *v1, spx_vector_t *v2, spx_vector_t *v3, spx_value_t num) { axpby(v3, v1, v2, 1.0, num, 0, v1->size); }
void spx_vec_scale_add_part(spx_vector_t *v1, spx_vector_t *v2, spx_vector_t *v3, spx_value_t num, spx_index_t start,
                            spx_index_t end) {
  axpby(v3, v1, v2, 1.0, num, (size_t)start, (size_t)end);
}
void spx_vec_add(spx_vector_t *v1, spx_vector_t *v2, spx_vector_t *v3) { axpby(v3, v1, v2, 1.0, 1.0, 0, v1->size); }
void spx_vec_add_part(spx_vector_t *v1, spx_vector_t *v2, spx_vector_t *v3, spx_index_t start, spx_index_t end) {
  axpby(v3, v1, v2, 1.0, 1.0, (size_t)start, (size_t)end);
}
void spx_vec_sub(spx_vector_t *v1, spx_vector_t *v2, spx_vector_t *v3) { axpby(v3, v1, v2, 1.0, -1.0, 0, v1->size); }
void spx_vec_sub_part(spx_vector_t *v1, spx_vector_t *v2, spx_vector_t *v3, spx_index_t start, spx_index_t end) {
  axpby(v3, v1, v2, 1.0, -1.0, (size_t)start, (size_t)end);
}
spx_value_t spx_vec_mul(const spx_vector_t *v1, const spx_vector_t *v2) { return dot(v1, v2, 0, v1->size); }
spx_value_t spx_vec_mul_part(const spx_vector_t *v1, const spx_vector_t *v2, spx_index_t start, spx_index_t end) {
  return dot(v1, v2, (size_t)start, (size_t)end);
}
spx_error_t spx_vec_reorder(spx_vector_t *v, spx_perm_t *p) {  // matvec.c:934-958
  if (p == SPX_INVALID_PERM) { SETERROR_1(SPX_ERR_ARG_INVALID, "invalid permutation"); return SPX_FAILURE; }
  spx_value_t *tmp = (spx_value_t *)malloc(v->size * sizeof(spx_value_t));
  for (size_t i = 0; i < v->size; i++) tmp[p[i]] = v->elements[i];
  memcpy(v->elements, tmp, v->size * sizeof(spx_value_t));
  free(tmp);
  return SPX_SUCCESS;
}
spx_error_t spx_vec_inv_reorder(spx_vector_t *v, spx_perm_t *p) {
  if (p == SPX_INVALID_PERM) { SETERROR_1(SPX_ERR_ARG_INVALID, "invalid permutation"); return SPX_FAILURE; }
  spx_value_t *tmp = (spx_value_t *)malloc(v->size * sizeof(spx_value_t));
  for (size_t i = 0; i < v->size; i++) tmp[i] = v->elements[p[i]];
  memcpy(v->elements, tmp, v->size * sizeof(spx_value_t));
  free(tmp);
  return SPX_SUCCESS;
}
void spx_vec_copy(const spx_vector_t *v1, spx_vector_t *v2) { memcpy(v2->elements, v1->elements, v1->size * sizeof(spx_value_t)); }
int spx_vec_compare(const spx_vector_t *v1, const spx_vector_t *v2) {  // Vector.cpp:51-57, 396-413
  if (v1->size != v2->size) { fprintf(stderr, "v1->size=%lu v2->size=%lu differ\n", v1->size, v2->size); return -2; }
  for (size_t i = 0; i < v1->size; i++) {
    if (fabs((v1->elements[i] - v2->elements[i]) / v1->elements[i]) > 1.e-6) {
      fprintf(stderr, "element %ld differs: %10.20f != %10.20f\n", (long)i, v1->elements[i], v2->elements[i]);
      return -1;
    }
  }
  return 0;
}
void spx_vec_print(const spx_vector_t *v) {
  printf("[ ");
  for (size_t i = 0; i < v->size; i++) printf("%g ", v->elements[i]);
  printf("]\n");
}

}  // extern "C"
