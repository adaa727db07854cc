/*
 * csx_b200.h — thin C-ABI of the B200 CSX SpMV engine.
 *
 * This is the boundary between host code (C, C++, ctypes, cgo, JNI ...) and the
 * CUDA kernels: plain pointers and sizes, no C++ or torch types.  The SparseX
 * public API (include/sparsex/sparsex.h, spx_* functions) is implemented on top
 * of these entry points in sparsex_b200/csrc/api.cpp; each entry point below
 * names the reference interface it stands in for (file:line into the SparseX
 * tree).
 *
 * Threading: like the reference (global RtConfig/ThreadPool singletons,
 * Runtime.hpp:74-78), one caller thread per matrix handle.
 */
#ifndef CSX_B200_H
#define CSX_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct csxb_matrix csxb_matrix_t;

/* ---- tuning (host) ------------------------------------------------------
 * Replaces TuneCSR / TuneMMF -> SparseMatrix::CreateCsx()
 * (src/internals/Facade.cpp:86-122, SparseMatrix.hpp:123-255) and everything
 * below it (BuildPartitions, EncodingManager, CsxManager).
 *
 * `options` is a ';'-separated list of "mnemonic=value" pairs using the
 * reference's property names (src/internals/Runtime.cpp:65-95), e.g.
 * "spx.preproc.xform=all;spx.rt.nr_threads=8".  spx.rt.nr_threads is the number
 * of row partitions.  Partitions [part_lo, part_hi) are encoded by this call
 * (one process per GPU encodes only its own partition); pass 0, -1 for all.
 * CSR arrays are zero-based and are only read during the call.
 * Returns NULL and fills `err` on failure (the reference calls exit(1)).
 */
csxb_matrix_t *csxb_tune_csr(const int32_t *rowptr, const int32_t *colind, const double *values,
                             int64_t nrows, int64_t ncols, const char *options,
                             int part_lo, int part_hi, char *err, size_t errlen);
csxb_matrix_t *csxb_tune_mmf(const char *path, const char *options, int part_lo, int part_hi,
                             char *err, size_t errlen);
/* One process per GPU on matrices too large for one host: the CSR arrays hold exactly the rows
 * [row_start, row_start + slab_rows) of partition `part` of the spx.rt.nr_threads-way split of a matrix
 * with nrows_total rows (rowptr is relative to the slab; the caller applies the split rule of
 * SparseInternal.hpp:119-152 to the row lengths).  The partition is encoded from its own rows alone, like
 * the reference's per-thread preprocessing (CsxBuild.hpp:134-288), and equals what csxb_tune_csr yields
 * for it on the whole matrix.  CSX-Sym: no reduction map (it needs every partition). */
csxb_matrix_t *csxb_tune_csr_slab(const int32_t *rowptr, const int32_t *colind, const double *values,
                                  int64_t slab_rows, int64_t nrows_total, int64_t ncols, int64_t row_start,
                                  int part, const char *options, char *err, size_t errlen);
void csxb_destroy(csxb_matrix_t *m);

/* Matrix-level queries (spx_mat_get_nrows/ncols/nnz, src/api/matvec.c:447-476). */
enum { CSXB_NROWS = 0, CSXB_NCOLS = 1, CSXB_NNZ = 2, CSXB_SYMMETRIC = 3, CSXB_NPARTS = 4,
       CSXB_NPARTS_TOTAL = 5, CSXB_PART_LO = 6, CSXB_FULL_COLIND = 7,
       /* CSX-Sym with only some partitions local (valid after csxb_upload): rows [LO, HI) of y belong to
        * other devices; csxb_spmv zeroes them and adds this device's transposed contributions there, the
        * caller sends them to their owners and adds (sparsex_b200/dist.py: SymHaloReduce). */
       CSXB_SYM_HALO_LO = 8, CSXB_SYM_HALO_HI = 9,
       /* csxb_spmv_host: bytes of dynamic shared memory that cap the resident CTAs of the slab kernels (chosen by timing
        * the first calls), and the number of calls so far */
       CSXB_HOST_CAP = 10, CSXB_HOST_CALLS = 11,
       CSXB_DEVICE = 12 /* the device the matrix was uploaded to, -1 before csxb_upload */ };
int64_t csxb_info(const csxb_matrix_t *m, int what);

/* Per-partition CSX arrays == csx_matrix_t / csx_sym_matrix_t / map_t
 * (include/sparsex/internals/Csx.hpp:29-53, Map.hpp:23-27).  `part` is local
 * (0 .. CSXB_NPARTS-1).  Used by spx_mat_get_partition and by the parity tests. */
enum { CSXB_P_NNZ = 0, CSXB_P_NROWS = 1, CSXB_P_NCOLS = 2, CSXB_P_ROW_START = 3, CSXB_P_CTL_SIZE = 4,
       CSXB_P_ROW_JUMPS = 5, CSXB_P_ID_MAP_LEN = 6, CSXB_P_MAP_LEN = 7, CSXB_P_DVALUES_LEN = 8,
       CSXB_P_ROWS_INFO_LEN = 9, CSXB_P_SAMPLING_UNDEFINED = 10,
       CSXB_P_COL_MIN = 11, CSXB_P_COL_MAX = 12 /* zero-based column window the partition reads */ };
int64_t csxb_part_info(const csxb_matrix_t *m, int part, int what);
/* what: values f64[nnz] | ctl u8[ctl_size] | id_map i64[len] | rows_info {i64 rowptr,i64 valptr,i32 span,i32 pad}[nrows]
 *       | dvalues f64 | map_cpus u32 | map_pos u32 */
enum { CSXB_A_VALUES = 0, CSXB_A_CTL = 1, CSXB_A_ID_MAP = 2, CSXB_A_ROWS_INFO = 3, CSXB_A_DVALUES = 4,
       CSXB_A_MAP_CPUS = 5, CSXB_A_MAP_POS = 6 };
int csxb_part_copy(const csxb_matrix_t *m, int part, int what, void *dst);
/* Human-readable encoding sequence chosen for a partition, e.g. "d{1} h{1} ". */
const char *csxb_part_log(const csxb_matrix_t *m, int part);

/* ---- device ---------------------------------------------------------------
 * Replaces the per-partition JIT (CsxJit::GenCode, CsxJit.hpp:675-732) and
 * CreatePool (Facade.cpp:207-212): derives the GPU side tables from the ctl
 * stream and copies values/ctl/tables to `device`.  `free_host` != 0 drops the
 * host copies of values afterwards (ctl/id_map stay for introspection).
 * Returns 0 or a negative error (message via csxb_last_error). */
int csxb_upload(csxb_matrix_t *m, int device, int free_host);
const char *csxb_last_error(void);
/* Builds the GPU tables on the host only (no device needed) and reports their sizes, 12 numbers per row owner
 * (local partitions, then the CSX-Sym halo pseudo-partition): rows, tiles, table descriptors, stream chunks, stream
 * units, fix-up entries, gaps, entries of block tables 0..4.  Returns the number of row owners, -1 on error. */
int csxb_layout_stats(csxb_matrix_t *m, int64_t *out, int max_owners);

/* Device footprint and algorithmic traffic of one SpMV over the local
 * partitions, in bytes (SURVEY.md section 8d): */
enum { CSXB_B_VALUES = 0, CSXB_B_CTL = 1, CSXB_B_TABLES = 2, CSXB_B_X = 3, CSXB_B_Y = 4, CSXB_B_TOTAL = 5,
       CSXB_B_LAUNCHES = 6 /* kernels launched per SpMV */ };
int64_t csxb_traffic(const csxb_matrix_t *m, int what);

/* y[rows of the local partitions] = alpha * A_local * x (+ beta * y).
 * Replaces MatVecMult / MatVecKernel and their _sym variants
 * (src/internals/CsxKernels.cpp:35-129) plus the generated
 * spm_csx_multiply / spm_csx_sym_multiply (src/templates/csx_spmv_tmpl.c:66-101,
 * csx_sym_spmv_tmpl.c:60-106).
 *   d_x : device pointer, ncols doubles (the whole x vector)
 *   d_y : device pointer, nrows doubles (the whole y vector; only local rows are written)
 *   overwrite != 0 : spx_matvec_mult semantics (y := alpha*A*x, beta ignored, CsxKernels.cpp:93)
 *   overwrite == 0 : spx_matvec_kernel semantics (y := alpha*A*x + beta*y, CsxSpmv.cpp:52-65)
 *   stream : cudaStream_t (NULL = default stream).  Asynchronous.
 * CSX-Sym with a partition range: see CSXB_SYM_HALO_LO/HI. */
int csxb_spmv(csxb_matrix_t *m, double alpha, const double *d_x, double beta, double *d_y,
              int overwrite, void *stream);

/* Host-buffer convenience used by spx_matvec_* for vectors the library does
 * not own: H2D x (and y when beta matters), SpMV, D2H of the local y rows.
 * Synchronous. */
int csxb_spmv_host(csxb_matrix_t *m, double alpha, const double *h_x, double beta, double *h_y,
                   int overwrite);

/* ---- transposed product y = alpha * A^T * x (+ beta * y) ----------------------------
 * What BiCG, QMR, CGLS / LSQR and adjoint solves need next to A*x, without tuning A^T as a second matrix: the
 * transposed tables list the image y[col] += v * x[row] of every unit under the tiles of its columns and read the
 * values the forward product reads (set_entry updates reach both; only table bytes are added).
 *   prepare : builds and uploads the transposed tables (after csxb_upload; idempotent).  The first transposed product
 *             calls it; call it yourself to keep the set-up out of a timing.  Freed with the matrix.
 *   spmv_t  : d_x has nrows doubles, d_y ncols doubles.  overwrite as in csxb_spmv: every column of the window
 *             [CSXB_T_COL_LO, CSXB_T_COL_HI) is written exactly once (0 / beta*y where the column has no entry);
 *             other columns are not touched.  Asynchronous.  CSX-Sym: A^T = A, runs csxb_spmv (bit-identical).
 *   spmv_t_host : host buffers, unpipelined (x in, product, the window of y out).  Synchronous.
 * Partial handles (part_lo..part_hi, csxb_tune_csr_slab): the window is the columns the local partitions read and
 * y[c] = alpha * (A_local^T x)[c] + beta * y[c] there; summing the partials of all processes is the caller's job (as
 * for the CSX-Sym halo rows, CSXB_SYM_HALO_LO/HI).
 * csxb_transpose_info (after prepare, else -1): column window [LO, HI), device bytes of the transposed tables,
 * algorithmic bytes of one product with overwrite (values + tables read + 8*nrows for x + 8 per window column for y;
 * add 8 per window column when beta matters), kernels launched per product, heavy columns and their segments (columns
 * whose many single entries are summed by whole warps), host build time in microseconds.
 * csxb_decode_coords_t: parity aid; for every device-wide value index (partitions in order, as csxb_decode_coords
 * numbers them after each partition's value base) the (row, col) of A at which the transposed tables gather it.
 * A host walk of the host copy of the tables: needs no device and no upload. */
enum { CSXB_T_COL_LO = 0, CSXB_T_COL_HI = 1, CSXB_T_DEVICE_BYTES = 2, CSXB_T_ALG_BYTES = 3, CSXB_T_LAUNCHES = 4,
       CSXB_T_HEAVY_COLS = 5, CSXB_T_SEGMENTS = 6, CSXB_T_BUILD_US = 7 };
int csxb_transpose_prepare(csxb_matrix_t *m);
int csxb_spmv_t(csxb_matrix_t *m, double alpha, const double *d_x, double beta, double *d_y, int overwrite,
                void *stream);
int csxb_spmv_t_host(csxb_matrix_t *m, double alpha, const double *h_x, double beta, double *h_y, int overwrite);
int64_t csxb_transpose_info(const csxb_matrix_t *m, int what);
int csxb_decode_coords_t(const csxb_matrix_t *m, int32_t *rows, int32_t *cols);

/* ---- tuned-matrix container, single entries -------------------------------------
 * csxb_save / csxb_load replace SaveTuned / LoadTuned (src/internals/Facade.cpp,
 * CsxSaveRestore.hpp:77-370, a boost::archive) with a Boost-free container of the
 * CSX arrays (values, ctl, id_map, rows_info, dvalues, reduction map, options);
 * a loaded matrix is uploaded with csxb_upload like a freshly tuned one (the GPU
 * tables are rebuilt from ctl).  csxb_get_entry / csxb_set_entry replace GetValue /
 * SetValue (CsxGetSet.hpp:84-537): zero-based (row, col); return 0, 1 when the
 * entry is not stored (or the row is not local), < 0 on error.  set updates the
 * host copy and the device copy, so the next SpMV sees it without re-tuning. */
int csxb_save(csxb_matrix_t *m, const char *path);
csxb_matrix_t *csxb_load(const char *path, char *err, size_t errlen);
int csxb_get_entry(csxb_matrix_t *m, int64_t row, int64_t col, double *value);
int csxb_set_entry(csxb_matrix_t *m, int64_t row, int64_t col, double value);

/* ---- several GPUs behind one handle, one process ------------------------------------
 * Replaces the reference's worker-thread pool over the nr_threads partitions of one matrix (CsxKernels.cpp:35-129
 * MatVecMult / MatVecMult_sym, the CSX-Sym local buffers and their reduction, CsxSpmv.cpp:37-50): the partitions of a
 * tuned (or loaded) matrix that has not been uploaded are dealt out, in contiguous ranges, to the listed devices
 * (a device may be listed more than once: logical members on one GPU).  csxb_group_create consumes `whole` on success.
 * csxb_group_spmv: y = alpha*A*x (+ beta*y unless overwrite); x and y may be host, pinned, managed or device memory;
 * synchronous.  CSX-Sym: the sums for rows of lower members are added by their owners in member order (no atomics).
 * (Repeated SpMV with the exchange inside the kernels is csxb_xchg_*; this is the one-call form behind spx_matvec_*.) */
typedef struct csxb_group csxb_group_t;
csxb_group_t *csxb_group_create(csxb_matrix_t *whole, const int *devices, int ndev, int free_host, char *err, size_t errlen);
void csxb_group_destroy(csxb_group_t *g);
int csxb_group_size(const csxb_group_t *g);
csxb_matrix_t *csxb_group_member(csxb_group_t *g, int i);
int csxb_group_device(const csxb_group_t *g, int i);
int csxb_group_spmv(csxb_group_t *g, double alpha, const double *x, double beta, double *y, int overwrite);
/* y = alpha*A^T*x (+ beta*y unless overwrite): x has nrows, y ncols entries, same memory kinds as csxb_group_spmv;
 * synchronous.  Every member computes its partial over its column window; the partials are added in member order on
 * the first member's device (deterministic).  CSX-Sym: csxb_group_spmv. */
int csxb_group_spmv_t(csxb_group_t *g, double alpha, const double *x, double beta, double *y, int overwrite);
int csxb_group_save(csxb_group_t *g, const char *path);
int csxb_group_get_entry(csxb_group_t *g, int64_t row, int64_t col, double *value);
int csxb_group_set_entry(csxb_group_t *g, int64_t row, int64_t col, double value);
int csxb_group_set_perm(csxb_group_t *g, const int32_t *perm, int64_t n);

/* ---- reverse Cuthill-McKee reordering ------------------------------------------------
 * Replaces ReorderCSR (src/internals/Facade.cpp:56-69 -> Rcm.hpp:318-340 DoReorder_RCM, FindPerm :116-153 on
 * boost::cuthill_mckee_ordering).  Host code.  csxb_rcm_csr: zero-based square CSR; perm[old] = new (what
 * spx_mat_get_perm returns); bandwidth[0/1] (may be NULL) = bandwidth before / after.  Returns 0, 1 when the matrix
 * has no off-diagonal element ("no reordering available for this matrix", the input stays as it is), < 0 on bad
 * arguments.  csxb_rcm_edges: the same ordering for an explicit list of undirected edges (added in the given order); start >= 0
 * names the starting vertex of a connected graph (boost's cuthill_mckee_ordering(G, s, ...)), -1 lets the algorithm pick.
 * csxb_permute_csr: B = P A P^T into caller-allocated arrays of the same sizes (row i of B = row
 * inv_perm[i] of A, columns through perm, sorted; Rcm.hpp:289-316, Csr.hpp:270-360). */
int csxb_rcm_csr(const int32_t *rowptr, const int32_t *colind, int64_t nrows, int64_t ncols, int32_t *perm,
                 int64_t *bandwidth);
int csxb_rcm_edges(const int32_t *eu, const int32_t *ev, int64_t nedges, int64_t n, int64_t start, int32_t *perm,
                   int64_t *bandwidth);
/* The permutation is kept with the tuned matrix and stored by csxb_save (matvec.c:298, 422, 445).  get returns the
 * length (0 = none) and copies when perm is not NULL. */
int csxb_set_perm(csxb_matrix_t *m, const int32_t *perm, int64_t n);
int64_t csxb_get_perm(const csxb_matrix_t *m, int32_t *perm);
int csxb_permute_csr(const int32_t *rowptr, const int32_t *colind, const double *values, int64_t nrows,
                     const int32_t *perm, int32_t *out_rowptr, int32_t *out_colind, double *out_values);

/* ---- BLAS-1 on device-resident vectors -------------------------------------------
 * What a solver iteration needs next to the SpMV, so that it stays on the GPU
 * (VecScale / VecScaleAdd / VecAdd / VecSub / VecMult, src/internals/Vector.cpp:259-377).
 * Pointers are device-accessible (cudaMalloc or managed memory).
 *   axpby : out[i] = alpha*a[i] + beta*b[i]   (b may be NULL with beta ignored; out may alias a or b)
 *   dot   : *result = sum a[i]*b[i]           (synchronises `stream`; fixed reduction order) */
int csxb_vec_axpby(double *d_out, const double *d_a, const double *d_b, double alpha, double beta, int64_t n, void *stream);
int csxb_vec_dot(const double *d_a, const double *d_b, int64_t n, double *result, void *stream);

/* ---- repeated SpMV across GPUs, exchange over peer memory -------------------
 * Replaces the shared-memory x vector of the reference's thread pool
 * (CsxKernels.cpp:35-129: all threads read one x) for one process per GPU.
 * Every rank owns one partition (csxb_tune_* with part_lo = rank) and holds two
 * full-length vectors in a block the other ranks map through CUDA IPC.  Step k
 * computes vec[(k+1)&1][own rows] = alpha * A_local * vec[k&1]; the kernel
 * stores the rows that other ranks read (their column windows,
 * CSXB_P_COL_MIN/MAX) directly into their vectors over NVLink, and device-side
 * flags order the steps, so a step is kernel launches only (no host
 * synchronisation, CUDA-graph capturable).  CSX-Sym is not covered here.
 *   create  : after csxb_upload; allocates the block on the matrix's device
 *   handle  : 64-byte CUDA IPC handle of the block, to be all-gathered by the caller
 *   connect : handles = world * 64 bytes in rank order; row_lo/row_n = row range of every rank;
 *             win_lo/win_hi = first/last column every rank reads
 *   vector  : device pointer of vec[which]; fill vec[0] with the initial x (all columns the rank reads)
 *   spmv    : one step (asynchronous on `stream`).  The host alternates the two vectors from call to call, so a
 *             CUDA graph that is replayed must capture an even number of steps
 *   status  : what = 0 steps finished, 1 error word (non-zero: a wait for a neighbour timed out — device-side waits
 *             give up after about three seconds, so ranks have to issue their steps within that time of each other),
 *             2 protocol (1: edge tiles first — the tiles that touch other ranks run first in every step and
 *             publish it at once, nothing else waits; 0: one sync kernel at the end of every step), 3 edge tiles */
typedef struct csxb_xchg csxb_xchg_t;
csxb_xchg_t *csxb_xchg_create(csxb_matrix_t *m, int rank, int world);
int csxb_xchg_handle(csxb_xchg_t *x, void *handle64);
int csxb_xchg_connect(csxb_xchg_t *x, const void *handles, const int64_t *row_lo, const int64_t *row_n,
                      const int64_t *win_lo, const int64_t *win_hi);
/* Same plan for ranks that live in one process (peer access enabled by the caller, or one device): bases[q] =
 * csxb_xchg_base of rank q. */
int csxb_xchg_connect_ptr(csxb_xchg_t *x, void *const *bases, const int64_t *row_lo, const int64_t *row_n,
                          const int64_t *win_lo, const int64_t *win_hi);
void *csxb_xchg_base(csxb_xchg_t *x);
double *csxb_xchg_vector(csxb_xchg_t *x, int which);
int csxb_xchg_spmv(csxb_xchg_t *x, double alpha, void *stream);
int64_t csxb_xchg_status(csxb_xchg_t *x, int what);
void csxb_xchg_destroy(csxb_xchg_t *x);

/* Debug/parity aid: decode the device-side tables back into (row, col) pairs
 * in values order for partition `part` (0-based global coordinates), running
 * the same ctl walk the kernels use but on the host copy of the tables. */
int csxb_decode_coords(const csxb_matrix_t *m, int part, int32_t *rows, int32_t *cols);

#ifdef __cplusplus
}
#endif
#endif /* CSX_B200_H */
