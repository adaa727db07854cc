/* sparsex/matvec.h — matrix, vector and SpMV routines of the drop-in API.
 * Names, argument meaning and error behaviour follow
 * include/sparsex/matvec.h:39-535 and src/api/matvec.c of SparseX; the
 * implementation (sparsex_b200/csrc/api.cpp) runs the SpMV on a B200. */
#ifndef SPARSEX_MATVEC_H
#define SPARSEX_MATVEC_H

#include <sparsex/common.h>

#ifdef __cplusplus
extern "C" {
#endif

/* input: CSR arrays are wrapped, not copied, and must outlive spx_mat_tune().
 * As in the reference, the optional indexing argument is ignored: CSR input is
 * always zero-based (matvec.c:171-177). */
spx_input_t *spx_input_load_csr(const spx_index_t *rowptr, const spx_index_t *colind, const spx_value_t *values,
                                spx_index_t nr_rows, spx_index_t nr_cols, ...);
spx_input_t *spx_input_load_mmf(const char *filename);
spx_error_t spx_input_destroy(spx_input_t *input);

/* tuning: CSX / CSX-Sym encoding + upload to the GPU.  Options are read from
 * the global property map (spx_option_set). */
spx_matrix_t *spx_mat_tune(spx_input_t *input, ...);
spx_error_t spx_mat_get_entry(const spx_matrix_t *A, spx_index_t row, spx_index_t column, spx_value_t *value, ...);
spx_error_t spx_mat_set_entry(spx_matrix_t *A, spx_index_t row, spx_index_t column, spx_value_t value, ...);
spx_error_t spx_mat_save(const spx_matrix_t *A, const char *filename);
spx_matrix_t *spx_mat_restore(const char *filename);
spx_index_t spx_mat_get_nrows(const spx_matrix_t *A);
spx_index_t spx_mat_get_ncols(const spx_matrix_t *A);
spx_index_t spx_mat_get_nnz(const spx_matrix_t *A);
spx_partition_t *spx_mat_get_partition(const spx_matrix_t *A);
spx_index_t *spx_partition_get_rs(const spx_partition_t *p);
spx_index_t *spx_partition_get_re(const spx_partition_t *p);
spx_perm_t *spx_mat_get_perm(const spx_matrix_t *A);

/* y <- alpha*A*x */
spx_error_t spx_matvec_mult(spx_value_t alpha, const spx_matrix_t *A, const spx_vector_t *x, spx_vector_t *y);
/* y <- alpha*A*x + beta*y */
spx_error_t spx_matvec_kernel(spx_value_t alpha, const spx_matrix_t *A, const spx_vector_t *x, spx_value_t beta,
                              spx_vector_t *y);
spx_error_t spx_matvec_kernel_csr(spx_matrix_t **A, spx_index_t nr_rows, spx_index_t nr_cols,
                                  const spx_index_t *rowptr, const spx_index_t *colind, const spx_value_t *values,
                                  spx_value_t alpha, const spx_vector_t *x, spx_value_t beta, spx_vector_t *y);
spx_error_t spx_mat_destroy(spx_matrix_t *A);

spx_partition_t *spx_partition_csr(const spx_index_t *rowptr, spx_index_t nr_rows, size_t nr_threads);
spx_error_t spx_partition_destroy(spx_partition_t *p);

void spx_option_set(const char *option, const char *string);
void spx_options_set_from_env(void);

spx_vector_t *spx_vec_create(size_t size, const spx_partition_t *p);
spx_vector_t *spx_vec_create_from_buff(spx_value_t *buff, spx_value_t **tuned, size_t size, const spx_partition_t *p,
                                       spx_vecmode_t mode);
spx_vector_t *spx_vec_create_random(size_t size, const spx_partition_t *p);
void spx_vec_init(spx_vector_t *v, spx_value_t val);
void spx_vec_init_part(spx_vector_t *v, spx_value_t val, spx_index_t start, spx_index_t end);
void spx_vec_init_rand_range(spx_vector_t *v, spx_value_t max, spx_value_t min);
spx_error_t spx_vec_set_entry(spx_vector_t *v, spx_index_t idx, spx_value_t val, ...);
void spx_vec_scale(spx_vector_t *v1, spx_vector_t *v2, spx_value_t num);
void spx_vec_scale_add(spx_vector_t *v1, spx_vector_t *v2, spx_vector_t *v3, spx_value_t num);
void spx_vec_scale_add_part(spx_vector_t *v1, spx_vector_t *v2, spx_vector_t *v3, spx_value_t num,
                            spx_index_t start, spx_index_t end);
void spx_vec_add(spx_vector_t *v1, spx_vector_t *v2, spx_vector_t *v3);
void spx_vec_add_part(spx_vector_t *v1, spx_vector_t *v2, spx_vector_t *v3, spx_index_t start, spx_index_t end);
void spx_vec_sub(spx_vector_t *v1, spx_vector_t *v2, spx_vector_t *v3);
void spx_vec_sub_part(spx_vector_t *v1, spx_vector_t *v2, spx_vector_t *v3, spx_index_t start, spx_index_t end);
spx_value_t spx_vec_mul(const spx_vector_t *v1, const spx_vector_t *v2);
spx_value_t spx_vec_mul_part(const spx_vector_t *v1, const spx_vector_t *v2, spx_index_t start, spx_index_t end);
spx_error_t spx_vec_reorder(spx_vector_t *v, spx_perm_t *p);
spx_error_t spx_vec_inv_reorder(spx_vector_t *v, spx_perm_t *p);
void spx_vec_copy(const spx_vector_t *v1, spx_vector_t *v2);
int spx_vec_compare(const spx_vector_t *v1, const spx_vector_t *v2);
void spx_vec_print(const spx_vector_t *v);
void spx_vec_destroy(spx_vector_t *v);

/* ---- engine additions (not in the reference API) ------------------------ */
/* The csxb_matrix_t (include/csx_b200.h) behind a tuned matrix: CSX arrays,
 * side tables, traffic figures. */
struct csxb_matrix;
struct csxb_matrix *spx_mat_get_engine(const spx_matrix_t *A);
/* Transposed product, y = alpha * A^T * x and y = alpha * A^T * x + beta * y: x has nrows and y ncols entries
 * (SPX_ERR_DIM otherwise).  Same vectors, groups and asynchrony as spx_matvec_mult / spx_matvec_kernel; an
 * SPX_MAT_REORDER matrix works in the permuted numbering, as they do.  The values are the forward product's, so
 * spx_mat_set_entry updates reach both. */
spx_error_t spx_matvec_mult_trans(spx_value_t alpha, const spx_matrix_t *A, const spx_vector_t *x, spx_vector_t *y);
spx_error_t spx_matvec_kernel_trans(spx_value_t alpha, const spx_matrix_t *A, const spx_vector_t *x, spx_value_t beta,
                                    spx_vector_t *y);
/* Block until all SpMVs issued on library vectors have completed. */
void spx_device_synchronize(void);

#ifdef __cplusplus
}
#endif
#endif /* SPARSEX_MATVEC_H */
