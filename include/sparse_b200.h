/*
 * sparse_b200.h -- C ABI of libsparse_b200.so, the B200 (sm_100a) implementation
 * of pydata/sparse's data-parallel hot path.
 *
 * The reference has no C/FFI seam for this path: its "native" layer is a set of
 * numba-JIT closures called only from sparse/numba_backend/_common.py::_dot,
 * _umath.py::_Elemwise and _coo/core.py::_grouped_reduce.  Each entry point below
 * replaces one of those closures; the reference call site it substitutes is cited
 * on every declaration (paths relative to /root/reference/sparse/numba_backend/).
 *
 * Conventions
 *  - extern "C", plain pointers and sizes; no torch / Python / C++ types.
 *  - every function returns 0 on success, a negative b2s_status otherwise;
 *    b2s_last_error() returns a thread-local message for the last failure.
 *  - "_dev" pointers are device (HBM) pointers on the current CUDA device,
 *    "_host" pointers are host pointers.  `stream` is a cudaStream_t passed as
 *    void* (NULL = legacy default stream).  Calls are asynchronous on `stream`
 *    unless stated otherwise; functions that return a data-dependent size
 *    synchronise the stream once.
 *  - inputs are borrowed and never written; outputs are caller-allocated
 *    (the two-phase count -> fill pattern of the reference's own kernels,
 *    e.g. _csr_csr_count_nnz + _dot_csr_csr).
 *  - index arrays are int32 or int64 (`idx_bytes` = 4 or 8); value arrays are
 *    described by b2s_dtype.  Mixed-dtype products are promoted by the caller
 *    (the reference promotes to _dot_dtype(dt1, dt2), _common.py:635-636).
 *  - there is NO CPU fallback anywhere in this library.
 */
#ifndef SPARSE_B200_H_
#define SPARSE_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B2S_ABI_VERSION 1

typedef enum {
    B2S_OK = 0,
    B2S_ERR_INVALID = -1,     /* bad argument (dtype, alignment, negative size ...) */
    B2S_ERR_CUDA = -2,        /* a CUDA runtime call failed; see b2s_last_error()   */
    B2S_ERR_UNSUPPORTED = -3, /* dtype / op outside the supported matrix            */
    B2S_ERR_OVERFLOW = -4,    /* sizes do not fit the chosen index width            */
    B2S_ERR_NO_DEVICE = -5    /* no CUDA device visible                             */
} b2s_status;

typedef enum {
    B2S_F32 = 0, B2S_F64 = 1, B2S_I32 = 2, B2S_I64 = 3, B2S_BOOL = 4,
    /* storage-only integer widths: accepted by b2s_cast alone (every arithmetic entry point rejects them) */
    B2S_I8 = 5, B2S_I16 = 6, B2S_U8 = 7, B2S_U16 = 8, B2S_U32 = 9, B2S_U64 = 10
} b2s_dtype;

/* ---- runtime ---------------------------------------------------------- */
int b2s_abi_version(void);
const char *b2s_last_error(void);
int b2s_device_count(int *count);
/* name_buf may be NULL. sm = 10*major+minor (100 on B200). */
int b2s_device_info(int device, char *name_buf, size_t name_len, int *sm, int *n_sms, size_t *hbm_bytes,
                    size_t *l2_bytes);
int b2s_set_device(int device);
int b2s_malloc(void **dev_ptr, size_t nbytes);
int b2s_free(void *dev_ptr);
int b2s_host_register(void *host_ptr, size_t nbytes); /* pin caller memory so H2D/D2H run at link rate */
int b2s_host_unregister(void *host_ptr);
int b2s_memcpy_h2d(void *dst_dev, const void *src_host, size_t nbytes, void *stream);
int b2s_memcpy_d2h(void *dst_host, const void *src_dev, size_t nbytes, void *stream);
int b2s_memset(void *dst_dev, int value, size_t nbytes, void *stream);
int b2s_stream_sync(void *stream);
/* Number of kernels this library has launched since load (bench.py's gpu_launches). */
int64_t b2s_launch_count(void);

/* ---- CSR x dense -> dense (K1) ---------------------------------------- */
/*
 * Replaces _dot_csr_ndarray_type(dt1, dt2)(out_shape, a_data, a_indices, a_indptr, b)
 * (_common.py:720-755, called at _common.py:389 and :440): out[M,N] = CSR(A)[M,K] . B[K,N].
 * Bit-exact contract: every out[i,j] is accumulated in dtype arithmetic, in the
 * stored order of row i, product and sum rounded separately (no FMA), starting
 * from +0 -- the same operation sequence as the reference loop.
 * ldb / ldc are row strides in ELEMENTS (>= N).  Rows without entries are
 * written as zeros (out needs no pre-initialisation).
 */
int b2s_spmm_csr_dense(int dtype, int idx_bytes, int64_t M, int64_t K, int64_t N, const void *a_data_dev,
                       const void *a_indices_dev, const void *a_indptr_dev, const void *b_dev, int64_t ldb,
                       void *out_dev, int64_t ldc, void *stream);

/*
 * Same product through HOST buffers (the reference-facing call: numpy arrays in, numpy array out).
 * A three-stream pipeline overlaps the uploads of A (in nnz-balanced row chunks), K1 on the rows that have landed
 * and the download of finished rows of C; synchronous on return.  Host buffers should be pinned
 * (b2s_host_register) for full link rate.  a_indices/a_indptr have idx_bytes (8 = np.intp as the reference holds
 * them, narrowed to int32 on the device when K and nnz allow; 4 = int32, e.g. arrays that came from SciPy).
 */
int b2s_spmm_csr_dense_host(int dtype, int idx_bytes, int64_t M, int64_t K, int64_t N, int64_t nnz,
                            const void *a_data_host, const void *a_indices_host, const void *a_indptr_host,
                            const void *b_host, void *out_host);
/* Host threads that narrow int64 column indices to int32 into pinned staging before the upload of
 * b2s_spmm_csr_dense_host (-1 = auto, 0 = upload the raw int64 indices and narrow on the device). */
int b2s_spmm_host_set_threads(int n);
/* Pipeline shape of b2s_spmm_csr_dense_host: number of nnz-balanced row chunks and of pinned staging slots. */
int b2s_spmm_host_set_pipeline(int chunks, int slots);
/* The host-side narrowing step on its own (same thread pool): dst[i] = (int32) src[i]. */
int b2s_host_narrow_i64_i32(const int64_t *src_host, int32_t *dst_host, int64_t n);

/* 1 if every row of the CSR has non-decreasing column indices (precondition of the panel passes). Synchronises. */
int b2s_csr_rows_sorted(int idx_bytes, int64_t M, const void *indptr_dev, const void *indices_dev, int *sorted_host,
                        void *stream);
/*
 * K1 with explicit scheduling: n_panels <= 1 -> the one-pass kernel; n_panels >= 2 -> column-panel passes that keep
 * the active slice of B resident in L2 (rows must be sorted by column: rows_sorted = 1; bit-identical results);
 * n_panels == 0 -> choose from the size of B (~48 MB per panel) and nnz / M.  nnz < 0 = unknown.
 */
int b2s_spmm_csr_dense_ex(int dtype, int idx_bytes, int64_t M, int64_t K, int64_t N, int64_t nnz,
                          const void *a_data_dev, const void *a_indices_dev, const void *a_indptr_dev,
                          const void *b_dev, int64_t ldb, void *out_dev, int64_t ldc, int n_panels, int rows_sorted,
                          int long_rows, void *stream);
/* Largest number of stored entries in a row: callers enable `long_rows` (nnz-balanced mode: rows longer than
 * max(512, 4 x mean) go to the column-split shared-memory-ring kernel, run concurrently on a side stream) only for
 * matrices whose longest row exceeds max(512, 8 x mean). */
int b2s_csr_max_row_nnz(int idx_bytes, int64_t M, const void *indptr_dev, int64_t *max_host, void *stream);

/* Tuning knob for K1 (0 = default).  variant: 1 = register-staged LDG gather with DYNAMIC row assignment (persistent
 * warps draw rows from a counter; the default), 3 = the same gather on the static one-row-per-warp grid,
 * 2 = 1-D bulk-TMA (cp.async.bulk) gather through a shared-memory ring. */
int b2s_spmm_set_variant(int variant, int unroll);
/* process-wide default of the nnz-balanced long-row path used by b2s_spmm_csr_dense (default off; b2s_spmm_csr_dense_ex
 * selects it per call; results stay bit-identical). */
int b2s_spmm_set_skew(int enabled);


/* ---- streaming primitives (prims.cu): COO canonicalisation / format conversion ------------ */
/* linear_loc (_coo/common.py:56-64) with an arbitrary axis permutation folded into `strides_host`:
 * keys[i] = sum_d coords[d][i] * strides_host[d]. coords is [ndim, nnz] with row stride `row_stride` elements. */
int b2s_coo_linearize(int idx_bytes, int ndim, int64_t nnz, const void *coords_dev, int64_t row_stride,
                      const int64_t *strides_host, int64_t *keys_out_dev, void *stream);
/* trace selector of _einsum_single (_common.py:1378-1392): flags[i] = 1 iff coords[d][i] == coords[first_host[d]][i]
 * for every d (first_host[d] = first axis carrying the same subscript label, == d for unrepeated labels). */
int b2s_coo_diag_flags(int idx_bytes, int ndim, int64_t nnz, const void *coords_dev, int64_t row_stride,
                       const int32_t *first_host, uint8_t *flags_out_dev, void *stream);
/* basic indexing x[ints / slices] (_coo/indexing.py:12-133: _mask + the coordinate transform `(c - start) // step`).
 * keys_dev: C-order linear keys over shape_host.  Axis d keeps coordinate c iff c = start + j*step for some
 * 0 <= j < count (an integer index is start = i, step = 1, count = 1); flags[i] = all axes keep, and
 * keys_out[i] = sum_d j_d * out_stride_host[d] (out_stride 0 drops the axis).  Compaction is the caller's. */
int b2s_coo_slice_keys(int ndim, int64_t nnz, const int64_t *keys_dev, const int64_t *shape_host,
                       const int64_t *start_host, const int64_t *step_host, const int64_t *count_host,
                       const int64_t *out_stride_host, uint8_t *flags_out_dev, int64_t *keys_out_dev, void *stream);
/* inverse of linear_loc for C-order `shape_host`; writes coords [ndim, nnz] of width idx_bytes. */
int b2s_coo_unravel(int idx_bytes, int ndim, int64_t nnz, const int64_t *keys_dev, const int64_t *shape_host,
                    void *coords_out_dev, int64_t row_stride, void *stream);
/* COO._sort_indices' test `(np.diff(linear) >= 0).all()` and _sum_duplicates' uniqueness test
 * (_coo/core.py:1310-1313, 1340-1343). Synchronises the stream. */
int b2s_keys_flags(const int64_t *keys_dev, int64_t n, int *unsorted_host, int *has_dups_host, void *stream);
/* stable argsort of non-negative int64 keys over their low `key_bits` bits (np.argsort(kind="mergesort"),
 * _coo/core.py:1315): keys_out = sorted keys, perm_out = source positions. */
int b2s_sort_keys(const int64_t *keys_in_dev, int64_t n, int key_bits, int64_t *keys_out_dev, int64_t *perm_out_dev,
                  void *stream);
/* Element movers (gather, compact, scatter, fill, flag_not_fill, transpose_dense): elem_bytes = 1, 2, 4, 8 or 16 -- they
 * move and compare raw bits, so every value dtype a container can hold passes through them (complex128 = 16 bytes). */
int b2s_gather(int elem_bytes, const void *in_dev, const int64_t *perm_dev, int64_t n, void *out_dev, void *stream);
int b2s_flag_heads(const int64_t *keys_dev, int64_t n, uint8_t *flags_out_dev, void *stream);
/* keep-flags of COO._prune / GCXS._prune: bits(data[i]) != bits(fill) (`equivalent`, _utils.py:448-452). */
int b2s_flag_not_fill(int elem_bytes, const void *data_dev, int64_t n, const void *fill_host, uint8_t *flags_out_dev,
                      void *stream);
/* exclusive scan of 0/1 flags; returns the number of set flags on the host (synchronises). */
int b2s_scan_flags(const uint8_t *flags_dev, int64_t n, int64_t *pos_out_dev, int64_t *total_host, void *stream);
int b2s_exclusive_scan_i64(const int64_t *in_dev, int64_t n, int64_t *out_dev, void *stream);
int b2s_compact(int elem_bytes, const void *in_dev, const uint8_t *flags_dev, const int64_t *pos_dev, int64_t n,
                void *out_dev, void *stream);
int b2s_compact_rows(int elem_bytes, int nrows, const void *in_dev, int64_t in_stride, const uint8_t *flags_dev,
                     const int64_t *pos_dev, int64_t n, void *out_dev, int64_t out_stride, void *stream);
/* COO._sum_duplicates (np.add.reduceat over runs, _coo/core.py:1350): out[pos[i]] = sum of the run headed at i. */
int b2s_segment_sum(int dtype, const void *data_dev, const uint8_t *heads_dev, const int64_t *pos_dev, int64_t n,
                    void *out_dev, void *stream);
/* bincount + cumsum of _from_coo (_compressed/compressed.py:72-74) and of _dot's COO branch (_common.py:452-458). */
int b2s_indptr_from_sorted(int in_idx_bytes, const void *rows_dev, int64_t n, int64_t nrows, int out_idx_bytes,
                           void *indptr_out_dev, void *stream);
/* sorted 2-D linear keys -> (rows?, indices, indptr?) of the compressed (nrows x ncols) view (_from_coo :66-75). */
int b2s_csr_from_keys(const int64_t *keys_dev, int64_t n, int64_t nrows, int64_t ncols, int out_idx_bytes,
                      void *rows_out_dev_or_null, void *indices_out_dev, void *indptr_out_dev, void *stream);
/* uncompress_dimension (_compressed/convert.py:81-87). */
int b2s_rows_from_indptr(int in_idx_bytes, const void *indptr_dev, int64_t nrows, int out_idx_bytes,
                         void *rows_out_dev, void *stream);
/* todense (COO.todense, _coo/core.py): out[keys[i]] = data[i] over a buffer pre-filled with the fill value. */
int b2s_scatter(int elem_bytes, const void *data_dev, const int64_t *keys_dev, int64_t n, void *out_dev, void *stream);
int b2s_fill(int elem_bytes, void *out_dev, int64_t n, const void *value_host, void *stream);
int b2s_cast(int src_dtype, int dst_dtype, const void *in_dev, int64_t n, void *out_dev, void *stream);
int b2s_transpose_dense(int elem_bytes, const void *in_dev, int64_t rows, int64_t cols, int64_t ld_in, void *out_dev,
                        int64_t ld_out, void *stream);
/* nan_check (_common.py:51-69), used for matmul's RuntimeWarning. Synchronises. */
int b2s_any_nan(int dtype, const void *data_dev, int64_t n, int *result_host, void *stream);

/* ---- CSR x CSR -> CSR / COO x COO -> COO (K4, spgemm.cu) ---------------------------------- */
/*
 * Replaces _dot_csr_csr_type(dt1,dt2)(out_shape, a_data, b_data, a_indices, b_indices, a_indptr, b_indptr)
 * (_common.py:639-717, called at :359-373) and _dot_coo_coo (:907-976, called at :459-461).
 * begin(): runs the whole numeric product (one pass over the products, warp per row, shared-memory hash) into an
 * upper-bound layout and returns the structural nnz and the nnz after dropping sums bitwise equal to +0 -- the count
 * pass of the reference (_csr_csr_count_nnz, :543-570) is not a separate pass here.  finish(): compacts into
 * caller-allocated outputs (indptr[M+1] or NULL, indices[nnz], rows[nnz] or NULL, data[nnz]) and frees the plan.
 * sorted_order = 0: reverse-first-touch column order per row, bit-identical to the reference's linked list
 * (incl. the all-dense row flip); 1: ascending columns (canonical COO order).
 * wide_accumulate = 1: float64 accumulator and "skip if sum == 0" of _dot_csc_ndarray_sparse (:835, :852).
 */
int b2s_spgemm_begin(int dtype, int idx_bytes, int64_t M, int64_t K, int64_t n_col, const void *a_indptr_dev,
                     const void *a_indices_dev, const void *a_data_dev, const void *b_indptr_dev,
                     const void *b_indices_dev, const void *b_data_dev, int sorted_order, int wide_accumulate,
                     void **plan_out, int64_t *nnz_struct_out, int64_t *nnz_pruned_out, void *stream);
int b2s_spgemm_finish(void *plan, int prune, int64_t *indptr_out_dev, int64_t *indices_out_dev,
                      int64_t *rows_out_dev, void *data_out_dev);
int b2s_spgemm_abort(void *plan);
/* test hook: rows with more than t1 (<= 256) products take the CTA-per-row path */
int b2s_spgemm_set_thresholds(int64_t t0, int64_t t1);

/* ---- sparse-output sparse x dense (K3, spmm_sparse.cu) ------------------------------------ */
/* _dot_csr_ndarray_sparse arithmetic (_common.py:758-804): product rounded to dtype, running sum in the type
 * numba unifies `val = 0` with (f64 for floats, i64 for ints); flags[i,j] = structural test of
 * _csr_ndarray_count_nnz (:573-600).  out and flags are dense (M x N, contiguous). */
int b2s_spmm_csr_dense_flagged(int dtype, int idx_bytes, int64_t M, int64_t K, int64_t N, const void *a_data_dev,
                               const void *a_indices_dev, const void *a_indptr_dev, const void *b_dev, int64_t ldb,
                               void *out_dev, uint8_t *flags_out_dev, void *stream);
/* dense (M x N) -> CSR/COO entries.  flags_or_null: externally computed keep flags; else mode 0: x != 0
 * (`if data_curr != 0`, _common.py:1062,1149), mode 1: bits(x) != bits(+0) (prune). */
int b2s_dense_to_csr_begin(int dtype, int64_t M, int64_t N, const void *x_dev, const uint8_t *flags_or_null_dev,
                           int mode, void **plan_out, int64_t *nnz_out, void *stream);
int b2s_dense_to_csr_finish(void *plan, int64_t *rows_out_or_null_dev, int64_t *cols_out_dev, void *data_out_dev,
                            int64_t *indptr_out_or_null_dev);
/* GCXS._prune's indptr rebuild (_compressed/compressed.py:836-842): new_indptr[r] = pos[old_indptr[r]]. */
int b2s_indptr_remap(int idx_bytes, const void *old_indptr_dev, int64_t nrows, const int64_t *pos_dev, int64_t n,
                     int64_t total, void *new_indptr_dev, void *stream);

/* ---- broadcasting element-wise coiteration (K5, elemwise.cu) ------------------------------ */
/* Operator codes: binary 0..13 value ops (add sub mul div maximum minimum fmax fmin pow floordiv mod band bor bxor),
 * 14 nan_replace, 15 / 16 the two selections of a three-operand where, 17 OR of the raw bit patterns, 18 left_shift and
 * 19 right_shift (integers; a count outside [0, bits) gives 0, or -1 for a negative value shifted right, as NumPy),
 * 32..40 predicates (gt ge lt le eq ne land lor lxor); unary 0..31 value ops, 64..68 predicates (see elemwise.cu). */
/* Replaces _Elemwise._match_coo + _match_arrays + _get_func_coords_data (_umath.py:656-751, 53-92, 576-654) for two
 * COO operands: merge-path union of two sorted key streams, each optionally expanded virtually by a trailing
 * broadcast factor R; the operator is applied and results equal to the output fill value are dropped in the same
 * pass.  SINGLE pass (decoupled look-back instead of count + scan + emit): the caller passes output buffers with room
 * for `capacity` >= na*Ra + nb*Rb entries (the union can never be larger); kept (key, value) pairs are written
 * densely from offset 0 in key order and their number is returned in *nnz_out (synchronises the stream once).
 * Coordinates are b2s_coo_unravel of the keys. */
int b2s_ew_merge_single(int dtype, int op, const int64_t *keys_a_dev, const void *data_a_dev, int64_t na, int64_t Ra,
                        const int64_t *keys_b_dev, const void *data_b_dev, int64_t nb, int64_t Rb,
                        const void *fill_a_host, const void *fill_b_host, const void *out_fill_host, int64_t capacity,
                        void *vals_out_dev, int64_t *keys_out_dev, int64_t *nnz_out, void *stream);
/* COO (x) scalar (mode 0: f(x,s), 1: f(s,x)) and unary maps (mode 2). */
int b2s_ew_map(int dtype, int op, int mode, const void *x_dev, int64_t n, const void *scalar_host,
               const void *out_fill_host, void *out_vals_dev, uint8_t *out_flags_dev, void *stream);
/* COO (x) dense ndarray: the mask (True, None) branch, np.broadcast_to(arg, shape)[coords] (_umath.py:606-608). */
int b2s_ew_dense(int dtype, int op, int swap, const int64_t *keys_a_dev, const void *data_a_dev, int64_t na,
                 int64_t Ra, const void *dense_dev, int ndim, const int64_t *shape_host,
                 const int64_t *dense_strides_host, const void *out_fill_host, int64_t *out_keys_dev,
                 void *out_vals_dev, uint8_t *out_flags_dev, void *stream);
/* _get_expanded_coords_data (_umath.py:220-277) for arbitrary broadcast axes: n*R (key, source index) pairs. */
int b2s_ew_expand(int idx_bytes, const void *coords_dev, int64_t row_stride, int64_t n, int ndim,
                  const int64_t *result_shape_host, const int32_t *is_bcast_host, const int32_t *src_row_host,
                  int64_t *out_keys_dev, int64_t *out_src_dev, void *stream);

/* ---- grouped reductions (K7, reduce_fused.cu) ------------------------------------------------ */
/* Operator codes: 0 add, 1 multiply, 2 maximum, 3 minimum, 4 logical_and, 5 logical_or, 6..8 bitwise and/or/xor.
 * Replaces _grouped_reduce = _calc_counts_invidx + ufunc.reduceat (_coo/core.py:1601-1661). */
/* Hand-written SINGLE-pass segmented-scan reduction (reduce_fused.cu; replaces _grouped_reduce / _calc_counts_invidx +
 * ufunc.reduceat, _coo/core.py:1601-1661, and the fill-value correction of _sparse_array.py:405-422): runs of equal
 * group id (= key / ncols) of the sorted keys are reduced with `op` (0 add, 1 mul, 2 max, 3 min, 4 and, 5 or, 6 band,
 * 7 bor, 8 bxor, 9 fmax, 10 fmin); group ids (= linear index over the kept axes) and values are written densely from
 * offset 0 into caller buffers of `capacity` >= n entries; tile carries come from a decoupled look-back.  Returns the
 * number of groups and how many results are bitwise equal to result_fill (so the prune compaction of
 * _coo/core.py:713-723 can be skipped when 0).  Synchronises the stream once. */
int b2s_reduce_single(int dtype, int op, const int64_t *keys_dev, const void *vals_dev, int64_t n, int64_t ncols,
                      const void *fill_host, int apply_fill_fix, const void *result_fill_host, int64_t capacity,
                      int64_t *gid_out_dev, void *vals_out_dev, int64_t *n_groups_out, int64_t *n_equal_fill_out,
                      void *stream);

/* test hook: 0 = choose the form of b2s_reduce_single by ncols (count / scan / emit without inter-tile communication
 * when a run cannot be longer than one tile, single-pass look-back otherwise), 1 / 2 = force one of them */
int b2s_reduce_set_form(int form);

/* ---- fused example paths (K8 / K9, fused.cu) ---------------------------------------------- */
/* examples/sddmm_example.py:51-52  s * (a @ b): out_vals[p] = s_vals[p] * dot(A[i_p,:], Bt[j_p,:]). */
int b2s_sddmm(int dtype, int idx_bytes, int64_t M, int64_t N, int64_t K, const void *indptr_dev,
              const void *cols_dev, const void *s_vals_dev, const void *a_dev, int64_t lda, const void *bt_dev,
              int64_t ldbt, void *out_vals_dev, void *stream);
/* examples/mttkrp_example.py:51-52: out[i,j] = sum_{k,l} B[i,k,l] * D[l,j] * C[k,j]. */
int b2s_mttkrp(int dtype, int idx_bytes, int64_t I_, int64_t J, const void *indptr_dev, const void *k_dev,
               const void *l_dev, const void *vals_dev, const void *d_dev, int64_t ldd, const void *c_dev, int64_t ldc,
               void *out_dev, int64_t ldo, void *stream);

/* ---- masked sparse product (K10, masked_spgemm.cu) ----------------------------------------- */
/* examples/triangles_example.py `a @ a * a`, i.e. s * (a @ b) with sparse a and b, without forming a @ b:
 * out_vals[p] = s_vals[p] * sum_k A[i_p,k] * Bt[j_p,k] over the k stored in both rows, summed in ascending k.  S, A and
 * Bt (b compressed by column) are CSR with sorted rows; s_vals / out_vals are dtype_out, a_data / bt_data dtype_ab.
 * Pairs (dtype_ab, dtype_out): (F32,F32) (F32,F64) (F64,F64) (I64,I64) (I64,F64) (BOOL, BOOL|I64|F32|F64). */
int b2s_masked_spgemm(int dtype_ab, int dtype_out, int idx_bytes, int64_t M, int64_t N, int64_t K,
                      const void *s_indptr_dev, const void *s_cols_dev, const void *s_vals_dev,
                      const void *a_indptr_dev, const void *a_indices_dev, const void *a_data_dev,
                      const void *bt_indptr_dev, const void *bt_indices_dev, const void *bt_data_dev,
                      void *out_vals_dev, void *stream);

/* ---- copy-engine exchange of a row-sharded dense operand (peer.cu; SURVEY.md s8(e), no reference counterpart: the
 * reference is single-process) ------------------------------------------------------------------------------------
 * b2s_peer_alloc: cudaMalloc'ed (IPC-exportable) device buffer; b2s_peer_export writes its 64-byte CUDA IPC handle;
 * b2s_peer_open maps a peer process's buffer (peer access enabled lazily); b2s_peer_gather copies every rank's shard
 * (shards_dev[r], r = 0..world-1, entry `rank` = the local shard) to dst_full_dev + r*shard_bytes with
 * cudaMemcpyAsync -- DMA over NVLink, no kernel, no SM taken from the product kernel it overlaps -- round-robin over
 * `streams`, starting at rank+1. */
int b2s_peer_alloc(void **dev_ptr, int64_t nbytes);
int b2s_peer_free(void *dev_ptr);
int b2s_peer_export(void *dev_ptr, void *handle64);
int b2s_peer_open(const void *handle64, void **dev_ptr);
int b2s_peer_close(void *dev_ptr);
int b2s_peer_gather(void *dst_full_dev, const void *const *shards_dev, int world, int rank, int64_t shard_bytes,
                    void *const *streams, int n_streams);

#ifdef __cplusplus
}
#endif
#endif /* SPARSE_B200_H_ */
