/*
 * libxsmm_b200.h -- stream-ordered, device-pointer entry points of the B200-native SPMDM/FSSPMDM
 * library (libxsmm_b200.so) plus a few service calls.  These are ADDITIONS to the reference
 * interface declared in libxsmm_spmdm.h / libxsmm_fsspmdm.h: one call covers the whole problem
 * (all createSparseSlice blocks / all compute blocks) and is asynchronous on `stream`.
 * `stream` is a cudaStream_t passed as void* so that this header needs no CUDA headers.
 */
#ifndef LIBXSMM_B200_H
#define LIBXSMM_B200_H

#include <stddef.h>
#include "libxsmm_spmdm.h"
#include "libxsmm_fsspmdm.h"

/* All block ids of reference samples/spmdm/spmdm.c:100-104 in one launch.  d_a is a DEVICE pointer. */
LIBXSMM_API void libxsmm_spmdm_createSparseSlice_fp32_stream(const libxsmm_spmdm_handle* handle, char transa,
  const float* d_a, libxsmm_CSR_sparseslice* libxsmm_output_csr_a, void* stream);
LIBXSMM_API void libxsmm_spmdm_createSparseSlice_bfloat16_stream(const libxsmm_spmdm_handle* handle, char transa,
  const libxsmm_bfloat16* d_a, libxsmm_CSR_sparseslice* libxsmm_output_csr_a, void* stream);

/* A (M x K, the handle's shape) in CSR form: row_ptr[M + 1], col_idx[nnz], values[nnz], all DEVICE pointers, 0-based,
 * column indices strictly ascending within each row.  Fills the handle's slices exactly as createSparseSlice_*_stream would
 * for the dense matrix holding these entries (transa = 'N'); asynchronous on stream.  The compute entries then take the
 * slices unchanged.  Errors (sticky, nothing launched): -90 NULL row_ptr, or NULL col_idx / values with nnz > 0;
 * -91 nnz < 0 or nnz > 2^32 - 1.  Malformed arrays on the device give unspecified slices, never writes outside them. */
LIBXSMM_API void libxsmm_spmdm_createSparseSlice_csr_fp32_stream(const libxsmm_spmdm_handle* handle,
  const unsigned int* d_row_ptr, const unsigned int* d_col_idx, const float* d_values, long long nnz,
  libxsmm_CSR_sparseslice* libxsmm_output_csr_a, void* stream);
LIBXSMM_API void libxsmm_spmdm_createSparseSlice_csr_bfloat16_stream(const libxsmm_spmdm_handle* handle,
  const unsigned int* d_row_ptr, const unsigned int* d_col_idx, const libxsmm_bfloat16* d_values, long long nnz,
  libxsmm_CSR_sparseslice* libxsmm_output_csr_a, void* stream);

/* A (M x K, the handle's shape) in CSC form: col_ptr[K + 1], row_idx[nnz], values[nnz], all DEVICE pointers, 0-based, row
 * indices strictly ascending within each column.  These are also the CSR arrays of A stored K x M (a kernel kept as
 * in x out and multiplied with transpose_a).  Fills the handle's slices exactly as createSparseSlice_*_stream would with
 * transa = 'T' for the K x M array holding these entries, and as the CSR entry would for A's CSR arrays; asynchronous on
 * stream.  The compute entries then take the slices unchanged.  Errors (sticky, nothing launched): -90 NULL col_ptr, or NULL
 * row_idx / values with nnz > 0; -91 nnz < 0 or nnz > 2^32 - 1.  Malformed arrays on the device give unspecified slices,
 * never writes outside them. */
LIBXSMM_API void libxsmm_spmdm_createSparseSlice_csc_fp32_stream(const libxsmm_spmdm_handle* handle,
  const unsigned int* d_col_ptr, const unsigned int* d_row_idx, const float* d_values, long long nnz,
  libxsmm_CSR_sparseslice* libxsmm_output_csr_a, void* stream);
LIBXSMM_API void libxsmm_spmdm_createSparseSlice_csc_bfloat16_stream(const libxsmm_spmdm_handle* handle,
  const unsigned int* d_col_ptr, const unsigned int* d_row_idx, const libxsmm_bfloat16* d_values, long long nnz,
  libxsmm_CSR_sparseslice* libxsmm_output_csr_a, void* stream);

/* All block ids of reference samples/spmdm/spmdm.c:106-110 in one launch.  d_b, d_c are DEVICE pointers;
 * alpha and beta are HOST pointers read at call time (alpha is ignored like in the reference). */
LIBXSMM_API void libxsmm_spmdm_compute_fp32_stream(const libxsmm_spmdm_handle* handle, char transa, char transb,
  const float* alpha, libxsmm_CSR_sparseslice* a_sparse, const float* d_b, char transc, const float* beta,
  float* d_c, void* stream);
LIBXSMM_API void libxsmm_spmdm_compute_bfloat16_stream(const libxsmm_spmdm_handle* handle, char transa, char transb,
  const libxsmm_bfloat16* alpha, libxsmm_CSR_sparseslice* a_sparse, const libxsmm_bfloat16* d_b, char transc,
  const libxsmm_bfloat16* beta, float* d_c, void* stream);

/* Whole multiply with HOST buffers: copies A and B (and C if *beta != 0) to the device, slices,
 * multiplies and copies C back; returns when C is complete.  This is what one repetition of the
 * reference sample does (samples/spmdm/spmdm.c:88-111).  datatype selects the element type of a, b
 * (the reference never fills handle->datatype, so it is an argument here); beta points at a float
 * (F32) or at a libxsmm_bfloat16 bit pattern (BFLOAT16).  Host buffers should be page-locked
 * (libxsmm_b200_host_alloc) for full PCIe speed; pageable memory works but is slower. */
LIBXSMM_API void libxsmm_spmdm_exec_host(const libxsmm_spmdm_handle* handle, libxsmm_CSR_sparseslice* slices,
  libxsmm_spmdm_datatype datatype, char transa, char transb, char transc, const void* a, const void* b,
  const void* beta, float* c);
/* Same two phases on DEVICE matrices, asynchronous on stream (slice creation, then compute). */
LIBXSMM_API void libxsmm_spmdm_exec_stream(const libxsmm_spmdm_handle* handle, libxsmm_CSR_sparseslice* slices,
  libxsmm_spmdm_datatype datatype, char transa, char transb, char transc, const void* d_a, const void* d_b,
  const void* beta, float* d_c, void* stream);

/* execute() on DEVICE pointers, asynchronous on stream (reference src/libxsmm_fsspmdm.c:260-291). */
LIBXSMM_API void libxsmm_dfsspmdm_execute_stream(const libxsmm_dfsspmdm* handle, const double* d_B, double* d_C, void* stream);
LIBXSMM_API void libxsmm_sfsspmdm_execute_stream(const libxsmm_sfsspmdm* handle, const float* d_B, float* d_C, void* stream);

/* 1 if the reference would have taken its sparse_reg branch for this operator (rows without
 * nonzeros are then left untouched, reference src/generator_spgemm_csr_asparse_reg.c:229,287). */
LIBXSMM_API int libxsmm_dfsspmdm_is_sparse(const libxsmm_dfsspmdm* handle);
LIBXSMM_API int libxsmm_sfsspmdm_is_sparse(const libxsmm_sfsspmdm* handle);
/* 1 if the operator was baked into a specialised kernel at create time, 0 = generic kernel. */
LIBXSMM_API int libxsmm_dfsspmdm_is_baked(const libxsmm_dfsspmdm* handle);
LIBXSMM_API int libxsmm_sfsspmdm_is_baked(const libxsmm_sfsspmdm* handle);
/* 1 if execute() of this float operator runs on the tensor cores (dense operators; the reference's dense
 * SMM branch, src/libxsmm_fsspmdm.c:240-248). */
LIBXSMM_API int libxsmm_sfsspmdm_is_tensor_core(const libxsmm_sfsspmdm* handle);

/* Sticky error state (the reference entry points return void and are mute unless LIBXSMM_VERBOSE). */
LIBXSMM_API int libxsmm_b200_last_error(void);
LIBXSMM_API const char* libxsmm_b200_last_error_string(void);
LIBXSMM_API void libxsmm_b200_clear_error(void);

/* Number of kernels this library has launched so far in this process. */
LIBXSMM_API unsigned long long libxsmm_b200_launch_count(void);
/* name of the kernel the last spmdm compute / fsspmdm execute call enqueued for the bulk of its work (static string) */
LIBXSMM_API const char* libxsmm_b200_last_compute_kernel(void);

/* Page-locked host memory for callers that want full PCIe speed on the host-pointer paths. */
LIBXSMM_API void* libxsmm_b200_host_alloc(size_t bytes);
LIBXSMM_API void libxsmm_b200_host_free(void* p);

/* Thin device-memory helpers so that C callers and the test harness need no CUDA headers. */
LIBXSMM_API void* libxsmm_b200_device_alloc(size_t bytes);
LIBXSMM_API void libxsmm_b200_device_free(void* p);
LIBXSMM_API int libxsmm_b200_memcpy_h2d(void* dst_device, const void* src_host, size_t bytes);
LIBXSMM_API int libxsmm_b200_memcpy_d2h(void* dst_host, const void* src_device, size_t bytes);
LIBXSMM_API int libxsmm_b200_memset(void* dst_device, int value, size_t bytes);
LIBXSMM_API int libxsmm_b200_synchronize(void);
LIBXSMM_API int libxsmm_b200_device_count(void);
LIBXSMM_API int libxsmm_b200_set_device(int device);

/* Streams, events, asynchronous copies and graph capture, again so that plain C callers (and the
 * ctypes harness) can drive the stream entries without CUDA headers.  A stream/event/graph is an
 * opaque pointer (cudaStream_t / cudaEvent_t / cudaGraphExec_t underneath). */
LIBXSMM_API void* libxsmm_b200_stream_create(void);
LIBXSMM_API void libxsmm_b200_stream_destroy(void* stream);
LIBXSMM_API int libxsmm_b200_stream_synchronize(void* stream);
LIBXSMM_API void* libxsmm_b200_event_create(void);
LIBXSMM_API void libxsmm_b200_event_destroy(void* event);
LIBXSMM_API int libxsmm_b200_event_record(void* event, void* stream);
LIBXSMM_API int libxsmm_b200_event_synchronize(void* event);
LIBXSMM_API float libxsmm_b200_event_elapsed_ms(void* start, void* stop);
LIBXSMM_API int libxsmm_b200_memcpy_h2d_async(void* dst_device, const void* src_host, size_t bytes, void* stream);
LIBXSMM_API int libxsmm_b200_memcpy_d2h_async(void* dst_host, const void* src_device, size_t bytes, void* stream);
LIBXSMM_API int libxsmm_b200_memset_async(void* dst_device, int value, size_t bytes, void* stream);
/* Capture everything enqueued on stream between begin and end into an executable graph. */
LIBXSMM_API int libxsmm_b200_graph_begin(void* stream);
LIBXSMM_API void* libxsmm_b200_graph_end(void* stream);
LIBXSMM_API int libxsmm_b200_graph_launch(void* graph_exec, void* stream);
LIBXSMM_API void libxsmm_b200_graph_destroy(void* graph_exec);

/* Fused caller step: C = A.B (+ beta.C) on DEVICE matrices in ONE stream-ordered call -- handle lookup, slice
 * creation and compute.  This is the wrapper TensorFlow's sparse_matmul_op keeps around the reference
 * (reference documentation/tensorflow.md:241-250; in-tree model samples/spmdm/spmdm.c:74-154): handles are cached
 * by (M, N, K, max_threads, stream), at most 16, least recently used evicted.  Arguments as
 * libxsmm_spmdm_exec_stream; returns 0 or the library's error code. */
LIBXSMM_API int libxsmm_b200_sparse_matmul(libxsmm_spmdm_datatype datatype, char transa, char transb, char transc,
  int M, int N, int K, int max_threads, const void* d_a, const void* d_b, const void* beta, float* d_c, void* stream);
LIBXSMM_API int libxsmm_b200_sparse_matmul_cache_entries(void);
LIBXSMM_API void libxsmm_b200_sparse_matmul_cache_clear(void);

/* MatrixMarket coordinate files (the operator format of samples/pyfr/mats and samples/edge/mats; reference reader
 * src/generator_spgemm_csr_reader.c:46-169): read into CSR (malloc'ed arrays, release with libxsmm_b200_csr_free;
 * returns 0 or a negative error code), or straight into a fixed operator (lda = K = columns of the file, alpha = 1).
 * Host-only parsing; create_mtx then calls the ordinary create(). */
LIBXSMM_API int libxsmm_b200_csr_read_mtx(const char* path, unsigned int** row_ptr, unsigned int** col_idx, double** values,
  unsigned int* rows, unsigned int* cols, unsigned int* nnz);
LIBXSMM_API void libxsmm_b200_csr_free(unsigned int* row_ptr, unsigned int* col_idx, double* values);
LIBXSMM_API libxsmm_dfsspmdm* libxsmm_b200_dfsspmdm_create_mtx(const char* path, int N, int ldb, int ldc, double beta, int* M, int* K);
LIBXSMM_API libxsmm_sfsspmdm* libxsmm_b200_sfsspmdm_create_mtx(const char* path, int N, int ldb, int ldc, float beta, int* M, int* K);

/* CSR x dense SoA kernels (SURVEY.md section 8f-1): the GPU counterpart of
 *     kernel = libxsmm_create_xcsr_soa(descriptor(m, n, k, lda, ldb, ldc, alpha = 1, beta), row_ptr, column_idx, values)
 *     kernel(a, b, c)                                        once per mesh element
 * (reference src/template/libxsmm.h:283-293, src/libxsmm_main.c:2423-2447, src/generator_spgemm_csr_asparse_soa.c,
 * src/generator_spgemm_csr_bsparse_soa.c; callers samples/edge/asparse_srsoa.c:148-160, samples/edge/bsparse_srsoa.c:160-176).
 * As in the reference's descriptor exactly one of lda / ldb is 0 and names the SPARSE operand (CSR):
 *   lda == 0  A sparse (CSR over its m rows), B dense [k][ldb][soa_width], C [m][ldc][soa_width]:
 *             C[m][n][s] = (beta == 0 ? 0 : C[m][n][s]) + sum over row m's nonzeros z, in CSR order, of values[z] * B[column_idx[z]][n][s];
 *             rows of A WITHOUT nonzeros leave their C rows untouched, like the reference's emitted code;
 *   ldb == 0  B sparse (CSR over its k rows), A dense [m][lda][soa_width], C [m][ldc][soa_width]:
 *             C[m][n][s] = (beta == 0 ? 0 : C[m][n][s]) + sum over k ascending, over row k's nonzeros (k, n), of A[m][k][s] * values[z];
 *             columns 0 .. ncols-1 of C are written, ncols = 1 + the largest column index any nonzero of B holds (an empty
 *             column below ncols gives beta * C; columns from ncols on are never touched, not even for beta = 0 -- the
 *             reference's generator, generator_spgemm_csr_bsparse_soa.c:161-167); nonzeros with column >= n are not
 *             multiplied; ncols > ldc is rejected.
 * One fused multiply-add per nonzero; beta is 0 or 1, as for the reference's descriptor.  soa_width is a property of the caller's
 * tensors (the reference's generator fixes it per host: 8 doubles / 16 floats with AVX-512, 4 / 8 otherwise).  One element is far
 * too small for a launch, so execute is BATCHED: n_elements elements, the dense operand of element e at d_X + e * stride_x and its
 * C at d_C + e * stride_c (strides in scalars), asynchronous on `stream`.  The sparse operand's values are fixed at create (the
 * reference's kernel re-reads them at every call; its callers pass the same array). */
typedef struct libxsmm_b200_csr_soa libxsmm_b200_csr_soa;
LIBXSMM_API libxsmm_b200_csr_soa* libxsmm_b200_dcsr_soa_create(int M, int N, int K, int lda, int ldb, int ldc, int soa_width, double beta,
  const unsigned int* row_ptr, const unsigned int* column_idx, const double* values);
LIBXSMM_API libxsmm_b200_csr_soa* libxsmm_b200_scsr_soa_create(int M, int N, int K, int lda, int ldb, int ldc, int soa_width, float beta,
  const unsigned int* row_ptr, const unsigned int* column_idx, const float* values);
/* libxsmm_create_xcsc_soa + kernel(a, values, c) (reference src/template/libxsmm.h:283-293, src/libxsmm_main.c:2450-2474,
 * src/generator_spgemm_csc_bsparse_soa.c; caller samples/edge/bsparse_scsoa.c:327-354): B sparse in CSC (column_ptr over its n
 * columns, row_idx = k), A dense [m][lda][soa_width], C [m][ldc][soa_width];
 *     C[m][n][s] = (beta == 0 ? 0 : C[m][n][s]) + sum over k ascending of A[m][k][s] * (the first entry of column n with row index k).
 * All n columns are written.  The handle is executed (d_X = A) and destroyed with the csr_soa entries below. */
LIBXSMM_API libxsmm_b200_csr_soa* libxsmm_b200_dcsc_soa_create(int M, int N, int K, int lda, int ldc, int soa_width, double beta,
                                                               const unsigned int* column_ptr, const unsigned int* row_idx, const double* values);
LIBXSMM_API libxsmm_b200_csr_soa* libxsmm_b200_scsc_soa_create(int M, int N, int K, int lda, int ldc, int soa_width, float beta,
                                                               const unsigned int* column_ptr, const unsigned int* row_idx, const float* values);
LIBXSMM_API void libxsmm_b200_csr_soa_execute(const libxsmm_b200_csr_soa* handle, const void* d_X, void* d_C, long long n_elements,
  long long stride_x, long long stride_c, void* stream);
LIBXSMM_API int libxsmm_b200_csr_soa_is_baked(const libxsmm_b200_csr_soa* handle);
LIBXSMM_API void libxsmm_b200_csr_soa_destroy(libxsmm_b200_csr_soa* handle);

/* Dense x SoA kernels: the GPU counterparts of
 *     kernel = libxsmm_create_rm_ac_soa(descriptor(m, n, k, lda, ldb, ldc, alpha = 1, beta))   or   libxsmm_create_rm_bc_soa(...)
 *     kernel(a, b, c)                                        once per mesh element
 * (reference src/libxsmm_main.c:2477,2500).  Layout as for the csr_soa entries: an SoA operand with R rows and pitch ld is
 * [R][ld][soa_width], a plain operand is row-major with pitch ld, strides count scalars.
 *   ac form  A [M][lda][soa_width], b K x N (pitch ldb), C [M][ldc][soa_width]:
 *            C[m][n][s] = chain over k = 0 .. K-1 ascending of acc = fma(A[m][k][s], b[k][n], acc);
 *   bc form  a M x K (pitch lda), B [K][ldb][soa_width], C [M][ldc][soa_width]:
 *            C[m][n][s] = chain over k = 0 .. K-1 ascending of acc = fma(a[m][k], B[k][n][s], acc);
 * acc starts from C[m][n][s] for beta = 1 and from +0 for beta = 0 (C is then never read).  One rounding per k; zeros are not
 * skipped (0 * Inf gives NaN).  Exactly the columns 0 .. N-1 of every C row are written.  alpha is 1; beta must be 0 or 1.
 * Create is host only (no CUDA call) and returns NULL with the sticky error set for an empty shape (-80), a pitch smaller than
 * its extent (lda < K, ldb < N, ldc < N: -81) or another beta (-82).  Execute is BATCHED and asynchronous on `stream`: element e
 * has its operands at d_a + e * stride_a, d_b + e * stride_b and d_c + e * stride_c (DEVICE pointers, strides in scalars).  An
 * input stride of 0 shares that operand among all elements.  n_elements = 0 does nothing; a negative count or stride, or
 * n_elements > 1 with stride_c below one element's C extent ((M-1) * ldc + N) * soa_width, sets error -83 and launches nothing.
 * All operands are read at call time. */
typedef struct libxsmm_b200_rm_soa libxsmm_b200_rm_soa;
LIBXSMM_API libxsmm_b200_rm_soa* libxsmm_b200_drm_ac_soa_create(int M, int N, int K, int lda, int ldb, int ldc, int soa_width, double beta);
LIBXSMM_API libxsmm_b200_rm_soa* libxsmm_b200_srm_ac_soa_create(int M, int N, int K, int lda, int ldb, int ldc, int soa_width, float beta);
LIBXSMM_API libxsmm_b200_rm_soa* libxsmm_b200_drm_bc_soa_create(int M, int N, int K, int lda, int ldb, int ldc, int soa_width, double beta);
LIBXSMM_API libxsmm_b200_rm_soa* libxsmm_b200_srm_bc_soa_create(int M, int N, int K, int lda, int ldb, int ldc, int soa_width, float beta);
LIBXSMM_API void libxsmm_b200_rm_soa_execute(const libxsmm_b200_rm_soa* handle, const void* d_a, const void* d_b, void* d_c,
  long long n_elements, long long stride_a, long long stride_b, long long stride_c, void* stream);
LIBXSMM_API void libxsmm_b200_rm_soa_destroy(libxsmm_b200_rm_soa* handle);

/* Indexed execution of the batched SoA entries: per-element slots, so that neighbour (flux) terms and element subsets need no
 * gather copy.  Define slot_x(e) = d_x_index ? d_x_index[e] : e, and the same for every operand.  Element e (0 <= e < n_elements)
 * computes exactly what the strided entry computes for one element whose operands sit at base + slot(e) * stride: the same chain
 * of fused multiply-adds, the same bits.
 *   - A NULL index is the identity.  A stride of 0 still shares that operand among all elements, with or without an index.
 *   - An element whose index in some operand is at or past that operand's *_slots is skipped on the device: nothing of it is
 *     read, its C slot is untouched.  Input indices may repeat.  If C indices repeat, the C of those slots is unspecified;
 *     nothing is written outside slots 0 .. c_slots - 1 (0 .. n_elements - 1 without a C index).
 *   - Index arrays are DEVICE arrays of n_elements entries, read at execute time on `stream` (a graph replay reads their
 *     current contents).
 *   - One call is one launch; n_elements = 0 does nothing.  Rejected on the host, before any CUDA call, with error -84 and
 *     nothing launched: a NULL handle, a negative count or stride, a non-NULL index with *_slots < 1 or > 2^32, a NULL operand
 *     (n_elements > 0), and C slots that overlap: stride_c below one element's C extent with a C index and c_slots > 1, or
 *     without a C index and n_elements > 1. */
LIBXSMM_API void libxsmm_b200_csr_soa_execute_indexed(const libxsmm_b200_csr_soa* handle, const void* d_X, void* d_C,
  long long n_elements, long long stride_x, long long stride_c,
  const unsigned int* d_x_index, long long x_slots, const unsigned int* d_c_index, long long c_slots, void* stream);
LIBXSMM_API void libxsmm_b200_rm_soa_execute_indexed(const libxsmm_b200_rm_soa* handle, const void* d_a, const void* d_b, void* d_c,
  long long n_elements, long long stride_a, long long stride_b, long long stride_c,
  const unsigned int* d_a_index, long long a_slots, const unsigned int* d_b_index, long long b_slots,
  const unsigned int* d_c_index, long long c_slots, void* stream);

/* A fixed 2:4-sparse bf16 operator (M x K, row-major, pitch lda; HOST or DEVICE pointer, read only during create).
 * An element is kept iff it is an ordered nonzero (+-0 and NaN dropped, as the spmdm slicing kernels do).  Every aligned
 * group of four along k (k = 4g .. 4g+3; the last group of a row may be partial) must keep at most two elements.
 * create compresses A on the GPU into [M_pad][K_pad / 2] kept values plus the metadata image the sparse tensor-core
 * instruction takes (M_pad, K_pad: multiples of 128, zero-padded), then synchronises once to read the 2:4 check.
 * NULL + sticky error: -95 M < 1, K < 1, lda < K or NULL a (checked on the host, before any CUDA call);
 *                      -96 A is not 2:4 (the message names the first offending row and group).
 * execute: C = A . op(B) + beta . C, accumulated in fp32 on the tensor cores (same contract as the bf16 spmdm path).
 *   transb 'N': B is K x N (d_b[k * ldb + n]);  'T': B is stored N x K (d_b[n * ldb + k]; y = x . W^T with x tokens x K)
 *   transc 'N': C is M x N (d_c[m * ldc + n]);  'T': C is stored N x M (d_c[n * ldc + m])
 *   beta = 0: C is not read.  Any other beta: C = fmaf(beta, C, acc).
 *   One launch, asynchronous on stream, no allocation, no host synchronisation (graph-capturable); N = 0 does nothing.
 *   -97 (nothing launched): NULL handle, a trans flag outside N/n/T/t, N < 0, ldb or ldc below its extent, NULL d_b / d_c
 *   with N > 0, d_b not 16-byte aligned or ldb % 8 != 0 (B goes through TMA), a current device other than create's. */
typedef struct libxsmm_b200_sp24 libxsmm_b200_sp24;
LIBXSMM_API libxsmm_b200_sp24* libxsmm_b200_sp24_create_bfloat16(int M, int K, int lda, const libxsmm_bfloat16* a);
LIBXSMM_API void libxsmm_b200_sp24_execute(const libxsmm_b200_sp24* handle, char transb, char transc, int N,
  const libxsmm_bfloat16* d_b, int ldb, float beta, float* d_c, int ldc, void* stream);
LIBXSMM_API void libxsmm_b200_sp24_destroy(libxsmm_b200_sp24* handle);   /* either kind; NULL does nothing */

/* A fixed 2:4-sparse FP8 operator: A is M x K bytes, row-major, pitch lda, HOST or DEVICE pointer, in one format:
 *   format 0 = e4m3 (OCP E4M3, "fn": no Inf, NaN = 0x7F / 0xFF), 1 = e5m2.
 * Same keep rule as the bf16 operator: ordered nonzeros, so +-0 and NaN are dropped and e5m2 +-Inf is kept; a group of four
 * keeping three or four elements is -96 (first row and group named), and a group of two values and two NaN is legal.
 * The multiply runs on the 8-bit structured-sparse tensor-core instruction (twice the rate of the bf16 one).
 * NULL + sticky error: -95 M < 1, K < 1, lda < K, NULL a or a format other than 0 / 1 (on the host, before any CUDA call).
 * execute_fp8: C = alpha . (A . op(B)) + beta . C with fp32 C and fp32 accumulation, per element fmaf(beta, C, alpha * acc);
 *   beta = 0: C is not read.  alpha carries the per-tensor scales (scale_a * scale_b).  b_format (0 / 1) may differ from A's.
 *   transb / transc, launch behaviour and N = 0 as for execute.
 *   -97 (nothing launched): NULL handle or a bf16 handle (and execute rejects an FP8 handle), a trans flag outside N/n/T/t,
 *   b_format not 0 / 1, N < 0, ldb or ldc below its extent, NULL d_b / d_c with N > 0, d_b not 16-byte aligned or
 *   ldb % 16 != 0 (B goes through TMA), a current device other than create's. */
LIBXSMM_API libxsmm_b200_sp24* libxsmm_b200_sp24_create_fp8(int M, int K, int lda, const unsigned char* a, int format);
LIBXSMM_API void libxsmm_b200_sp24_execute_fp8(const libxsmm_b200_sp24* handle, char transb, char transc, int N,
  const unsigned char* d_b, int b_format, int ldb, float alpha, float beta, float* d_c, int ldc, void* stream);

/* bf16 C with an optional per-row bias, for either kind of 2:4 operator: y = x . W^T + b of a pruned linear layer in one call.
 * acc is the fp32 accumulator the fp32-output entries produce for (m, n).  Per element of C:
 *   1. v = acc for a bf16 operator; v = alpha * acc (one fp32 multiply, as in execute_fp8) for an FP8 operator.
 *   2. If d_bias is not NULL, v = v + (float)d_bias[m], one fp32 addition.  If d_bias is NULL, no addition is made at all
 *      (adding +0 would turn a -0 into +0; C stays bit-identical to rounding the fp32 entry's output).
 *   3. If beta != 0, v = fmaf(beta, (float)C[m][n], v), where C is the old bf16 value.  If beta == 0, C is not read.
 *   4. C[m][n] = bf16_round_to_nearest_even(v).  NaN stays NaN (the payload is not part of the contract); overflow gives +-Inf.
 * d_bias is a DEVICE array of M bf16 values, indexed by A's row, read at execute time on stream (a graph replay reads its
 * current contents).  transb, transc, pitches (in bf16 elements for C), N = 0 and launch behaviour as for execute.
 * -97 (nothing launched): every case of execute / execute_fp8 (the bf16 entry rejects an FP8 handle and the FP8 entry a bf16
 * handle), and d_c or d_bias not 2-byte aligned. */
/* bf16 operator (sp24_create_bfloat16), bf16 C */
LIBXSMM_API void libxsmm_b200_sp24_execute_bf16out(const libxsmm_b200_sp24* handle, char transb, char transc, int N,
  const libxsmm_bfloat16* d_b, int ldb, const libxsmm_bfloat16* d_bias, float beta, libxsmm_bfloat16* d_c, int ldc, void* stream);
/* FP8 operator (sp24_create_fp8), bf16 C */
LIBXSMM_API void libxsmm_b200_sp24_execute_fp8_bf16out(const libxsmm_b200_sp24* handle, char transb, char transc, int N,
  const unsigned char* d_b, int b_format, int ldb, float alpha, const libxsmm_bfloat16* d_bias, float beta,
  libxsmm_bfloat16* d_c, int ldc, void* stream);

/* Dense SMM dispatch for row-major operators with very many columns (SURVEY.md section 8f-3): the GPU counterpart of
 *     kernel = libxsmm_dmmdispatch(nblock, M_op, K_op, &ldb_panel, &lda_op, &ldc_panel, alpha, beta, flags, prefetch)
 *     for (i = 0; i < N; i += nblock) kernel(B_panel + i, A_op, C_panel + i)
 * (reference src/libxsmm_main.c:2166-2195; caller samples/pyfr/pyfr_gemm_rm.c:98-122).  Same argument meaning as
 * libxsmm_[sd]mmdispatch: column-major C(m x n) = A(m x k) B(k x n) + beta C with NULL lda / ldb / ldc = m / k / m and
 * NULL alpha / beta = 1; like the reference's JIT it exists for alpha = 1 and beta in {0, 1} only (NULL otherwise).
 * execute covers m_total rows of A and C -- all the chunks of the caller's loop -- in one asynchronous call: d_a, d_c
 * are DEVICE pointers, b (the small k x n operand = the row-major operator, pitch ldb) may be a host or a device
 * pointer and is read at every call; the handle keeps the kernel baked for the operand's current content and re-bakes when
 * it changes.  Per output element: an in-order chain of fused multiply-adds over k starting from C (beta = 1) or 0. */
typedef struct libxsmm_b200_mm libxsmm_b200_mm;
LIBXSMM_API libxsmm_b200_mm* libxsmm_b200_dmmdispatch(int m, int n, int k, const int* lda, const int* ldb, const int* ldc,
  const double* alpha, const double* beta);
LIBXSMM_API libxsmm_b200_mm* libxsmm_b200_smmdispatch(int m, int n, int k, const int* lda, const int* ldb, const int* ldc,
  const float* alpha, const float* beta);
LIBXSMM_API void libxsmm_b200_mm_execute(libxsmm_b200_mm* handle, const void* d_a, const void* b, void* d_c, long long m_total, void* stream);
LIBXSMM_API const char* libxsmm_b200_mm_kernel(const libxsmm_b200_mm* handle);   /* which kernel the handle currently holds */
LIBXSMM_API void libxsmm_b200_mm_release(libxsmm_b200_mm* handle);

/* Host-only planning entries (no CUDA call is made; they work on a machine without a GPU).
 * geometry: the block geometry libxsmm_spmdm_init would choose (reference src/libxsmm_spmdm.c:552-608)
 *   for bn = 48 | 96 | 6; geom[9] = m n k bm bn bk mb nb kb.  Returns 0 on success.
 * plan: what create() decides for an operator (reference src/libxsmm_fsspmdm.c:88-143 and
 *   src/generator_spgemm_csr_asparse_reg.c:111-150): info[6] = nnz, unique values, 1 if the reference
 *   takes its sparse_reg branch, bytes of x86 code it would emit (0 if not evaluated), N_chunksize, and the
 *   form of the kernel create() bakes (0 none: generic kernel, 1 B rows in registers, 2 B strip in shared memory).
 * kernel_source: the CUDA source create() would bake for the operator (free with free_string). */
LIBXSMM_API int libxsmm_b200_spmdm_geometry(int M, int N, int K, int max_threads, int bn, int* geom);
LIBXSMM_API int libxsmm_b200_fsspmdm_plan(int is_double, int M, int N, int K, int lda, int ldb, int ldc, double beta,
  const void* a_dense, long long* info);
LIBXSMM_API char* libxsmm_b200_fsspmdm_kernel_source(int is_double, int M, int N, int K, int lda, int ldb, int ldc,
  double beta, const void* a_dense);
LIBXSMM_API void libxsmm_b200_free_string(char* s);

#endif /*LIBXSMM_B200_H*/
