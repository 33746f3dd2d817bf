/*
 * bhsparse_b200.h -- C-ABI of the B200-native CSR SpGEMM (C = A*B) library.
 *
 * This is the drop-in boundary for the hot path of
 * weifengliu-ssslab/Benchmark_SpGEMM_using_CSR: everything behind the public
 * methods of class `bhsparse` (SpGEMM_cuda/bhsparse.h:17-34) and its CUDA
 * back-end `bhsparse_cuda` (SpGEMM_cuda/bhsparse_cuda.h:17-90).  Plain C types
 * only; no STL, torch, Thrust, CUB, cuSPARSE or CUSP types cross it.  The
 * header-only C++ forwarder include/bhsparse.h rebuilds the reference class on
 * top of these entry points; Python binds them with ctypes.
 *
 * CSR layout (bhsparse.h:22-25, common.h:30-31): int32 row pointers and column
 * indices, 0-based; float or double values.  Rows of B must be sorted by column
 * and duplicate-free (the reference's merge kernels assume the same,
 * bhsparse_cuda.h:1730,1762).  Argument order is val, rowptr, colidx, as in the
 * reference.
 *
 * Values (DESIGN.md §2, "The value contract").  For an entry C_ij with p products a_ik*b_kj, let
 * s = sum |a_ik*b_kj| (exact), u the unit roundoff (2^-53 for f64, 2^-24 for f32), lam the smallest normal
 * number (2^-1022 / 2^-126) and gamma(p) = p*u / (1 - p*u).
 *  - Finite inputs whose exact partial sums cannot overflow: |c_hat - c| <= gamma(p)*s + 2*p*lam, in every
 *    kernel and summation order.  The 2*p*lam term covers gradual underflow and the two f32 kernels that flush
 *    subnormal products and partial sums to zero: k_num_large<float> and k_mask_global<float> add into global
 *    memory with atomics that flush subnormals (RED/ATOMG.E.ADD.F32.FTZ on sm_100a).
 *  - Integers with |a|, |b| <= 2^q and p * 2^(2q) <= 2^(t-1) (t = 53 for f64, 24 for f32) are summed exactly
 *    in any order: the values are equal to the exact ones.
 *  - Non-finite: any NaN product, or both a +inf and a -inf product, gives NaN; otherwise a +inf or -inf
 *    product gives that infinity (products in the value type; inf * stored 0 is NaN).  An entry whose
 *    products are all finite is finite.  Overflow of finite partial sums is unspecified.
 *  - Not promised: the sign of a zero result, and bitwise identical results from two identical calls (some
 *    kernels sum in the order atomics decide).
 *  - complex64 (BHB200_DTYPE_C64): each component of C_ij is a real sum of 2p real products of f32 values,
 *    Re: ar*br and (-ai)*bi, Im: ar*bi and ai*br.  The f32 rules above hold per component with p replaced by
 *    2p and s by the sum of the magnitudes of those 2p products: |c_hat - c| <= gamma(2p)*s + 4*p*lam.
 *    Gaussian integers within the f32 budget for 2p products come back equal.  The class of a non-finite
 *    component follows the real rule applied to its 2p products, provided no finite real product overflows
 *    (otherwise it is unspecified): this is the naive formula's behaviour, not C99 Annex G's recovery of
 *    infinities (inf * (0 + 1i) gives NaN components here).
 *  - complex128 (BHB200_DTYPE_C128): the same per-component rule with the f64 values and constants: each
 *    component is a real sum of 2p f64 products, |c_hat - c| <= gamma(2p)*s + 4*p*lam with u = 2^-53 and
 *    lam = 2^-1022.  Gaussian integers within the f64 budget for 2p products come back equal; non-finite
 *    components follow the naive formula, as for complex64.
 *
 * Every function returns BHB200_SUCCESS (0 == BHSPARSE_SUCCESS, common.h:26) or
 * a negative error code; nothing calls exit().  Not thread-safe per context
 * (the reference is not either, bhsparse_cuda.h:100-101); distinct contexts may
 * be used from distinct threads.
 */
#ifndef BHSPARSE_B200_H
#define BHSPARSE_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define BHB200_API __attribute__((visibility("default")))
#else
#define BHB200_API
#endif

#define BHB200_SUCCESS 0
#define BHB200_ERR_INVALID (-1)      /* bad argument / call order                      */
#define BHB200_ERR_CUDA (-2)         /* CUDA runtime error (see bhb200_last_error)     */
#define BHB200_ERR_OVERFLOW (-3)     /* nnz(C) or a row does not fit the int32 API     */
#define BHB200_ERR_ALLOC (-4)        /* device or host allocation failed               */
#define BHB200_ERR_NO_DEVICE (-5)    /* no sm_100 device / device index out of range   */

#define BHB200_DTYPE_F32 0
#define BHB200_DTYPE_F64 1
/* structure only: operands and C have row pointers and columns, no values (see "structure-only
 * products" below) */
#define BHB200_DTYPE_NONE 2
/* value 3 is not a type (and stays invalid) */
/* single-precision complex: two floats (re, im) per value, 8 bytes, 8-byte aligned -- the layout of C99
 * float _Complex, std::complex<float>, cuFloatComplex, numpy / torch complex64.  Value arrays are passed
 * as float * holding 2*nnz interleaved floats (or void * to the same bytes); see "complex64 products" below. */
#define BHB200_DTYPE_C64 4
/* double-precision complex: two doubles (re, im) per value, 16 bytes, 16-byte aligned -- the layout of C99
 * double _Complex, std::complex<double>, cuDoubleComplex, numpy / torch complex128.  Value arrays are passed
 * as double * holding 2*nnz interleaved doubles (or void * to the same bytes); see "complex128 products" below. */
#define BHB200_DTYPE_C128 5

/* op(X) of bhb200_init_data_op_* / bhb200_init_data_device_op: X as stored, its transpose, or its conjugate
 * transpose X^H (complex64 and complex128 operands only: with f32, f64 or structure-only operands OP_C is
 * BHB200_ERR_INVALID) */
#define BHB200_OP_N 0
#define BHB200_OP_T 1
#define BHB200_OP_C 2

#define BHB200_NUM_SYM_BINS 24
#define BHB200_NUM_NUM_BINS 24
#define BHB200_NUM_MASK_BINS 9

typedef struct bhb200_ctx bhb200_ctx;

/* Per-call statistics of the last bhb200_spgemm (replaces the reference's
 * stdout chatter: stage times bhsparse.h:307-336, "allocated size ... out of
 * full size ..." :432, GFLOPS :286-289). */
typedef struct bhb200_stats {
    int64_t m, k, n, nnzA, nnzB;
    int64_t products;        /* sum over rows of intermediate products = _nnzCt_full (bhsparse.h:368-406) */
    int64_t nnzC;
    int64_t max_row_products;
    int64_t sym_bin_rows[BHB200_NUM_SYM_BINS]; /* rows per symbolic bin (by upper bound)       */
    int64_t num_bin_rows[BHB200_NUM_NUM_BINS]; /* rows per numeric bin (by exact nnz(C_i))     */
    float ms_total;          /* device time of the whole call (CUDA events)                    */
    float ms_count;          /* stage 1: per-row upper bound + binning                         */
    float ms_symbolic;       /* stage 2: per-bin symbolic kernels                              */
    float ms_scan;           /* stage 3: row-pointer scan + numeric binning + C allocation     */
    float ms_numeric;        /* stage 4: per-bin numeric kernels                               */
    int32_t kernel_launches; /* kernels launched by the last call                              */
    int32_t dtype;           /* BHB200_DTYPE_*                                                 */
    int64_t bytes_algorithmic; /* stream-gather model, SURVEY.md 8(d)                          */
    int64_t bytes_compulsory;  /* bytes(A)+bytes(B)+bytes(C)                                   */
    int64_t workspace_bytes;   /* device memory currently held by the context                  */
    /* per numeric bin: work done by that bin's kernel (always filled) */
    int64_t num_bin_products[BHB200_NUM_NUM_BINS];
    int64_t num_bin_nnzC[BHB200_NUM_NUM_BINS];
    int64_t num_bin_nnzA[BHB200_NUM_NUM_BINS];
    /* per-bin kernel times in ms (CUDA events; only with bhb200_set_profiling(ctx, 1)) */
    float ms_sym_bin[BHB200_NUM_SYM_BINS];
    float ms_num_bin[BHB200_NUM_NUM_BINS];
    /* direct (single-pass) mode: rows computed without a symbolic pass, rows among them that
     * overflowed the speculated capacity and were redone, size of the staging buffer (Ct) */
    int64_t direct_rows, direct_retry_rows, direct_ct_bytes;
    int64_t direct_bin_mask;   /* bit b: symbolic bin b ran in direct mode (its ms_sym_bin is the numeric kernel) */
    /* diagonal-pattern mode (operands with <= 64 distinct diagonals each, <= 256 in the product):
     * 1 if the last product ran through it (ms_count then includes the offset sets + codes,
     * ms_symbolic the mask kernel, ms_numeric the one numeric kernel), and the number of distinct
     * diagonals of A, B and C and the accumulator length. */
    int64_t pattern_mode, pattern_nDA, pattern_nDB, pattern_nD, pattern_acc_len;
    /* host-memory spill: bytes of C / of the staging buffer that live in pinned, device-mapped host
     * memory because the device could not hold them (0 normally) */
    int64_t spill_bytes;
    /* transposed operands: bit 0 = op(A) is A^T, bit 1 = op(B) is B^T.  ms_transpose: device time of the
     * transposition (or value re-gather) this call ran, included in ms_total; its kernels count in
     * kernel_launches */
    int64_t transposed_ops;
    float ms_transpose;
    /* masked product (bhb200_set_mask): 1 if the last product was masked, nnz(M), and the rows per
     * masked kernel bin: 0 no products or no mask entries (no kernel), 1 <= 32 products (warp, binary
     * search), 2-4 warp per row with a table for <= 32 / 128 / 512 mask entries (<= 2048 products),
     * 5-7 CTA per row with a table for <= 512 / 2048 / 8192 mask entries, 8 more mask entries (binary
     * search, values in global memory).  The stage times then read: ms_count = stage 1 + mask binning,
     * ms_symbolic = the masked kernels (ms_sym_bin[b]: masked bin b, with profiling), ms_scan = scan +
     * allocation of C, ms_numeric = the copy of the staged rows into C. */
    int64_t masked;
    int64_t nnzM;
    int64_t mask_bin_rows[BHB200_NUM_MASK_BINS];
} bhb200_stats;

/* -- platform --------------------------------------------------------------
 * bhb200_create replaces bhsparse::initPlatform (bhsparse.h:96-124) and
 * bhsparse_cuda::initPlatform (bhsparse_cuda.h:96-113, which hard-wires device
 * 0).  bhb200_destroy replaces freePlatform (bhsparse.h:126-148). */
BHB200_API int bhb200_create(bhb200_ctx **ctx, int device);
BHB200_API int bhb200_destroy(bhb200_ctx *ctx);
/* Run all work of this context on the caller's cudaStream_t (0 = the context's
 * own non-blocking stream).  No reference counterpart (default stream only). */
BHB200_API int bhb200_set_stream(bhb200_ctx *ctx, void *cuda_stream);
BHB200_API const char *bhb200_last_error(const bhb200_ctx *ctx);
BHB200_API const char *bhb200_device_name(const bhb200_ctx *ctx);
BHB200_API int bhb200_sm_count(const bhb200_ctx *ctx);

/* -- operands ----------------------------------------------------------------
 * bhb200_init_data_{f64,f32} replace bhsparse::initData (bhsparse.h:180-258)
 * -> bhsparse_cuda::initData (bhsparse_cuda.h:151-203): HOST pointers, copied
 * to the device before the call returns; the caller keeps ownership.  A is
 * m x k, B is k x n.  f64/f32 replaces the compile-time value_type typedef
 * (common.h:31). */
BHB200_API int bhb200_init_data_f64(bhb200_ctx *ctx, int m, int k, int n,
                                    int nnzA, const double *valA, const int32_t *rowptrA, const int32_t *colA,
                                    int nnzB, const double *valB, const int32_t *rowptrB, const int32_t *colB);
BHB200_API int bhb200_init_data_f32(bhb200_ctx *ctx, int m, int k, int n,
                                    int nnzA, const float *valA, const int32_t *rowptrA, const int32_t *colA,
                                    int nnzB, const float *valB, const int32_t *rowptrB, const int32_t *colB);
/* C = op(A)*op(B) with op(X) = X (BHB200_OP_N) or X^T (BHB200_OP_T), as the transpose flags of
 * cuSPARSE's legacy csrgemm: m, k, n are the dimensions of op(A) (m x k) and op(B) (k x n); the stored
 * arrays have the stored row count + 1 row pointers (rowptrA: k+1 entries for opA = T, rowptrB: n+1 for
 * opB = T).  The library transposes on the device (stable: the rows of X^T in increasing column order,
 * whatever the order inside the stored rows, so with opB = T the rows of the stored B need not be
 * sorted; they must still be duplicate-free).  A column of a stored operand outside its range makes
 * bhb200_spgemm return BHB200_ERR_INVALID naming the operand.  When the transposition runs:
 *   host operands (bhb200_init_data_op_*): once, at the first bhb200_warmup or bhb200_spgemm after
 *     init_data; bhb200_update_values_* carries new values into the transposed copies;
 *   borrowed operands (bhb200_init_data_device_op): at every bhb200_spgemm (the caller may have rewritten
 *     them); bhb200_spgemm_numeric re-gathers the values of the transposed copies from the caller's arrays,
 *     so values rewritten in place take effect with the structure kept.
 * With the same host arrays for A and B (A*A^T, A^T*A) they are uploaded once; with both ops T one
 * transposed copy serves both operands.  The two functions without _op are the OP_N, OP_N case. */
BHB200_API int bhb200_init_data_op_f64(bhb200_ctx *ctx, int opA, int opB, int m, int k, int n,
                                       int nnzA, const double *valA, const int32_t *rowptrA, const int32_t *colA,
                                       int nnzB, const double *valB, const int32_t *rowptrB, const int32_t *colB);
BHB200_API int bhb200_init_data_op_f32(bhb200_ctx *ctx, int opA, int opB, int m, int k, int n,
                                       int nnzA, const float *valA, const int32_t *rowptrA, const int32_t *colA,
                                       int nnzB, const float *valB, const int32_t *rowptrB, const int32_t *colB);
/* 1 if the last bhb200_init_data_{f64,f32} (or _op_) received the SAME host arrays for A and B (C = A*A as
 * the reference driver's stock workloads set it up, main.cu:32-51; also A*A^T, A^T*A): they are uploaded
 * once and both operands share the device copy.  bhb200_update_values_* then takes one set of values. */
BHB200_API int bhb200_operands_aliased(const bhb200_ctx *ctx);
/* The operands as the library holds them on the device (borrowed views, valid until the next
 * init_data / dist_setup / free_mem): dims = {m, k, n, nnzA, nnzB, dtype}.  These are the effective
 * operands op(A) and op(B): the transposed copies for BHB200_OP_T.  After
 * bhb200_dist_setup_square this is the rank's row block of A and its replica of B.  Any pointer may
 * be NULL. */
BHB200_API int bhb200_get_operands_device(const bhb200_ctx *ctx, int32_t *dims, const int32_t **rowptrA,
                                          const int32_t **colA, const void **valA, const int32_t **rowptrB,
                                          const int32_t **colB, const void **valB);
/* Same, but the six arrays are DEVICE pointers on the context's device and are
 * borrowed (not copied, not freed) until bhb200_free_mem: the device-resident
 * operand API of SURVEY.md 8(f).3, used by the multi-GPU row-block driver. */
BHB200_API int bhb200_init_data_device(bhb200_ctx *ctx, int dtype, int m, int k, int n,
                                       int nnzA, const void *valA, const int32_t *rowptrA, const int32_t *colA,
                                       int nnzB, const void *valB, const int32_t *rowptrB, const int32_t *colB);
/* Device operands with transpose flags (see bhb200_init_data_op_f64 above for m, k, n and the rules). */
BHB200_API int bhb200_init_data_device_op(bhb200_ctx *ctx, int dtype, int opA, int opB, int m, int k, int n,
                                          int nnzA, const void *valA, const int32_t *rowptrA, const int32_t *colA,
                                          int nnzB, const void *valB, const int32_t *rowptrB, const int32_t *colB);

/* -- structure-only products: the sparsity pattern of op(A)*op(B) (GraphBLAS's boolean product, the
 * symbolic stage of MKL sp2m / cuSPARSE SpGEMMreuse) -----------------------------------------------------
 * Operands of type BHB200_DTYPE_NONE have row pointers and columns only, and so has C: C_ij is present iff
 * some product A_ik*B_kj exists, so rowptrC / colC are bit for bit those of the valued product of the same
 * operands.  No value is read, multiplied, staged or stored.
 *   bhb200_init_data_structure  HOST arrays, copied before the call returns; the rules of
 *                               bhb200_init_data_op_* (transpose flags, stored row counts, the same host
 *                               arrays for A and B uploaded once).
 *   bhb200_init_data_device / _device_op with dtype BHB200_DTYPE_NONE: valA / valB are never read and may
 *                               be NULL; with the arrays of valued device operands this gives their pattern
 *                               without a copy.
 *   bhb200_get_C_structure      rowptrC (m+1) and colC (nnzC) into HOST arrays, for any product (valued
 *                               too); the NULL, BHB200_ERR_INVALID and BHB200_ERR_OVERFLOW rules of
 *                               bhb200_get_C_f64.
 * After a structure-only product, bhb200_get_C_f64 / _f32, bhb200_update_values_*, bhb200_spgemm_numeric,
 * and bhb200_get_C_range / bhb200_copy_C_to_device with a non-NULL valC return BHB200_ERR_INVALID;
 * bhb200_get_C_device sets *valC = NULL.  Masks and the row pointer, range and device getters work as for
 * valued products; bhb200_stats.dtype is BHB200_DTYPE_NONE and its byte counts take 0 bytes per value.
 * Multi-GPU products (bhb200_dist_setup_square) are valued only. */
BHB200_API int bhb200_init_data_structure(bhb200_ctx *ctx, int opA, int opB, int m, int k, int n,
                                          int nnzA, const int32_t *rowptrA, const int32_t *colA,
                                          int nnzB, const int32_t *rowptrB, const int32_t *colB);
BHB200_API int bhb200_get_C_structure(bhb200_ctx *ctx, int32_t *rowptrC, int32_t *colC);

/* -- complex64 products: C = op(A)*op(B) over single-precision complex values ------------------------------
 * Values are BHB200_DTYPE_C64 (two floats per value, see the define).  Every path of the real types runs:
 * the same bins, direct-mode plans, diagonal-pattern mode and masked kernels as f64 (a complex64 value has the
 * size of a double), with the product of the value contract above.
 *   bhb200_init_data_op_c64    HOST arrays, the rules of bhb200_init_data_op_f64; valA / valB hold 2*nnz
 *                              floats.  opA / opB may also be BHB200_OP_C: op(X) = X^H, the transpose with
 *                              every value conjugated (the imaginary part's sign flipped, which keeps NaN, inf
 *                              and zero).  With the same host arrays for A and B they are uploaded once; one
 *                              transposed copy serves both operands when both ops are equal (T, T or C, C), so
 *                              A*A^H takes one upload and one transposition.
 *   bhb200_update_values_c64   new values of the host operands (conjugated again into X^H copies).
 *   bhb200_get_C_c64           rowptrC, colC and valC (2*nnzC floats) into HOST arrays.
 *   bhb200_init_data_device / _device_op with BHB200_DTYPE_C64: borrowed device operands; value pointers that
 *                              are not 8-byte aligned return BHB200_ERR_INVALID from the init call.
 *                              bhb200_spgemm_numeric re-gathers (and re-conjugates) the values of op = T / C
 *                              operands from the caller's arrays.
 * bhb200_get_C_range, bhb200_get_C_device, bhb200_copy_C_to_device, masks and the structure getters work with
 * 8-byte values; bhb200_stats.dtype is BHB200_DTYPE_C64 and its byte counts take 8 bytes per value.
 * bhb200_dist_setup_square takes BHB200_DTYPE_C64 (values broadcast as 8-byte words).  The real getters and
 * update_values_f64 / _f32 on a complex64 context, and the _c64 ones on a real context, return
 * BHB200_ERR_INVALID; so do they on a complex128 context. */
BHB200_API int bhb200_init_data_op_c64(bhb200_ctx *ctx, int opA, int opB, int m, int k, int n,
                                       int nnzA, const float *valA, const int32_t *rowptrA, const int32_t *colA,
                                       int nnzB, const float *valB, const int32_t *rowptrB, const int32_t *colB);
BHB200_API int bhb200_update_values_c64(bhb200_ctx *ctx, const float *valA, const float *valB);
BHB200_API int bhb200_get_C_c64(bhb200_ctx *ctx, int32_t *rowptrC, int32_t *colC, float *valC);

/* -- complex128 products: C = op(A)*op(B) over double-precision complex values -----------------------------
 * Values are BHB200_DTYPE_C128 (two doubles per value, see the define).  The entry points follow the _c64 ones:
 *   bhb200_init_data_op_c128   HOST arrays, the rules of bhb200_init_data_op_c64; valA / valB hold 2*nnz
 *                              doubles; opA / opB may be BHB200_OP_C.
 *   bhb200_update_values_c128  new values of the host operands (conjugated again into X^H copies).
 *   bhb200_get_C_c128          rowptrC, colC and valC (2*nnzC doubles) into HOST arrays.
 *   bhb200_init_data_device / _device_op with BHB200_DTYPE_C128: borrowed device operands; value pointers that
 *                              are not 16-byte aligned return BHB200_ERR_INVALID from the init call.
 * bhb200_get_C_range, bhb200_get_C_device, bhb200_copy_C_to_device, masks and the structure getters work with
 * 16-byte values; bhb200_stats.dtype is BHB200_DTYPE_C128 and its byte counts take 16 bytes per value.
 * bhb200_dist_setup_square takes BHB200_DTYPE_C128.  The on-chip tables sized for 8-byte values do not all hold
 * 16-byte ones, so some rows run in another kernel than they would in f64 (DESIGN.md 4.13); the statistics
 * (num_bin_rows, mask_bin_rows, direct_bin_mask) report the kernels that ran.  The real and _c64 getters and
 * updaters return BHB200_ERR_INVALID on a complex128 context, and the _c128 ones on any other context. */
BHB200_API int bhb200_init_data_op_c128(bhb200_ctx *ctx, int opA, int opB, int m, int k, int n,
                                        int nnzA, const double *valA, const int32_t *rowptrA, const int32_t *colA,
                                        int nnzB, const double *valB, const int32_t *rowptrB, const int32_t *colB);
BHB200_API int bhb200_update_values_c128(bhb200_ctx *ctx, const double *valA, const double *valB);
BHB200_API int bhb200_get_C_c128(bhb200_ctx *ctx, int32_t *rowptrC, int32_t *colC, double *valC);

/* -- masked products: C = M .* (op(A)*op(B)) (GraphBLAS C<M> = A*B) ----------------------------------
 * M is m x n and structural: row pointers (m+1) and column indices, no values; its rows must be sorted
 * and duplicate-free with columns in [0, n), as the rows of B.  C_ij is present iff M_ij is present and
 * at least one product A_ik*B_kj exists; its value is the sum of those products (explicit zeros from
 * cancellation are kept).  So C is the unmasked C restricted to the pattern of M.  Rows of C are
 * sorted; the row pointers, get_C*, get_C_range, get_C_device and copy_C_to_device work as for
 * unmasked products.  Only nnz(M) entries are staged and no product is sorted.
 *   bhb200_set_mask         HOST arrays, copied before the call returns.  Needs operands (m, n).
 *   bhb200_set_mask_device  DEVICE arrays, borrowed and read by every bhb200_spgemm, like borrowed
 *                           operands; they may be the operands' own arrays (triangle counting: L as A,
 *                           B and M).
 *   bhb200_clear_mask       back to unmasked products.
 * The mask is checked on the device by bhb200_spgemm: unsorted or duplicate columns, a column outside
 * [0, n), row pointers that do not rise from 0 to nnzM all return BHB200_ERR_INVALID naming the mask.
 * Every init_data*, init_data_device*, dist_setup_square and free_mem clears the mask.  Setting or
 * clearing it leaves an existing C readable, but bhb200_spgemm_numeric returns BHB200_ERR_INVALID until
 * the next bhb200_spgemm; after a masked bhb200_spgemm, update_values_* + spgemm_numeric recompute the
 * masked values with the structure kept.  A masked product never takes the diagonal-pattern mode.
 * Complemented masks and masks with values are not supported; on a multi-GPU context (after
 * bhb200_dist_init) bhb200_set_mask* returns BHB200_ERR_INVALID. */
BHB200_API int bhb200_set_mask(bhb200_ctx *ctx, int nnzM, const int32_t *rowptrM, const int32_t *colM);
BHB200_API int bhb200_set_mask_device(bhb200_ctx *ctx, int nnzM, const int32_t *rowptrM, const int32_t *colM);
BHB200_API int bhb200_clear_mask(bhb200_ctx *ctx);

/* -- the hot path --------------------------------------------------------------
 * bhb200_warmup replaces bhsparse::warmup (bhsparse.h:341-363): runs the
 * per-row upper-bound kernel once; an existing result (C, nnzC) stays valid.
 * bhb200_spgemm replaces bhsparse::spgemm (bhsparse.h:260-339): all four stages
 * on the device.  Unlike the reference it may be called repeatedly.  It returns
 * after the last kernel has been enqueued and the sizes are known; results are
 * complete after bhb200_synchronize or any bhb200_get_* call. */
BHB200_API int bhb200_warmup(bhb200_ctx *ctx);
BHB200_API int bhb200_spgemm(bhb200_ctx *ctx);
BHB200_API int bhb200_synchronize(bhb200_ctx *ctx);

/* -- repeated products with the same patterns (SURVEY.md 8(f).3; no reference
 * counterpart: the reference recomputes everything, bhsparse.h:260-339) --------
 * bhb200_update_values_* replaces the VALUES of A and/or B (host arrays of nnzA /
 * nnzB entries; NULL keeps the current ones); row pointers and column indices
 * stay those of the last bhb200_init_data_*.  With bhb200_init_data_device the
 * caller owns the device arrays and simply overwrites them (the call returns
 * BHB200_ERR_INVALID).
 * bhb200_spgemm_numeric recomputes the values of C after a completed
 * bhb200_spgemm on the same operands: row pointers and column indices of C are
 * kept, the upper-bound, symbolic, scan and allocation stages are skipped, the
 * numeric kernels overwrite the values in place.  Returns BHB200_ERR_INVALID if
 * there is no completed product to reuse. */
BHB200_API int bhb200_update_values_f64(bhb200_ctx *ctx, const double *valA, const double *valB);
BHB200_API int bhb200_update_values_f32(bhb200_ctx *ctx, const float *valA, const float *valB);
BHB200_API int bhb200_spgemm_numeric(bhb200_ctx *ctx);

/* -- results -------------------------------------------------------------------
 * bhb200_get_nnzC replaces bhsparse::get_nnzC (bhsparse_cuda.h:3006-3009) with
 * a 64-bit count.  bhb200_get_C_{f64,f32} replace bhsparse::get_C
 * (bhsparse_cuda.h:3011-3020): device->host copy of rowptrC (m+1), colC and valC
 * (nnzC each) into caller-allocated HOST arrays; any pointer may be NULL to skip
 * it.  Returns BHB200_ERR_OVERFLOW if nnz(C) > INT32_MAX (use the _i64 row
 * pointer variant then). */
BHB200_API int64_t bhb200_get_nnzC(const bhb200_ctx *ctx);
BHB200_API int bhb200_get_C_f64(bhb200_ctx *ctx, int32_t *rowptrC, int32_t *colC, double *valC);
BHB200_API int bhb200_get_C_f32(bhb200_ctx *ctx, int32_t *rowptrC, int32_t *colC, float *valC);
BHB200_API int bhb200_get_rowptrC_i64(bhb200_ctx *ctx, int64_t *rowptrC64);
/* Entries [first, first+count) of colC / valC into HOST arrays (value type of initData; either
 * pointer may be NULL).  With the int64 row pointers this serves results beyond INT32_MAX
 * entries piecewise (the reference's int get_C cannot, bhsparse_cuda.h:3011-3020). */
BHB200_API int bhb200_get_C_range(bhb200_ctx *ctx, int64_t first, int64_t count, int32_t *colC, void *valC);
/* Device-resident result (borrowed until the next spgemm / free_mem):
 * rowptr32 is NULL-valued when nnz(C) > INT32_MAX. */
BHB200_API int bhb200_get_C_device(bhb200_ctx *ctx, const int32_t **rowptr32, const int64_t **rowptr64,
                                   const int32_t **colC, const void **valC);
/* Copy the result into caller-owned DEVICE buffers (rowptrC64: m+1 int64, colC / valC:
 * nnzC entries; any may be NULL).  Device-to-device on the context's stream, complete on
 * return. */
BHB200_API int bhb200_copy_C_to_device(bhb200_ctx *ctx, int64_t *rowptrC64, int32_t *colC, void *valC);
/* Host copies of the per-row intermediate-product counts (int32[m], the
 * reference's csrRowPtrCt contents, bhsparse_cuda.h:210-237) -- test hook. */
BHB200_API int bhb200_get_row_products(bhb200_ctx *ctx, int32_t *row_products);
BHB200_API int bhb200_get_stats(const bhb200_ctx *ctx, bhb200_stats *out);
/* Per-bin kernel timing (one CUDA event per launch; off by default).  Replaces the
 * reference's dead `_profiling` switch (bhsparse_cuda.h:205-208, 728-733). */
BHB200_API int bhb200_set_profiling(bhb200_ctx *ctx, int enabled);

/* -- multi-GPU: 1-D row blocks of A, B replicated (SURVEY.md 8e; the reference is single-GPU,
 * bhsparse_cuda.h:100-101).  One process per GPU, one context per process; NCCL is called
 * directly by the library (dlopen of libnccl.so.2 at the first call).
 *   bhb200_dist_unique_id   any one rank produces the 128-byte NCCL id; the caller hands it to every
 *                           rank by its own means (MPI, a TCP store, a file).
 *   bhb200_dist_init        ncclCommInitRank on the context's device; collective.
 *   bhb200_dist_setup_square  C = B*B: on `root` the three arrays are DEVICE pointers to B (n x n,
 *                           nnz entries; borrowed), ignored elsewhere.  The root computes the per-row
 *                           products and the block boundaries on its device (blocks hold equal shares
 *                           of the intermediate products; a row is never split), then B is
 *                           broadcast -- boundaries, rowptr, col, and val on a second stream so that it
 *                           overlaps stage 1 of the first product.  Every rank ends with B replicated
 *                           and its row block of A set as operands.  Collective.
 *   bhb200_dist_spgemm      the single-GPU pipeline on the block + ncclAllGather of the int64 nnz(C)
 *                           of every rank + a device kernel that writes the GLOBAL row pointers of the
 *                           block (local + offset): no host round trip.  Collective.
 *   bhb200_dist_get_layout  host view: global rows [row_begin, row_end) of this rank, its first
 *                           global entry and the total nnz(C) (these two copy nranks int64 from the
 *                           device), total intermediate products.  Any pointer may be NULL.
 *   bhb200_dist_get_block_products  intermediate products of every rank's block (nranks int64).
 *   bhb200_dist_get_global_rowptr_device  device pointer to rows+1 int64 global row pointers.
 *   bhb200_dist_broadcast_ms  device time of the last set-up (partition + broadcast of B).
 * C stays row-sharded: rank r's colC / valC (bhb200_get_C_device, bhb200_get_C_range) are the global
 * entries [nnz_offset, nnz_offset + nnzC_local). */
#define BHB200_DIST_ID_BYTES 128
BHB200_API int bhb200_dist_unique_id(void *id);
BHB200_API int bhb200_dist_init(bhb200_ctx *ctx, int rank, int nranks, const void *id);
/* dist_setup_square takes BHB200_DTYPE_F32, BHB200_DTYPE_F64, BHB200_DTYPE_C64 or BHB200_DTYPE_C128 (structure-only products are
 * single-GPU) */
BHB200_API int bhb200_dist_setup_square(bhb200_ctx *ctx, int root, int dtype, int n, int64_t nnz, const int32_t *rowptr,
                                        const int32_t *col, const void *val);
BHB200_API int bhb200_dist_spgemm(bhb200_ctx *ctx);
BHB200_API int bhb200_dist_get_layout(bhb200_ctx *ctx, int64_t *row_begin, int64_t *row_end, int64_t *nnz_offset,
                                      int64_t *nnz_total, int64_t *products_total);
BHB200_API int bhb200_dist_get_block_products(bhb200_ctx *ctx, int64_t *block_products);
BHB200_API int bhb200_dist_get_global_rowptr_device(bhb200_ctx *ctx, const int64_t **rowptr_global);
BHB200_API int bhb200_dist_broadcast_ms(bhb200_ctx *ctx, float *ms);
BHB200_API int bhb200_dist_finalize(bhb200_ctx *ctx);

/* Host-only probe of the diagonal-pattern mode (no reference counterpart; no GPU needed): the plan
 * the library would build for operands whose entries sit on the diagonals offsA (nA values of
 * column - row) and offsB.  info[0] = 1 if the mode applies (at most 64 diagonals per operand and 256
 * in the product), then info[1..5] = diagonals of C, mask words per row, accumulator length,
 * shared-memory wavefronts of one pass over all (A diagonal, lane group) pairs with the chosen
 * accumulator layout, and their conflict-free minimum.  position (nA*nB bytes, optional): accumulator
 * slot of product (ja, jb), diagonals in ascending order; offsC (<= 256 ints, optional): diagonals of C.
 * value_size is 4, 8 or 16 (f32; f64 and complex64; complex128): a lane group is the 128 bytes of one
 * shared-memory wavefront, 32, 16 or 8 lanes. */
BHB200_API int bhb200_pattern_plan_probe(const int32_t *offsA, int nA, const int32_t *offsB, int nB, int value_size,
                                         int32_t *info, uint8_t *position, int32_t *offsC);

/* bhb200_free_mem replaces bhsparse::free_mem (bhsparse.h:150-177,
 * bhsparse_cuda.h:121-149): releases operands, results and workspace. */
BHB200_API int bhb200_free_mem(bhb200_ctx *ctx);

/* Library identification: "bhsparse_b200 <version> sm_100a". */
BHB200_API const char *bhb200_version(void);

#ifdef __cplusplus
}
#endif
#endif /* BHSPARSE_B200_H */
