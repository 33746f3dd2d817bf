/*
 * bhsparse.h -- drop-in replacement for the reference's `bhsparse` class
 * (weifengliu-ssslab/Benchmark_SpGEMM_using_CSR, SpGEMM_cuda/bhsparse.h:17-34):
 * same public methods, argument order (val, rowptr, colidx) and int error
 * convention, forwarding to the C-ABI of libbhsparse_b200 (bhsparse_b200.h).
 * Header-only and all-inline (the reference defines non-inline members in its
 * header, an ODR hazard: bhsparse.h:91).
 *
 *     #include "bhsparse.h"          // instead of the reference's header
 *     bhsparse *bh = new bhsparse();
 *     bh->initPlatform(platforms);   // platforms[BHSPARSE_CUDA] = true
 *     bh->initData(m, k, n, nnzA, valA, rowptrA, colA, nnzB, valB, rowptrB, colB, rowptrC);
 *     bh->warmup(); bh->spgemm();
 *     int nnzC = bh->get_nnzC();  bh->get_C(colC, valC);
 *     bh->free_mem(); bh->freePlatform();
 *
 * value_type follows the reference's typedef (common.h:31): double unless
 * BHSPARSE_VALUE_FLOAT (float), BHSPARSE_VALUE_COMPLEX_FLOAT (std::complex<float>, the _c64 entry points) or
 * BHSPARSE_VALUE_COMPLEX_DOUBLE (std::complex<double>, the _c128 entry points) is defined before including this header.
 */
#ifndef BHSPARSE_H
#define BHSPARSE_H

#include <cstdio>
#if defined(BHSPARSE_VALUE_COMPLEX_FLOAT) || defined(BHSPARSE_VALUE_COMPLEX_DOUBLE)
#include <complex>
#endif

#include "bhsparse_b200.h"

#define BHSPARSE_SUCCESS 0   /* common.h:26 */
#define NUM_PLATFORMS 9      /* common.h:33 */
#define NAIVE 0
#define BHSPARSE_CUDA 1      /* common.h:36 */
#define BHSPARSE_OPENCL 2

typedef int index_type;      /* common.h:30 */
#if defined(BHSPARSE_VALUE_COMPLEX_DOUBLE)
typedef std::complex<double> value_type;   /* two doubles (re, im): BHB200_DTYPE_C128 */
#elif defined(BHSPARSE_VALUE_COMPLEX_FLOAT)
typedef std::complex<float> value_type;   /* two floats (re, im): BHB200_DTYPE_C64 */
#elif defined(BHSPARSE_VALUE_FLOAT)
typedef float value_type;
#else
typedef double value_type;   /* common.h:31 */
#endif

class bhsparse {
public:
    bhsparse() : _ctx(nullptr), _rowptrC(nullptr), _verbose(true) {}
    ~bhsparse()
    {
        if (_ctx) bhb200_destroy(_ctx);
    }
    bhsparse(const bhsparse &) = delete;
    bhsparse &operator=(const bhsparse &) = delete;

    /* The reference prints stage times and GFLOPS from spgemm() (bhsparse.h:286-336);
     * keep that for CLI users, switch it off for library use. */
    void set_verbose(bool v) { _verbose = v; }

    /* bhsparse.h:96-124.  Only the CUDA platform exists. */
    int initPlatform(bool *spgemm_platform)
    {
        if (!spgemm_platform || !spgemm_platform[BHSPARSE_CUDA]) return BHB200_ERR_INVALID;
        if (_ctx) return BHSPARSE_SUCCESS;
        int err = bhb200_create(&_ctx, 0);   /* device 0, like bhsparse_cuda.h:100-101 */
        if (err == BHSPARSE_SUCCESS && _verbose)
            printf("Device [0] %s. %d SMs.\n", bhb200_device_name(_ctx), bhb200_sm_count(_ctx));
        return err;
    }

    /* bhsparse.h:180-258.  csrRowPtrC (m+1 ints) is caller-owned and written by get_C.
     * Addition: transA / transB compute C = op(A)*op(B) with op(X) = X^T (bhb200_init_data_op_*);
     * m, k, n are then the dimensions of op(A) (m x k) and op(B) (k x n), the arrays hold A / B as stored. */
    int initData(int m, int k, int n, int nnzA, value_type *csrValA, index_type *csrRowPtrA, index_type *csrColIndA,
                 int nnzB, value_type *csrValB, index_type *csrRowPtrB, index_type *csrColIndB,
                 index_type *csrRowPtrC, bool transA = false, bool transB = false)
    {
        if (!_ctx) return BHB200_ERR_INVALID;
        _rowptrC = csrRowPtrC;
        const int opA = transA ? BHB200_OP_T : BHB200_OP_N, opB = transB ? BHB200_OP_T : BHB200_OP_N;
#if defined(BHSPARSE_VALUE_COMPLEX_DOUBLE)
        return bhb200_init_data_op_c128(_ctx, opA, opB, m, k, n, nnzA, reinterpret_cast<const double *>(csrValA), csrRowPtrA,
                                        csrColIndA, nnzB, reinterpret_cast<const double *>(csrValB), csrRowPtrB, csrColIndB);
#elif defined(BHSPARSE_VALUE_COMPLEX_FLOAT)
        return bhb200_init_data_op_c64(_ctx, opA, opB, m, k, n, nnzA, reinterpret_cast<const float *>(csrValA), csrRowPtrA,
                                       csrColIndA, nnzB, reinterpret_cast<const float *>(csrValB), csrRowPtrB, csrColIndB);
#elif defined(BHSPARSE_VALUE_FLOAT)
        return bhb200_init_data_op_f32(_ctx, opA, opB, m, k, n, nnzA, csrValA, csrRowPtrA, csrColIndA, nnzB, csrValB,
                                       csrRowPtrB, csrColIndB);
#else
        return bhb200_init_data_op_f64(_ctx, opA, opB, m, k, n, nnzA, csrValA, csrRowPtrA, csrColIndA, nnzB, csrValB,
                                       csrRowPtrB, csrColIndB);
#endif
    }

    /* Addition: structure-only products (bhb200_init_data_structure): the pattern of op(A)*op(B) from operands
     * without values; spgemm() fills csrRowPtrC and get_C(colC, nullptr) the columns. */
    int initDataStructure(int m, int k, int n, int nnzA, index_type *csrRowPtrA, index_type *csrColIndA, int nnzB,
                          index_type *csrRowPtrB, index_type *csrColIndB, index_type *csrRowPtrC, bool transA = false,
                          bool transB = false)
    {
        if (!_ctx) return BHB200_ERR_INVALID;
        _rowptrC = csrRowPtrC;
        return bhb200_init_data_structure(_ctx, transA ? BHB200_OP_T : BHB200_OP_N, transB ? BHB200_OP_T : BHB200_OP_N, m, k,
                                          n, nnzA, csrRowPtrA, csrColIndA, nnzB, csrRowPtrB, csrColIndB);
    }

    /* Addition: masked products C = M .* (op(A)*op(B)) on the structure of M (host arrays, copied;
     * bhb200_set_mask), until clearMask() or the next initData. */
    int setMask(int nnzM, index_type *csrRowPtrM, index_type *csrColIndM)
    {
        return _ctx ? bhb200_set_mask(_ctx, nnzM, csrRowPtrM, csrColIndM) : BHB200_ERR_INVALID;
    }
    int clearMask() { return _ctx ? bhb200_clear_mask(_ctx) : BHB200_ERR_INVALID; }

    int warmup() { return _ctx ? bhb200_warmup(_ctx) : BHB200_ERR_INVALID; }   /* bhsparse.h:341-363 */

    /* bhsparse.h:260-339 */
    int spgemm()
    {
        if (!_ctx) return BHB200_ERR_INVALID;
        int err = bhb200_spgemm(_ctx);
        if (err != BHSPARSE_SUCCESS) {
            printf("spgemm error = %d (%s)\n", err, bhb200_last_error(_ctx));
            return err;
        }
        /* create_C leaves the row pointers of C in the caller's array at the end of spgemm()
         * (bhsparse_cuda.h:2787-2808); get_C writes them again (:3016).  Results beyond
         * INT32_MAX entries have no int32 row pointers (get_nnzC() == -1). */
        if (_rowptrC && bhb200_get_nnzC(_ctx) <= 0x7fffffffLL) {
            err = bhb200_get_C_structure(_ctx, _rowptrC, nullptr);   /* (valued and structure-only products) */
            if (err != BHSPARSE_SUCCESS) return err;
        }
        if (_verbose) {
            bhb200_stats st;
            bhb200_get_stats(_ctx, &st);
            printf("STAGE 1 time: %g ms.\nSTAGE 2 time: %g ms.\nSTAGE 3 time: %g ms.\nSTAGE 4 time: %g ms.\n",
                   st.ms_count, st.ms_symbolic, st.ms_scan, st.ms_numeric);
            printf("[ CUDA ] SpGEMM time: %g ms. Gflops = %g\n", st.ms_total,
                   2.0 * (double)st.products / (st.ms_total * 1.0e+6));
        }
        return err;
    }

    int get_nnzC()   /* bhsparse_cuda.h:3006-3009; -1 if it does not fit an int */
    {
        long long c = _ctx ? bhb200_get_nnzC(_ctx) : -1;
        return (c < 0 || c > 0x7fffffffLL) ? -1 : (int)c;
    }

    /* Additions (no reference counterpart): new values, same patterns -> values of C only. */
    int update_values(const value_type *csrValA, const value_type *csrValB)
    {
        if (!_ctx) return BHB200_ERR_INVALID;
#if defined(BHSPARSE_VALUE_COMPLEX_DOUBLE)
        return bhb200_update_values_c128(_ctx, reinterpret_cast<const double *>(csrValA), reinterpret_cast<const double *>(csrValB));
#elif defined(BHSPARSE_VALUE_COMPLEX_FLOAT)
        return bhb200_update_values_c64(_ctx, reinterpret_cast<const float *>(csrValA), reinterpret_cast<const float *>(csrValB));
#elif defined(BHSPARSE_VALUE_FLOAT)
        return bhb200_update_values_f32(_ctx, csrValA, csrValB);
#else
        return bhb200_update_values_f64(_ctx, csrValA, csrValB);
#endif
    }
    int spgemm_numeric() { return _ctx ? bhb200_spgemm_numeric(_ctx) : BHB200_ERR_INVALID; }

    int get_C(index_type *csrColIndC, value_type *csrValC)   /* bhsparse_cuda.h:3011-3020 */
    {
        if (!_ctx) return BHB200_ERR_INVALID;
        if (!csrValC) return bhb200_get_C_structure(_ctx, _rowptrC, csrColIndC);   /* (structure-only products too) */
#if defined(BHSPARSE_VALUE_COMPLEX_DOUBLE)
        return bhb200_get_C_c128(_ctx, _rowptrC, csrColIndC, reinterpret_cast<double *>(csrValC));
#elif defined(BHSPARSE_VALUE_COMPLEX_FLOAT)
        return bhb200_get_C_c64(_ctx, _rowptrC, csrColIndC, reinterpret_cast<float *>(csrValC));
#elif defined(BHSPARSE_VALUE_FLOAT)
        return bhb200_get_C_f32(_ctx, _rowptrC, csrColIndC, csrValC);
#else
        return bhb200_get_C_f64(_ctx, _rowptrC, csrColIndC, csrValC);
#endif
    }

    int free_mem() { return _ctx ? bhb200_free_mem(_ctx) : BHSPARSE_SUCCESS; }   /* bhsparse.h:150-177 */

    int freePlatform()   /* bhsparse.h:126-148 */
    {
        int err = _ctx ? bhb200_destroy(_ctx) : BHSPARSE_SUCCESS;
        _ctx = nullptr;
        return err;
    }

    bhb200_ctx *native_handle() { return _ctx; }

private:
    bhb200_ctx *_ctx;
    index_type *_rowptrC;
    bool _verbose;
};

#endif /* BHSPARSE_H */
