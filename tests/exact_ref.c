/*
 * exact_ref.c -- quad-precision reference for the values of C = A * B (CSR x CSR -> CSR).
 *
 * Test infrastructure: tests/exact_ref.py compiles it with gcc and loads it with ctypes.
 *
 * Row-wise Gustavson with the column order of oracle/spgemm_oracle.c (columns in first-touch
 * order, sorted per row).  Every product a_ik * b_kj of two f32 or f64 values is exact in
 * __float128 (113-bit significand, exponent range far beyond f64's), and the products are summed
 * in __float128.  For each entry of C it returns
 *   hi, lo   the sum as hi + lo (two doubles: 106 bits of the quad sum),
 *   s        sum of |a_ik * b_kj|, rounded to double,
 *   p        the number of products,
 *   cls      the class the value type gives the entry (EXACT_FINITE / _NAN / _PINF / _NINF),
 *            from the products rounded to the value type, since that is what a kernel multiplies:
 *            any NaN product, or both a +inf and a -inf product, is NaN; otherwise an infinite
 *            product gives its infinity.
 * The operands arrive as doubles; f32 operands are widened exactly by the caller.
 */
#include <stdint.h>
#include <stdlib.h>
#ifdef _OPENMP
#include <omp.h>
#endif

#define EXACT_API __attribute__((visibility("default")))

enum { EXACT_FINITE = 0, EXACT_NAN = 1, EXACT_PINF = 2, EXACT_NINF = 3 };
enum { SEEN_NAN = 1, SEEN_PINF = 2, SEEN_NINF = 4 };

/* Threads for a pass whose every thread holds `bytes_per_col` bytes for each of n columns: at most 1 GiB of
 * such scratch in all, so that the footprint does not grow with the host's core count. */
static int threads_for(int n, size_t bytes_per_col)
{
    size_t per = bytes_per_col * (size_t)(n > 0 ? n : 1);
    size_t cap = ((size_t)1 << 30) / per;
    int t = 1;
#ifdef _OPENMP
    t = omp_get_max_threads();
#endif
    return cap < 1 ? 1 : cap < (size_t)t ? (int)cap : t;
}

static void sort_i32(int32_t *a, int64_t n)
{
    /* shell sort: rows are short */
    static const int64_t gaps[] = {1750, 701, 301, 132, 57, 23, 10, 4, 1};
    for (int g = 0; g < 9; g++) {
        int64_t h = gaps[g];
        for (int64_t i = h; i < n; i++) {
            int32_t v = a[i];
            int64_t j = i;
            for (; j >= h && a[j - h] > v; j -= h) a[j] = a[j - h];
            a[j] = v;
        }
    }
}

/* rowptrC64[m+1]; returns nnz(C), or -1 on allocation failure */
EXACT_API int64_t exact_symbolic(int m, int n, const int32_t *rowptrA, const int32_t *colA,
                                 const int32_t *rowptrB, const int32_t *colB, int64_t *rowptrC64)
{
    int fail = 0;
    rowptrC64[0] = 0;
#pragma omp parallel num_threads(threads_for(n, sizeof(int32_t)))
    {
        int32_t *mark = (int32_t *)malloc(sizeof(int32_t) * (size_t)(n > 0 ? n : 1));
        if (!mark) {
#pragma omp atomic write
            fail = 1;
        } else {
            for (int j = 0; j < n; j++) mark[j] = -1;
#pragma omp for schedule(dynamic, 64)
            for (int i = 0; i < m; i++) {
                int64_t cnt = 0;
                for (int32_t pa = rowptrA[i]; pa < rowptrA[i + 1]; pa++)
                    for (int32_t q = rowptrB[colA[pa]]; q < rowptrB[colA[pa] + 1]; q++)
                        if (mark[colB[q]] != i) {
                            mark[colB[q]] = i;
                            cnt++;
                        }
                rowptrC64[i + 1] = cnt;
            }
            free(mark);
        }
    }
    if (fail) return -1;
    for (int i = 0; i < m; i++) rowptrC64[i + 1] += rowptrC64[i];
    return rowptrC64[m];
}

/* f32 != 0: the operands are f32 values and their products are rounded to f32 for the class */
EXACT_API int exact_numeric(int m, int n, int f32, const int32_t *rowptrA, const int32_t *colA, const double *valA,
                            const int32_t *rowptrB, const int32_t *colB, const double *valB,
                            const int64_t *rowptrC64, int32_t *colC, double *hi, double *lo, double *s,
                            int64_t *p, int8_t *cls)
{
    int fail = 0;
#pragma omp parallel num_threads(threads_for(n, sizeof(int32_t) + 2 * sizeof(__float128) + sizeof(int64_t) + 1))
    {
        size_t nn = (size_t)(n > 0 ? n : 1);
        int32_t *mark = (int32_t *)malloc(sizeof(int32_t) * nn);
        __float128 *acc = (__float128 *)malloc(sizeof(__float128) * nn);
        __float128 *abs_acc = (__float128 *)malloc(sizeof(__float128) * nn);
        int64_t *cnt_acc = (int64_t *)malloc(sizeof(int64_t) * nn);
        int8_t *seen = (int8_t *)malloc(nn);
        if (!mark || !acc || !abs_acc || !cnt_acc || !seen) {
#pragma omp atomic write
            fail = 1;
        } else {
            for (int j = 0; j < n; j++) mark[j] = -1;
#pragma omp for schedule(dynamic, 64)
            for (int i = 0; i < m; i++) {
                int64_t base = rowptrC64[i], cnt = 0;
                for (int32_t pa = rowptrA[i]; pa < rowptrA[i + 1]; pa++) {
                    int32_t k = colA[pa];
                    double a = valA[pa];
                    for (int32_t q = rowptrB[k]; q < rowptrB[k + 1]; q++) {
                        int32_t j = colB[q];
                        double b = valB[q];
                        __float128 prod = (__float128)a * (__float128)b;
                        double vt = f32 ? (double)((float)a * (float)b) : a * b;
                        int8_t flag = vt != vt ? SEEN_NAN : vt > 0 && vt - vt != 0 ? SEEN_PINF
                                      : vt < 0 && vt - vt != 0 ? SEEN_NINF : 0;
                        if (mark[j] != i) {
                            mark[j] = i;
                            acc[j] = prod;
                            abs_acc[j] = prod < 0 ? -prod : prod;
                            cnt_acc[j] = 1;
                            seen[j] = flag;
                            colC[base + cnt++] = j;
                        } else {
                            acc[j] += prod;
                            abs_acc[j] += prod < 0 ? -prod : prod;
                            cnt_acc[j] += 1;
                            seen[j] |= flag;
                        }
                    }
                }
                sort_i32(colC + base, cnt);
                for (int64_t t = 0; t < cnt; t++) {
                    int32_t j = colC[base + t];
                    double h = (double)acc[j];
                    int8_t f = seen[j];
                    hi[base + t] = h;
                    lo[base + t] = f ? 0.0 : (double)(acc[j] - (__float128)h);
                    s[base + t] = (double)abs_acc[j];
                    p[base + t] = cnt_acc[j];
                    cls[base + t] = (f & SEEN_NAN) || (f & (SEEN_PINF | SEEN_NINF)) == (SEEN_PINF | SEEN_NINF) ? EXACT_NAN
                                    : f & SEEN_PINF ? EXACT_PINF : f & SEEN_NINF ? EXACT_NINF : EXACT_FINITE;
                }
            }
        }
        free(mark);
        free(acc);
        free(abs_acc);
        free(cnt_acc);
        free(seen);
    }
    return fail ? -1 : 0;
}
