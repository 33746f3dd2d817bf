// common.cuh -- shared definitions of the B200 SpGEMM pipeline (sm_100a).
//
// Pipeline (replaces bhsparse::spgemm_cuda, SpGEMM_cuda/bhsparse.h:297-339):
//   1. k_row_products     per-row intermediate-product upper bound + symbolic bins
//   2. k_bin_scatter      rows -> per-bin queues (device prefix sums, no host pass)
//   3. symbolic kernels   exact nnz(C_i) per row, one kernel family per bin
//   4. scan kernels       nnz(C_i) -> rowptrC (int32 + int64), numeric bins
//   5. numeric kernels    C rows written sorted, directly at rowptrC[i]
// The reference's over-allocated Ct + compaction (create_Ct / copyCt2C,
// bhsparse_cuda.h:285-301, 2813-2911) and its host re-allocation loop
// (:2527-2780) do not exist here: step 3 sizes C exactly.
#pragma once
#include "../../include/bhsparse_b200.h"   // BHB200_DTYPE_*
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>
#include <type_traits>

namespace bhb {

constexpr int EMPTY_KEY = -1;
constexpr int SORT_PAD = 0x7fffffff;
constexpr unsigned FULL = 0xffffffffu;

// ---- value types -------------------------------------------------------------
// The numeric kernels are templates on the value type VT (float, double, c64 and c128 below).  Structure-only
// products (BHB200_DTYPE_NONE) instantiate them with NoVal: an empty type whose arithmetic,
// shuffles, loads and atomics do nothing, so every value load, store and shared-memory access
// compiles away and only the column work is left.  Shared-memory layouts are sized with
// value_bytes<VT> (0 for NoVal, not sizeof = 1) and step over value arrays with vslots<VT>.
namespace novalue {   // (its own namespace: the overloads below would hide CUDA's for int and float inside bhb)
struct NoVal {
    __host__ __device__ constexpr NoVal() {}
    __host__ __device__ constexpr explicit NoVal(int) {}
    __host__ __device__ constexpr NoVal operator*(NoVal) const { return NoVal(); }
    __host__ __device__ constexpr NoVal operator+(NoVal) const { return NoVal(); }
    __host__ __device__ NoVal &operator+=(NoVal) { return *this; }
};
// found by argument-dependent lookup from the kernel templates
__device__ __forceinline__ NoVal __shfl_sync(unsigned, NoVal, int, int = 32) { return NoVal(); }
__device__ __forceinline__ NoVal __shfl_down_sync(unsigned, NoVal, unsigned, int = 32) { return NoVal(); }
__device__ __forceinline__ NoVal __ldg(const NoVal *) { return NoVal(); }
__device__ __forceinline__ NoVal atomicAdd(NoVal *, NoVal) { return NoVal(); }
}  // namespace novalue
using novalue::NoVal;

// Complex products (BHB200_DTYPE_C64) instantiate them with c64: two floats (re, im), 8 bytes and 8-byte
// aligned like float _Complex / std::complex<float> / torch.complex64, so every table, bin and plan sized for
// double holds it unchanged.  The product is the naive formula (re = ar*br - ai*bi, im = ar*bi + ai*br; the
// compiler may contract it into FMAs): each component is a real sum of the 2p real products, which is what the
// value contract bounds.  Gauss's three-multiplication form would not keep that per-component bound.
namespace cplx {   // (its own namespace, as novalue: the overloads below are found by argument-dependent lookup)
struct __align__(8) c64 {
    float re, im;
    c64() = default;   // (trivial: c64 lives in extern shared memory and in __shared__ variables)
    __host__ __device__ constexpr explicit c64(int v) : re((float)v), im(0.f) {}
    __host__ __device__ constexpr c64(float r, float i) : re(r), im(i) {}
    __host__ __device__ c64 operator*(const c64 b) const { return c64(re * b.re - im * b.im, re * b.im + im * b.re); }
    __host__ __device__ c64 operator+(const c64 b) const { return c64(re + b.re, im + b.im); }
    __host__ __device__ c64 &operator+=(const c64 b)
    {
        re += b.re;
        im += b.im;
        return *this;
    }
};
// a*b + c, as fma does for the real types (the pattern kernel's long-row path)
__device__ __forceinline__ c64 fma(const c64 a, const c64 b, const c64 c)
{
    return c64(fmaf(a.re, b.re, fmaf(-a.im, b.im, c.re)), fmaf(a.re, b.im, fmaf(a.im, b.re, c.im)));
}
__device__ __forceinline__ c64 __shfl_sync(unsigned mask, const c64 v, int src, int width = 32)
{
    return c64(::__shfl_sync(mask, v.re, src, width), ::__shfl_sync(mask, v.im, src, width));
}
__device__ __forceinline__ c64 __shfl_down_sync(unsigned mask, const c64 v, unsigned d, int width = 32)
{
    return c64(::__shfl_down_sync(mask, v.re, d, width), ::__shfl_down_sync(mask, v.im, d, width));
}
__device__ __forceinline__ c64 __ldg(const c64 *p)   // one 64-bit read-only load
{
    const float2 t = ::__ldg(reinterpret_cast<const float2 *>(p));
    return c64(t.x, t.y);
}
// per component: two float atomics (shared or global memory); returns the old value
__device__ __forceinline__ c64 atomicAdd(c64 *p, const c64 v)
{
    const float r = ::atomicAdd(&p->re, v.re);
    return c64(r, ::atomicAdd(&p->im, v.im));
}
// complex double: the column-by-column reduction of k_num_bucket_heavy sums in double, as it does for the real types
struct cdbl {
    double re, im;
    cdbl() = default;
    __host__ __device__ constexpr cdbl(double r) : re(r), im(0.0) {}
    __host__ __device__ constexpr cdbl(double r, double i) : re(r), im(i) {}
    __host__ __device__ explicit cdbl(const c64 v) : re(v.re), im(v.im) {}
    __host__ __device__ explicit operator c64() const { return c64((float)re, (float)im); }
    __host__ __device__ cdbl &operator+=(const cdbl b)
    {
        re += b.re;
        im += b.im;
        return *this;
    }
    __host__ __device__ bool operator!=(const double b) const { return re != b || im != 0.0; }
};
__device__ __forceinline__ cdbl __shfl_xor_sync(unsigned mask, const cdbl v, int d, int width = 32)
{
    return cdbl(::__shfl_xor_sync(mask, v.re, d, width), ::__shfl_xor_sync(mask, v.im, d, width));
}
__device__ __forceinline__ cdbl atomicAdd(cdbl *p, const cdbl v)
{
    const double r = ::atomicAdd(&p->re, v.re);
    return cdbl(r, ::atomicAdd(&p->im, v.im));
}

// Complex products in double (BHB200_DTYPE_C128) instantiate them with c128: two doubles (re, im), 16 bytes and
// 16-byte aligned like double _Complex / std::complex<double> / cuDoubleComplex / torch.complex128.  The product is
// the naive formula, as for c64.  Constructible from a double (a real zero or a real sum), so it is also the type
// k_num_bucket_heavy reduces a column in (WideSum below): its components are double already.  The on-chip layouts
// sized for 8-byte values do not all hold it: see the routing next to the bin enums.
struct __align__(16) c128 {
    double re, im;
    c128() = default;   // (trivial, as c64)
    __host__ __device__ constexpr c128(double r) : re(r), im(0.0) {}
    __host__ __device__ constexpr c128(double r, double i) : re(r), im(i) {}
    __host__ __device__ c128 operator*(const c128 b) const { return c128(re * b.re - im * b.im, re * b.im + im * b.re); }
    __host__ __device__ c128 operator+(const c128 b) const { return c128(re + b.re, im + b.im); }
    __host__ __device__ c128 &operator+=(const c128 b)
    {
        re += b.re;
        im += b.im;
        return *this;
    }
    __host__ __device__ bool operator!=(const double b) const { return re != b || im != 0.0; }
};
__device__ __forceinline__ c128 fma(const c128 a, const c128 b, const c128 c)
{
    return c128(::fma(a.re, b.re, ::fma(-a.im, b.im, c.re)), ::fma(a.re, b.im, ::fma(a.im, b.re, c.im)));
}
__device__ __forceinline__ c128 __shfl_sync(unsigned mask, const c128 v, int src, int width = 32)
{
    return c128(::__shfl_sync(mask, v.re, src, width), ::__shfl_sync(mask, v.im, src, width));
}
__device__ __forceinline__ c128 __shfl_down_sync(unsigned mask, const c128 v, unsigned d, int width = 32)
{
    return c128(::__shfl_down_sync(mask, v.re, d, width), ::__shfl_down_sync(mask, v.im, d, width));
}
__device__ __forceinline__ c128 __shfl_xor_sync(unsigned mask, const c128 v, int d, int width = 32)
{
    return c128(::__shfl_xor_sync(mask, v.re, d, width), ::__shfl_xor_sync(mask, v.im, d, width));
}
__device__ __forceinline__ c128 __ldg(const c128 *p)   // one 128-bit read-only load
{
    const double2 t = ::__ldg(reinterpret_cast<const double2 *>(p));
    return c128(t.x, t.y);
}
// per component: two double atomics (shared or global memory); returns the old value
__device__ __forceinline__ c128 atomicAdd(c128 *p, const c128 v)
{
    const double r = ::atomicAdd(&p->re, v.re);
    return c128(r, ::atomicAdd(&p->im, v.im));
}
}  // namespace cplx
using cplx::c64;
using cplx::c128;
static_assert(sizeof(c64) == 8 && alignof(c64) == 8, "complex64 is two floats, 8-byte aligned");
static_assert(sizeof(c128) == 16 && alignof(c128) == 16, "complex128 is two doubles, 16-byte aligned");

// the type k_num_bucket_heavy sums one column's products in: double for the real types, cdbl for c64
template <typename VT>
struct WideSum {
    using type = double;
};
template <>
struct WideSum<c64> {
    using type = cplx::cdbl;
};
template <>
struct WideSum<c128> {
    using type = c128;
};

template <typename VT>
constexpr size_t value_bytes = sizeof(VT);
template <>
constexpr size_t value_bytes<NoVal> = 0;

// elements per value slot when stepping over a value array: p + n * vslots<VT> (NoVal's arrays take no space)
template <typename VT>
constexpr int vslots = value_bytes<VT> ? 1 : 0;

// ---- bins ------------------------------------------------------------------
// Symbolic bins are chosen by p = upper bound of the row (products) and by the row's
// column span; numeric bins by c = exact nnz(C_i), p and the span.  They play the role
// of the reference's 128 segments (bhsparse.h:373-407) but the boundaries follow the
// B200's 227 KB shared memory instead of 32/64/128/256/512/2304.
//
// "span" = (max column - min column + 1) any product of the row can have, from the
// first/last column of every referenced B row.  Rows whose span fits a shared-memory
// bitmap (stencil / banded / FEM rows) take the *range* kernels: a column's position in
// the sorted output row is a popcount prefix of that bitmap, so there is no hashing,
// no probing and no sort.  Everything else takes the hash kernels.
constexpr int SPAN_SMALL = 12288 - 64;    // bitmap of 6 x 2048 columns   (1.5 KB)
constexpr int SPAN_LARGE = 69632 - 64;    // bitmap of 34 x 2048 columns  (8.5 KB)
constexpr int NSUM_SMALL = 6;             // summary words (one bit per 64-column word)
constexpr int NSUM_LARGE = 34;
constexpr int RANGE_NACC_MAX = 512;       // largest nnz(C_i) a range kernel accumulates

enum SymBin {
    SB_ZERO = 0,   // p == 0            -> nnz(C_i) = 0, no kernel   (ESC_0, bhsparse_cuda.h:1582)
    SB_ONE = 1,    // p == 1            -> nnz(C_i) = 1, no kernel   (ESC_1, :1597)
    SB_ESC = 2,    // 2 <= p <= 32      -> warp-shuffle ESC          (ESC_2heap, :653)
    SB_G128 = 3,   // p <= 96           -> group hash, T = 128       (ESC_bitonic, :1400)
    SB_G256 = 4,   // p <= 192
    SB_G512 = 5,   // p <= 384
    SB_G1024 = 6,  // p <= 768
    SB_G2048 = 7,  // p <= 1536
    SB_G4096 = 8,  // p <= 3072
    SB_B8192 = 9,  // p <= 6144         -> block hash                (EM_mergepath, :1902)
    SB_B16384 = 10, // p <= 12288
    SB_B32768 = 11, // p <= 24576
    SB_LARGE = 12,  // beyond           -> global bitmap             (EM_mergepath_global, :2270)
    SB_RANGE_S = 13, // p > 32, span <= SPAN_SMALL -> shared-memory bitmap
    SB_RANGE_L = 14, // p > 32, span <= SPAN_LARGE
    SB_COUNT = 15
};
enum NumBin {
    NB_ZERO = 0,   // c == 0
    NB_ONE = 1,    // p == 1
    NB_ESC = 2,    // 2 <= p <= 32
    NB_G64 = 3,    // c <= 32   T = 64
    NB_G128 = 4,   // c <= 64
    NB_G256 = 5,   // c <= 128
    NB_G512 = 6,   // c <= 256
    NB_G1024 = 7,  // c <= 512
    NB_G2048 = 8,  // c <= 1024
    NB_B4096 = 9,  // c <= 2048  block hash
    NB_B8192 = 10, // c <= 4096
    NB_B16384 = 11, // c <= 8192
    NB_LARGE = 12,  // beyond    global bitmap-rank accumulation
    NB_RANGE_S128 = 13, // span <= SPAN_SMALL, c <= 128  -> bitmap-rank in shared memory
    NB_RANGE_S512 = 14, // span <= SPAN_SMALL, c <= 512
    NB_RANGE_L128 = 15, // span <= SPAN_LARGE, c <= 128
    NB_RANGE_L512 = 16, // span <= SPAN_LARGE, c <= 512
    NB_COPY = 17,       // row already computed by the direct (single-pass) mode: Ct -> C copy only
    NB_COUNT = 18
};
constexpr int MAX_BINS = 24;

// Values of more than 8 bytes (complex128).  The bins above are the rows' shape, computed on the device by kernels
// that do not know the value type; the largest shared-memory tables are sized for 8-byte values and do not hold
// 16-byte ones (k_num_block with T = 16384: 352 KB).  So the host runs the rows of every numeric bin after
// num_hash_last() in the global-bitmap kernel of NB_LARGE: the bins NB_B16384 and NB_LARGE are neighbours in the
// queue, one launch takes both.  bhb200_stats.num_bin_rows counts those rows under NB_LARGE, where they ran.
constexpr size_t SMEM_BLOCK_MAX = 227 * 1024;   // dynamic shared memory of one CTA on sm_100a
inline int num_hash_last(size_t value_size)
{
    return value_size > 8 ? NB_B8192 : NB_B16384;
}

// Masked products (stage_masked.cu): the table size follows m = nnz(M_i), the parallelism p = products
enum MaskBin {
    MB_ZERO = 0,     // p == 0 or m == 0    -> nnz(C_i) = 0, no kernel
    MB_ESC = 1,      // p <= 32             -> warp per row, one product per lane
    MB_W64 = 2,      // m <= 32, p <= MASK_WARP_MAX_P -> warp per row, T = 64
    MB_W256 = 3,     // m <= 128
    MB_W1024 = 4,    // m <= 512
    MB_C1024 = 5,    // m <= 512, more products -> CTA per row, T = 1024
    MB_C4096 = 6,    // m <= 2048
    MB_C16384 = 7,   // m <= 8192
    MB_GLOBAL = 8,   // beyond the shared-memory tables: binary search in M_i, values in global scratch
    MB_COUNT = 9
};
// Values of more than 8 bytes: the table of MB_C16384 (264 KB for 16-byte values) does not fit, its rows run in the
// kernel of MB_GLOBAL (its neighbour in the queue: one launch); bhb200_stats.mask_bin_rows counts them there.
inline int mask_table_last(size_t value_size)
{
    return value_size > 8 ? MB_C4096 : MB_C16384;
}
constexpr int MASK_WARP_MAX_P = 2048;
constexpr int MASK_TABLE_MAX = 8192;
__host__ __device__ __forceinline__ int mask_bin_of(int p, int m)
{
    if (p == 0 || m == 0) return MB_ZERO;
    if (p <= 32) return MB_ESC;
    if (m > MASK_TABLE_MAX) return MB_GLOBAL;
    if (p <= MASK_WARP_MAX_P && m <= 512) return m <= 32 ? MB_W64 : m <= 128 ? MB_W256 : MB_W1024;
    return m <= 512 ? MB_C1024 : m <= 2048 ? MB_C4096 : MB_C16384;
}
// Counters::bad_M bits
constexpr int MASK_BAD_ROWPTR = 1, MASK_BAD_ORDER = 2, MASK_BAD_COL = 4;

__host__ __device__ __forceinline__ int sym_bin_of(int p, int span)
{
    if (p <= 1) return p;
    if (p <= 32) return SB_ESC;
    if (span <= SPAN_SMALL) return SB_RANGE_S;
    if (span <= SPAN_LARGE) return SB_RANGE_L;
    if (p <= 96) return SB_G128;
    if (p <= 192) return SB_G256;
    if (p <= 384) return SB_G512;
    if (p <= 768) return SB_G1024;
    if (p <= 1536) return SB_G2048;
    if (p <= 3072) return SB_G4096;
    if (p <= 6144) return SB_B8192;
    if (p <= 12288) return SB_B16384;
    if (p <= 24576) return SB_B32768;
    return SB_LARGE;
}
__host__ __device__ __forceinline__ int num_bin_of(int p, int c, int span)
{
    if (p <= 1) return p;
    if (p <= 32) return NB_ESC;
    if (c <= RANGE_NACC_MAX) {
        if (span <= SPAN_SMALL) return c <= 128 ? NB_RANGE_S128 : NB_RANGE_S512;
        if (span <= SPAN_LARGE) return c <= 128 ? NB_RANGE_L128 : NB_RANGE_L512;
    }
    if (c <= 32) return NB_G64;
    if (c <= 64) return NB_G128;
    if (c <= 128) return NB_G256;
    if (c <= 256) return NB_G512;
    if (c <= 512) return NB_G1024;
    if (c <= 1024) return NB_G2048;
    if (c <= 2048) return NB_B4096;
    if (c <= 4096) return NB_B8192;
    if (c <= 8192) return NB_B16384;
    return NB_LARGE;
}

// Device-side counters of one spgemm call (one small struct, zeroed per call,
// copied back once after stage 1 and once after the scan).
struct Counters {
    unsigned long long products;   // sum of per-row products (_nnzCt_full, bhsparse.h:368)
    unsigned long long nnzC;       // set by the scan
    unsigned long long pool_cursor;  // word-list pool: entries handed out by the symbolic range kernel
    int max_row_products;
    int row_overflow;              // a row's product count did not fit int32
    int bad_B;                     // a row of B is not strictly ascending / has a column outside [0, n)
    int bad_A;                     // a column of A is outside [0, k)
    int pat_miss;                  // pattern mode: an entry's offset is not in the (cached) offset lists
    int a_col_range[2];            // pattern mode: {max column of A, INT_MAX - min column of A} (which rows of B matter)
    int sym_bin[MAX_BINS];
    int num_bin[MAX_BINS];
    int sym_cursor[MAX_BINS];
    int num_cursor[MAX_BINS];
    int sample_max[MAX_BINS];      // direct mode: largest nnz(C_i) among the sampled rows of a symbolic bin
    int retry_cnt[MAX_BINS];       // direct mode: rows of a bin that overflowed their speculated capacity
    unsigned long long sample_sum[MAX_BINS];   // direct mode: sum of nnz(C_i) over the sampled rows
    unsigned long long sym_bin_products[MAX_BINS];   // intermediate products per symbolic bin (sizes the heavy rows' staging)
    unsigned long long heavy_cursor;                 // bump allocator of k_num_bucket_heavy's staging
    unsigned long long num_bin_products[MAX_BINS];
    unsigned long long num_bin_nnzc[MAX_BINS];
    unsigned long long num_bin_nnza[MAX_BINS];
    int mask_bin[MB_COUNT];        // masked product: rows per masked bin (k_mask_bins)
    int mask_cursor[MB_COUNT];
    int bad_M;                     // masked product: MASK_BAD_* of the mask
    // transposed operands (stage_transpose.cu): bit 0 / 1 = a column of the stored A / B outside its range.
    // Last member: written by the transposition only, so a transposition done by bhb200_warmup is still
    // reported by the next bhb200_spgemm (the per-call zeroing stops at CTR_ZERO_BYTES)
    int bad_T;
};
constexpr size_t CTR_ZERO_BYTES = offsetof(Counters, bad_T);
struct BinOffsets {
    int off[MAX_BINS + 1];
};

// Direct (single-pass) mode.  For a symbolic bin whose sampled rows all have nnz(C_i) <= cap
// the numeric kernel runs without a symbolic pass: table sized for `cap`, each row written
// sorted into a staging buffer at ct_off[row] (cap entries per row -- the reference's
// over-allocated Ct, bhsparse_cuda.h:285-301), nnz(C_i) into rc[row]; after the row-pointer
// scan k_copy_ct moves the rows to their final place (copyCt2C, :2813-2911).  A row with more
// than `cap` distinct columns is detected while it is accumulated, gets ct_off = -1 and goes
// to its bin's retry queue, i.e. through the ordinary symbolic + numeric kernels.
struct DirectOut {
    int *rc;                 // [m] nnz(C_i)
    long long *ct_off;       // [m] first staging entry of the row, or -1
    int *ctcol;              // staging columns
    void *ctval;             // staging values
    long long ct_base;       // first staging entry of this bin
    int *retry_queue;        // this bin's retry rows
    int *retry_cnt;          // their number (device)
    // wide bins run as two launches over the same queue, each with the table size its rows need:
    // a launch takes the rows with p_lo < products <= p_hi and stages row q at ct_base + q*ct_stride
    const int *prod = nullptr;
    int p_lo = 0, p_hi = 0x7fffffff;
    int ct_stride = 0;       // 0: the kernel's own capacity
    unsigned long long *bump = nullptr;   // k_num_bucket3: stage rows by atomic bump of this cursor (products each) instead of q * ct_stride
    const int *count_dev = nullptr;       // k_num_bucket_heavy as the retry kernel: number of queued rows, on the device
};

// Word lists: the symbolic range kernel stores, per row, the non-empty 64-column words of
// the row's bitmap (index + bits) in a device pool; the numeric range kernel rebuilds its
// bitmap and the rank prefixes from that list instead of walking all products a second
// time.  wl_cnt[row] < 0: the pool was full, the numeric kernel marks the row itself.
struct WordLists {
    long long *off;                  // [m] first pool entry of the row
    int *cnt;                        // [m] entries, or -1
    unsigned *idx;                   // [cap] word index inside the row's bitmap
    unsigned long long *bits;        // [cap]
    long long cap;
};

// ---- hashing ---------------------------------------------------------------
template <int LOG2T>
__device__ __forceinline__ int hash_slot(int c)
{
    return (int)(((unsigned)c * 2654435761u) >> (32 - LOG2T));
}

// Insert column c into an open-addressing table (linear probing).  Returns the
// slot; is_new is true for the thread whose CAS claimed an empty slot.
// Words of a per-CTA column bitmap for n columns (large-row kernels), padded to 16 bytes.
__host__ __device__ __forceinline__ int large_nwords(int n)
{
    return (int)((((long long)n + 31) / 32 + 3) & ~3LL);
}

// Dynamic B-row scheduling for CTA-per-row kernels: the warps of a CTA take the row's A entries
// from a shared-memory counter instead of a fixed stride, so a warp that drew a long B row
// does not hold the others at the next barrier.
__device__ __forceinline__ int take_next(int *counter, int lane)
{
    int j = 0;
    if (lane == 0) j = atomicAdd(counter, 1);
    return __shfl_sync(FULL, j, 0);
}

__device__ __forceinline__ int take_next_n(int *counter, int lane, int n)
{
    int j = 0;
    if (lane == 0) j = atomicAdd(counter, n);
    return __shfl_sync(FULL, j, 0);
}

// B rows of one A row, for the CTA-per-row kernels that accumulate in GLOBAL memory (large rows).
// Warps take B rows from a shared counter; a B row longer than LONG_B would keep one warp busy for
// hundreds of dependent global-memory round trips (R-MAT hub columns: thousands of elements), so
// it is listed and afterwards strided over by the whole CTA. f(j, p_first, p_end, p_stride)
// handles the elements p_first, p_first + p_stride, ... < p_end of the B row of A entry j.
// s_next / s_nlong must be zero on entry (and a barrier passed); all threads must call.
constexpr int LONG_B = 256;
constexpr int LONG_CAP = 96;
template <typename F>
__device__ __forceinline__ void cta_for_each_b_row(const int a0, const int a1, const int *__restrict__ colA,
                                                   const int *__restrict__ rowptrB, int *s_next, int *s_nlong,
                                                   int *s_long, F &&f)
{
    const int lane = threadIdx.x & 31;
    for (int j = a0 + take_next(s_next, lane); j < a1; j = a0 + take_next(s_next, lane)) {
        const int k = colA[j];
        const int bs = rowptrB[k], be = rowptrB[k + 1];
        if (be - bs > LONG_B) {
            int idx = 0;
            if (lane == 0) idx = atomicAdd(s_nlong, 1);
            idx = __shfl_sync(FULL, idx, 0);
            if (idx < LONG_CAP) {
                if (lane == 0) s_long[idx] = j;
                continue;
            }
        }
        f(j, bs + lane, be, 32);
    }
    __syncthreads();
    const int nlong = min(*s_nlong, LONG_CAP);
    for (int i = 0; i < nlong; ++i) {
        const int j = s_long[i];
        const int k = colA[j];
        f(j, rowptrB[k] + (int)threadIdx.x, rowptrB[k + 1], (int)blockDim.x);
    }
}


template <int LOG2T>
__device__ __forceinline__ int table_insert(int *keys, int c, bool &is_new)
{
    constexpr int MASK = (1 << LOG2T) - 1;
    volatile int *vk = keys;
    int h = hash_slot<LOG2T>(c);
    is_new = false;
    while (true) {
        int k = vk[h];
        if (k == c) return h;
        if (k == EMPTY_KEY) {
            int old = atomicCAS(&keys[h], EMPTY_KEY, c);
            if (old == EMPTY_KEY) {
                is_new = true;
                return h;
            }
            if (old == c) return h;
        }
        h = (h + 1) & MASK;
    }
}
template <int LOG2T>
__device__ __forceinline__ int table_find(const int *keys, int c)
{
    constexpr int MASK = (1 << LOG2T) - 1;
    int h = hash_slot<LOG2T>(c);
    while (keys[h] != c) h = (h + 1) & MASK;
    return h;
}

// ---- sub-warp groups ---------------------------------------------------------
template <int G>
__device__ __forceinline__ unsigned group_mask(int lane)
{
    if (G == 32) return FULL;
    return ((1u << (G & 31)) - 1u) << (lane & ~(G - 1));
}

// Bitonic sort of N = G*R keys held R per lane in blocked order (element index
// i = gl*R + r), ascending.  Strides below R are register compare-exchanges,
// strides of R and above are one __shfl_xor + one min/max per key.
template <int G, int R>
__device__ __forceinline__ void bitonic_sort_regs(int (&x)[R], const int gl, const unsigned gmask)
{
    constexpr int N = G * R;
#pragma unroll
    for (int k = 2; k <= N; k <<= 1) {
#pragma unroll
        for (int j = k >> 1; j > 0; j >>= 1) {
            if (j >= R) {
                const int d = j / R;
                const bool lower = (gl & d) == 0;
#pragma unroll
                for (int r = 0; r < R; ++r) {
                    const int i = gl * R + r;
                    const bool asc = (k == N) ? true : ((i & k) == 0);
                    const int y = __shfl_xor_sync(gmask, x[r], d, G);
                    x[r] = (lower == asc) ? min(x[r], y) : max(x[r], y);
                }
            } else {
#pragma unroll
                for (int r = 0; r < R; ++r) {
                    if ((r & j) == 0) {
                        const int i = gl * R + r;
                        const bool asc = (k == N) ? true : ((i & k) == 0);
                        const int lo = min(x[r], x[r + j]);
                        const int hi = max(x[r], x[r + j]);
                        x[r] = asc ? lo : hi;
                        x[r + j] = asc ? hi : lo;
                    }
                }
            }
        }
    }
}

// Bitonic sort of sk[0..N) (N a power of two) in shared memory by one group.
template <int G>
__device__ __forceinline__ void bitonic_sort_smem_group(int *sk, const int N, const int gl, const unsigned gmask)
{
    for (int k = 2; k <= N; k <<= 1) {
        for (int j = k >> 1; j > 0; j >>= 1) {
            for (int t = gl; t < (N >> 1); t += G) {
                const int i = ((t & ~(j - 1)) << 1) | (t & (j - 1));
                const int p = i | j;
                const int a = sk[i], b = sk[p];
                const bool asc = (i & k) == 0;
                if ((a > b) == asc) {
                    sk[i] = b;
                    sk[p] = a;
                }
            }
            __syncwarp(gmask);
        }
    }
}

// Same network with the stage loops rolled (only the per-key work is unrolled): for R >= 16
// the fully unrolled version is 30-70 KB of straight-line code and thrashes the
// instruction cache (measured: the R=16 CTA sort got slower when unrolled).
template <int G, int R>
__device__ __forceinline__ void bitonic_sort_regs_rolled(int (&x)[R], const int gl)
{
    constexpr int N = G * R;
#pragma unroll 1
    for (int k = 2; k <= N; k <<= 1) {
#pragma unroll 1
        for (int j = k >> 1; j >= R; j >>= 1) {
            const int d = j / R;
            const bool lower = (gl & d) == 0;
#pragma unroll
            for (int r = 0; r < R; ++r) {
                const bool asc = (((gl * R + r) & k) == 0);
                const int y = __shfl_xor_sync(FULL, x[r], d, G);
                x[r] = (lower == asc) ? min(x[r], y) : max(x[r], y);
            }
        }
#pragma unroll
        for (int j = R >> 1; j > 0; j >>= 1) {
            if (j < k) {
#pragma unroll
                for (int r = 0; r < R; ++r) {
                    if ((r & j) == 0) {
                        const bool asc = (((gl * R + r) & k) == 0);
                        const int lo = min(x[r], x[r + j]);
                        const int hi = max(x[r], x[r + j]);
                        x[r] = asc ? lo : hi;
                        x[r + j] = asc ? hi : lo;
                    }
                }
            }
        }
    }
}

// Bitonic sort of N = THREADS*K keys by a whole CTA, K keys per thread in blocked order
// (element index i = tid*K + r), ascending.  Strides < K are register compare-exchanges,
// strides < 32*K one __shfl_xor per key, and only the log2(THREADS/32) largest strides go
// through shared memory (`xchg`, N ints, stored transposed so the exchange is bank-conflict
// free) -- 2 barriers for each of those instead of one per stage for an in-smem network.
// Stage loops are rolled (see above).
template <int K, int THREADS>
__device__ __forceinline__ void block_bitonic_sort_regs(int (&x)[K], int *xchg)
{
    constexpr int N = THREADS * K;
    const int tid = threadIdx.x;
#pragma unroll 1
    for (int k = 2; k <= N; k <<= 1) {
#pragma unroll 1
        for (int j = k >> 1; j >= K; j >>= 1) {
            const int dt = j / K;   // partner thread = tid ^ dt
            const bool lower = (tid & dt) == 0;
            if (dt >= 32) {         // another warp: through shared memory
                __syncthreads();
#pragma unroll
                for (int r = 0; r < K; ++r) xchg[r * THREADS + tid] = x[r];
                __syncthreads();
#pragma unroll
                for (int r = 0; r < K; ++r) {
                    const bool asc = (((tid * K + r) & k) == 0);
                    const int y = xchg[r * THREADS + (tid ^ dt)];
                    x[r] = (lower == asc) ? min(x[r], y) : max(x[r], y);
                }
            } else {
#pragma unroll
                for (int r = 0; r < K; ++r) {
                    const bool asc = (((tid * K + r) & k) == 0);
                    const int y = __shfl_xor_sync(FULL, x[r], dt);
                    x[r] = (lower == asc) ? min(x[r], y) : max(x[r], y);
                }
            }
        }
#pragma unroll
        for (int j = K >> 1; j > 0; j >>= 1) {
            if (j < k) {
#pragma unroll
                for (int r = 0; r < K; ++r) {
                    if ((r & j) == 0) {
                        const bool asc = (((tid * K + r) & k) == 0);
                        const int lo = min(x[r], x[r + j]);
                        const int hi = max(x[r], x[r + j]);
                        x[r] = asc ? lo : hi;
                        x[r + j] = asc ? hi : lo;
                    }
                }
            }
        }
    }
}

// Fully unrolled variant for small K (measured faster than the rolled one for K = 4).
template <int K, int THREADS>
__device__ __forceinline__ void block_bitonic_sort_regs_unrolled(int (&x)[K], int *xchg)
{
    constexpr int N = THREADS * K;
    const int tid = threadIdx.x;
#pragma unroll
    for (int k = 2; k <= N; k <<= 1) {
#pragma unroll
        for (int j = k >> 1; j > 0; j >>= 1) {
            if (j >= 32 * K) {
                const int dt = j / K;
                const bool lower = (tid & dt) == 0;
                __syncthreads();
#pragma unroll
                for (int r = 0; r < K; ++r) xchg[r * THREADS + tid] = x[r];
                __syncthreads();
#pragma unroll
                for (int r = 0; r < K; ++r) {
                    const bool asc = (k == N) ? true : (((tid * K + r) & k) == 0);
                    const int y = xchg[r * THREADS + (tid ^ dt)];
                    x[r] = (lower == asc) ? min(x[r], y) : max(x[r], y);
                }
            } else if (j >= K) {
                const int d = j / K;
                const bool lower = (tid & d) == 0;
#pragma unroll
                for (int r = 0; r < K; ++r) {
                    const bool asc = (k == N) ? true : (((tid * K + r) & k) == 0);
                    const int y = __shfl_xor_sync(FULL, x[r], d);
                    x[r] = (lower == asc) ? min(x[r], y) : max(x[r], y);
                }
            } else {
#pragma unroll
                for (int r = 0; r < K; ++r) {
                    if ((r & j) == 0) {
                        const bool asc = (k == N) ? true : (((tid * K + r) & k) == 0);
                        const int lo = min(x[r], x[r + j]);
                        const int hi = max(x[r], x[r + j]);
                        x[r] = asc ? lo : hi;
                        x[r + j] = asc ? hi : lo;
                    }
                }
            }
        }
    }
}

__device__ __forceinline__ int next_pow2(int v)
{
    return v <= 2 ? 2 : 1 << (32 - __clz(v - 1));
}

template <typename T>
__device__ __forceinline__ T warp_sum(T v)
{
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) v += __shfl_xor_sync(FULL, v, d);
    return v;
}

// Block-wide sum; every thread gets the result.  `red` holds >= 33 elements.
template <typename T>
__device__ __forceinline__ T block_sum(T v, T *red)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    v = warp_sum(v);
    __syncthreads();
    if (lane == 0) red[warp] = v;
    __syncthreads();
    if (warp == 0) {
        T w = (lane < (int)((blockDim.x + 31) >> 5)) ? red[lane] : T(0);
        w = warp_sum(w);
        if (lane == 0) red[32] = w;
    }
    __syncthreads();
    return red[32];
}

// Resident CTAs per SM for a launch configuration (registers, shared memory and thread
// limits together).  Persistent grids are sized with this: a grid sized from shared memory
// alone ran a second, nearly empty wave when registers were the tighter limit.
template <typename KernelT>
inline int resident_blocks(KernelT kernel, int threads, size_t smem)
{
    int nb = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, kernel, threads, smem) != cudaSuccess || nb < 1) {
        cudaGetLastError();
        nb = 1;
    }
    return nb;
}

// ---- launch interface (defined in the stage_*.cu files, called by context.cu) -
struct Csr {
    const int *rowptr;
    const int *col;
    const void *val;
};
struct LaunchCtx {
    cudaStream_t stream;
    int sm_count;
    int *launches;   // incremented per kernel launch
    int max_span = SPAN_SMALL;   // rows with a wider column span never take the range kernels
};

// stage_count.cu
cudaError_t launch_b_row_ranges(const LaunchCtx &lc, int k, int n, Csr B, int4 *brange, Counters *ctr);
cudaError_t launch_row_products(const LaunchCtx &lc, int m, int k, int nnzA, Csr A, Csr B, const int4 *brange, int *prod,
                                int *rc, int *rlo, int *rspan, Counters *ctr);
// spec_mask: bit b set = symbolic bin b ran in direct mode (rows with ct_off >= 0 go to NB_COPY)
cudaError_t launch_bin_scatter(const LaunchCtx &lc, bool numeric, int m, const int *prod, const int *rc,
                               const int *rspan, unsigned spec_mask, const long long *ct_off, const BinOffsets &offs,
                               Counters *ctr, int *queue);
cudaError_t launch_scan(const LaunchCtx &lc, int m, const int *rowptrA, const int *prod, const int *rc,
                        const int *rspan, unsigned spec_mask, const long long *ct_off, int64_t *rowoff64,
                        int *rowptr32, long long *blocksums, Counters *ctr);
size_t scan_blocksum_count(int m);
// stage_transpose.cu: X (rows x cols, nnz entries, int32 CSR) -> X^T (cols x rows) and perm with
// out.val[p] = X.val[perm[p]]; a stored column outside [0, cols) is replaced by 0 and raises bad_bit in *bad
struct TransposeOut {
    int *rowptr;   // [cols + 1]
    int *col;      // [nnz]
    void *val;     // [nnz]
    int *perm;     // [nnz]
};
size_t transpose_scratch_bytes(int nnz, int cols);
int transpose_passes(int cols);
// conj: complex values are conjugated as they move (BHB200_OP_C)
cudaError_t launch_transpose(const LaunchCtx &lc, int dtype, bool conj, int rows, int cols, int nnz, Csr X, TransposeOut out,
                             void *scratch, int *bad, int bad_bit);
// values again through the permutation of the last transposition: valT[p] = val[perm[p]] (conjugated with conj)
cudaError_t launch_regather(const LaunchCtx &lc, int dtype, bool conj, int nnz, const void *val, const int *perm, void *valT);
// stage_masked.cu: the mask M (m x n, structural) and where the masked kernels put their rows
struct MaskCsr {
    const int *rowptr;
    const int *col;
    int nnz;
};
struct MaskOut {
    int *rc;                // [m] nnz(C_i)
    long long *ct_off;      // [m] = rowptrM[i]: rows are staged at their mask offsets
    int *ctcol;             // staging columns (nnzM)
    void *ctval;            // staging values (nnzM)
    void *acc;              // MB_GLOBAL: values per mask entry (nnzM), or null
    unsigned char *hit;     // MB_GLOBAL: hit flag per mask entry (nnzM), or null
};
cudaError_t launch_mask_bins(const LaunchCtx &lc, int m, int n, MaskCsr M, const int *prod, Counters *ctr);
cudaError_t launch_mask_scatter(const LaunchCtx &lc, int m, MaskCsr M, const int *prod, const BinOffsets &offs, Counters *ctr,
                                int *queue, int *rc, long long *ct_off);
cudaError_t launch_mask_bin(const LaunchCtx &lc, int dtype, int bin, const int *queue, int count, Csr A, Csr B,
                            const int4 *brange, MaskCsr M, MaskOut o);
// stage_small.cu
cudaError_t launch_sym_esc(const LaunchCtx &lc, const int *queue, int count, int n, Csr A, Csr B, int *rc);
cudaError_t launch_num_single(const LaunchCtx &lc, int dtype, const int *queue, int count, Csr A, Csr B,
                              const int64_t *rowoff, int *colC, void *valC);
cudaError_t launch_num_esc(const LaunchCtx &lc, int dtype, const int *queue, int count, int n, Csr A, Csr B,
                           const int64_t *rowoff, int *colC, void *valC);
// stage_symbolic.cu
// qstride > 1: only every qstride-th row of the queue (sampling); bin_max / bin_sum: atomicMax / sum of
// the counts; dcount: the number of rows is read from device memory (retry queues), `count` is its upper bound
cudaError_t launch_sym_hash(const LaunchCtx &lc, int bin, int G, const int *queue, int count, Csr A, Csr B, int *rc,
                            int qstride = 1, int *bin_max = nullptr, const int *dcount = nullptr,
                            unsigned long long *bin_sum = nullptr);
cudaError_t launch_sym_large(const LaunchCtx &lc, const int *queue, int count, int n, Csr A, Csr B, int *rc,
                             unsigned *bitmap_scratch, int scratch_blocks);
// column CDF of the intermediate products (stage_bucket.cu): colcountA [k+1] ints, hist [4096] u64, cdf [4097] u32
cudaError_t launch_build_cdf(const LaunchCtx &lc, int m, int k, int n, int nnzA, Csr A, Csr B, int *colcountA,
                             unsigned long long *hist, unsigned *cdf, int *shift_out);
// resident CTAs (= private scratch sets) of the large-row kernels for n columns
int large_scratch_blocks(int sm_count, int n);
// stage_range.cu (symbolic) / stage_numeric (numeric) -- shared-memory bitmap kernels
// (the launchers pick the 128-bit vectorised kernels of stage_range_vec.cuh when B is 16-byte aligned)
cudaError_t launch_sym_range(const LaunchCtx &lc, int nsum, const int *queue, int count, Csr A, Csr B, const int *rlo,
                             int *rc, Counters *ctr, WordLists wl);

// The numeric kernels of one value type (stage_numeric_f32.cu / _f64.cu / _none.cu / _c64.cu / _c128.cu); values
// are float, double, complex64 or complex128 as the operands are, or none (NoVal: columns only, value pointers never
// read).  The five types compile in five translation units, in parallel.
struct ColumnCdf {
    const unsigned *cdf;   // [CDF_KNOTS + 1], non-decreasing, cdf[0] = 0
    int shift;             // column >> shift < CDF_KNOTS
};
struct NumericKernels {
    cudaError_t (*hash)(const LaunchCtx &lc, int bin, int G, const int *queue, int count, Csr A, Csr B,
                        const int64_t *rowoff, int *colC, void *valC);
    cudaError_t (*large)(const LaunchCtx &lc, const int *queue, int count, int n, Csr A, Csr B, const int64_t *rowoff,
                         int *colC, void *valC, unsigned *bitmap_scratch, int *prefix_scratch, int scratch_blocks);
    cudaError_t (*range)(const LaunchCtx &lc, int nsum, int nacc, const int *queue, int count, Csr A, Csr B,
                         const int *rlo, const int64_t *rowoff, int *colC, void *valC, WordLists wl);
    // direct mode: cap in {32, 64, 128} speculated (rows may overflow into the retry queue), or
    // {256, ..., 8192} for bins whose product bound is below cap (no overflow possible)
    cudaError_t (*direct)(const LaunchCtx &lc, int cap, int G, const int *queue, int count, Csr A, Csr B, DirectOut d);
    // bucket-sort ESC for rows that barely compress (stage_bucket.cuh): wide direct bins, cap >= 512
    cudaError_t (*bucket)(const LaunchCtx &lc, int cap, const int *queue, int count, Csr A, Csr B, DirectOut d,
                          ColumnCdf cdf);
    // warp-per-row bucket sort (k_num_bucket3w): bins SB_G128 (capw 128) / SB_G256 (capw 256) whose rows barely compress;
    // sg = lanes per B row (8 | 32); rows staged `stride` apart, rows with more outputs go to d.retry_queue
    cudaError_t (*bucket3w)(const LaunchCtx &lc, int capw, int sg, const int *queue, int count, Csr A, Csr B, DirectOut d,
                            ColumnCdf cdf, int stride);
    // heavy rows (more products than fit on chip): sliced bucket sort, staged at ct_base + bump(cursor, products)
    cudaError_t (*heavy)(const LaunchCtx &lc, const int *queue, int count, Csr A, Csr B, DirectOut d, ColumnCdf cdf,
                         unsigned long long *cursor);
    // second formulation (k_num_bucket_heavy2): rows with more than d.p_lo products, partitioned by slice through their own
    // staging area; rows it cannot slice go to d.retry_queue / d.retry_cnt for `heavy` (d.count_dev)
    cudaError_t (*heavy2)(const LaunchCtx &lc, const int *queue, int count, Csr A, Csr B, DirectOut d, ColumnCdf cdf,
                          unsigned long long *cursor);
    // staged rows -> C; avg_row = staged entries per row of the launch: short rows are copied 32 rows per warp
    cudaError_t (*copy_ct)(const LaunchCtx &lc, const int *queue, int count, const int64_t *rowoff, const long long *ct_off,
                           const int *ctcol, const void *ctval, int *colC, void *valC, double avg_row);
};
extern const NumericKernels NUMERIC_F32, NUMERIC_F64, NUMERIC_NONE, NUMERIC_C64, NUMERIC_C128;

// The one place a BHB200_DTYPE_* becomes a value type: f(VT()) with VT = float, double, NoVal, c64 or c128 (host code;
// the launchers call it with a generic lambda and take the type as decltype of its argument).
template <typename F>
inline decltype(auto) dispatch_value_type(int dtype, F &&f)
{
    switch (dtype) {
    case BHB200_DTYPE_F64: return f(double());
    case BHB200_DTYPE_NONE: return f(NoVal());
    case BHB200_DTYPE_C64: return f(c64());
    case BHB200_DTYPE_C128: return f(c128());
    default: return f(float());
    }
}

inline const NumericKernels &numeric_kernels(int dtype)
{
    return dispatch_value_type(dtype, [](auto v) -> const NumericKernels & {
        using VT = decltype(v);
        if constexpr (std::is_same_v<VT, double>) return NUMERIC_F64;
        else if constexpr (std::is_same_v<VT, NoVal>) return NUMERIC_NONE;
        else if constexpr (std::is_same_v<VT, c64>) return NUMERIC_C64;
        else if constexpr (std::is_same_v<VT, c128>) return NUMERIC_C128;
        else return NUMERIC_F32;
    });
}

}  // namespace bhb
