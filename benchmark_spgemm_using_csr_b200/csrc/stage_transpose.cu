// stage_transpose.cu -- stable CSR transpose on the device: the effective operands op(A) = A^T and
// op(B) = B^T of bhb200_init_data_op_* / bhb200_init_data_device_op (no reference counterpart: the
// reference multiplies the operands as stored, bhsparse.h:180-258).
//
// LSD radix sort of the column keys with the entry index as payload.  The stored entries are in
// row-major order and every pass is stable, so the result is in (column, row) order whatever the
// order inside the stored rows.  Per pass of <= 11 bits (two passes up to 2^22 columns):
//   k_tr_hist     per tile of 8192 entries: digit counts (shared memory, warp-aggregated with
//                 __match_any_sync: a hub column costs one shared atomic per warp step)
//   k_tr_scan     one CTA per digit: exclusive scan of its tile counts + the digit total
//   k_tr_scatter  per tile: per-warp digit counts (warp-private, no atomics), their prefix over the
//                 warps, then the stable scatter with the rank of each lane among its digit peers;
//                 the last pass writes perm, the columns of X^T (rows of X) and gathers the values
// The row of each entry comes from an expanded row index (k_tr_rows), the row pointers of X^T from a
// lower bound per column in the sorted keys (k_tr_rowptr).  A column outside [0, cols) is replaced by
// 0 (so every array written stays in bounds) and raises `bad_bit` in *bad.
#include "common.cuh"

#include <algorithm>

namespace bhb {

namespace {

constexpr int TR_THREADS = 512;
constexpr int TR_WARPS = TR_THREADS / 32;
constexpr int TR_ITEMS = 16;                      // entries per lane and tile
constexpr int TR_TILE = TR_THREADS * TR_ITEMS;    // 8192 entries
constexpr int TR_MAX_BITS = 11;
constexpr int TR_MAX_BINS = 1 << TR_MAX_BITS;

__device__ __forceinline__ unsigned lanemask_lt()
{
    unsigned m;
    asm("mov.u32 %0, %%lanemask_lt;" : "=r"(m));
    return m;
}

// Values only move here.  The conjugate transpose of complex64 operands (BHB200_OP_C) moves them as Conj8: 8-byte words
// with the sign bit of the imaginary part (bit 63) flipped, which conjugates NaN, inf and zero exactly.
struct Conj8 {
    unsigned long long bits;
};
template <typename V>
__device__ __forceinline__ V moved(const V v)
{
    return v;
}
__device__ __forceinline__ Conj8 moved(const Conj8 v) { return Conj8{v.bits ^ 0x8000000000000000ull}; }
// complex128 moves as 16-byte words (Move16); its conjugate as Conj16, bit 63 of the imaginary double flipped
struct __align__(16) Move16 {
    unsigned long long re, im;
};
struct __align__(16) Conj16 {
    unsigned long long re, im;
};
__device__ __forceinline__ Conj16 moved(const Conj16 v) { return Conj16{v.re, v.im ^ 0x8000000000000000ull}; }

__device__ __forceinline__ int masked_key(int key, int cols)
{
    return (unsigned)key < (unsigned)cols ? key : 0;
}

// row index of every stored entry (one warp per row; entries outside [0, nnz) are not written)
__global__ void __launch_bounds__(256) k_tr_rows(const int rows, const int nnz, const int *__restrict__ rowptr,
                                                 int *__restrict__ rowidx)
{
    const long long r = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (r >= rows) return;
    const int lane = threadIdx.x & 31;
    const int s = max(rowptr[r], 0), e = min(rowptr[r + 1], nnz);
    for (int p = s + lane; p < e; p += 32) rowidx[p] = (int)r;
}

__global__ void __launch_bounds__(TR_THREADS) k_tr_hist(const int nnz, const int cols, const int *__restrict__ keys,
                                                        const int shift, const int nbins, const int ntiles,
                                                        unsigned *__restrict__ counts, int *__restrict__ bad,
                                                        const int bad_bit)
{
    __shared__ unsigned h[TR_MAX_BINS];
    __shared__ int s_bad;
    for (int d = threadIdx.x; d < nbins; d += TR_THREADS) h[d] = 0u;
    if (threadIdx.x == 0) s_bad = 0;
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const long long base = (long long)blockIdx.x * TR_TILE + warp * (32 * TR_ITEMS);
    const unsigned dmask = (unsigned)nbins - 1u;
    bool badl = false;
#pragma unroll 4
    for (int i = 0; i < TR_ITEMS; ++i) {
        const long long e = base + i * 32 + lane;
        const bool act = e < nnz;
        const int raw = act ? keys[e] : 0;
        badl |= act && (unsigned)raw >= (unsigned)cols;
        const unsigned d = act ? ((unsigned)masked_key(raw, cols) >> shift) & dmask : 0xffffffffu;
        const unsigned peers = __match_any_sync(FULL, d);
        if (act && (peers & lanemask_lt()) == 0u) atomicAdd(&h[d], (unsigned)__popc(peers));
    }
    if (__any_sync(FULL, badl) && lane == 0) s_bad = 1;
    __syncthreads();
    for (int d = threadIdx.x; d < nbins; d += TR_THREADS) counts[(size_t)d * ntiles + blockIdx.x] = h[d];
    if (threadIdx.x == 0 && s_bad && bad) atomicOr(bad, bad_bit);
}

// one CTA per digit: counts[d][0 .. ntiles) -> exclusive prefix in place, totals[d] = their sum
__global__ void __launch_bounds__(256) k_tr_scan(const int ntiles, unsigned *__restrict__ counts,
                                                 unsigned *__restrict__ totals)
{
    __shared__ unsigned s_w[8];
    __shared__ unsigned s_carry;
    unsigned *row = counts + (size_t)blockIdx.x * ntiles;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (threadIdx.x == 0) s_carry = 0u;
    __syncthreads();
    for (int t0 = 0; t0 < ntiles; t0 += 256 * 4) {
        const int t = t0 + threadIdx.x * 4;
        unsigned v[4], sum = 0u;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            v[j] = t + j < ntiles ? row[t + j] : 0u;
            sum += v[j];
        }
        unsigned incl = sum;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const unsigned y = __shfl_up_sync(FULL, incl, d);
            if (lane >= d) incl += y;
        }
        if (lane == 31) s_w[warp] = incl;
        __syncthreads();
        unsigned woff = 0u, tot = 0u;
#pragma unroll
        for (int w = 0; w < 8; ++w) {
            const unsigned x = s_w[w];
            woff += w < warp ? x : 0u;
            tot += x;
        }
        unsigned run = s_carry + woff + incl - sum;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            if (t + j < ntiles) row[t + j] = run;
            run += v[j];
        }
        __syncthreads();
        if (threadIdx.x == 0) s_carry += tot;
        __syncthreads();
    }
    if (threadIdx.x == 0) totals[blockIdx.x] = s_carry;
}

// Stable scatter of one tile.  Warp w owns the tile's entries [w*512, (w+1)*512), lane l the entries
// w*512 + 32*i + l, so a warp's steps follow the stored order.  LAST: the final pass -- writes perm
// (idx_out), the sorted keys, the columns of X^T and the gathered values.
template <bool LAST, typename V>
__global__ void __launch_bounds__(TR_THREADS) k_tr_scatter(const int nnz, const int cols, const int *__restrict__ keys_in,
                                                           const int *__restrict__ idx_in, const int shift, const int nbins,
                                                           const int ntiles, const unsigned *__restrict__ counts,
                                                           const unsigned *__restrict__ totals, int *__restrict__ keys_out,
                                                           int *__restrict__ idx_out, const int *__restrict__ rowidx,
                                                           int *__restrict__ colT, const V *__restrict__ val,
                                                           V *__restrict__ valT)
{
    extern __shared__ __align__(16) unsigned char tr_smem[];
    unsigned *s_g = reinterpret_cast<unsigned *>(tr_smem);                  // [nbins] first position of digit d in this tile
    unsigned short *s_w = reinterpret_cast<unsigned short *>(s_g + nbins);  // [TR_WARPS][nbins] per-warp counts -> offsets
    __shared__ unsigned s_red[TR_WARPS];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const unsigned lt = lanemask_lt();
    const unsigned dmask = (unsigned)nbins - 1u;

    // digit bases (exclusive scan of the totals) + this tile's offset inside each digit
    {
        const int per = (nbins + TR_THREADS - 1) / TR_THREADS;   // 1 .. 4
        const int d0 = tid * per;
        unsigned loc[4], sum = 0u;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            loc[j] = (j < per && d0 + j < nbins) ? totals[d0 + j] : 0u;
            sum += loc[j];
        }
        unsigned incl = sum;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const unsigned y = __shfl_up_sync(FULL, incl, d);
            if (lane >= d) incl += y;
        }
        if (lane == 31) s_red[warp] = incl;
        __syncthreads();
        unsigned run = incl - sum;
        for (int w = 0; w < warp; ++w) run += s_red[w];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            if (j < per && d0 + j < nbins) {
                s_g[d0 + j] = run + counts[(size_t)(d0 + j) * ntiles + blockIdx.x];
                run += loc[j];
            }
        }
    }
    for (int i = tid; i < TR_WARPS * nbins; i += TR_THREADS) s_w[i] = 0;
    __syncthreads();

    const long long base = (long long)blockIdx.x * TR_TILE + warp * (32 * TR_ITEMS);
    unsigned short *my = s_w + warp * nbins;
    int key[TR_ITEMS];
#pragma unroll
    for (int i = 0; i < TR_ITEMS; ++i) {
        const long long e = base + i * 32 + lane;
        const bool act = e < nnz;
        key[i] = act ? masked_key(keys_in[e], cols) : -1;
        const unsigned d = act ? ((unsigned)key[i] >> shift) & dmask : 0xffffffffu;
        const unsigned peers = __match_any_sync(FULL, d);
        if (act && (peers & lt) == 0u) my[d] += (unsigned short)__popc(peers);
        __syncwarp();
    }
    __syncthreads();
    for (int d = tid; d < nbins; d += TR_THREADS) {
        unsigned run = 0u;
#pragma unroll
        for (int w = 0; w < TR_WARPS; ++w) {
            const unsigned c = s_w[w * nbins + d];
            s_w[w * nbins + d] = (unsigned short)run;
            run += c;
        }
    }
    __syncthreads();
#pragma unroll
    for (int i = 0; i < TR_ITEMS; ++i) {
        const long long e = base + i * 32 + lane;
        const bool act = key[i] >= 0;
        const unsigned d = act ? ((unsigned)key[i] >> shift) & dmask : 0xffffffffu;
        const unsigned peers = __match_any_sync(FULL, d);
        unsigned pos = 0u;
        if (act) pos = s_g[d] + my[d] + (unsigned)__popc(peers & lt);
        __syncwarp();
        if (act && (peers & lt) == 0u) my[d] += (unsigned short)__popc(peers);
        __syncwarp();
        if (act) {
            const int src = idx_in ? idx_in[e] : (int)e;
            keys_out[pos] = key[i];
            idx_out[pos] = src;
            if (LAST) {
                colT[pos] = rowidx[src];
                valT[pos] = moved(val[src]);
            }
        }
    }
}

// no pass (cols <= 1): X^T keeps the stored order; the columns of X^T were written by k_tr_rows
template <typename V>
__global__ void __launch_bounds__(256) k_tr_identity(const int nnz, const int cols, const int *__restrict__ col,
                                                     const V *__restrict__ val, V *__restrict__ valT,
                                                     int *__restrict__ perm, int *__restrict__ rowptrT,
                                                     int *__restrict__ bad, const int bad_bit)
{
    bool badl = false;
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < nnz; e += (long long)gridDim.x * blockDim.x) {
        badl |= (unsigned)col[e] >= (unsigned)cols;
        perm[e] = (int)e;
        valT[e] = moved(val[e]);
    }
    if (badl && bad) atomicOr(bad, bad_bit);
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        rowptrT[0] = 0;
        if (cols == 1) rowptrT[1] = nnz;
    }
}

// rowptrT[c] = first position of a key >= c in the sorted keys (c = 0 .. cols)
__global__ void __launch_bounds__(256) k_tr_rowptr(const int cols, const int nnz, const int *__restrict__ skeys,
                                                   int *__restrict__ rowptrT)
{
    const long long c = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (c > cols) return;
    int lo = 0, hi = nnz;
    while (lo < hi) {
        const int mid = (int)(((unsigned)lo + (unsigned)hi) >> 1);
        if (skeys[mid] < c) lo = mid + 1;
        else hi = mid;
    }
    rowptrT[c] = lo;
}

template <typename V>
__global__ void __launch_bounds__(256) k_tr_gather(const int nnz, const V *__restrict__ val, const int *__restrict__ perm,
                                                   V *__restrict__ valT)
{
    for (long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x; p < nnz; p += (long long)gridDim.x * blockDim.x)
        valT[p] = moved(val[perm[p]]);
}

int pass_count(int cols, int *bits_out)
{
    const int bits = cols <= 1 ? 0 : 32 - __builtin_clz((unsigned)(cols - 1));
    if (bits_out) *bits_out = bits;
    return (bits + TR_MAX_BITS - 1) / TR_MAX_BITS;
}

size_t align256(size_t b)
{
    return (b + 255) & ~(size_t)255;
}

int grid_for(long long n, int threads, int sm_count)
{
    const long long b = (n + threads - 1) / threads;
    const long long cap = (long long)sm_count * 16;
    return (int)std::max<long long>(1, std::min(b, cap));
}

template <typename V>
cudaError_t transpose_typed(const LaunchCtx &lc, int rows, int cols, int nnz, Csr X, TransposeOut out, void *scratch,
                            int *bad, int bad_bit)
{
    cudaStream_t s = lc.stream;
    int bits = 0;
    const int passes = pass_count(cols, &bits);
    const V *val = static_cast<const V *>(X.val);
    V *valT = static_cast<V *>(out.val);
    unsigned char *sc = static_cast<unsigned char *>(scratch);
    const size_t nb = align256((size_t)nnz * 4 + 4);
    int *rowidx = passes == 0 ? out.col : reinterpret_cast<int *>(sc);
    if (rows > 0 && nnz > 0) {
        ++*lc.launches;
        k_tr_rows<<<(int)(((long long)rows * 32 + 255) / 256), 256, 0, s>>>(rows, nnz, X.rowptr, rowidx);
    }
    if (passes == 0) {
        ++*lc.launches;
        k_tr_identity<V><<<grid_for(nnz, 256, lc.sm_count), 256, 0, s>>>(nnz, cols, X.col, val, valT, out.perm, out.rowptr, bad,
                                                                         bad_bit);
        return cudaGetLastError();
    }
    int *kbuf[2] = {reinterpret_cast<int *>(sc + nb), reinterpret_cast<int *>(sc + 2 * nb)};
    int *idx_x = reinterpret_cast<int *>(sc + 3 * nb);
    const int ntiles = (int)(((long long)nnz + TR_TILE - 1) / TR_TILE);
    unsigned *counts = reinterpret_cast<unsigned *>(sc + 4 * nb);
    unsigned *totals = counts + align256((size_t)TR_MAX_BINS * ntiles * 4) / 4;
    const int *keys_in = X.col;
    const int *idx_in = nullptr;
    int shift = 0;
    for (int p = 0; p < passes; ++p) {
        const int pb = bits / passes + (p < bits % passes ? 1 : 0);
        const int nbins = 1 << pb;
        const bool last = p == passes - 1;
        int *keys_out = kbuf[p & 1];
        int *idx_out = ((passes - 1 - p) & 1) == 0 ? out.perm : idx_x;
        if (ntiles > 0) {
            *lc.launches += 3;
            k_tr_hist<<<ntiles, TR_THREADS, 0, s>>>(nnz, cols, keys_in, shift, nbins, ntiles, counts, p == 0 ? bad : nullptr,
                                                    bad_bit);
            k_tr_scan<<<nbins, 256, 0, s>>>(ntiles, counts, totals);
            const size_t smem = (size_t)nbins * 4 + (size_t)TR_WARPS * nbins * 2;
            if (last) {
                cudaError_t e = cudaFuncSetAttribute(k_tr_scatter<true, V>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
                if (e != cudaSuccess) return e;
                k_tr_scatter<true, V><<<ntiles, TR_THREADS, smem, s>>>(nnz, cols, keys_in, idx_in, shift, nbins, ntiles, counts,
                                                                       totals, keys_out, idx_out, rowidx, out.col, val, valT);
            } else {
                cudaError_t e = cudaFuncSetAttribute(k_tr_scatter<false, V>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
                if (e != cudaSuccess) return e;
                k_tr_scatter<false, V><<<ntiles, TR_THREADS, smem, s>>>(nnz, cols, keys_in, idx_in, shift, nbins, ntiles, counts,
                                                                        totals, keys_out, idx_out, nullptr, nullptr, nullptr,
                                                                        nullptr);
            }
        }
        keys_in = keys_out;
        idx_in = idx_out;
        shift += pb;
    }
    ++*lc.launches;
    k_tr_rowptr<<<(int)(((long long)cols + 1 + 255) / 256), 256, 0, s>>>(cols, nnz, keys_in, out.rowptr);
    return cudaGetLastError();
}

}  // namespace

size_t transpose_scratch_bytes(int nnz, int cols)
{
    if (pass_count(cols, nullptr) == 0) return 0;
    const size_t nb = align256((size_t)nnz * 4 + 4);
    const size_t ntiles = ((size_t)nnz + TR_TILE - 1) / TR_TILE;
    return 4 * nb + align256((size_t)TR_MAX_BINS * ntiles * 4) + (size_t)TR_MAX_BINS * 4;
}

int transpose_passes(int cols)
{
    return pass_count(cols, nullptr);
}

// the type the values move as: complex64 as double (8-byte words), Conj8 for conjugation; complex128 as Move16,
// Conj16 for conjugation (conj is only ever set for complex operands: check_ops)
template <typename F>
cudaError_t with_mover(int dtype, bool conj, F &&f)
{
    if (conj) return dtype == BHB200_DTYPE_C128 ? f(Conj16()) : f(Conj8());
    return dispatch_value_type(dtype, [&](auto v) {
        using V = decltype(v);
        if constexpr (std::is_same_v<V, c128>) return f(Move16());
        else return f(std::conditional_t<std::is_same_v<V, c64>, double, V>());
    });
}

cudaError_t launch_transpose(const LaunchCtx &lc, int dtype, bool conj, int rows, int cols, int nnz, Csr X, TransposeOut out,
                             void *scratch, int *bad, int bad_bit)
{
    return with_mover(dtype, conj, [&](auto v) {
        return transpose_typed<decltype(v)>(lc, rows, cols, nnz, X, out, scratch, bad, bad_bit);
    });
}

cudaError_t launch_regather(const LaunchCtx &lc, int dtype, bool conj, int nnz, const void *val, const int *perm, void *valT)
{
    if (nnz <= 0) return cudaSuccess;
    return with_mover(dtype, conj, [&](auto v) {
        using V = decltype(v);
        if constexpr (value_bytes<V> > 0) {
            ++*lc.launches;
            k_tr_gather<V><<<grid_for(nnz, 256, lc.sm_count), 256, 0, lc.stream>>>(nnz, static_cast<const V *>(val), perm,
                                                                                 static_cast<V *>(valT));
            return cudaGetLastError();
        }
        return cudaSuccess;   // (structure-only operands have no values to gather)
    });
}

}  // namespace bhb
