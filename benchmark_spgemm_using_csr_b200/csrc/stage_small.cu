// stage_small.cu -- rows with 1..32 intermediate products.
//
// k_num_single  : p == 1, one thread per row           (ESC_1_cudakernel, bhsparse_cuda.h:1597-1640)
// k_esc<...>    : 2 <= p <= 32, one warp per row, expand - sort - compress entirely in
//                 registers: one product per lane, a 32-wide warp-shuffle bitonic network on
//                 (column, lane) keys, duplicate runs summed with a segmented shuffle
//                 reduction.  Replaces the per-thread shared-memory heap of
//                 ESC_2heap_noncoalesced (bhsparse_cuda.h:520-722) -- which needs one launch
//                 per distinct row size and reads B uncoalesced -- with one launch for the
//                 whole bin and coalesced reads of B segments.
#include "common.cuh"
#include <type_traits>

namespace bhb {

template <typename VT>
__global__ void __launch_bounds__(256) k_num_single(const int *__restrict__ queue, const int count,
                                                    const int *__restrict__ rowptrA, const int *__restrict__ colA,
                                                    const VT *__restrict__ valA, const int *__restrict__ rowptrB,
                                                    const int *__restrict__ colB, const VT *__restrict__ valB,
                                                    const int64_t *__restrict__ rowoff, int *__restrict__ colC,
                                                    VT *__restrict__ valC)
{
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= count) return;
    const int row = queue[q];
    const int a1 = rowptrA[row + 1];
    for (int j = rowptrA[row]; j < a1; ++j) {
        const int k = colA[j];
        const int bs = rowptrB[k];
        if (rowptrB[k + 1] > bs) {
            const int64_t o = rowoff[row];
            colC[o] = colB[bs];
            valC[o] = valA[j] * valB[bs];
            return;
        }
    }
}

// One product per lane.  WIDE=false packs (column << 5 | lane) into 32 bits
// (needs n <= 2^26); WIDE=true uses 64-bit keys.  The lane tag makes the sort
// stable, so duplicate columns stay in A-row order.
template <typename VT, bool NUMERIC, bool WIDE>
__global__ void __launch_bounds__(256) k_esc(const int *__restrict__ queue, const int count,
                                             const int *__restrict__ rowptrA, const int *__restrict__ colA,
                                             const VT *__restrict__ valA, const int *__restrict__ rowptrB,
                                             const int *__restrict__ colB, const VT *__restrict__ valB,
                                             int *__restrict__ rc, const int64_t *__restrict__ rowoff,
                                             int *__restrict__ colC, VT *__restrict__ valC)
{
    typedef typename std::conditional<WIDE, unsigned long long, unsigned>::type KT;
    const KT KPAD = ~(KT)0;
    const int lane = threadIdx.x & 31;
    const int warps_per_block = blockDim.x >> 5;
    for (int q = blockIdx.x * warps_per_block + (threadIdx.x >> 5); q < count; q += gridDim.x * warps_per_block) {
        const int row = queue[q];
        const int a0 = rowptrA[row], a1 = rowptrA[row + 1];
        KT key = KPAD;
        VT val = VT(0);
        int filled = 0;   // products placed so far (warp-uniform, <= 32)
        for (int base = a0; base < a1; base += 32) {
            const int j = base + lane;
            int bs = 0, len = 0;
            VT av = VT(0);
            if (j < a1) {
                const int k = colA[j];
                bs = rowptrB[k];
                len = rowptrB[k + 1] - bs;
                if (NUMERIC) av = valA[j];
            }
            int incl = len;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const int y = __shfl_up_sync(FULL, incl, d);
                if (lane >= d) incl += y;
            }
            const int tot = __shfl_sync(FULL, incl, 31);
            // lane `filled + t` takes product t of this chunk: owner = #lanes with incl <= t
            const int t = lane - filled;
            int owner = 0;
#pragma unroll
            for (int step = 16; step > 0; step >>= 1) {
                const int v = __shfl_sync(FULL, incl, (owner + step - 1) & 31);
                if (v <= t) owner += step;
            }
            owner &= 31;
            const int o_incl = __shfl_sync(FULL, incl, owner);
            const int o_len = __shfl_sync(FULL, len, owner);
            const int o_bs = __shfl_sync(FULL, bs, owner);
            VT o_av = VT(0);
            if (NUMERIC) o_av = __shfl_sync(FULL, av, owner);
            if (t >= 0 && t < tot) {
                const int p = o_bs + (t - (o_incl - o_len));
                const int c = colB[p];
                key = WIDE ? (KT)(((unsigned long long)(unsigned)c << 32) | (unsigned)lane)
                           : (KT)(((unsigned)c << 5) | (unsigned)lane);
                if (NUMERIC) val = o_av * valB[p];
            }
            filled += tot;
        }
        // 32-wide bitonic sort of the keys across the warp
#pragma unroll
        for (int k = 2; k <= 32; k <<= 1) {
#pragma unroll
            for (int j = k >> 1; j > 0; j >>= 1) {
                const KT y = __shfl_xor_sync(FULL, key, j);
                const bool lower = (lane & j) == 0;
                const bool asc = (k == 32) ? true : ((lane & k) == 0);
                const KT lo = key < y ? key : y, hi = key < y ? y : key;
                key = (lower == asc) ? lo : hi;
            }
        }
        const bool valid = key != KPAD;
        const int col = WIDE ? (int)(key >> 32) : (int)(key >> 5);
        const int src = (int)(key & 31);
        const int prev = __shfl_up_sync(FULL, col, 1);
        const bool head = valid && (lane == 0 || prev != col);
        const unsigned heads = __ballot_sync(FULL, head);
        if (!NUMERIC) {
            if (lane == 0) rc[row] = __popc(heads);
        } else {
            VT v = __shfl_sync(FULL, val, src);
            if (!valid) v = VT(0);
            // segmented sum over runs of equal columns (runs are contiguous after the sort)
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const VT v2 = __shfl_down_sync(FULL, v, d);
                const int c2 = __shfl_down_sync(FULL, col, d);
                const bool ok2 = __shfl_down_sync(FULL, (int)valid, d) != 0;
                if (lane + d < 32 && ok2 && valid && c2 == col) v += v2;
            }
            if (head) {
                const int64_t o = rowoff[row] + __popc(heads & ((1u << lane) - 1u));
                colC[o] = col;
                valC[o] = v;
            }
        }
    }
}

static int esc_blocks(const LaunchCtx &lc, int count, int threads)
{
    const int wpb = threads / 32;
    long long blocks = ((long long)count + wpb - 1) / wpb;
    const long long cap = (long long)lc.sm_count * 32;
    return (int)(blocks > cap ? cap : blocks);
}

cudaError_t launch_sym_esc(const LaunchCtx &lc, const int *queue, int count, int n, Csr A, Csr B, int *rc)
{
    if (count <= 0) return cudaSuccess;
    const int threads = 256;
    const int blocks = esc_blocks(lc, count, threads);
    ++*lc.launches;
    if (n <= (1 << 26))
        k_esc<float, false, false><<<blocks, threads, 0, lc.stream>>>(queue, count, A.rowptr, A.col, nullptr, B.rowptr,
                                                                       B.col, nullptr, rc, nullptr, nullptr, nullptr);
    else
        k_esc<float, false, true><<<blocks, threads, 0, lc.stream>>>(queue, count, A.rowptr, A.col, nullptr, B.rowptr,
                                                                      B.col, nullptr, rc, nullptr, nullptr, nullptr);
    return cudaGetLastError();
}

template <typename VT>
static cudaError_t launch_num_esc_t(const LaunchCtx &lc, const int *queue, int count, int n, Csr A, Csr B,
                                    const int64_t *rowoff, int *colC, VT *valC)
{
    const int threads = 256;
    const int blocks = esc_blocks(lc, count, threads);
    ++*lc.launches;
    if (n <= (1 << 26))
        k_esc<VT, true, false><<<blocks, threads, 0, lc.stream>>>(queue, count, A.rowptr, A.col, (const VT *)A.val,
                                                                   B.rowptr, B.col, (const VT *)B.val, nullptr, rowoff,
                                                                   colC, valC);
    else
        k_esc<VT, true, true><<<blocks, threads, 0, lc.stream>>>(queue, count, A.rowptr, A.col, (const VT *)A.val,
                                                                  B.rowptr, B.col, (const VT *)B.val, nullptr, rowoff,
                                                                  colC, valC);
    return cudaGetLastError();
}

cudaError_t launch_num_esc(const LaunchCtx &lc, int dtype, const int *queue, int count, int n, Csr A, Csr B,
                           const int64_t *rowoff, int *colC, void *valC)
{
    if (count <= 0) return cudaSuccess;
    return dispatch_value_type(dtype, [&](auto v) {
        using VT = decltype(v);
        return launch_num_esc_t<VT>(lc, queue, count, n, A, B, rowoff, colC, (VT *)valC);
    });
}

template <typename VT>
static cudaError_t launch_num_single_t(const LaunchCtx &lc, const int *queue, int count, Csr A, Csr B,
                                       const int64_t *rowoff, int *colC, VT *valC)
{
    const int threads = 256;
    const int blocks = (count + threads - 1) / threads;
    ++*lc.launches;
    k_num_single<VT><<<blocks, threads, 0, lc.stream>>>(queue, count, A.rowptr, A.col, (const VT *)A.val, B.rowptr,
                                                        B.col, (const VT *)B.val, rowoff, colC, valC);
    return cudaGetLastError();
}

cudaError_t launch_num_single(const LaunchCtx &lc, int dtype, const int *queue, int count, Csr A, Csr B,
                              const int64_t *rowoff, int *colC, void *valC)
{
    if (count <= 0) return cudaSuccess;
    return dispatch_value_type(dtype, [&](auto v) {
        using VT = decltype(v);
        return launch_num_single_t<VT>(lc, queue, count, A, B, rowoff, colC, (VT *)valC);
    });
}

}  // namespace bhb
