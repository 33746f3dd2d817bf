// stage_range_vec.cuh -- 128-bit vectorised variants of the range kernels' product loops.
//
// A warp step covers FOUR rows of B at once: 8 lanes per B row, each lane one aligned
// 16-byte vector of column indices (4 columns) and the matching 16/32 bytes of values, head
// and tail elements outside [rowptrB[k], rowptrB[k+1]) redirected to sink words.  A 27-entry
// stencil row costs one LDG.128 per lane instead of 27 scalar steps per warp, and the loop
// overhead (broadcasts, bounds, address arithmetic) is paid once per 4 B rows.
//
// In the numeric kernel the four B rows in flight may contain the same column, so each
// 8-lane group adds into its own private accumulator array (shared-memory FP atomics are
// CAS loops on sm_100a); the four arrays are summed when the row is stored.
//
// Requires colB / valB 16-byte aligned (true for cudaMalloc and torch allocations); the
// launchers fall back to the scalar kernels of stage_range.cuh otherwise.
#pragma once
#include "stage_range.cuh"

namespace bhb {

constexpr int RANGE_NG = 4;   // B rows per warp step (8 lanes each)

__host__ __device__ inline size_t num_range_vec_warp_bytes(int nsum, int nacc, size_t vsize)
{
    return ((size_t)nsum * 32 + 2) * 8                       // bitmap + sinks
           + (size_t)RANGE_NG * ((size_t)nacc + 4) * vsize   // private accumulators (+ sink slot, pad)
           + ((size_t)nacc + 4) * 4                          // sorted columns
           + ((size_t)nsum * 32 + 8) * 2;                    // rank prefixes (+ sink, pad)
}

// Columns e0..e0+3 of a B row [lo, hi); elements outside the row become `sink`.
// Returns true if the vector was loaded (at least one valid element).
__device__ __forceinline__ bool load_cols4(const int *__restrict__ colB, const unsigned e0, const unsigned lo,
                                           const unsigned hi, const int sink, int (&c)[4])
{
    c[0] = c[1] = c[2] = c[3] = sink;
    const bool ld = (e0 < hi) && (e0 + 3u >= lo);
    if (ld) {
        const int4 q = __ldg(reinterpret_cast<const int4 *>(colB + e0));
        if (e0 >= lo) c[0] = q.x;
        if (e0 + 1u >= lo && e0 + 1u < hi) c[1] = q.y;
        if (e0 + 2u >= lo && e0 + 2u < hi) c[2] = q.z;
        if (e0 + 3u < hi) c[3] = q.w;
    }
    return ld;
}
__device__ __forceinline__ void load_vals4(const double *__restrict__ valB, const unsigned e0, const unsigned hi,
                                           double (&v)[4])
{
    const double2 a = __ldg(reinterpret_cast<const double2 *>(valB + e0));
    v[0] = a.x;
    v[1] = a.y;
    if (e0 + 2u < hi) {   // never touch a 16-byte chunk that holds no element of the row
        const double2 b = __ldg(reinterpret_cast<const double2 *>(valB + e0) + 1);
        v[2] = b.x;
        v[3] = b.y;
    }
}
// complex64: 16 bytes hold two values, as for double
__device__ __forceinline__ void load_vals4(const c64 *__restrict__ valB, const unsigned e0, const unsigned hi, c64 (&v)[4])
{
    const float4 a = __ldg(reinterpret_cast<const float4 *>(valB + e0));
    v[0] = c64(a.x, a.y);
    v[1] = c64(a.z, a.w);
    if (e0 + 2u < hi) {
        const float4 b = __ldg(reinterpret_cast<const float4 *>(valB + e0) + 1);
        v[2] = c64(b.x, b.y);
        v[3] = c64(b.z, b.w);
    }
}
__device__ __forceinline__ void load_vals4(const float *__restrict__ valB, const unsigned e0, const unsigned,
                                           float (&v)[4])
{
    const float4 a = __ldg(reinterpret_cast<const float4 *>(valB + e0));
    v[0] = a.x;
    v[1] = a.y;
    v[2] = a.z;
    v[3] = a.w;
}

__device__ __forceinline__ void mark4(const int (&c)[4], const int base, unsigned *bm32)
{
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int rel = c[i] - base;
        atomicOr(&bm32[rel >> 5], 1u << (rel & 31));
    }
}

// Vectorised marking of all products of one row.  Warp-collective.
__device__ __forceinline__ void range_mark_row_vec(const int a0, const int a1, const int base, const int sink_c,
                                                   const int lane, const int *__restrict__ colA,
                                                   const int *__restrict__ rowptrB, const int *__restrict__ colB,
                                                   unsigned *bm32)
{
    const int gi = lane >> 3;
    const unsigned gl4 = (unsigned)(lane & 7) * 4u;
    for (int cb = a0; cb < a1; cb += 32) {
        const int j = cb + lane;
        unsigned bs = 0, len = 0;   // lanes past the row keep len = 0: nothing valid
        if (j < a1) {
            const int k = colA[j];
            bs = (unsigned)rowptrB[k];
            len = (unsigned)rowptrB[k + 1] - bs;
        }
        const int cnt = min(32, a1 - cb);
        unsigned nbs = __shfl_sync(FULL, bs, gi), nlen = __shfl_sync(FULL, len, gi);
        int nc[4];
        load_cols4(colB, (nbs & ~3u) + gl4, nbs, nbs + nlen, sink_c, nc);
        for (int s4 = 0; s4 < cnt; s4 += RANGE_NG) {
            const unsigned cbs = nbs, cend = nbs + nlen;
            int c[4] = {nc[0], nc[1], nc[2], nc[3]};
            const int tn = s4 + RANGE_NG + gi;   // this group's B row in the next step
            nbs = __shfl_sync(FULL, bs, tn & 31);
            nlen = __shfl_sync(FULL, len, tn & 31);
            if (tn >= 32) nlen = 0;
            load_cols4(colB, (nbs & ~3u) + gl4, nbs, nbs + nlen, sink_c, nc);
            mark4(c, base, bm32);
            // B rows longer than one 32-element window (group-uniform trip count)
            for (unsigned w0 = (cbs & ~3u) + 32u; w0 < cend; w0 += 32u) {
                int d[4];
                load_cols4(colB, w0 + gl4, cbs, cend, sink_c, d);
                mark4(d, base, bm32);
            }
        }
    }
}

template <typename VT>
__device__ __forceinline__ void accum4(const int (&c)[4], const VT (&v)[4], const VT a, const int base,
                                       const unsigned long long *bm64, const unsigned short *prefix16, VT *acc)
{
#pragma unroll
    for (int i = 0; i < 4; ++i) range_accum<VT>(c[i], a * v[i], base, bm64, prefix16, acc);
}

template <typename VT>
__device__ __forceinline__ void range_accumulate_row_vec(const int a0, const int a1, const int base,
                                                         const int sink_c, const int lane,
                                                         const int *__restrict__ colA, const VT *__restrict__ valA,
                                                         const int *__restrict__ rowptrB,
                                                         const int *__restrict__ colB, const VT *__restrict__ valB,
                                                         const unsigned long long *bm64,
                                                         const unsigned short *prefix16, VT *acc_g)
{
    const int gi = lane >> 3;
    const unsigned gl4 = (unsigned)(lane & 7) * 4u;
    for (int cb = a0; cb < a1; cb += 32) {
        const int j = cb + lane;
        unsigned bs = 0, len = 0;
        VT av = VT(0);
        if (j < a1) {
            const int k = colA[j];
            bs = (unsigned)rowptrB[k];
            len = (unsigned)rowptrB[k + 1] - bs;
            av = valA[j];
        }
        const int cnt = min(32, a1 - cb);
        unsigned nbs = __shfl_sync(FULL, bs, gi), nlen = __shfl_sync(FULL, len, gi);
        int nc[4];
        VT nv[4] = {VT(0), VT(0), VT(0), VT(0)};
        if (load_cols4(colB, (nbs & ~3u) + gl4, nbs, nbs + nlen, sink_c, nc))
            load_vals4(valB, (nbs & ~3u) + gl4, nbs + nlen, nv);
        for (int s4 = 0; s4 < cnt; s4 += RANGE_NG) {
            const unsigned cbs = nbs, cend = nbs + nlen;
            int c[4] = {nc[0], nc[1], nc[2], nc[3]};
            VT v[4] = {nv[0], nv[1], nv[2], nv[3]};
            const int t = s4 + gi, tn = t + RANGE_NG;
            nbs = __shfl_sync(FULL, bs, tn & 31);
            nlen = __shfl_sync(FULL, len, tn & 31);
            if (tn >= 32) nlen = 0;
            if (load_cols4(colB, (nbs & ~3u) + gl4, nbs, nbs + nlen, sink_c, nc))
                load_vals4(valB, (nbs & ~3u) + gl4, nbs + nlen, nv);
            const VT a_t = __shfl_sync(FULL, av, t & 31);
            accum4<VT>(c, v, a_t, base, bm64, prefix16, acc_g);
            for (unsigned w0 = (cbs & ~3u) + 32u; w0 < cend; w0 += 32u) {
                int d[4];
                VT dv[4] = {VT(0), VT(0), VT(0), VT(0)};
                if (load_cols4(colB, w0 + gl4, cbs, cend, sink_c, d)) load_vals4(valB, w0 + gl4, cend, dv);
                accum4<VT>(d, dv, a_t, base, bm64, prefix16, acc_g);
            }
            __syncwarp();   // this group's next B row may add into the same positions
        }
    }
}

// Numeric range kernel, vectorised (nacc <= 128 class: 4 private accumulator arrays).
template <typename VT>
__global__ void __launch_bounds__(512)
k_num_range_vec(const int *__restrict__ queue, const int count, const int *__restrict__ rowptrA,
                const int *__restrict__ colA, const VT *__restrict__ valA, const int *__restrict__ rowptrB,
                const int *__restrict__ colB, const VT *__restrict__ valB, const int *__restrict__ rlo,
                const int nsum, const int nacc, const int64_t *__restrict__ rowoff, int *__restrict__ colC,
                VT *__restrict__ valC, const WordLists wl)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
    const int nwords = nsum * 32;
    const int astride = nacc + 4;
    unsigned char *mine = smem_raw + (size_t)warp * num_range_vec_warp_bytes(nsum, nacc, value_bytes<VT>);
    unsigned long long *bm64 = reinterpret_cast<unsigned long long *>(mine);   // [nwords] + zero sink + garbage sink
    unsigned *bm32 = reinterpret_cast<unsigned *>(mine);
    VT *acc = reinterpret_cast<VT *>(bm64 + nwords + 2);                        // RANGE_NG x ([nacc] + sink slot)
    int *ocol = reinterpret_cast<int *>(acc + RANGE_NG * astride);              // [nacc]
    unsigned short *prefix16 = reinterpret_cast<unsigned short *>(ocol + nacc + 4);   // [nwords] + sink
    VT *acc_g = acc + (lane >> 3) * astride;

    for (int i = lane; i < nwords + 2; i += 32) bm64[i] = 0ull;
    if (lane == 0) prefix16[nwords] = (unsigned short)nacc;   // zero sink word -> sink accumulator slot
    __syncwarp();

    for (int q = blockIdx.x * nwarps + warp; q < count; q += gridDim.x * nwarps) {
        const int row = queue[q];
        const int base = rlo[row] & ~63;
        const int sink_zero = base + (nwords << 6);
        const int sink_garbage = sink_zero + 64;
        const int64_t o = rowoff[row];
        const int cntc = (int)(rowoff[row + 1] - o);
        const int a0 = rowptrA[row], a1 = rowptrA[row + 1];
        for (int i = lane; i < cntc; i += 32) {
#pragma unroll
            for (int g = 0; g < RANGE_NG; ++g) acc[g * astride + i] = VT(0);
        }
        const int lc = wl.cnt[row];
        const long long loff = wl.off[row];
        if (lc >= 0) {
            int run = 0;
            for (int e0 = 0; e0 < lc; e0 += 32) {
                const int e = e0 + lane;
                int w = nwords + 1;
                unsigned long long bits = 0ull;
                if (e < lc) {
                    w = (int)wl.idx[loff + e];
                    bits = wl.bits[loff + e];
                }
                const int pcnt = __popcll(bits);
                const int incl = warp_incl_scan(pcnt, lane);
                int pos = run + incl - pcnt;
                bm64[w] = bits;
                prefix16[w] = (unsigned short)pos;   // (the garbage sink's prefix is never read)
                const int cbase = base + (w << 6);
                for (unsigned long long b = bits; b; b &= b - 1) ocol[pos++] = cbase + __ffsll((long long)b) - 1;
                run += __shfl_sync(FULL, incl, 31);
            }
        } else {
            range_mark_row_vec(a0, a1, base, sink_garbage, lane, colA, rowptrB, colB, bm32);
            __syncwarp();
            const int w0 = lane * nsum;
            int tl = 0;
            for (int jw = 0; jw < nsum; ++jw) tl += __popcll(bm64[w0 + jw]);
            const int incl = warp_incl_scan(tl, lane);
            int pos = incl - tl;
            for (int jw = 0; jw < nsum; ++jw) {
                const unsigned long long bits = bm64[w0 + jw];
                if (bits) {
                    prefix16[w0 + jw] = (unsigned short)pos;
                    const int cbase = base + ((w0 + jw) << 6);
                    for (unsigned long long b = bits; b; b &= b - 1) ocol[pos++] = cbase + __ffsll((long long)b) - 1;
                }
            }
        }
        __syncwarp();
        range_accumulate_row_vec<VT>(a0, a1, base, sink_zero, lane, colA, valA, rowptrB, colB, valB, bm64, prefix16,
                                     acc_g);
        __syncwarp();
        for (int i = lane; i < cntc; i += 32) {
            const int c = ocol[i];
            colC[o + i] = c;
            valC[o + i] = ((acc[i] + acc[astride + i]) + acc[2 * astride + i]) + acc[3 * astride + i];
            bm64[(c - base) >> 6] = 0ull;   // restore the all-zero bitmap (only the words that were set)
        }
        __syncwarp();
    }
}

template <typename VT>
static cudaError_t launch_num_range_vec_t(const LaunchCtx &lc, int nsum, int nacc, const int *queue, int count, Csr A,
                                          Csr B, const int *rlo, const int64_t *rowoff, int *colC, void *valC,
                                          WordLists wl)
{
    if (count <= 0) return cudaSuccess;
    const size_t wb = num_range_vec_warp_bytes(nsum, nacc, value_bytes<VT>);
    int wpb, bps;
    range_launch_shape(wb, wpb, bps);
    const size_t smem = wb * wpb;
    cudaError_t e = cudaFuncSetAttribute(k_num_range_vec<VT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    bps = resident_blocks(k_num_range_vec<VT>, wpb * 32, smem);
    long long blocks = ((long long)count + wpb - 1) / wpb;
    const long long cap = (long long)lc.sm_count * bps;
    if (blocks > cap) blocks = cap;
    ++*lc.launches;
    k_num_range_vec<VT><<<(int)blocks, wpb * 32, smem, lc.stream>>>(queue, count, A.rowptr, A.col, (const VT *)A.val,
                                                                    B.rowptr, B.col, (const VT *)B.val, rlo, nsum, nacc,
                                                                    rowoff, colC, (VT *)valC, wl);
    return cudaGetLastError();
}

inline bool range_vec_aligned(const Csr &B)
{
    return (((uintptr_t)B.col | (uintptr_t)B.val) & 15u) == 0;
}

// numeric range bins: the vectorised kernel for rows of at most 128 outputs when B is 16-byte aligned (its 128-bit loads
// carry values: structure-only products take the scalar kernel, and so do complex128 ones, whose 128-bit load would
// carry one value where the kernel's four-column step wants four)
template <typename VT>
static cudaError_t launch_num_range_pick_t(const LaunchCtx &lc, int nsum, int nacc, const int *queue, int count, Csr A,
                                           Csr B, const int *rlo, const int64_t *rowoff, int *colC, void *valC,
                                           WordLists wl)
{
    if constexpr (value_bytes<VT> > 0 && value_bytes<VT> <= 8) {
        if (nacc <= 128 && range_vec_aligned(B))
            return launch_num_range_vec_t<VT>(lc, nsum, nacc, queue, count, A, B, rlo, rowoff, colC, valC, wl);
    }
    return launch_num_range_t<VT>(lc, nsum, nacc, queue, count, A, B, rlo, rowoff, colC, valC, wl);
}

}  // namespace bhb
