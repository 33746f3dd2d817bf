// stage_range.cuh -- "range" kernels: rows of C whose column span fits a shared-memory
// bitmap (stencil / banded / FEM rows; BASELINE config 2's 27-point rows span 66 053
// columns).  One warp owns a row.
//
//   bitmap  : one bit per column of [base, base + nsum*2048), base = row's min column & ~63,
//             as 32*nsum 64-bit words; lane l owns words [l*nsum, (l+1)*nsum) in the sweeps
//   rank(c) : prefix16[word(c)] + popc(bits below c)  = position of c in the sorted row
//
// symbolic  k_sym_range : mark every product's column (ATOMS.OR -- measured on B200 at the
//           cost of a plain STS, tools/smem_ubench.cu), sweep the bitmap (LDS.128, bank
//           conflict free), count the set bits and hand the non-empty words (index, bits)
//           to the numeric kernel through a device pool.
// numeric   k_num_range : rebuild bitmap + prefixes + the sorted column list from the word
//           list (or mark + sweep again if the pool was full), then for every product
//           acc[rank(c)] += a*b in shared memory -- columns of one B row are distinct, so
//           no atomics -- and store the row at rowptrC[row], coalesced.
//
// The step loops are branch free: inactive lanes and padding steps are redirected to sink
// words / a sink accumulator slot instead of being predicated off (the first version of
// these kernels spent 60 SASS instructions per B row on reconvergence and predicates).
// B rows are fetched RANGE_U steps ahead into registers (one B row per step, coalesced
// segment loads): 12.5 KB of shared memory per warp leaves ~18 warps per SM.
// Replaces, for these rows, ESC_bitonic_scan / EM_mergepath (bhsparse_cuda.h:1400-1518,
// 1902-2157) and the Ct -> C compaction (:2813-2911).
#pragma once
#include "common.cuh"

namespace bhb {

constexpr int RANGE_U = 4;   // B rows in flight per warp

// per-warp shared-memory footprints (multiples of 16 bytes)
__host__ __device__ inline size_t sym_range_warp_bytes(int nsum)
{
    return ((size_t)nsum * 32 + 2) * 8;                      // bitmap + 2 sink words
}
__host__ __device__ inline size_t num_range_warp_bytes(int nsum, int nacc, size_t vsize)
{
    return ((size_t)nsum * 32 + 2) * 8                       // bitmap + sinks
           + ((size_t)nacc + 4) * vsize                      // accumulators + sink slot (+pad)
           + ((size_t)nacc + 4) * 4                          // sorted columns
           + ((size_t)nsum * 32 + 8) * 2;                    // rank prefixes (+ sink, pad)
}

__device__ __forceinline__ int warp_incl_scan(int v, const int lane)
{
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const int y = __shfl_up_sync(FULL, v, d);
        if (lane >= d) v += y;
    }
    return v;
}

// Mark the columns of all products of one row.  Warp-collective, branch free per step.
// sink_c: a column value that lands in the bitmap's garbage sink word.
__device__ __forceinline__ void range_mark_row(const int a0, const int a1, const int base, const int sink_c,
                                               const int lane, const int *__restrict__ colA,
                                               const int *__restrict__ rowptrB, const int *__restrict__ colB_lane,
                                               unsigned *bm32)
{
    for (int cb = a0; cb < a1; cb += 32) {
        const int j = cb + lane;
        unsigned bs = 0;
        int len = 0;
        if (j < a1) {
            const int k = colA[j];
            bs = (unsigned)rowptrB[k];
            len = rowptrB[k + 1] - (int)bs;
        }
        const int cnt = min(32, a1 - cb);
        int pc[RANGE_U], pl[RANGE_U];
        unsigned pb[RANGE_U];
#pragma unroll
        for (int u = 0; u < RANGE_U; ++u) {
            pb[u] = __shfl_sync(FULL, bs, u);
            pl[u] = (u < cnt) ? __shfl_sync(FULL, len, u) : 0;
            pc[u] = sink_c;
            if (lane < pl[u]) pc[u] = __ldg(colB_lane + pb[u]);
        }
        for (int t0 = 0; t0 < cnt; t0 += RANGE_U) {
#pragma unroll
            for (int u = 0; u < RANGE_U; ++u) {
                const int c = pc[u], tl = pl[u];
                const unsigned tb = pb[u];
                const int tn = t0 + u + RANGE_U;   // refill this slot with the B row RANGE_U steps ahead
                pb[u] = __shfl_sync(FULL, bs, tn & 31);
                const int nl = __shfl_sync(FULL, len, tn & 31);
                pl[u] = (tn < cnt) ? nl : 0;
                pc[u] = sink_c;
                if (lane < pl[u]) pc[u] = __ldg(colB_lane + pb[u]);
                const int rel = c - base;
                atomicOr(&bm32[rel >> 5], 1u << (rel & 31));
                if (tl > 32) {   // long B row (warp-uniform, rare): the rest without prefetch
                    for (int p = 32 + lane; p < tl; p += 32) {
                        const int r2 = __ldg(colB_lane + tb + p - lane) - base;
                        atomicOr(&bm32[r2 >> 5], 1u << (r2 & 31));
                    }
                }
            }
        }
    }
}

// ---------------------------------------------------------------------------------------
template <typename VT>
__device__ __forceinline__ void range_accum(const int c, const VT x, const int base,
                                            const unsigned long long *bm64, const unsigned short *prefix16,
                                            VT *acc)
{
    const int rel = c - base;
    const int w = rel >> 6;
    const unsigned long long bits = bm64[w];
    const int pos = (int)prefix16[w] + __popcll(bits & ((1ull << (rel & 63)) - 1ull));
    acc[pos] += x;
}

// sink_c: a column whose bitmap word is always zero and whose prefix is the sink slot nacc.
template <typename VT>
__device__ __forceinline__ void range_accumulate_row(const int a0, const int a1, const int base, const int sink_c,
                                                     const int lane, const int *__restrict__ colA,
                                                     const VT *__restrict__ valA, const int *__restrict__ rowptrB,
                                                     const int *__restrict__ colB_lane,
                                                     const VT *__restrict__ valB_lane,
                                                     const unsigned long long *bm64,
                                                     const unsigned short *prefix16, VT *acc)
{
    for (int cb = a0; cb < a1; cb += 32) {
        const int j = cb + lane;
        unsigned bs = 0;
        int len = 0;
        VT av = VT(0);
        if (j < a1) {
            const int k = colA[j];
            bs = (unsigned)rowptrB[k];
            len = rowptrB[k + 1] - (int)bs;
            av = valA[j];
        }
        const int cnt = min(32, a1 - cb);
        int pc[RANGE_U], pl[RANGE_U];
        unsigned pb[RANGE_U];
        VT pv[RANGE_U];
#pragma unroll
        for (int u = 0; u < RANGE_U; ++u) {
            pb[u] = __shfl_sync(FULL, bs, u);
            pl[u] = (u < cnt) ? __shfl_sync(FULL, len, u) : 0;
            pc[u] = sink_c;
            pv[u] = VT(0);
            if (lane < pl[u]) {
                pc[u] = __ldg(colB_lane + pb[u]);
                pv[u] = __ldg(valB_lane + pb[u]);
            }
        }
        for (int t0 = 0; t0 < cnt; t0 += RANGE_U) {
#pragma unroll
            for (int u = 0; u < RANGE_U; ++u) {
                const int c = pc[u], tl = pl[u];
                const unsigned tb = pb[u];
                const VT v = pv[u];
                const int t = t0 + u, tn = t + RANGE_U;
                pb[u] = __shfl_sync(FULL, bs, tn & 31);
                const int nl = __shfl_sync(FULL, len, tn & 31);
                pl[u] = (tn < cnt) ? nl : 0;
                pc[u] = sink_c;
                pv[u] = VT(0);
                if (lane < pl[u]) {
                    pc[u] = __ldg(colB_lane + pb[u]);
                    pv[u] = __ldg(valB_lane + pb[u]);
                }
                const VT a_t = __shfl_sync(FULL, av, t & 31);
                range_accum<VT>(c, a_t * v, base, bm64, prefix16, acc);
                if (tl > 32) {
                    for (int p = 32 + lane; p < tl; p += 32)
                        range_accum<VT>(__ldg(colB_lane + tb + p - lane), a_t * __ldg(valB_lane + tb + p - lane), base,
                                        bm64, prefix16, acc);
                }
                __syncwarp();   // the next B row may add into the same positions
            }
        }
    }
}

template <typename VT>
__global__ void __launch_bounds__(512)
k_num_range(const int *__restrict__ queue, const int count, const int *__restrict__ rowptrA,
            const int *__restrict__ colA, const VT *__restrict__ valA, const int *__restrict__ rowptrB,
            const int *__restrict__ colB, const VT *__restrict__ valB, const int *__restrict__ rlo, const int nsum,
            const int nacc, const int64_t *__restrict__ rowoff, int *__restrict__ colC, VT *__restrict__ valC,
            const WordLists wl)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
    const int nwords = nsum * 32;
    unsigned char *mine = smem_raw + (size_t)warp * num_range_warp_bytes(nsum, nacc, value_bytes<VT>);
    unsigned long long *bm64 = reinterpret_cast<unsigned long long *>(mine);   // [nwords] + zero sink + garbage sink
    unsigned *bm32 = reinterpret_cast<unsigned *>(mine);
    VT *acc = reinterpret_cast<VT *>(bm64 + nwords + 2);                        // [nacc] + sink slot
    int *ocol = reinterpret_cast<int *>(acc + (nacc + 4) * vslots<VT>);         // [nacc]
    unsigned short *prefix16 = reinterpret_cast<unsigned short *>(ocol + nacc + 4);   // [nwords] + sink
    const int *colB_lane = colB + lane;
    const VT *valB_lane = valB + lane;

    for (int i = lane; i < nwords + 2; i += 32) bm64[i] = 0ull;
    if (lane == 0) prefix16[nwords] = (unsigned short)nacc;   // zero sink word -> sink accumulator slot
    __syncwarp();

    for (int q = blockIdx.x * nwarps + warp; q < count; q += gridDim.x * nwarps) {
        const int row = queue[q];
        const int base = rlo[row] & ~63;
        const int sink_zero = base + (nwords << 6);         // word nwords: always zero
        const int sink_garbage = sink_zero + 64;            // word nwords+1: write-only
        const int64_t o = rowoff[row];
        const int cntc = (int)(rowoff[row + 1] - o);
        const int a0 = rowptrA[row], a1 = rowptrA[row + 1];
        for (int i = lane; i < cntc; i += 32) acc[i] = VT(0);
        const int lc = wl.cnt[row];
        const long long loff = wl.off[row];
        if (lc >= 0) {
            // ---- rebuild bitmap, rank prefixes and the sorted column list from the word list ----
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
                prefix16[min(w, nwords + 1)] = (unsigned short)pos;   // (garbage sink prefix is never read)
                const int cbase = base + (w << 6);
                for (unsigned long long b = bits; b; b &= b - 1) ocol[pos++] = cbase + __ffsll((long long)b) - 1;
                run += __shfl_sync(FULL, incl, 31);
            }
        } else {
            // ---- the pool was full for this row: mark here, then sweep this lane's words ----
            range_mark_row(a0, a1, base, sink_garbage, lane, colA, rowptrB, colB_lane, bm32);
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
        range_accumulate_row<VT>(a0, a1, base, sink_zero, lane, colA, valA, rowptrB, colB_lane, valB_lane, bm64,
                                 prefix16, acc);
        __syncwarp();
        for (int i = lane; i < cntc; i += 32) {
            colC[o + i] = ocol[i];
            valC[o + i] = acc[i];
        }
        // ---- restore the all-zero bitmap (only the words that were set) ----
        for (int i = lane; i < cntc; i += 32) bm64[(ocol[i] - base) >> 6] = 0ull;
        __syncwarp();
    }
}

// warps per block / blocks per SM that maximise resident warps for a per-warp footprint
inline void range_launch_shape(size_t warp_bytes, int &wpb, int &blocks_per_sm)
{
    int best_w = 0, best_wpb = 4, best_b = 1;
    for (int w = 4; w <= 16; ++w) {
        const size_t smem = warp_bytes * w;
        if (smem > 227 * 1024) break;
        int b = (int)((228 * 1024) / (smem + 1024));
        if (b > 32) b = 32;
        if (b * w > 64) b = 64 / w;
        if (b < 1) continue;
        if (b * w > best_w) {
            best_w = b * w;
            best_wpb = w;
            best_b = b;
        }
    }
    wpb = best_wpb;
    blocks_per_sm = best_b;
}

template <typename VT>
static cudaError_t launch_num_range_t(const LaunchCtx &lc, int nsum, int nacc, const int *queue, int count, Csr A,
                                      Csr B, const int *rlo, const int64_t *rowoff, int *colC, void *valC, WordLists wl)
{
    if (count <= 0) return cudaSuccess;
    const size_t wb = num_range_warp_bytes(nsum, nacc, value_bytes<VT>);
    int wpb, bps;
    range_launch_shape(wb, wpb, bps);
    const size_t smem = wb * wpb;
    cudaError_t e = cudaFuncSetAttribute(k_num_range<VT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    bps = resident_blocks(k_num_range<VT>, wpb * 32, smem);
    long long blocks = ((long long)count + wpb - 1) / wpb;
    const long long cap = (long long)lc.sm_count * bps;
    if (blocks > cap) blocks = cap;
    ++*lc.launches;
    k_num_range<VT><<<(int)blocks, wpb * 32, smem, lc.stream>>>(queue, count, A.rowptr, A.col, (const VT *)A.val,
                                                                B.rowptr, B.col, (const VT *)B.val, rlo, nsum, nacc,
                                                                rowoff, colC, (VT *)valC, wl);
    return cudaGetLastError();
}

}  // namespace bhb
