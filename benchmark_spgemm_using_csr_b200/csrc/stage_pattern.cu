// stage_pattern.cu -- kernels of the diagonal-pattern mode (see stage_pattern.cuh).
#include "stage_pattern.cuh"

namespace bhb {

// ---------------------------------------------------------------------------------------------
// k_offset_set: the set of (column - row) over all entries of a CSR matrix.  Every CTA filters
// through a private shared-memory set, so only the first sighting of an offset per CTA reaches the
// global set (a structured matrix: a few dozen global probes per CTA, everything else is LDS hits).
// More than PAT_MAX_OFFS distinct offsets -- in a CTA or globally -- raise `overflow`; every
// entry checks the flag, so an unstructured matrix costs a few microseconds.
// ---------------------------------------------------------------------------------------------
constexpr int PAT_LOCAL_SLOTS = 256;

__device__ __forceinline__ void pat_set_insert_global(PatSet *set, const int d)
{
    unsigned h = ((unsigned)d * 2654435761u) >> (32 - 9);
    static_assert(PAT_SET_SLOTS == 512, "hash shift");
    volatile int *vs = set->slot;
    for (int probe = 0; probe < PAT_SET_SLOTS; ++probe) {
        const int v = vs[h];
        if (v == d) return;
        if (v == PAT_EMPTY) {
            const int old = atomicCAS(&set->slot[h], PAT_EMPTY, d);
            if (old == PAT_EMPTY) {
                if (atomicAdd(&set->count, 1) + 1 > PAT_MAX_OFFS) set->overflow = 1;
                return;
            }
            if (old == d) return;
        }
        if (*(volatile int *)&set->overflow) return;
        h = (h + 1) & (PAT_SET_SLOTS - 1);
    }
    set->overflow = 1;
}

__global__ void __launch_bounds__(256) k_offset_set(const int rows, const int *__restrict__ rowptr,
                                                    const int *__restrict__ col, PatSet *__restrict__ set)
{
    __shared__ int s_slot[PAT_LOCAL_SLOTS];
    __shared__ int s_count, s_stop;
    for (int i = threadIdx.x; i < PAT_LOCAL_SLOTS; i += blockDim.x) s_slot[i] = PAT_EMPTY;
    if (threadIdx.x == 0) {
        s_count = 0;
        s_stop = *(volatile int *)&set->overflow;
    }
    __syncthreads();
    const int gl = threadIdx.x & 7;
    const long long stride = (long long)gridDim.x * (blockDim.x >> 3);
    int c0 = PAT_EMPTY, c1 = PAT_EMPTY, c2 = PAT_EMPTY, c3 = PAT_EMPTY;
    for (long long r = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 3; r < rows; r += stride) {
        if (*(volatile int *)&s_stop) return;
        if (gl == 0 && *(volatile int *)&set->overflow) *(volatile int *)&s_stop = 1;
        const int s = rowptr[r], e = rowptr[r + 1];
        for (int p = s + gl; p < e; p += 8) {
            const int d = col[p] - (int)r;
            // lane gl of a row sees entries gl, gl + 8, ...: in a structured matrix the same few offsets row
            // after row -- four registers catch them before shared memory is touched
            if (d == c0 || d == c1 || d == c2 || d == c3) continue;
            c3 = c2, c2 = c1, c1 = c0, c0 = d;
            if (*(volatile int *)&s_stop) return;
            if (d == PAT_EMPTY) {   // (an offset no int32-indexed matrix of sane size has)
                set->overflow = 1;
                *(volatile int *)&s_stop = 1;
                return;
            }
            unsigned h = ((unsigned)d * 2654435761u) >> (32 - 8);
            static_assert(PAT_LOCAL_SLOTS == 256, "hash shift");
            while (true) {
                const int v = *(volatile int *)&s_slot[h];
                if (v == d) break;
                if (v == PAT_EMPTY) {
                    const int old = atomicCAS(&s_slot[h], PAT_EMPTY, d);
                    if (old == PAT_EMPTY) {
                        // first sighting in this CTA
                        // (an unstructured matrix: some CTA overflows within microseconds; the others must not
                        // queue up on the global set's atomics -- measured 260 us on a random 4M-row matrix before)
                        if (*(volatile int *)&set->overflow) {
                            *(volatile int *)&s_stop = 1;
                        } else if (atomicAdd(&s_count, 1) + 1 > PAT_MAX_OFFS) {
                            set->overflow = 1;
                            *(volatile int *)&s_stop = 1;
                        } else {
                            pat_set_insert_global(set, d);
                        }
                        break;
                    }
                    if (old == d) break;
                }
                if (*(volatile int *)&s_stop) return;
                h = (h + 1) & (PAT_LOCAL_SLOTS - 1);
            }
        }
    }
}

cudaError_t launch_offset_set(const LaunchCtx &lc, int rows, const int *rowptr, const int *col, PatSet *set)
{
    if (rows <= 0) return cudaSuccess;
    long long blocks = ((long long)rows * 8 + 255) / 256;
    const long long cap = (long long)lc.sm_count * 8;
    if (blocks > cap) blocks = cap;
    ++*lc.launches;
    k_offset_set<<<(int)blocks, 256, 0, lc.stream>>>(rows, rowptr, col, set);
    return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------
// k_pat_codes: code[p] = index of (col[p] - row) in the sorted offset list (binary search in
// shared memory); rowmask[r] = OR of 1 << code over the row (B only).
// ---------------------------------------------------------------------------------------------
// DIRECT: the offsets span at most PAT_DIRECT_SPAN values: a byte table indexed by (offset - smallest
// offset) in shared memory replaces the binary search (one LDS.U8 per entry instead of six LDS + compares).
constexpr int PAT_DIRECT_SPAN = 40 * 1024;

template <bool DIRECT>
__global__ void __launch_bounds__(256) k_pat_codes(const int rows, const int ncols, const int *__restrict__ rowptr,
                                                   const int *__restrict__ col, const int *__restrict__ offs,
                                                   const int noffs, const int span, unsigned char *__restrict__ code,
                                                   unsigned long long *__restrict__ rowmask, int *__restrict__ bad,
                                                   int *__restrict__ miss, int *__restrict__ col_range_out,
                                                   const int *__restrict__ row_range)
{
    __shared__ int s_offs[PAT_MAX_OFFS];
    extern __shared__ unsigned char s_tab[];
    if (threadIdx.x < PAT_MAX_OFFS) s_offs[threadIdx.x] = threadIdx.x < noffs ? offs[threadIdx.x] : 0x7fffffff;
    if constexpr (DIRECT) {
        for (int i = threadIdx.x * 16; i < span; i += blockDim.x * 16) *reinterpret_cast<uint4 *>(s_tab + i) = make_uint4(~0u, ~0u, ~0u, ~0u);
    }
    __syncthreads();
    const int dmin = s_offs[0];
    if constexpr (DIRECT) {
        if (threadIdx.x < noffs) s_tab[s_offs[threadIdx.x] - dmin] = (unsigned char)threadIdx.x;
        __syncthreads();
    }
    const int gl = threadIdx.x & 7;
    const long long stride = (long long)gridDim.x * (blockDim.x >> 3);
    // row_range (B in a multi-GPU row block): only the rows of B that the block of A references are coded
    // and checked -- {largest column of A, INT_MAX - smallest column of A} as written by the pass over A
    long long r_first = 0, r_end = rows;
    if (row_range) {
        r_first = 0x7fffffffLL - (long long)row_range[1];
        r_end = min((long long)rows, (long long)row_range[0] + 1);
    }
    int cmax = 0, cnegmax = 0;
    for (long long r = r_first + (((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 3); r < r_end; r += stride) {
        const int s = rowptr[r], e = rowptr[r + 1];
        unsigned long long mask = 0ull;
        bool wrong = e < s, unknown = false;
        for (int p = s + gl; p < e; p += 8) {
            const int c = col[p];
            cmax = max(cmax, c);
            cnegmax = max(cnegmax, 0x7fffffff - c);
            // the operand preconditions (see k_b_row_ranges): columns inside the matrix; for B
            // (rowmask != nullptr) strictly ascending along the row
            wrong |= (unsigned)c >= (unsigned)ncols;
            if (rowmask) wrong |= (p > s && col[p - 1] >= c);
            const int d = c - (int)r;
            int lo = 0;   // index of d in the sorted offset list
            if constexpr (DIRECT) {
                const unsigned rel = (unsigned)(d - dmin);
                lo = rel < (unsigned)span ? s_tab[rel] : 0xff;
            } else {
#pragma unroll
                for (int step = PAT_MAX_OFFS / 2; step > 0; step >>= 1)
                    if (s_offs[lo + step - 1] < d) lo += step;
                if (s_offs[lo] != d) lo = 0xff;
            }
            // an offset that is not in the list: the (cached) plan does not describe this matrix any
            // more -- flagged, the caller re-runs the detection; a valid code keeps the later kernels in bounds
            if (lo >= noffs) {
                unknown = true;
                lo = 0;
            }
            code[p] = (unsigned char)lo;
            mask |= 1ull << lo;
        }
        if (wrong) *bad = 1;
        if (unknown) *miss = 1;
        if (rowmask) {
            mask |= __shfl_xor_sync(group_mask<8>(threadIdx.x & 31), mask, 1, 8);
            mask |= __shfl_xor_sync(group_mask<8>(threadIdx.x & 31), mask, 2, 8);
            mask |= __shfl_xor_sync(group_mask<8>(threadIdx.x & 31), mask, 4, 8);
            if (gl == 0) rowmask[r] = mask;
        }
    }
    if (col_range_out) {   // column range of the matrix (a pass over A): which rows of B matter
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) {
            cmax = max(cmax, __shfl_xor_sync(FULL, cmax, d));
            cnegmax = max(cnegmax, __shfl_xor_sync(FULL, cnegmax, d));
        }
        if ((threadIdx.x & 31) == 0) {
            atomicMax(&col_range_out[0], cmax);
            atomicMax(&col_range_out[1], cnegmax);
        }
    }
}

// one bit per row of B: the row holds every offset of DB (then its image under any A offset is the
// precomputed P[ja] and k_pat_symbolic does not need the 8-byte mask)
__global__ void __launch_bounds__(256) k_pat_fullbits(const int rows, const unsigned long long *__restrict__ rowmask,
                                                      const unsigned long long full, unsigned *__restrict__ bits)
{
    const long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const bool f = r < rows && rowmask[r] == full;
    const unsigned b = __ballot_sync(FULL, f);
    if ((threadIdx.x & 31) == 0 && (r >> 5) <= ((long long)rows - 1) >> 5) bits[r >> 5] = b;
}

cudaError_t launch_pat_codes(const LaunchCtx &lc, int rows, int ncols, const int *rowptr, const int *col, const int *offs,
                             int noffs, long long span, unsigned char *code, unsigned long long *rowmask, int *bad, int *miss,
                             unsigned long long full, unsigned *fullbits, int *col_range_out, const int *row_range)
{
    if (rows <= 0) return cudaSuccess;
    long long blocks = ((long long)rows * 8 + 255) / 256;
    const long long cap = (long long)lc.sm_count * 4;
    if (blocks > cap) blocks = cap;
    ++*lc.launches;
    if (span > 0 && span <= PAT_DIRECT_SPAN) {
        const size_t smem = ((size_t)span + 15) & ~(size_t)15;
        k_pat_codes<true><<<(int)blocks, 256, smem, lc.stream>>>(rows, ncols, rowptr, col, offs, noffs, (int)span, code, rowmask, bad,
                                                                  miss, col_range_out, row_range);
    } else {
        k_pat_codes<false><<<(int)blocks, 256, 0, lc.stream>>>(rows, ncols, rowptr, col, offs, noffs, 0, code, rowmask, bad, miss,
                                                                col_range_out, row_range);
    }
    if (rowmask && fullbits) {
        ++*lc.launches;
        k_pat_fullbits<<<(rows + 255) / 256, 256, 0, lc.stream>>>(rows, rowmask, full, fullbits);
    }
    return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------
// k_pat_symbolic: 8 lanes per row of A.  The output-offset mask of row i is the OR over its
// entries (ja, k) of the image of B row k's offset mask under jb -> M[ja][jb]; for a B row that
// holds every offset of DB (all interior rows of a stencil) that image is the precomputed
// P[ja].  nnz(C_i) = popcount.  The mask is kept for the numeric kernel.
// ---------------------------------------------------------------------------------------------
template <int NW>
__global__ void __launch_bounds__(256) k_pat_symbolic(const int m, const int *__restrict__ rowptrA,
                                                      const int *__restrict__ colA,
                                                      const unsigned char *__restrict__ ta,
                                                      const unsigned long long *__restrict__ maskB, const PatTables t,
                                                      unsigned *__restrict__ outmask, int *__restrict__ rc,
                                                      int *__restrict__ prod, Counters *__restrict__ ctr, const int k,
                                                      const unsigned *__restrict__ fullbits)
{
    __shared__ unsigned long long s_total;
    __shared__ int s_max;
    __shared__ unsigned s_pfull[PAT_MAX_OFFS * NW];
    __shared__ unsigned char s_mlog[PAT_MAX_OFFS * PAT_MAX_OFFS];
    if (threadIdx.x == 0) {
        s_total = 0ull;
        s_max = 0;
    }
    for (int i = threadIdx.x; i < t.nDA * NW; i += blockDim.x) s_pfull[i] = t.pfull[i];
    for (int i = threadIdx.x; i < t.nDA * t.nDB; i += blockDim.x) s_mlog[i] = t.mlog[i];
    __syncthreads();
    const int gl = threadIdx.x & 7;
    const unsigned gmask = group_mask<8>(threadIdx.x & 31);
    const long long stride = (long long)gridDim.x * (blockDim.x >> 3);
    unsigned long long my_total = 0ull;
    int my_max = 0;
    for (long long r = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 3; r < m; r += stride) {
        const int a0 = rowptrA[r], a1 = rowptrA[r + 1];
        unsigned mk[NW];
#pragma unroll
        for (int w = 0; w < NW; ++w) mk[w] = 0u;
        int p = 0;   // intermediate products of the row: a B row holds popcount(mask) entries
        // four entries per lane and step: the dependent gathers colA -> maskB of up to 32 entries of the
        // row are in flight together (the kernel is bound by their latency, not by instructions)
        for (int j0 = a0 + gl; j0 < a1; j0 += 32) {
            int ja[4], ck[4];
            unsigned long long mb[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int j = j0 + 8 * u;
                const bool in = j < a1;
                ja[u] = in ? ta[j] : 0;
                ck[u] = in ? colA[j] : -1;
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) {   // (bad columns are flagged by k_pat_codes)
                const bool okc = (unsigned)ck[u] < (unsigned)k;
                const bool isfull = okc && ((__ldg(fullbits + (ck[u] >> 5)) >> (ck[u] & 31)) & 1u);
                mb[u] = isfull ? t.fullB : (okc ? maskB[ck[u]] : 0ull);   // the 8-byte mask only for partial rows
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                unsigned long long m1 = mb[u];
                p += __popcll(m1);
                if (m1 == t.fullB) {
#pragma unroll
                    for (int w = 0; w < NW; ++w) mk[w] |= s_pfull[ja[u] * NW + w];
                } else if (m1) {
                    // partial B row (boundary cells of a grid): the image of its offset set.  Walk whichever is
                    // shorter, the offsets present (set their output bits) or the ones missing (clear them
                    // from the full-row image; for a fixed A offset jb -> output is injective).
                    const unsigned long long miss = t.fullB & ~m1;
                    const bool by_missing = __popcll(miss) < __popcll(m1);
                    unsigned long long walk = by_missing ? miss : m1;
                    unsigned img[NW];
#pragma unroll
                    for (int w = 0; w < NW; ++w) img[w] = by_missing ? s_pfull[ja[u] * NW + w] : 0u;
                    const unsigned char *mrow = s_mlog + ja[u] * t.nDB;
                    while (walk) {
                        const int jb = __ffsll((long long)walk) - 1;
                        walk &= walk - 1;
                        const int o = mrow[jb];
#pragma unroll
                        for (int w = 0; w < NW; ++w) img[w] ^= ((o >> 5) == w) ? (1u << (o & 31)) : 0u;   // set, or clear from the full image
                    }
#pragma unroll
                    for (int w = 0; w < NW; ++w) mk[w] |= img[w];
                }
            }
        }
        int cnt = 0;
#pragma unroll
        for (int w = 0; w < NW; ++w) {
            mk[w] |= __shfl_xor_sync(gmask, mk[w], 1, 8);
            mk[w] |= __shfl_xor_sync(gmask, mk[w], 2, 8);
            mk[w] |= __shfl_xor_sync(gmask, mk[w], 4, 8);
            cnt += __popc(mk[w]);
            if (gl == (w & 7)) outmask[r * NW + w] = mk[w];
        }
        p += __shfl_xor_sync(gmask, p, 1, 8);
        p += __shfl_xor_sync(gmask, p, 2, 8);
        p += __shfl_xor_sync(gmask, p, 4, 8);
        if (gl == 0) {
            rc[r] = cnt;
            prod[r] = p;       // (<= 64 * 64: no overflow)
            my_total += (unsigned long long)p;
            my_max = max(my_max, p);
        }
    }
    my_total = warp_sum(my_total);
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) my_max = max(my_max, __shfl_xor_sync(FULL, my_max, d));
    if ((threadIdx.x & 31) == 0) {
        atomicAdd(&s_total, my_total);
        atomicMax(&s_max, my_max);
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        if (s_total) atomicAdd(&ctr->products, s_total);
        atomicMax(&ctr->max_row_products, s_max);
    }
}

// Warp-per-row variant (rows of A with more than 8 entries on average): one entry per lane, so the
// dependent gathers colA -> maskB of a row are all in flight together, and the OR / sum over the
// row are single REDUX instructions.
template <int NW>
__global__ void __launch_bounds__(256) k_pat_symbolic_warp(const int m, const int *__restrict__ rowptrA,
                                                           const int *__restrict__ colA,
                                                           const unsigned char *__restrict__ ta,
                                                           const unsigned long long *__restrict__ maskB, const PatTables t,
                                                           unsigned *__restrict__ outmask, int *__restrict__ rc,
                                                           int *__restrict__ prod, Counters *__restrict__ ctr, const int k,
                                                           const unsigned *__restrict__ fullbits)
{
    (void)fullbits;
    __shared__ unsigned long long s_total;
    __shared__ int s_max;
    __shared__ unsigned s_pfull[PAT_MAX_OFFS * NW];
    if (threadIdx.x == 0) {
        s_total = 0ull;
        s_max = 0;
    }
    for (int i = threadIdx.x; i < t.nDA * NW; i += blockDim.x) s_pfull[i] = t.pfull[i];
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const long long nwarps = (long long)gridDim.x * (blockDim.x >> 5);
    unsigned long long my_total = 0ull;
    int my_max = 0;
    for (long long r = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); r < m; r += nwarps) {
        const int a0 = rowptrA[r], a1 = rowptrA[r + 1];
        unsigned mk[NW];
#pragma unroll
        for (int w = 0; w < NW; ++w) mk[w] = 0u;
        int p = 0;
        for (int j = a0 + lane; j < a1; j += 32) {
            const int ja = ta[j];
            const int ck = colA[j];
            if ((unsigned)ck >= (unsigned)k) continue;   // (flagged by k_pat_codes; not followed)
            unsigned long long mb = maskB[ck];
            p += __popcll(mb);
            if (mb == t.fullB) {
#pragma unroll
                for (int w = 0; w < NW; ++w) mk[w] |= s_pfull[ja * NW + w];
            } else {
                while (mb) {
                    const int jb = __ffsll((long long)mb) - 1;
                    mb &= mb - 1;
                    const int o = t.mlog[ja * t.nDB + jb];
#pragma unroll
                    for (int w = 0; w < NW; ++w) mk[w] |= ((o >> 5) == w) ? (1u << (o & 31)) : 0u;
                }
            }
        }
        int cnt = 0;
#pragma unroll
        for (int w = 0; w < NW; ++w) {
            mk[w] = __reduce_or_sync(FULL, mk[w]);
            cnt += __popc(mk[w]);
            if (lane == w) outmask[r * NW + w] = mk[w];
        }
        p = __reduce_add_sync(FULL, p);
        if (lane == 0) {
            rc[r] = cnt;
            prod[r] = p;
            my_total += (unsigned long long)p;
            my_max = max(my_max, p);
        }
    }
    if (lane == 0) {
        atomicAdd(&s_total, my_total);
        atomicMax(&s_max, my_max);
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        if (s_total) atomicAdd(&ctr->products, s_total);
        atomicMax(&ctr->max_row_products, s_max);
    }
}

cudaError_t launch_pat_symbolic(const LaunchCtx &lc, int m, Csr A, const unsigned char *ta, const unsigned long long *maskB,
                                PatTables t, unsigned *outmask, int *rc, int *prod, Counters *ctr, int k, double avg_row,
                                const unsigned *fullbits)
{
    if (m <= 0) return cudaSuccess;
    ++*lc.launches;
    const long long cap = (long long)lc.sm_count * 8;
    if (avg_row > 40.0) {   // (measured: the 8-lane kernel wins up to 27 entries per row, profiles/r02_notes.md)
        long long blocks = ((long long)m + 7) / 8;
        if (blocks > cap) blocks = cap;
        switch (t.nw) {
        case 1: k_pat_symbolic_warp<1><<<(int)blocks, 256, 0, lc.stream>>>(m, A.rowptr, A.col, ta, maskB, t, outmask, rc, prod, ctr, k, fullbits); break;
        case 2: k_pat_symbolic_warp<2><<<(int)blocks, 256, 0, lc.stream>>>(m, A.rowptr, A.col, ta, maskB, t, outmask, rc, prod, ctr, k, fullbits); break;
        case 4: k_pat_symbolic_warp<4><<<(int)blocks, 256, 0, lc.stream>>>(m, A.rowptr, A.col, ta, maskB, t, outmask, rc, prod, ctr, k, fullbits); break;
        case 8: k_pat_symbolic_warp<8><<<(int)blocks, 256, 0, lc.stream>>>(m, A.rowptr, A.col, ta, maskB, t, outmask, rc, prod, ctr, k, fullbits); break;
        default: return cudaErrorInvalidValue;
        }
        return cudaGetLastError();
    }
    long long blocks = ((long long)m * 8 + 255) / 256;
    if (blocks > cap * 2) blocks = cap * 2;
    switch (t.nw) {
    case 1: k_pat_symbolic<1><<<(int)blocks, 256, 0, lc.stream>>>(m, A.rowptr, A.col, ta, maskB, t, outmask, rc, prod, ctr, k, fullbits); break;
    case 2: k_pat_symbolic<2><<<(int)blocks, 256, 0, lc.stream>>>(m, A.rowptr, A.col, ta, maskB, t, outmask, rc, prod, ctr, k, fullbits); break;
    case 4: k_pat_symbolic<4><<<(int)blocks, 256, 0, lc.stream>>>(m, A.rowptr, A.col, ta, maskB, t, outmask, rc, prod, ctr, k, fullbits); break;
    case 8: k_pat_symbolic<8><<<(int)blocks, 256, 0, lc.stream>>>(m, A.rowptr, A.col, ta, maskB, t, outmask, rc, prod, ctr, k, fullbits); break;
    default: return cudaErrorInvalidValue;
    }
    return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------
// k_pat_numeric: a group of G lanes owns a row of C (G = 32 unless B rows have <= 8 / <= 16
// entries).  The row's A entries are staged as 16-byte records {B row start, length | ja << 16,
// value} in shared memory and read back as one broadcast LDS.128 per B row (four shuffles in the
// hash kernels).  Per product: one byte of B's offset codes, one value of B, one byte of the
// position table, LDS/FMA/STS on the dense accumulator.  The accumulator layout (PatTables::pos)
// is chosen on the host so that the products of one B row fall into distinct banks.
// Rows are taken in natural order: neighbouring rows read the same rows of B.
// All loops are warp-uniform (see k_num_group).
// ---------------------------------------------------------------------------------------------
// Shared-memory accesses by 32-bit shared-space address: the hot loop below is bound by instruction
// issue, and generic-pointer arithmetic on the dynamic shared window costs three uniform-datapath
// instructions per access (S2UR / UMOV / ULEA in the first version's SASS).
__device__ __forceinline__ unsigned sm_addr(const void *p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ int lds_u8(unsigned a)
{
    unsigned v;
    asm volatile("ld.shared.u8 %0, [%1];" : "=r"(v) : "r"(a) : "memory");
    return (int)v;
}
__device__ __forceinline__ int4 lds_v4(unsigned a)
{
    int4 v;
    asm volatile("ld.shared.v4.s32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(a) : "memory");
    return v;
}
__device__ __forceinline__ double lds_val(unsigned a, double)
{
    double v;
    asm volatile("ld.shared.f64 %0, [%1];" : "=d"(v) : "r"(a) : "memory");
    return v;
}
__device__ __forceinline__ float lds_val(unsigned a, float)
{
    float v;
    asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(a) : "memory");
    return v;
}
__device__ __forceinline__ void sts_val(unsigned a, double v) { asm volatile("st.shared.f64 [%0], %1;" ::"r"(a), "d"(v) : "memory"); }
__device__ __forceinline__ void sts_val(unsigned a, float v) { asm volatile("st.shared.f32 [%0], %1;" ::"r"(a), "f"(v) : "memory"); }
__device__ __forceinline__ c64 lds_val(unsigned a, c64)
{
    c64 v;
    asm volatile("ld.shared.v2.f32 {%0, %1}, [%2];" : "=f"(v.re), "=f"(v.im) : "r"(a) : "memory");
    return v;
}
__device__ __forceinline__ void sts_val(unsigned a, c64 v)
{
    asm volatile("st.shared.v2.f32 [%0], {%1, %2};" ::"r"(a), "f"(v.re), "f"(v.im) : "memory");
}
__device__ __forceinline__ c128 lds_val(unsigned a, c128)
{
    c128 v;
    asm volatile("ld.shared.v2.f64 {%0, %1}, [%2];" : "=d"(v.re), "=d"(v.im) : "r"(a) : "memory");
    return v;
}
__device__ __forceinline__ void sts_val(unsigned a, c128 v)
{
    asm volatile("st.shared.v2.f64 [%0], {%1, %2};" ::"r"(a), "d"(v.re), "d"(v.im) : "memory");
}

// Predicated (not branched) element load and accumulate of the hot loop: inactive lanes issue no memory
// access at all, and the warp stays converged.
__device__ __forceinline__ void pat_load_if(const bool on, const unsigned char *cp, const double *vp, int &jb, double &bv)
{
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.s32 p, %2, 0;\n"
        "@p ld.global.nc.u8 %0, [%3];\n"
        "@p ld.global.nc.f64 %1, [%4];\n"
        "}\n"
        : "+r"(jb), "+d"(bv)
        : "r"((int)on), "l"(cp), "l"(vp)
        : "memory");
}
__device__ __forceinline__ void pat_load_if(const bool on, const unsigned char *cp, const float *vp, int &jb, float &bv)
{
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.s32 p, %2, 0;\n"
        "@p ld.global.nc.u8 %0, [%3];\n"
        "@p ld.global.nc.f32 %1, [%4];\n"
        "}\n"
        : "+r"(jb), "+f"(bv)
        : "r"((int)on), "l"(cp), "l"(vp)
        : "memory");
}
// acc[ mphys[mp] ] += av * bv   (mp, acc_s: shared-space addresses)
__device__ __forceinline__ void pat_accum_if(const bool on, const unsigned mp, const unsigned acc_s, const double av, const double bv)
{
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        ".reg .u32 q, a;\n"
        ".reg .f64 v;\n"
        "setp.ne.s32 p, %0, 0;\n"
        "@p ld.shared.u8 q, [%1];\n"
        "@p mad.lo.u32 a, q, 8, %2;\n"
        "@p ld.shared.f64 v, [a];\n"
        "@p fma.rn.f64 v, %3, %4, v;\n"
        "@p st.shared.f64 [a], v;\n"
        "}\n" ::"r"((int)on),
        "r"(mp), "r"(acc_s), "d"(av), "d"(bv)
        : "memory");
}
__device__ __forceinline__ void pat_accum_if(const bool on, const unsigned mp, const unsigned acc_s, const float av, const float bv)
{
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        ".reg .u32 q, a;\n"
        ".reg .f32 v;\n"
        "setp.ne.s32 p, %0, 0;\n"
        "@p ld.shared.u8 q, [%1];\n"
        "@p mad.lo.u32 a, q, 4, %2;\n"
        "@p ld.shared.f32 v, [a];\n"
        "@p fma.rn.f32 v, %3, %4, v;\n"
        "@p st.shared.f32 [a], v;\n"
        "}\n" ::"r"((int)on),
        "r"(mp), "r"(acc_s), "f"(av), "f"(bv)
        : "memory");
}
// complex64: the 8-byte accumulator slot of a double, four FMAs (re += ar*br + (-ai)*bi, im += ar*bi + ai*br)
__device__ __forceinline__ void pat_accum_if(const bool on, const unsigned mp, const unsigned acc_s, const c64 av, const c64 bv)
{
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        ".reg .u32 q, a;\n"
        ".reg .f32 vr, vi;\n"
        "setp.ne.s32 p, %0, 0;\n"
        "@p ld.shared.u8 q, [%1];\n"
        "@p mad.lo.u32 a, q, 8, %2;\n"
        "@p ld.shared.v2.f32 {vr, vi}, [a];\n"
        "@p fma.rn.f32 vr, %3, %5, vr;\n"
        "@p fma.rn.f32 vr, %7, %6, vr;\n"
        "@p fma.rn.f32 vi, %3, %6, vi;\n"
        "@p fma.rn.f32 vi, %4, %5, vi;\n"
        "@p st.shared.v2.f32 [a], {vr, vi};\n"
        "}\n" ::"r"((int)on),
        "r"(mp), "r"(acc_s), "f"(av.re), "f"(av.im), "f"(bv.re), "f"(bv.im), "f"(-av.im)
        : "memory");
}
// complex128: a 16-byte accumulator slot, the same four FMAs in double
__device__ __forceinline__ void pat_accum_if(const bool on, const unsigned mp, const unsigned acc_s, const c128 av, const c128 bv)
{
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        ".reg .u32 q, a;\n"
        ".reg .f64 vr, vi;\n"
        "setp.ne.s32 p, %0, 0;\n"
        "@p ld.shared.u8 q, [%1];\n"
        "@p mad.lo.u32 a, q, 16, %2;\n"
        "@p ld.shared.v2.f64 {vr, vi}, [a];\n"
        "@p fma.rn.f64 vr, %3, %5, vr;\n"
        "@p fma.rn.f64 vr, %7, %6, vr;\n"
        "@p fma.rn.f64 vi, %3, %6, vi;\n"
        "@p fma.rn.f64 vi, %4, %5, vi;\n"
        "@p st.shared.v2.f64 [a], {vr, vi};\n"
        "}\n" ::"r"((int)on),
        "r"(mp), "r"(acc_s), "d"(av.re), "d"(av.im), "d"(bv.re), "d"(bv.im), "d"(-av.im)
        : "memory");
}

// The per-lane record of one A entry: its B row start bs, lj = length | (ja * nDB) << 16, and the value.  Values of
// at most 8 bytes share one 16-byte int4 with bs and lj; a complex128 value takes a 32-byte record of its own layout.
struct PatRec16 {
    using Rec = int4;
    static __device__ __forceinline__ Rec load(unsigned a) { return lds_v4(a); }
};
template <typename VT>
struct PatRec;
template <>
struct PatRec<double> : PatRec16 {
    static __device__ __forceinline__ int4 pack(int bs, int lj, double v)
    {
        return make_int4(bs, lj, __double2loint(v), __double2hiint(v));
    }
    static __device__ __forceinline__ double val(const int4 &r) { return __hiloint2double(r.w, r.z); }
};
template <>
struct PatRec<float> : PatRec16 {
    static __device__ __forceinline__ int4 pack(int bs, int lj, float v) { return make_int4(bs, lj, __float_as_int(v), 0); }
    static __device__ __forceinline__ float val(const int4 &r) { return __int_as_float(r.z); }
};
template <>
struct PatRec<c64> : PatRec16 {   // {bs, lj, re, im}
    static __device__ __forceinline__ int4 pack(int bs, int lj, c64 v)
    {
        return make_int4(bs, lj, __float_as_int(v.re), __float_as_int(v.im));
    }
    static __device__ __forceinline__ c64 val(const int4 &r) { return c64(__int_as_float(r.z), __int_as_float(r.w)); }
};
struct __align__(16) PatRec32 {   // {bs, lj, -, -, re, im}
    int x, y, z, w;
    double re, im;
};
template <>
struct PatRec<c128> {
    using Rec = PatRec32;
    static __device__ __forceinline__ Rec pack(int bs, int lj, c128 v) { return Rec{bs, lj, 0, 0, v.re, v.im}; }
    static __device__ __forceinline__ c128 val(const Rec &r) { return c128(r.re, r.im); }
    static __device__ __forceinline__ Rec load(unsigned a)
    {
        const int4 h = lds_v4(a);
        Rec r{h.x, h.y, h.z, h.w, 0.0, 0.0};
        asm volatile("ld.shared.v2.f64 {%0, %1}, [%2];" : "=d"(r.re), "=d"(r.im) : "r"(a + 16u) : "memory");
        return r;
    }
};

// LONGB: rows of B may hold more than G entries (only possible for G = 32 with more than 32 diagonals in B)
// 6 CTAs per SM (40 registers): per-warp memory-level parallelism beat 8 CTAs at 32 registers (profiles/r02_notes.md).
// complex128 takes 4 (64 registers): its 32-byte records and 16-byte values spill 72 / 124 bytes at 40.
template <typename VT, int G, bool LONGB>
__global__ void __launch_bounds__(256, value_bytes<VT> > 8 ? 4 : 6)
k_pat_numeric(const int m, const int *__restrict__ rowptrA, const int *__restrict__ colA, const VT *__restrict__ valA,
              const unsigned char *__restrict__ ta, const int *__restrict__ rowptrB, const unsigned char *__restrict__ tb,
              const VT *__restrict__ valB, const PatTables t, const unsigned *__restrict__ outmask,
              const int64_t *__restrict__ rowoff, int *__restrict__ colC, VT *__restrict__ valC)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    // CTA-wide tables: dcol int[nD] | mphys u8[nDA*nDB] | pos u8[nD]   (padded to 16 bytes)
    int *s_dcol = reinterpret_cast<int *>(smem_raw);
    unsigned char *s_mphys = smem_raw + (size_t)t.nD * 4;
    unsigned char *s_pos = s_mphys + (size_t)t.nDA * t.nDB;
    const size_t tab_bytes = ((size_t)t.nD * 4 + (size_t)t.nDA * t.nDB + (size_t)t.nD + 15) & ~(size_t)15;
    for (int i = threadIdx.x; i < t.nD; i += blockDim.x) {
        s_dcol[i] = t.dcol[i];
        s_pos[i] = t.pos[i];
    }
    for (int i = threadIdx.x; i < t.nDA * t.nDB; i += blockDim.x) s_mphys[i] = t.mphys[i];
    __syncthreads();

    constexpr int GPW = 32 / G;   // groups per warp
    const int lane = threadIdx.x & 31;
    const int gl = threadIdx.x & (G - 1);
    const int gib = threadIdx.x / G;
    const int groups_per_block = blockDim.x / G;
    const int gshift = lane & ~(G - 1);
    const unsigned gbits = (G == 32) ? FULL : ((1u << (G & 31)) - 1u);
    const int acc_len = t.acc_len;
    using Rec = typename PatRec<VT>::Rec;
    const size_t per_group = (size_t)acc_len * sizeof(VT) + (size_t)G * sizeof(Rec);   // accumulators | records
    unsigned char *mine = smem_raw + tab_bytes + (size_t)gib * per_group;
    VT *acc = reinterpret_cast<VT *>(mine);
    Rec *rec = reinterpret_cast<Rec *>(mine + (size_t)acc_len * sizeof(VT));
    const int nDB = t.nDB, nD = t.nD, nw = t.nw;
    (void)gshift;
    (void)gbits;
    const unsigned acc_s = sm_addr(acc), rec_s = sm_addr(rec), mphys_s = sm_addr(s_mphys);

    for (long long q0 = (long long)blockIdx.x * groups_per_block + (gib & ~(GPW - 1)); q0 < m;
         q0 += (long long)gridDim.x * groups_per_block) {
        const long long q = q0 + (gib & (GPW - 1));
        const bool active = q < m;
        const int row = active ? (int)q : 0;
        for (int s = gl; s < acc_len; s += G) acc[s] = VT(0);
        const int a0 = active ? rowptrA[row] : 0;
        const int na = active ? rowptrA[row + 1] - a0 : 0;
        const int max_na = (G == 32) ? na : __reduce_max_sync(FULL, na);
        for (int base = 0; base < max_na; base += G) {
            const int j = base + gl;
            if (j < na) {
                const int k = colA[a0 + j];
                const int bs = rowptrB[k];
                const int len = rowptrB[k + 1] - bs;
                rec[gl] = PatRec<VT>::pack(bs, len | (((int)ta[a0 + j] * nDB) << 16), valA[a0 + j]);   // (ja * nDB <= 63 * 64)
            } else {
                rec[gl] = Rec{};   // length 0: nothing to do for this slot
            }
            __syncwarp();
            const int cnt = min(G, max_na - base);   // warp-uniform
            // Software pipeline, two register sets in ping-pong: the loads of B row tt+1 (one code byte, one
            // value per lane) are issued before B row tt is accumulated.  Branch-free: lanes beyond the end of
            // their B row are predicated off (no memory access), the warp never diverges and every step is
            // straight-line code.
            Rec rA, rB;
            int jbA = 0, jbB = 0;
            VT bvA = VT(0), bvB = VT(0);
            bool onA = false, onB = false;
#define PAT_LOAD(R, JB, BV, ON, TT)                                      \
    do {                                                                  \
        R = PatRec<VT>::load(rec_s + (unsigned)(TT) * (unsigned)sizeof(Rec)); \
        ON = gl < (R.y & 0x7fff);                                         \
        /* lanes past the end re-read the row's first element (same cache line, no branch); empty row: element 0 */ \
        const int idx__ = ON ? R.x + gl : ((R.y & 0x7fff) ? R.x : 0);    \
        JB = tb[idx__]; /* (measured and dropped: skipping this load for B rows that hold every offset -- */ \
                        /*  code = lane -- the uniform branch cost more than the load: 3.8 -> 4.3 ms)   */ \
        BV = valB[idx__];                                                 \
    } while (0)
#define PAT_ACCUM(R, JB, BV, ON)                                                          \
    do {                                                                                   \
        pat_accum_if(ON, mphys_s + (unsigned)(R.y >> 16) + (unsigned)(JB), acc_s, PatRec<VT>::val(R), BV); \
        if constexpr (LONGB) {                                                             \
            const int len__ = R.y & 0x7fff;                                                \
            _Pragma("unroll 1") for (int off = G + gl; off < len__; off += G) {            \
                const int q__ = lds_u8(mphys_s + (unsigned)(R.y >> 16) + (unsigned)tb[R.x + off]); \
                const unsigned b__ = acc_s + (unsigned)q__ * (unsigned)sizeof(VT);         \
                sts_val(b__, fma(PatRec<VT>::val(R), valB[R.x + off], lds_val(b__, VT(0)))); \
            }                                                                              \
        }                                                                                  \
        __syncwarp(); /* the next B row may hit the same accumulators from other lanes */  \
    } while (0)
            PAT_LOAD(rA, jbA, bvA, onA, 0);
#pragma unroll 1
            for (int tt = 0; tt < cnt; tt += 2) {
                if (tt + 1 < cnt) PAT_LOAD(rB, jbB, bvB, onB, tt + 1);
                PAT_ACCUM(rA, jbA, bvA, onA);
                if (tt + 1 < cnt) {
                    if (tt + 2 < cnt) PAT_LOAD(rA, jbA, bvA, onA, tt + 2);
                    PAT_ACCUM(rB, jbB, bvB, onB);
                }
            }
#undef PAT_LOAD
#undef PAT_ACCUM
        }
        // ---- emit: output index o (ascending offset = ascending column) -> rank by popcount ----
        const int64_t o0 = active ? rowoff[row] : 0;
        const unsigned *mrow = outmask + (size_t)row * nw;
        int rank0 = 0;
        for (int ob = 0; ob < nD; ob += G) {
            const unsigned word = active ? __ldg(mrow + (ob >> 5)) : 0u;
            const unsigned bits = (G == 32) ? word : ((word >> (ob & 31)) & gbits);
            const int o = ob + gl;
            if ((bits >> gl) & 1u) {
                const int rnk = rank0 + __popc(bits & ((1u << gl) - 1u));
                colC[o0 + rnk] = row + s_dcol[o];
                valC[o0 + rnk] = acc[s_pos[o]];
            }
            rank0 += __popc(bits);
        }
        __syncwarp();
    }
}

template <typename VT, int G, bool LONGB>
static cudaError_t launch_pat_numeric_tbl(const LaunchCtx &lc, int m, Csr A, Csr B, const unsigned char *ta,
                                        const unsigned char *tb, const PatTables &t, const unsigned *outmask,
                                        const int64_t *rowoff, int *colC, VT *valC)
{
    const int threads = 256;
    const int groups = threads / G;
    const size_t tab_bytes = ((size_t)t.nD * 4 + (size_t)t.nDA * t.nDB + (size_t)t.nD + 15) & ~(size_t)15;
    const size_t smem = tab_bytes + (size_t)groups * ((size_t)t.acc_len * sizeof(VT) + (size_t)G * sizeof(typename PatRec<VT>::Rec));
    if (smem > SMEM_BLOCK_MAX) return cudaErrorInvalidValue;
    auto kern = k_pat_numeric<VT, G, LONGB>;
    if (smem > 48 * 1024) {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
    }
    long long blocks = ((long long)m + groups - 1) / groups;
    const long long cap = (long long)lc.sm_count * resident_blocks(kern, threads, smem);
    if (blocks > cap) blocks = cap;
    ++*lc.launches;
    kern<<<(int)blocks, threads, smem, lc.stream>>>(m, A.rowptr, A.col, (const VT *)A.val, ta, B.rowptr, tb,
                                                    (const VT *)B.val, t, outmask, rowoff, colC, valC);
    return cudaGetLastError();
}

template <typename VT, int G>
static cudaError_t launch_pat_numeric_t(const LaunchCtx &lc, int m, Csr A, Csr B, const unsigned char *ta,
                                        const unsigned char *tb, const PatTables &t, const unsigned *outmask,
                                        const int64_t *rowoff, int *colC, VT *valC)
{
    if constexpr (G == 32) {
        if (t.nDB > 32) return launch_pat_numeric_tbl<VT, G, true>(lc, m, A, B, ta, tb, t, outmask, rowoff, colC, valC);
    }
    return launch_pat_numeric_tbl<VT, G, false>(lc, m, A, B, ta, tb, t, outmask, rowoff, colC, valC);
}

// Structure-only products: row i of C is i + dcol[o] for the set bits o of its output mask, in ascending o (dcol is
// sorted, so the columns come out ascending) -- no operand is read and nothing is accumulated.  A warp per row: lane
// l of step w writes bit l of mask word w at the row's offset plus the popcount of the bits below it (coalesced).
__global__ void __launch_bounds__(256) k_pat_emit(const int m, const int nD, const int nw, const int *__restrict__ dcol,
                                                  const unsigned *__restrict__ outmask, const int64_t *__restrict__ rowoff,
                                                  int *__restrict__ colC)
{
    __shared__ int s_dcol[PAT_MAX_OUT];
    for (int i = threadIdx.x; i < nD; i += blockDim.x) s_dcol[i] = dcol[i];
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const unsigned below = (1u << lane) - 1u;
    const int warps = (int)((gridDim.x * blockDim.x) >> 5);
    for (int row = (int)((blockIdx.x * blockDim.x + threadIdx.x) >> 5); row < m; row += warps) {
        const unsigned mine = lane < nw ? __ldg(outmask + (size_t)row * nw + lane) : 0u;
        int64_t o = rowoff[row];
        for (int w = 0; w < nw; ++w) {
            const unsigned bits = __shfl_sync(FULL, mine, w);
            if ((bits >> lane) & 1u) colC[o + __popc(bits & below)] = row + s_dcol[(w << 5) + lane];
            o += __popc(bits);
        }
    }
}

cudaError_t launch_pat_numeric(const LaunchCtx &lc, int dtype, int m, Csr A, Csr B, const unsigned char *ta,
                               const unsigned char *tb, PatTables t, const unsigned *outmask, const int64_t *rowoff,
                               int *colC, void *valC)
{
    if (m <= 0) return cudaSuccess;
    if (dtype == BHB200_DTYPE_NONE) {
        const int threads = 256;
        long long blocks = ((long long)m * 32 + threads - 1) / threads;
        const long long cap = (long long)lc.sm_count * resident_blocks(k_pat_emit, threads, 0);
        if (blocks > cap) blocks = cap;
        ++*lc.launches;
        k_pat_emit<<<(int)blocks, threads, 0, lc.stream>>>(m, t.nD, t.nw, t.dcol, outmask, rowoff, colC);
        return cudaGetLastError();
    }
    const int G = t.nDB <= 8 ? 8 : t.nDB <= 16 ? 16 : 32;
    return dispatch_value_type(dtype, [&](auto val) {
        using VT = decltype(val);
        if constexpr (value_bytes<VT> == 0) {
            return cudaErrorInvalidValue;   // (handled above)
        } else {
            VT *v = (VT *)valC;
            if (G == 8) return launch_pat_numeric_t<VT, 8>(lc, m, A, B, ta, tb, t, outmask, rowoff, colC, v);
            if (G == 16) return launch_pat_numeric_t<VT, 16>(lc, m, A, B, ta, tb, t, outmask, rowoff, colC, v);
            return launch_pat_numeric_t<VT, 32>(lc, m, A, B, ta, tb, t, outmask, rowoff, colC, v);
        }
    });
}

}  // namespace bhb
