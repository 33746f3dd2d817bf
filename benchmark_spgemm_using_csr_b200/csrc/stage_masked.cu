// stage_masked.cu -- masked products C = M .* (op(A) op(B)) (DESIGN.md 4.10).
//
// M is structural (row pointers + sorted, duplicate-free columns).  Row i of C can only hold the
// columns of M_i, so nnz(M_i) bounds the row exactly: every row is computed in one pass and staged
// at rowptrM[i] in the staging buffer (Ct), then moved to C by k_copy_ct after the row-pointer
// scan, like the direct mode.  The slot of an output column is its rank in M_i, which is sorted:
// rows come out sorted by a ballot compaction of the hit flags, with no sort of the products.
//   k_mask_bins     after k_row_products: validates M, histogram of the masked bins (read back
//                   with the stage-1 counters)
//   k_mask_scatter  rows -> per-bin queue; rows without products or mask entries get nnz(C_i) = 0
//   k_mask_esc      p_i <= 32: one product per lane, binary search in M_i in global memory
//   k_mask_warp     warp per row, table of M_i in shared memory (p_i <= MASK_WARP_MAX_P)
//   k_mask_cta      CTA per row, table of M_i in shared memory (up to 8192 mask entries)
//   k_mask_global   CTA per row, binary search in M_i, values accumulated in global scratch
// The tables map mask column -> position in M_i; they are built once per row and only probed by
// the products.  A hit sets a per-position byte flag: a value of 0 cannot mark a hit, because
// explicit zeros from cancellation are kept.
#include "common.cuh"

namespace bhb {

namespace {

// slot of column c in a table built from M_i, or -1 (the table is at most half full: probing ends)
template <int LOG2T>
__device__ __forceinline__ int table_probe(const int *keys, int c)
{
    constexpr int MASK = (1 << LOG2T) - 1;
    int h = hash_slot<LOG2T>(c);
    while (true) {
        const int k = keys[h];
        if (k == c) return h;
        if (k == EMPTY_KEY) return -1;
        h = (h + 1) & MASK;
    }
}

// position of c in the sorted cols[0, len), or -1
__device__ __forceinline__ int mask_search(const int *__restrict__ cols, int len, int c)
{
    int lo = 0, hi = len - 1;
    while (lo <= hi) {
        const int mid = (lo + hi) >> 1;
        const int cm = cols[mid];
        if (cm == c) return mid;
        if (cm < c) lo = mid + 1;
        else hi = mid - 1;
    }
    return -1;
}

}  // namespace

// ---------------------------------------------------------------------------------------------
// k_mask_bins: 8 lanes per row.  Checks the row pointers (each row inside [0, nnzM] and ordered,
// first 0, last nnzM) and the columns (strictly ascending, inside [0, n)) and counts the rows per
// masked bin.  A bad row is not read beyond its row pointers and raises a bit of ctr->bad_M.
__global__ void __launch_bounds__(256) k_mask_bins(const int m, const int n, const MaskCsr M, const int *__restrict__ prod,
                                                   Counters *__restrict__ ctr)
{
    __shared__ int s_hist[MB_COUNT];
    if (threadIdx.x < MB_COUNT) s_hist[threadIdx.x] = 0;
    __syncthreads();
    const int gl = threadIdx.x & 7;
    const long long r = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 3;
    int bad = 0;
    if (r < m) {
        const int s = M.rowptr[r], e = M.rowptr[r + 1];
        if (s < 0 || e < s || e > M.nnz || (r == 0 && s != 0) || (r == m - 1 && e != M.nnz)) {
            bad = MASK_BAD_ROWPTR;
        } else {
            for (int p = s + gl; p < e; p += 8) {
                const int c = M.col[p];
                if ((unsigned)c >= (unsigned)n) bad |= MASK_BAD_COL;
                if (p > s && M.col[p - 1] >= c) bad |= MASK_BAD_ORDER;
            }
            if (gl == 0) atomicAdd(&s_hist[mask_bin_of(prod[r], e - s)], 1);
        }
    }
    if (m == 0 && blockIdx.x == 0 && threadIdx.x == 0 && (M.rowptr[0] != 0 || M.nnz != 0)) bad = MASK_BAD_ROWPTR;
    if (bad) atomicOr(&ctr->bad_M, bad);
    __syncthreads();
    if (threadIdx.x < MB_COUNT && s_hist[threadIdx.x]) atomicAdd(&ctr->mask_bin[threadIdx.x], s_hist[threadIdx.x]);
}

// rows -> queue by masked bin (bins contiguous, as k_bin_scatter); rows of MB_ZERO are settled here
constexpr int MSCATTER_ITEMS = 4;
__global__ void __launch_bounds__(256) k_mask_scatter(const int m, const MaskCsr M, const int *__restrict__ prod,
                                                      const BinOffsets offs, int *__restrict__ cursor,
                                                      int *__restrict__ queue, int *__restrict__ rc,
                                                      long long *__restrict__ ct_off)
{
    __shared__ int s_cnt[MB_COUNT];
    __shared__ int s_base[MB_COUNT];
    if (threadIdx.x < MB_COUNT) s_cnt[threadIdx.x] = 0;
    __syncthreads();
    const long long chunk0 = (long long)blockIdx.x * blockDim.x * MSCATTER_ITEMS;
    int bin[MSCATTER_ITEMS], rank[MSCATTER_ITEMS];
#pragma unroll
    for (int it = 0; it < MSCATTER_ITEMS; ++it) {
        const long long row = chunk0 + (long long)it * blockDim.x + threadIdx.x;
        bin[it] = -1;
        if (row < m) {
            const int b = mask_bin_of(prod[row], M.rowptr[row + 1] - M.rowptr[row]);
            if (b == MB_ZERO) {
                rc[row] = 0;
                ct_off[row] = -1;
            } else {
                bin[it] = b;
                rank[it] = atomicAdd(&s_cnt[b], 1);
            }
        }
    }
    __syncthreads();
    if (threadIdx.x < MB_COUNT) {
        const int c = s_cnt[threadIdx.x];
        s_base[threadIdx.x] = c ? offs.off[threadIdx.x] + atomicAdd(&cursor[threadIdx.x], c) : 0;
    }
    __syncthreads();
#pragma unroll
    for (int it = 0; it < MSCATTER_ITEMS; ++it)
        if (bin[it] >= 0) queue[s_base[bin[it]] + rank[it]] = (int)(chunk0 + (long long)it * blockDim.x + threadIdx.x);
}

// ---------------------------------------------------------------------------------------------
// p_i <= 32: warp per row, one product per lane.  Lanes find their column in M_i by binary search;
// equal positions are summed across lanes (__match_any_sync) and the leaders write in position order.
template <typename VT>
__global__ void __launch_bounds__(256) k_mask_esc(const int *__restrict__ queue, const int count, const Csr A, const Csr B,
                                                  const int4 *__restrict__ brange, const MaskCsr M, const MaskOut o)
{
    const int lane = threadIdx.x & 31;
    const VT *__restrict__ valA = static_cast<const VT *>(A.val);
    const VT *__restrict__ valB = static_cast<const VT *>(B.val);
    VT *__restrict__ ctval = static_cast<VT *>(o.ctval);
    const int wpb = blockDim.x >> 5;
    for (int q = blockIdx.x * wpb + (threadIdx.x >> 5); q < count; q += gridDim.x * wpb) {
        const int row = queue[q];
        const int ms = M.rowptr[row], mc = M.rowptr[row + 1] - ms;
        const int mlo = M.col[ms], mhi = M.col[ms + mc - 1];
        const int a0 = A.rowptr[row], a1 = A.rowptr[row + 1];
        int c = -1;
        VT v = VT(0);
        int off = 0;   // products placed so far (at most 32 in all)
        for (int j0 = a0; j0 < a1; j0 += 32) {
            const int j = j0 + lane;
            int bs = 0, len = 0;
            VT av = VT(0);
            if (j < a1) {
                const int4 br = __ldg(brange + A.col[j]);
                if (br.w >= mlo && br.z <= mhi) {
                    bs = br.x;
                    len = br.y;
                    av = valA[j];
                }
            }
            int incl = len;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const int y = __shfl_up_sync(FULL, incl, d);
                if (lane >= d) incl += y;
            }
            for (unsigned nz = __ballot_sync(FULL, len > 0); nz; nz &= nz - 1) {
                const int t = __ffs(nz) - 1;
                const int s_bs = __shfl_sync(FULL, bs, t), s_len = __shfl_sync(FULL, len, t);
                const int s_ex = __shfl_sync(FULL, incl - len, t);
                const VT s_av = __shfl_sync(FULL, av, t);
                const int e = lane - off - s_ex;
                if (e >= 0 && e < s_len) {
                    c = B.col[s_bs + e];
                    v = s_av * valB[s_bs + e];
                }
            }
            off += __shfl_sync(FULL, incl, 31);
        }
        const int pos = (c >= mlo && c <= mhi) ? mask_search(M.col + ms, mc, c) : -1;
        const unsigned same = __match_any_sync(FULL, pos);
        const bool leader = pos >= 0 && __ffs(same) - 1 == lane;
        const unsigned leaders = __ballot_sync(FULL, leader);
        VT sum = VT(0);
        int rank = 0;
#pragma unroll 8
        for (int s = 0; s < 32; ++s) {
            const int ps = __shfl_sync(FULL, pos, s);
            const VT vs = __shfl_sync(FULL, v, s);
            if (ps == pos) sum += vs;
            if (((leaders >> s) & 1u) && ps < pos) ++rank;
        }
        if (leader) {
            o.ctcol[ms + rank] = c;
            ctval[ms + rank] = sum;
        }
        if (lane == 0) {
            o.rc[row] = __popc(leaders);
            o.ct_off[row] = ms;
        }
    }
}

// ---------------------------------------------------------------------------------------------
// Warp per row, table of T = 2^LOG2T slots for nnz(M_i) <= T/2 in shared memory (8 warps per CTA,
// one table each).  B rows are streamed one per step: their columns are distinct, so the value at
// a found position is updated without an atomic.
template <typename VT, int LOG2T>
__host__ __device__ constexpr size_t mask_warp_bytes()
{
    return (size_t)(1 << LOG2T) / 2 * (value_bytes<VT> + 1) + (size_t)(1 << LOG2T) * 8;
}
constexpr int MASK_WARPS = 8;

template <typename VT, int LOG2T>
__global__ void __launch_bounds__(MASK_WARPS * 32) k_mask_warp(const int *__restrict__ queue, const int count, const Csr A,
                                                               const Csr B, const int4 *__restrict__ brange, const MaskCsr M,
                                                               const MaskOut o)
{
    constexpr int T = 1 << LOG2T, H = T / 2;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    unsigned char *mine = smem_raw + (size_t)warp * mask_warp_bytes<VT, LOG2T>();
    VT *vals = reinterpret_cast<VT *>(mine);
    int *keys = reinterpret_cast<int *>(mine + (size_t)H * value_bytes<VT>);
    int *posv = keys + T;
    unsigned char *flag = reinterpret_cast<unsigned char *>(posv + T);
    const VT *__restrict__ valA = static_cast<const VT *>(A.val);
    const VT *__restrict__ valB = static_cast<const VT *>(B.val);
    VT *__restrict__ ctval = static_cast<VT *>(o.ctval);
    for (int q = blockIdx.x * MASK_WARPS + warp; q < count; q += gridDim.x * MASK_WARPS) {
        const int row = queue[q];
        const int ms = M.rowptr[row], mc = M.rowptr[row + 1] - ms;
        for (int s = lane; s < T; s += 32) keys[s] = EMPTY_KEY;
        __syncwarp();
        for (int t = lane; t < mc; t += 32) {
            bool is_new;
            const int slot = table_insert<LOG2T>(keys, M.col[ms + t], is_new);
            posv[slot] = t;
            vals[t] = VT(0);
            flag[t] = 0;
        }
        __syncwarp();
        const int mlo = M.col[ms], mhi = M.col[ms + mc - 1];
        const int a0 = A.rowptr[row], a1 = A.rowptr[row + 1];
        for (int j0 = a0; j0 < a1; j0 += 32) {
            const int j = j0 + lane;
            int bs = 0, len = 0;
            VT av = VT(0);
            if (j < a1) {
                const int4 br = __ldg(brange + A.col[j]);
                if (br.w >= mlo && br.z <= mhi) {   // B rows outside [first, last] of M_i are skipped whole
                    bs = br.x;
                    len = br.y;
                    av = valA[j];
                }
            }
            for (unsigned nz = __ballot_sync(FULL, len > 0); nz; nz &= nz - 1) {
                const int t = __ffs(nz) - 1;
                const int s_bs = __shfl_sync(FULL, bs, t), s_len = __shfl_sync(FULL, len, t);
                const VT s_av = __shfl_sync(FULL, av, t);
                for (int e = lane; e < s_len; e += 32) {
                    const int c = B.col[s_bs + e];
                    if (c < mlo || c > mhi) continue;
                    const int slot = table_probe<LOG2T>(keys, c);
                    if (slot >= 0) {
                        const int p = posv[slot];
                        vals[p] += s_av * valB[s_bs + e];
                        flag[p] = 1;
                    }
                }
                __syncwarp();
            }
        }
        int cnt = 0;
        for (int t0 = 0; t0 < mc; t0 += 32) {
            const int t = t0 + lane;
            const bool hit = t < mc && flag[t];
            const unsigned bm = __ballot_sync(FULL, hit);
            if (hit) {
                const int r = ms + cnt + __popc(bm & ((1u << lane) - 1u));
                o.ctcol[r] = M.col[ms + t];
                ctval[r] = vals[t];
            }
            cnt += __popc(bm);
        }
        if (lane == 0) {
            o.rc[row] = cnt;
            o.ct_off[row] = ms;
        }
        __syncwarp();
    }
}

// ---------------------------------------------------------------------------------------------
// Hit positions of a row, compacted in position order by the whole CTA (ballot per warp, warp
// totals through shared memory).  hit(t) / put(t, r): is position t a hit / write it as entry r.
template <typename Hit, typename Put>
__device__ __forceinline__ int cta_compact(const int mc, int *s_wcnt, Hit &&hit, Put &&put)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
    int cnt = 0;
    for (int t0 = 0; t0 < mc; t0 += blockDim.x) {
        const int t = t0 + (int)threadIdx.x;
        const bool h = t < mc && hit(t);
        const unsigned bm = __ballot_sync(FULL, h);
        if (lane == 0) s_wcnt[warp] = __popc(bm);
        __syncthreads();
        int before = 0, total = 0;
        for (int w = 0; w < nwarps; ++w) {
            const int x = s_wcnt[w];
            before += w < warp ? x : 0;
            total += x;
        }
        if (h) put(t, cnt + before + __popc(bm & ((1u << lane) - 1u)));
        cnt += total;
        __syncthreads();
    }
    return cnt;
}

struct MaskCtaShared {
    int next, nlong, wcnt[32];
    int lng[LONG_CAP];
};

// CTA per row: the products of p_i > MASK_WARP_MAX_P or nnz(M_i) > 512, table of M_i in shared
// memory.  Warps take B rows dynamically and long B rows go to the whole CTA (cta_for_each_b_row);
// warps may meet at one position, so the value update is a shared-memory atomic.
template <typename VT, int LOG2T>
__host__ __device__ constexpr size_t mask_cta_bytes()
{
    return mask_warp_bytes<VT, LOG2T>();
}

template <typename VT, int LOG2T, int THREADS>
__global__ void __launch_bounds__(THREADS) k_mask_cta(const int *__restrict__ queue, const int count, const Csr A, const Csr B,
                                                      const int4 *__restrict__ brange, const MaskCsr M, const MaskOut o)
{
    constexpr int T = 1 << LOG2T, H = T / 2;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __shared__ MaskCtaShared sh;
    VT *vals = reinterpret_cast<VT *>(smem_raw);
    int *keys = reinterpret_cast<int *>(smem_raw + (size_t)H * value_bytes<VT>);
    int *posv = keys + T;
    unsigned char *flag = reinterpret_cast<unsigned char *>(posv + T);
    const VT *__restrict__ valA = static_cast<const VT *>(A.val);
    const VT *__restrict__ valB = static_cast<const VT *>(B.val);
    VT *__restrict__ ctval = static_cast<VT *>(o.ctval);
    for (int q = blockIdx.x; q < count; q += gridDim.x) {
        const int row = queue[q];
        const int ms = M.rowptr[row], mc = M.rowptr[row + 1] - ms;
        for (int s = threadIdx.x; s < T; s += THREADS) keys[s] = EMPTY_KEY;
        if (threadIdx.x == 0) {
            sh.next = 0;
            sh.nlong = 0;
        }
        __syncthreads();
        for (int t = threadIdx.x; t < mc; t += THREADS) {
            bool is_new;
            const int slot = table_insert<LOG2T>(keys, M.col[ms + t], is_new);
            posv[slot] = t;
            vals[t] = VT(0);
            flag[t] = 0;
        }
        __syncthreads();
        const int mlo = M.col[ms], mhi = M.col[ms + mc - 1];
        cta_for_each_b_row(A.rowptr[row], A.rowptr[row + 1], A.col, B.rowptr, &sh.next, &sh.nlong, sh.lng,
                           [&](int j, int p0, int pe, int pstride) {
                               const int4 br = __ldg(brange + A.col[j]);
                               if (br.w < mlo || br.z > mhi) return;
                               const VT av = valA[j];
                               for (int p = p0; p < pe; p += pstride) {
                                   const int c = B.col[p];
                                   if (c < mlo || c > mhi) continue;
                                   const int slot = table_probe<LOG2T>(keys, c);
                                   if (slot >= 0) {
                                       const int pos = posv[slot];
                                       atomicAdd(&vals[pos], av * valB[p]);
                                       flag[pos] = 1;
                                   }
                               }
                           });
        __syncthreads();
        const int cnt = cta_compact(mc, sh.wcnt, [&](int t) { return flag[t] != 0; },
                                    [&](int t, int r) {
                                        o.ctcol[ms + r] = M.col[ms + t];
                                        ctval[ms + r] = vals[t];
                                    });
        if (threadIdx.x == 0) {
            o.rc[row] = cnt;
            o.ct_off[row] = ms;
        }
    }
}

// CTA per row for nnz(M_i) beyond the shared-memory tables: binary search in M_i, values and hit
// flags in global scratch at the row's mask offsets (acc / hit, nnzM entries), zeroed here per row.
constexpr int MASK_GLOBAL_THREADS = 1024;
template <typename VT>
__global__ void __launch_bounds__(MASK_GLOBAL_THREADS) k_mask_global(const int *__restrict__ queue, const int count, const Csr A,
                                                                     const Csr B, const int4 *__restrict__ brange,
                                                                     const MaskCsr M, const MaskOut o)
{
    __shared__ MaskCtaShared sh;
    const VT *__restrict__ valA = static_cast<const VT *>(A.val);
    const VT *__restrict__ valB = static_cast<const VT *>(B.val);
    VT *__restrict__ ctval = static_cast<VT *>(o.ctval);
    for (int q = blockIdx.x; q < count; q += gridDim.x) {
        const int row = queue[q];
        const int ms = M.rowptr[row], mc = M.rowptr[row + 1] - ms;
        VT *acc = static_cast<VT *>(o.acc) + ms * vslots<VT>;
        unsigned char *hit = o.hit + ms;
        const int *mcol = M.col + ms;
        for (int t = threadIdx.x; t < mc; t += blockDim.x) {
            acc[t] = VT(0);
            hit[t] = 0;
        }
        if (threadIdx.x == 0) {
            sh.next = 0;
            sh.nlong = 0;
        }
        __syncthreads();
        const int mlo = mcol[0], mhi = mcol[mc - 1];
        cta_for_each_b_row(A.rowptr[row], A.rowptr[row + 1], A.col, B.rowptr, &sh.next, &sh.nlong, sh.lng,
                           [&](int j, int p0, int pe, int pstride) {
                               const int4 br = __ldg(brange + A.col[j]);
                               if (br.w < mlo || br.z > mhi) return;
                               const VT av = valA[j];
                               for (int p = p0; p < pe; p += pstride) {
                                   const int c = B.col[p];
                                   if (c < mlo || c > mhi) continue;
                                   const int pos = mask_search(mcol, mc, c);
                                   if (pos >= 0) {
                                       atomicAdd(&acc[pos], av * valB[p]);
                                       hit[pos] = 1;
                                   }
                               }
                           });
        __syncthreads();
        const int cnt = cta_compact(mc, sh.wcnt, [&](int t) { return hit[t] != 0; },
                                    [&](int t, int r) {
                                        o.ctcol[ms + r] = mcol[t];
                                        ctval[ms + r] = acc[t];
                                    });
        if (threadIdx.x == 0) {
            o.rc[row] = cnt;
            o.ct_off[row] = ms;
        }
    }
}

// ---------------------------------------------------------------------------------------------
cudaError_t launch_mask_bins(const LaunchCtx &lc, int m, int n, MaskCsr M, const int *prod, Counters *ctr)
{
    const long long blocks = ((long long)m * 8 + 255) / 256;
    ++*lc.launches;
    k_mask_bins<<<blocks > 0 ? (int)blocks : 1, 256, 0, lc.stream>>>(m, n, M, prod, ctr);
    return cudaGetLastError();
}

cudaError_t launch_mask_scatter(const LaunchCtx &lc, int m, MaskCsr M, const int *prod, const BinOffsets &offs, Counters *ctr,
                                int *queue, int *rc, long long *ct_off)
{
    if (m <= 0) return cudaSuccess;
    const long long per_block = 256LL * MSCATTER_ITEMS;
    ++*lc.launches;
    k_mask_scatter<<<(int)((m + per_block - 1) / per_block), 256, 0, lc.stream>>>(m, M, prod, offs, ctr->mask_cursor, queue, rc,
                                                                                  ct_off);
    return cudaGetLastError();
}

namespace {

template <typename KernelT>
cudaError_t launch_persistent(const LaunchCtx &lc, KernelT kern, int threads, size_t smem, long long units_per_block,
                              const int *queue, int count, const Csr &A, const Csr &B, const int4 *brange, const MaskCsr &M,
                              const MaskOut &o)
{
    if (smem > SMEM_BLOCK_MAX) return cudaErrorInvalidValue;
    if (smem > 48 * 1024) {
        const cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
    }
    long long blocks = ((long long)count + units_per_block - 1) / units_per_block;
    const long long cap = (long long)lc.sm_count * resident_blocks(kern, threads, smem);
    if (blocks > cap) blocks = cap;
    ++*lc.launches;
    kern<<<(int)blocks, threads, smem, lc.stream>>>(queue, count, A, B, brange, M, o);
    return cudaGetLastError();
}

template <typename VT>
cudaError_t launch_mask_bin_t(const LaunchCtx &lc, int bin, const int *queue, int count, Csr A, Csr B, const int4 *brange,
                              MaskCsr M, MaskOut o)
{
    switch (bin) {
    case MB_ESC: return launch_persistent(lc, k_mask_esc<VT>, 256, 0, 8, queue, count, A, B, brange, M, o);
    case MB_W64:
        return launch_persistent(lc, k_mask_warp<VT, 6>, MASK_WARPS * 32, MASK_WARPS * mask_warp_bytes<VT, 6>(), MASK_WARPS, queue,
                                 count, A, B, brange, M, o);
    case MB_W256:
        return launch_persistent(lc, k_mask_warp<VT, 8>, MASK_WARPS * 32, MASK_WARPS * mask_warp_bytes<VT, 8>(), MASK_WARPS, queue,
                                 count, A, B, brange, M, o);
    case MB_W1024:
        return launch_persistent(lc, k_mask_warp<VT, 10>, MASK_WARPS * 32, MASK_WARPS * mask_warp_bytes<VT, 10>(), MASK_WARPS,
                                 queue, count, A, B, brange, M, o);
    case MB_C1024:
        return launch_persistent(lc, k_mask_cta<VT, 10, 256>, 256, mask_cta_bytes<VT, 10>(), 1, queue, count, A, B, brange, M, o);
    case MB_C4096:
        return launch_persistent(lc, k_mask_cta<VT, 12, 512>, 512, mask_cta_bytes<VT, 12>(), 1, queue, count, A, B, brange, M, o);
    case MB_C16384:
        // (16-byte values: no such table, the host runs these rows in k_mask_global -- mask_table_last)
        if constexpr (value_bytes<VT> <= 8)
            return launch_persistent(lc, k_mask_cta<VT, 14, 1024>, 1024, mask_cta_bytes<VT, 14>(), 1, queue, count, A, B, brange,
                                     M, o);
        return cudaErrorInvalidValue;
    case MB_GLOBAL:
        return launch_persistent(lc, k_mask_global<VT>, MASK_GLOBAL_THREADS, 0, 1, queue, count, A, B, brange, M, o);
    default: return cudaErrorInvalidValue;
    }
}

}  // namespace

cudaError_t launch_mask_bin(const LaunchCtx &lc, int dtype, int bin, const int *queue, int count, Csr A, Csr B,
                            const int4 *brange, MaskCsr M, MaskOut o)
{
    if (count <= 0) return cudaSuccess;
    // (NoVal: hit flags only)
    return dispatch_value_type(dtype, [&](auto v) { return launch_mask_bin_t<decltype(v)>(lc, bin, queue, count, A, B, brange, M, o); });
}

}  // namespace bhb
