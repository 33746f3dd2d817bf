// stage_bucket.cuh -- expand / bucket-sort / compress for rows that barely compress.
//
// R-MAT rows (BASELINE configs 3 and 5): nnz(C_i) is within a fraction of a percent of the row's
// intermediate products, so hashing buys nothing and the work is a sort of p (column, value) pairs.
// The hash kernels sort with a bitonic network -- O(log^2 p) compare-exchanges per key, ~200 of their
// ~240 instructions per product at p = 1024 (profiles/r02_notes.md).  These kernels sort in O(1) passes:
//
//   * a MONOTONE bucket function  bucket(c) = floor(F(c) * NB),  F = the cumulative distribution of the
//     columns of all intermediate products of the whole multiplication (a 4096-knot piecewise-linear
//     table built once per product by k_cdf_*: every entry (k, c) of B weighted by the number of entries
//     of A in column k).  Under F the products of a row spread almost evenly over the buckets, whatever
//     the skew of the matrix (R-MAT: a third of all products fall into 1 % of the column range);
//   * the products of a row are counted per bucket (shared-memory integer atomics), a CTA-wide scan turns
//     the counts into segments, and the (column, a*b) pairs are placed into them;
//   * each bucket is sorted by column and equal columns are merged; the buckets are in column order, so the
//     row is sorted; a second scan gives the compacted positions.
//
// They play the role of the reference's EM_mergepath rounds (bhsparse_cuda.h:1902-2157) for these rows.
// Direct (single-pass) mode only: the row is staged in Ct (at ct_base + q*ct_stride, or by atomic bump),
// its length goes to rc[], k_copy_ct moves it to its final place after the scan.
#pragma once
#include "common.cuh"

namespace bhb {

constexpr int CDF_BITS = 12;
constexpr int CDF_KNOTS = 1 << CDF_BITS;   // cdf[0 .. CDF_KNOTS], cdf[i] = F(i << shift) scaled to 2^32 (ColumnCdf)

// exclusive scan of a[0..n) in place by the whole CTA; returns the total.  scratch: 33 ints.
template <int THREADS>
__device__ __forceinline__ int cta_exclusive_scan(int *a, const int n, int *scratch)
{
    const int per = (n + THREADS - 1) / THREADS;
    const int b0 = (int)threadIdx.x * per, b1 = min(b0 + per, n);
    int mine = 0;
    for (int i = b0; i < b1; ++i) mine += a[i];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int incl = mine;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const int y = __shfl_up_sync(FULL, incl, d);
        if (lane >= d) incl += y;
    }
    if (lane == 31) scratch[warp] = incl;
    __syncthreads();
    if (warp == 0) {
        int w = (lane < THREADS / 32) ? scratch[lane] : 0;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const int y = __shfl_up_sync(FULL, w, d);
            if (lane >= d) w += y;
        }
        scratch[lane] = w;   // inclusive warp totals; scratch[THREADS/32 - 1] = grand total
    }
    __syncthreads();
    int run = (warp ? scratch[warp - 1] : 0) + incl - mine;
    const int total = scratch[THREADS / 32 - 1];
    for (int i = b0; i < b1; ++i) {
        const int v = a[i];
        a[i] = run;
        run += v;
    }
    __syncthreads();
    return total;
}

// ---------------------------------------------------------------------------------------------------
// k_num_bucket3: one CTA per row, ONE pass over the B rows and no per-bucket loops by single threads.  A
// two-pass kernel with a thread per bucket measured (profiles/r02_ncu_bucket_v1.txt) L1TEX 74 % -- 7.5 sectors
// per global load request, because every product looked the CDF table up twice per pass through L1 (32 lanes,
// ~25 different sectors) -- and 45 % of its instructions ran at 3-4 active lanes.
//   * the CDF table sits in shared memory (all 4096 knots, or every fourth for the small capacities);
//   * the row's A entries are staged a chunk at a time as {B row start, length, first product index}: the
//     colA -> rowptrB -> colB chain of dependent loads is paid once per chunk by all threads in parallel,
//     not once per B row by one warp;
//   * pass 1 (the only one over B): product t = (column, a*b) is staged at its running index, its bucket's
//     counter gives (bucket, arrival) -- one shared-memory atomic per product instead of two;
//   * after the scan the columns are copied into bucket order (dense loop), every PRODUCT ranks itself
//     inside its bucket (1-2 members on average: nb = cap/2 buckets for rows of cap/2 .. cap products) and
//     writes its column and its index at the rank: the row is sorted;
//   * emit walks the sorted row with whole warps: heads of equal-column runs sum their run, a ballot scan
//     compacts, stores are coalesced.
// Members of buckets longer than B3_BIG (hub columns of skewed matrices, rows that do compress) are ranked
// by their whole warp, one member at a time, so one long bucket does not stretch every lane's loop.
// ---------------------------------------------------------------------------------------------------
constexpr int B3_LONG = 512;      // B rows longer than this are strided over by the whole CTA
constexpr int B3_LONG_CAP = 64;
constexpr int B3_BIG = 12;        // bucket sizes above this: warp-cooperative ranking
constexpr int B3_U = 2;           // B rows a warp takes (and loads) at a time
constexpr int B3_SCRATCH = 80;    // ints: [0,34) scan, 34 next, 35 nlong, 36 cursor, [40,72) heads per warp

template <int THREADS>
__host__ __device__ constexpr int b3_chunk()
{
    return THREADS < 512 ? THREADS : (THREADS == 768 ? 256 : 512);   // (768 threads: the variant sized for two CTAs per SM)
}

template <typename VT, int THREADS>
inline size_t b3_smem_bytes(const int cap, const int nb, const int knots)
{
    return (size_t)b3_chunk<THREADS>() * (16 + value_bytes<VT>) + (size_t)cap * (value_bytes<VT> + 12) + (size_t)(nb + 1) * 4 +
           (size_t)(knots + 1) * 4 + (size_t)(B3_SCRATCH + B3_LONG_CAP) * 4 + (size_t)cap * 2;
}

// The sort of k_num_bucket3 after the products are staged: c[t], v[t], meta[t] = bucket << 16 | arrival for the p
// products, cnt[0..nb] = products per bucket (cnt[nb] = 0); a barrier has been passed.  Scans the counts, copies
// the columns into bucket order, ranks every product inside its bucket, then emits the heads of equal-column
// runs (values summed) to ctcol/ctval[o ..).  Returns the number of entries written (CTA-uniform).  The caller
// needs a barrier before it touches the arrays again.
template <typename VT, int THREADS>
__device__ __forceinline__ int b3_sort_emit(VT *v, int *c, unsigned *meta, int *key2, int *cnt, unsigned short *perm, int *scratch,
                                            const int p, const int nb, int *__restrict__ ctcol, VT *__restrict__ ctval,
                                            const long long o)
{
    constexpr int NW = THREADS / 32;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    int *s_heads = scratch + 40;
    cta_exclusive_scan<THREADS>(cnt, nb + 1, scratch);   // cnt[b] = first slot of bucket b, cnt[nb] = p
    // ---- columns into bucket order ----
    for (int t = tid; t < p; t += THREADS) {
        const unsigned m = meta[t];
        key2[cnt[m >> 16] + (int)(m & 0xffffu)] = c[t];
    }
    __syncthreads();
    // ---- every product ranks itself inside its bucket (ties by arrival): sorted columns + permutation ----
    for (int t0 = warp * 32; t0 < p; t0 += THREADS) {   // warp-uniform
        const int t = t0 + lane;
        int s = 0, e = 0, mine = 0, cc = 0;
        bool big = false;
        if (t < p) {
            const unsigned m = meta[t];
            const int b = (int)(m >> 16);
            s = cnt[b];
            e = cnt[b + 1];
            mine = s + (int)(m & 0xffffu);
            cc = key2[mine];
            big = e - s > B3_BIG;
            if (!big) {
                // (a fixed, predicated trip count of 6 with the longer buckets on the warp path was measured
                // slower than this loop: too many members took the warp path)
                // (ci, i) < (cc, mine)  <=>  ci < cc + (i < mine): members before mine count when they are <= cc
                int r = s;
                for (int i = s; i < e; ++i) r += (key2[i] < cc + (i < mine ? 1 : 0)) ? 1 : 0;
                c[r] = cc;
                perm[r] = (unsigned short)t;
            }
        }
        unsigned bm = __ballot_sync(FULL, big);
        while (bm) {   // members of long buckets: the warp counts for one member at a time
            const int src = __ffs(bm) - 1;
            bm &= bm - 1;
            const int ss = __shfl_sync(FULL, s, src), ee = __shfl_sync(FULL, e, src);
            const int mm = __shfl_sync(FULL, mine, src), xc = __shfl_sync(FULL, cc, src);
            int part = 0;
            for (int i = ss + lane; i < ee; i += 32) {
                const int ci = key2[i];
                part += (ci < xc || (ci == xc && i < mm)) ? 1 : 0;
            }
            part = __reduce_add_sync(FULL, part);
            if (lane == src) {
                c[ss + part] = cc;
                perm[ss + part] = (unsigned short)t;
            }
        }
    }
    __syncthreads();
    // ---- emit: heads of equal-column runs, compacted by a ballot scan; warp w owns positions [w*L, (w+1)*L) ----
    const int L = (((p + NW - 1) / NW) + 31) & ~31;
    const int r0 = warp * L, r1 = min(r0 + L, p);
    int heads = 0;
    for (int rb = r0; rb < r1; rb += 32) {
        const int r = rb + lane;
        const bool head = r < r1 && (r == 0 || c[r] != c[r - 1]);
        heads += __popc(__ballot_sync(FULL, head));
    }
    if (lane == 0) s_heads[warp] = heads;
    __syncthreads();
    int incl = lane < NW ? s_heads[lane] : 0;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const int y = __shfl_up_sync(FULL, incl, d);
        if (lane >= d) incl += y;
    }
    const int total = __shfl_sync(FULL, incl, 31);
    int base = __shfl_sync(FULL, incl, warp > 0 ? warp - 1 : 0);
    if (warp == 0) base = 0;
    for (int rb = r0; rb < r1; rb += 32) {
        const int r = rb + lane;
        int cc = -1;
        bool head = false;
        if (r < r1) {
            cc = c[r];
            head = r == 0 || cc != c[r - 1];
        }
        const unsigned bal = __ballot_sync(FULL, head);
        if (head) {
            VT sum = v[perm[r]];
            for (int rr = r + 1; rr < p && c[rr] == cc; ++rr) sum += v[perm[rr]];
            const long long at = o + base + __popc(bal & ((1u << lane) - 1u));
            ctcol[at] = cc;
            ctval[at] = sum;
        }
        base += __popc(bal);
    }
    return total;
}

template <typename VT, int THREADS, int KB>
__global__ void __launch_bounds__(THREADS, THREADS >= 1024 ? 1 : 1536 / THREADS)   // 1536 threads per SM, or one full-size CTA
k_num_bucket3(const int *__restrict__ queue, const int count, const int *__restrict__ rowptrA, const int *__restrict__ colA,
              const VT *__restrict__ valA, const int *__restrict__ rowptrB, const int *__restrict__ colB,
              const VT *__restrict__ valB, const ColumnCdf cdf, const int cap, const int nb, int *__restrict__ rc,
              long long *__restrict__ ct_off, int *__restrict__ ctcol, VT *__restrict__ ctval, const long long ct_base,
              const int *__restrict__ prod, const int p_lo, const int p_hi, const int ct_stride,
              unsigned long long *__restrict__ cursor)   // cursor != nullptr: rows staged by atomic bump (p entries each) instead of q * ct_stride
{
    constexpr int K = 1 << KB;
    constexpr int ACH = b3_chunk<THREADS>();
    extern __shared__ __align__(16) unsigned char smem_raw[];
    int4 *arec = reinterpret_cast<int4 *>(smem_raw);                      // [ACH] {B row start, length, first product index, -}
    VT *aval = reinterpret_cast<VT *>(arec + ACH);                        // [ACH]
    VT *v = aval + ACH * vslots<VT>;                                      // [cap] a*b of product t
    int *c = reinterpret_cast<int *>(v + cap * vslots<VT>);               // [cap] column of product t; later the sorted columns
    unsigned *meta = reinterpret_cast<unsigned *>(c + cap);               // [cap] bucket << 16 | arrival
    int *key2 = reinterpret_cast<int *>(meta + cap);                      // [cap] columns in bucket order
    int *cnt = key2 + cap;                                                // [nb + 1] counts -> first slot of every bucket
    unsigned *scdf = reinterpret_cast<unsigned *>(cnt + nb + 1);          // [K + 1]
    int *scratch = reinterpret_cast<int *>(scdf + K + 1);                 // [B3_SCRATCH]
    int *s_long = scratch + B3_SCRATCH;                                   // [B3_LONG_CAP]
    unsigned short *perm = reinterpret_cast<unsigned short *>(s_long + B3_LONG_CAP);   // [cap] product at sorted position r
    int *s_next = scratch + 34, *s_nlong = scratch + 35, *s_cursor = scratch + 36;
    __shared__ long long s_bump[1];
    const int tid = threadIdx.x, lane = tid & 31;

    constexpr int DEC = CDF_BITS - KB;
    for (int i = tid; i <= K; i += THREADS) scdf[i] = cdf.cdf[i << DEC];
    const int sh = cdf.shift + DEC;
    const unsigned fmask = (1u << sh) - 1u;

    auto stage = [&](const int cc, const VT vv, const int t) {
        const int i = cc >> sh;
        const unsigned lo = scdf[i], hi = scdf[i + 1];
        const unsigned f = lo + (unsigned)(((unsigned long long)(hi - lo) * ((unsigned)cc & fmask)) >> sh);
        const unsigned b = __umulhi(f, (unsigned)nb);
        const unsigned arr = (unsigned)atomicAdd(&cnt[b], 1);
        c[t] = cc;
        v[t] = vv;
        meta[t] = (b << 16) | arr;
    };
    auto product = [&](const int e, const int t, const VT av) { stage(colB[e], av * valB[e], t); };

    for (int q = blockIdx.x; q < count; q += gridDim.x) {
        const int row = queue[q];
        const int p = prod[row];
        if (p <= p_lo || p > p_hi) continue;   // CTA-uniform
        for (int i = tid; i <= nb; i += THREADS) cnt[i] = 0;
        if (tid == 0) {
            *s_cursor = 0;
            if (cursor) s_bump[0] = ct_base + (long long)atomicAdd(cursor, (unsigned long long)p);
        }
        const int a0 = rowptrA[row], a1 = rowptrA[row + 1];
        // ---- the only pass over B: stage the products, count them per bucket ----
        for (int jb = a0; jb < a1; jb += ACH) {
            const int nch = min(ACH, a1 - jb);
            __syncthreads();   // the previous chunk (or the previous row's emit) is done with the staging arrays
            if (tid < nch) {
                const int k = colA[jb + tid];
                const int bs = rowptrB[k];
                const int len = rowptrB[k + 1] - bs;
                const int tb = len > 0 ? atomicAdd(s_cursor, len) : 0;
                arec[tid] = make_int4(bs, len, tb, 0);
                aval[tid] = valA[jb + tid];
            }
            if (tid == 0) {
                *s_next = 0;
                *s_nlong = 0;
            }
            __syncthreads();
            // warps take B3_U staged B rows at a time and issue the loads of their first 32 entries together: one B
            // row at a time left a warp with two loads in flight (ncu: half of the kernel's stall samples were
            // long-scoreboard waits in this loop, at a fifth of its instructions)
            for (int idx = take_next_n(s_next, lane, B3_U); idx < nch; idx = take_next_n(s_next, lane, B3_U)) {
                int4 r[B3_U];
                int cc[B3_U];
                VT bv[B3_U];
#pragma unroll
                for (int u = 0; u < B3_U; ++u) {
                    r[u] = idx + u < nch ? arec[idx + u] : make_int4(0, 0, 0, 0);
                    if (r[u].y > B3_LONG) {   // warp-uniform
                        int li = 0;
                        if (lane == 0) li = atomicAdd(s_nlong, 1);
                        li = __shfl_sync(FULL, li, 0);
                        if (li < B3_LONG_CAP) {
                            if (lane == 0) s_long[li] = idx + u;
                            r[u].y = 0;
                        }
                    }
                }
#pragma unroll
                for (int u = 0; u < B3_U; ++u) {
                    cc[u] = 0;
                    bv[u] = VT(0);
                    if (lane < r[u].y) {
                        cc[u] = colB[r[u].x + lane];
                        bv[u] = valB[r[u].x + lane];
                    }
                }
#pragma unroll
                for (int u = 0; u < B3_U; ++u)
                    if (lane < r[u].y) stage(cc[u], aval[idx + u] * bv[u], r[u].z + lane);
#pragma unroll
                for (int u = 0; u < B3_U; ++u) {
                    if (r[u].y > 32) {   // warp-uniform
                        const VT av = aval[idx + u];
                        for (int e = 32 + lane; e < r[u].y; e += 32) product(r[u].x + e, r[u].z + e, av);
                    }
                }
            }
            __syncthreads();
            const int nlong = min(*s_nlong, B3_LONG_CAP);
            for (int i = 0; i < nlong; ++i) {
                const int4 r = arec[s_long[i]];
                const VT av = aval[s_long[i]];
                for (int e = tid; e < r.y; e += THREADS) product(r.x + e, r.z + e, av);
            }
        }
        __syncthreads();
        const long long o = cursor ? s_bump[0] : ct_base + (long long)q * ct_stride;
        const int total = b3_sort_emit<VT, THREADS>(v, c, meta, key2, cnt, perm, scratch, p, nb, ctcol, ctval, o);
        if (tid == 0) {
            rc[row] = total;
            ct_off[row] = o;
        }
    }
}

// ---------------------------------------------------------------------------------------------------
// k_num_bucket3w: the same single-pass bucket sort with ONE WARP PER ROW, for the bins of at most 96 / 192 products
// (SB_G128, SB_G256) when their rows barely compress (uniform random operands: BASELINE config 4, 8 x 8 = 64
// products -> 64 outputs per row; the small rows of R-MAT).  The hash kernel spends ~700 warp instructions per
// 64-product row, most of them in the register bitonic network and the table re-lookup of the emit.
//   * SG lanes per B row (8 when the B rows are short: four B rows per warp step, all lanes busy for 8-entry rows);
//   * the row's A entries are read 32 at a time, their first product indices come from a warp scan;
//   * bucket / arrival / rank / emit as in k_num_bucket3, at warp scope (__syncwarp only), one emit sweep;
//   * tight direct bins (DirectOut: rows staged `stride` entries apart, stride < product bound): entries beyond the
//     stride are not written and the row goes to the retry queue, like k_num_direct.
// Shared memory per warp: CAPW * (value_bytes<VT> + 4 + 4 + 2 + 1) + (CAPW/2 + 1) * 4; the 1024-knot CDF once per CTA.
// ---------------------------------------------------------------------------------------------------
constexpr int B3W_KB = 10;
constexpr int B3W_WARPS = 8;

template <typename VT, int CAPW>
__host__ __device__ constexpr size_t b3w_per_warp()
{
    return (((size_t)CAPW * (value_bytes<VT> + 4 + 4 + 2 + 1) + (size_t)(CAPW / 2 + 1) * 4) + 15) & ~(size_t)15;
}

template <typename VT, int CAPW, int SG>
__global__ void __launch_bounds__(B3W_WARPS * 32, 6)
k_num_bucket3w(const int *__restrict__ queue, const int count, const int *__restrict__ rowptrA, const int *__restrict__ colA,
               const VT *__restrict__ valA, const int *__restrict__ rowptrB, const int *__restrict__ colB,
               const VT *__restrict__ valB, const ColumnCdf cdf, int *__restrict__ rc, long long *__restrict__ ct_off,
               int *__restrict__ ctcol, VT *__restrict__ ctval, const long long ct_base, const int stride,
               int *__restrict__ retry_queue, int *__restrict__ retry_cnt)
{
    constexpr int K = 1 << B3W_KB;
    constexpr int NB = CAPW / 2;
    constexpr int PER = (NB + 1 + 31) / 32;   // counters per lane in the warp scan
    static_assert(CAPW <= 256 && NB <= 256, "bucket and arrival are one byte each");
    extern __shared__ __align__(16) unsigned char smem_raw[];
    unsigned *scdf = reinterpret_cast<unsigned *>(smem_raw);   // [K + 1] (+ padding to 16 bytes)
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    unsigned char *mine = smem_raw + (((size_t)(K + 1) * 4 + 15) & ~(size_t)15) + (size_t)w * b3w_per_warp<VT, CAPW>();
    VT *v = reinterpret_cast<VT *>(mine);                                   // [CAPW]
    int *c = reinterpret_cast<int *>(v + CAPW * vslots<VT>);               // [CAPW] staged columns, later the sorted ones
    int *key2 = c + CAPW;                                                   // [CAPW]
    int *cnt = key2 + CAPW;                                                 // [NB + 1]
    unsigned short *meta = reinterpret_cast<unsigned short *>(cnt + NB + 1);   // [CAPW] bucket << 8 | arrival
    unsigned char *perm = reinterpret_cast<unsigned char *>(meta + CAPW);   // [CAPW]

    constexpr int DEC = CDF_BITS - B3W_KB;
    for (int i = threadIdx.x; i <= K; i += B3W_WARPS * 32) scdf[i] = cdf.cdf[i << DEC];
    __syncthreads();
    const int sh = cdf.shift + DEC;
    const unsigned fmask = (1u << sh) - 1u;

    // (Measured and dropped: issuing the queue -> rowptrA -> colA -> rowptrB chain of the NEXT row before the current row
    // is processed -- 8 more registers, one CTA less per SM: config 4 3.58 -> 3.87 ms.)
    for (int q = blockIdx.x * B3W_WARPS + w; q < count; q += gridDim.x * B3W_WARPS) {   // warp-uniform, no CTA barrier inside
        const int row = queue[q];
        for (int i = lane; i <= NB; i += 32) cnt[i] = 0;
        __syncwarp();
        const int a0 = rowptrA[row], a1 = rowptrA[row + 1];
        int p = 0;   // products staged so far (warp-uniform)
        for (int jr = a0; jr < a1; jr += 32) {
            const int j = jr + lane;
            int bs = 0, len = 0;
            VT av = VT(0);
            if (j < a1) {
                const int k = colA[j];
                bs = rowptrB[k];
                len = rowptrB[k + 1] - bs;
                av = valA[j];
            }
            int incl = len;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const int y = __shfl_up_sync(FULL, incl, d);
                if (lane >= d) incl += y;
            }
            const int tb = p + incl - len;
            p += __shfl_sync(FULL, incl, 31);
            const int nent = min(32, a1 - jr);
            constexpr int EPP = 32 / SG;   // A entries per warp step
            for (int e0 = 0; e0 < nent; e0 += EPP) {
                const int src = e0 + lane / SG;   // (entries past the row's end carry length 0)
                const int s_bs = __shfl_sync(FULL, bs, src & 31), s_len = (src < 32) ? __shfl_sync(FULL, len, src & 31) : 0;
                const int s_tb = __shfl_sync(FULL, tb, src & 31);
                const VT s_av = __shfl_sync(FULL, av, src & 31);
                const int max_len = (SG == 32) ? s_len : __reduce_max_sync(FULL, s_len);
                for (int off0 = 0; off0 < max_len; off0 += SG) {
                    const int off = off0 + (lane & (SG - 1));
                    if (off < s_len && s_tb + off < CAPW) {
                        const int cc = colB[s_bs + off];
                        const VT vv = s_av * valB[s_bs + off];
                        const int i = cc >> sh;
                        const unsigned lo = scdf[i], hi = scdf[i + 1];
                        const unsigned f = lo + (unsigned)(((unsigned long long)(hi - lo) * ((unsigned)cc & fmask)) >> sh);
                        const unsigned b = __umulhi(f, (unsigned)NB);
                        const unsigned arr = (unsigned)atomicAdd(&cnt[b], 1);
                        const int t = s_tb + off;
                        c[t] = cc;
                        v[t] = vv;
                        meta[t] = (unsigned short)((b << 8) | arr);
                    }
                }
            }
        }
        p = min(p, CAPW);   // (the bin's product bound is below CAPW; the guard above keeps a wrong bin from writing out of bounds)
        __syncwarp();
        // ---- warp scan of the counters: cnt[b] = first slot of bucket b, cnt[NB] = p ----
        {
            int run = 0;
#pragma unroll
            for (int u = 0; u < PER; ++u) {
                const int i = lane * PER + u;
                if (i <= NB) {
                    const int x = cnt[i];
                    cnt[i] = run;
                    run += x;
                }
            }
            int incl = run;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const int y = __shfl_up_sync(FULL, incl, d);
                if (lane >= d) incl += y;
            }
            const int before = incl - run;
#pragma unroll
            for (int u = 0; u < PER; ++u) {
                const int i = lane * PER + u;
                if (i <= NB) cnt[i] += before;
            }
        }
        __syncwarp();
        for (int t = lane; t < p; t += 32) {
            const unsigned m = meta[t];
            key2[cnt[m >> 8] + (int)(m & 0xffu)] = c[t];
        }
        __syncwarp();
        for (int t0 = 0; t0 < p; t0 += 32) {
            const int t = t0 + lane;
            int s = 0, e = 0, mine_slot = 0, cc = 0;
            bool big = false;
            if (t < p) {
                const unsigned m = meta[t];
                const int b = (int)(m >> 8);
                s = cnt[b];
                e = cnt[b + 1];
                mine_slot = s + (int)(m & 0xffu);
                cc = key2[mine_slot];
                big = e - s > B3_BIG;
                if (!big) {
                    int r = s;
                    for (int i = s; i < e; ++i) r += (key2[i] < cc + (i < mine_slot ? 1 : 0)) ? 1 : 0;
                    c[r] = cc;
                    perm[r] = (unsigned char)t;
                }
            }
            unsigned bm = __ballot_sync(FULL, big);
            while (bm) {
                const int src = __ffs(bm) - 1;
                bm &= bm - 1;
                const int ss = __shfl_sync(FULL, s, src), ee = __shfl_sync(FULL, e, src);
                const int mm = __shfl_sync(FULL, mine_slot, src), xc = __shfl_sync(FULL, cc, src);
                int part = 0;
                for (int i = ss + lane; i < ee; i += 32) part += (key2[i] < xc + (i < mm ? 1 : 0)) ? 1 : 0;
                part = __reduce_add_sync(FULL, part);
                if (lane == src) {
                    c[ss + part] = cc;
                    perm[ss + part] = (unsigned char)t;
                }
            }
        }
        __syncwarp();
        // ---- emit (one sweep: the warp walks the sorted row front to back) ----
        const long long o = ct_base + (long long)q * stride;
        int base = 0;
        for (int rb = 0; rb < p; rb += 32) {
            const int r = rb + lane;
            int cc = -1;
            bool head = false;
            if (r < p) {
                cc = c[r];
                head = r == 0 || cc != c[r - 1];
            }
            const unsigned bal = __ballot_sync(FULL, head);
            if (head) {
                VT sum = v[perm[r]];
                for (int rr = r + 1; rr < p && c[rr] == cc; ++rr) sum += v[perm[rr]];
                const int at = base + __popc(bal & ((1u << lane) - 1u));
                if (at < stride) {
                    ctcol[o + at] = cc;
                    ctval[o + at] = sum;
                }
            }
            base += __popc(bal);
        }
        if (lane == 0) {
            if (base > stride && retry_queue) {   // tight bin: more outputs than the speculated capacity -> two-pass path
                ct_off[row] = -1;
                retry_queue[atomicAdd(retry_cnt, 1)] = row;
            } else {
                ct_off[row] = o;
                rc[row] = base;
            }
        }
        __syncwarp();
    }
}

// ---------------------------------------------------------------------------------------------------
// k_num_bucket_heavy: the bucket sort for rows with MORE products than fit on chip (the rows the
// reference sends through EM_mergepath_global, bhsparse_cuda.h:2270-2525, and round 1 sent through a global
// column bitmap -- at n = 16.8 M columns, config 5, that kernel ran at 6 products/ns and held rank 0 at 99 ms
// while the other ranks finished in 67, profiles/r02_notes.md).  It runs the rows k_num_bucket_heavy2 (below)
// cannot slice, from that kernel's retry queue.  The row is cut into slices of the
// F-axis (F = the product-column CDF): 2^k equal slices sized for 1.5x headroom; a slice whose products
// exceed the capacity is halved, recursively (an explicit stack, CTA-uniform control flow).  Every slice takes
// two passes over the row's B rows: the first counts its products per bucket, a CTA scan turns the counts into
// segments, the second scatters (column, a*b) into them; then one thread per bucket insertion-sorts its entries
// and merges equal columns, and a second scan gives the compacted positions.  Slices are processed in ascending F,
// so their outputs concatenate into the sorted row.  The row's products are re-read once per slice and pass
// (they sit in L1/L2).  A slice of a single F value that still overflows (thousands of products in one
// column: possible only for rows of A with more entries than the capacity) is reduced column by column.
// (Measured and dropped: finding a long B row's share of a slice by a warp-wide 32-ary search of its sorted
// columns instead of scanning it with the filter -- 8 % slower on R-MAT 24 rank 0: the scans hit L1/L2, the searches
// are chains of dependent loads.)
// Direct mode: the row is staged at ct_base + [running sum of the products of the rows before it in the
// launch, by atomic bump]; its length goes to rc[row], its staging offset to ct_off[row].
// ---------------------------------------------------------------------------------------------------
template <typename VT, int THREADS>
__global__ void __launch_bounds__(THREADS)
k_num_bucket_heavy(const int *__restrict__ queue, const int count, const int *__restrict__ rowptrA,
                   const int *__restrict__ colA, const VT *__restrict__ valA, const int *__restrict__ rowptrB,
                   const int *__restrict__ colB, const VT *__restrict__ valB, const ColumnCdf cdf, const int cap,
                   const int nb, int *__restrict__ rc, long long *__restrict__ ct_off, int *__restrict__ ctcol,
                   VT *__restrict__ ctval, const long long ct_base, unsigned long long *__restrict__ cursor,
                   const int *__restrict__ prod, const int *__restrict__ count_dev)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    VT *vals = reinterpret_cast<VT *>(smem_raw);                              // [cap]
    int *keys = reinterpret_cast<int *>(smem_raw + (size_t)cap * value_bytes<VT>);   // [cap]
    int *cnt = keys + cap;                                                    // [nb]
    int *ocnt = cnt + nb;                                                     // [nb + 1]
    int *scratch = ocnt + nb + 1;                                             // [34]
    unsigned *scdf = reinterpret_cast<unsigned *>(scratch + 34);              // [CDF_KNOTS + 1]: the CDF table, looked up from shared memory
    for (int i = threadIdx.x; i <= CDF_KNOTS; i += THREADS) scdf[i] = cdf.cdf[i];
    const unsigned fmask = (1u << cdf.shift) - 1u;
    auto feval = [&](const int c) {
        const int i = c >> cdf.shift;
        const unsigned lo = scdf[i], hi = scdf[i + 1];
        return lo + (unsigned)(((unsigned long long)(hi - lo) * ((unsigned)c & fmask)) >> cdf.shift);
    };
    __shared__ unsigned s_stack_lo[40];
    __shared__ int s_stack_lg[40];
    __shared__ long long s_row_base;
    __shared__ int s_min;
    using Wide = typename WideSum<VT>::type;   // (double; two doubles for c64 and c128)
    __shared__ Wide s_sum;
    const int lane = threadIdx.x & 31;
    const int nrows = count_dev ? min(*count_dev, count) : count;   // (retry kernel: the queue was filled on the device)

    for (int q = blockIdx.x; q < nrows; q += gridDim.x) {
        const int row = queue[q];
        const int p = prod[row];
        const int a0 = rowptrA[row], a1 = rowptrA[row + 1];
        if (threadIdx.x == 0) s_row_base = ct_base + (long long)atomicAdd(cursor, (unsigned long long)p);
        // first cut: 2^lg0 slices with 1.5x headroom
        int lg0 = 0;
        while (lg0 < 20 && ((long long)cap << lg0) * 2 < (long long)p * 3) ++lg0;
        __syncthreads();
        const long long o = s_row_base;
        int written = 0;   // CTA-uniform
        for (unsigned first = 0; first < (1u << lg0); ++first) {
            int sp = 0;   // stack pointer (CTA-uniform: every thread tracks it)
            if (threadIdx.x == 0) {
                s_stack_lo[0] = lg0 ? first << (32 - lg0) : 0u;
                s_stack_lg[0] = 32 - lg0;
            }
            sp = 1;
            while (sp > 0) {
                __syncthreads();
                const unsigned lo = s_stack_lo[sp - 1];
                const int lgw = s_stack_lg[sp - 1];   // the slice is [lo, lo + 2^lgw) on the F axis (lgw = 32: everything)
                --sp;
                // ---- count ----
                for (int i = threadIdx.x; i < nb; i += THREADS) cnt[i] = 0;
                if (threadIdx.x == 0) scratch[33] = 0;
                __syncthreads();
                for (int j = a0 + take_next(&scratch[33], lane); j < a1; j = a0 + take_next(&scratch[33], lane)) {
                    const int k = colA[j];
                    const int bs = rowptrB[k], be = rowptrB[k + 1];
                    for (int e = bs + lane; e < be; e += 32) {
                        const unsigned rel = feval(colB[e]) - lo;
                        if (lgw == 32 || (rel >> lgw) == 0u) atomicAdd(&cnt[__umulhi(lgw == 32 ? rel : rel << (32 - lgw), (unsigned)nb)], 1);
                    }
                }
                __syncthreads();
                const int total = cta_exclusive_scan<THREADS>(cnt, nb, scratch);
                if (total == 0) continue;
                if (total > cap) {
                    if (lgw > 0) {   // halve the slice: lower half on top of the stack
                        if (threadIdx.x == 0) {
                            s_stack_lo[sp] = lo + (1u << (lgw - 1));
                            s_stack_lg[sp] = lgw - 1;
                            s_stack_lo[sp + 1] = lo;
                            s_stack_lg[sp + 1] = lgw - 1;
                        }
                        sp += 2;
                        continue;
                    }
                    // one F value with more products than the capacity: reduce it column by column (ascending)
                    int last = -1;
                    while (true) {
                        if (threadIdx.x == 0) {
                            s_min = 0x7fffffff;
                            s_sum = 0.0;
                        }
                        __syncthreads();
                        int mymin = 0x7fffffff;
                        for (int j = a0 + (int)(threadIdx.x >> 5); j < a1; j += THREADS / 32) {
                            const int k = colA[j];
                            for (int e = rowptrB[k] + lane; e < rowptrB[k + 1]; e += 32) {
                                const int c = colB[e];
                                if (c > last && feval(c) == lo) mymin = min(mymin, c);
                            }
                        }
                        mymin = min(mymin, __shfl_xor_sync(FULL, mymin, 16));
                        mymin = min(mymin, __shfl_xor_sync(FULL, mymin, 8));
                        mymin = min(mymin, __shfl_xor_sync(FULL, mymin, 4));
                        mymin = min(mymin, __shfl_xor_sync(FULL, mymin, 2));
                        mymin = min(mymin, __shfl_xor_sync(FULL, mymin, 1));
                        if (lane == 0) atomicMin(&s_min, mymin);
                        __syncthreads();
                        const int cmin = s_min;
                        if (cmin == 0x7fffffff) break;
                        if constexpr (value_bytes<VT> > 0) {
                            Wide part = 0.0;
                            for (int j = a0 + (int)(threadIdx.x >> 5); j < a1; j += THREADS / 32) {
                                const int k = colA[j];
                                const VT av = valA[j];
                                for (int e = rowptrB[k] + lane; e < rowptrB[k + 1]; e += 32)
                                    if (colB[e] == cmin) part += Wide(av * valB[e]);
                            }
                            part = warp_sum(part);
                            if (lane == 0 && part != 0.0) atomicAdd(&s_sum, part);
                            __syncthreads();
                        }
                        if (threadIdx.x == 0) {
                            ctcol[o + written] = cmin;
                            if constexpr (value_bytes<VT> > 0) ctval[o + written] = (VT)s_sum;
                        }
                        ++written;
                        last = cmin;
                        __syncthreads();
                    }
                    continue;
                }
                // ---- scatter ----
                if (threadIdx.x == 0) scratch[33] = 0;
                __syncthreads();
                for (int j = a0 + take_next(&scratch[33], lane); j < a1; j = a0 + take_next(&scratch[33], lane)) {
                    const int k = colA[j];
                    const VT av = valA[j];
                    const int bs = rowptrB[k], be = rowptrB[k + 1];
                    for (int e = bs + lane; e < be; e += 32) {
                        const int c = colB[e];
                        const unsigned rel = feval(c) - lo;
                        if (lgw == 32 || (rel >> lgw) == 0u) {
                            const int slot = atomicAdd(&cnt[__umulhi(lgw == 32 ? rel : rel << (32 - lgw), (unsigned)nb)], 1);
                            keys[slot] = c;
                            vals[slot] = av * valB[e];
                        }
                    }
                }
                __syncthreads();
                // ---- per bucket: insertion sort, merge equal columns ----
                for (int b = threadIdx.x; b < nb; b += THREADS) {
                    const int s = b ? cnt[b - 1] : 0, e = cnt[b];
                    for (int i = s + 1; i < e; ++i) {
                        const int kc = keys[i];
                        const VT kv = vals[i];
                        int j = i - 1;
                        while (j >= s && keys[j] > kc) {
                            keys[j + 1] = keys[j];
                            vals[j + 1] = vals[j];
                            --j;
                        }
                        keys[j + 1] = kc;
                        vals[j + 1] = kv;
                    }
                    int w = s;
                    for (int i = s; i < e; ++i) {
                        if (i > s && keys[i] == keys[w - 1]) {
                            vals[w - 1] += vals[i];
                        } else {
                            keys[w] = keys[i];
                            vals[w] = vals[i];
                            ++w;
                        }
                    }
                    ocnt[b] = w - s;
                }
                if (threadIdx.x == 0) ocnt[nb] = 0;
                __syncthreads();
                const int out = cta_exclusive_scan<THREADS>(ocnt, nb + 1, scratch);
                for (int b = threadIdx.x; b < nb; b += THREADS) {
                    const int s = b ? cnt[b - 1] : 0;
                    const int o0 = ocnt[b], n = ocnt[b + 1] - o0;
                    for (int i = 0; i < n; ++i) {
                        ctcol[o + written + o0 + i] = keys[s + i];
                        ctval[o + written + o0 + i] = vals[s + i];
                    }
                }
                written += out;
            }
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            rc[row] = written;
            ct_off[row] = o;
        }
        __syncthreads();
    }
}

// ---------------------------------------------------------------------------------------------------
// k_num_bucket_heavy2: rows with more products than fit on chip, second formulation.  k_num_bucket_heavy
// re-reads ALL of a row's B rows twice per slice (count + scatter with the slice's filter): a row of 200 000
// products in 40 slices is walked 80 times (R-MAT 24, rank 0: 31 of 62 ms in these rows).  Here the row is
//   1. counted per slice (one pass; a slice that would overflow the chip doubles the slice count, once),
//   2. scattered into its own staging area in global memory, partitioned by slice (one pass),
//   3. sorted slice by slice: the slice's segment is loaded densely, bucketed, ranked and emitted by
//      b3_sort_emit, compacted, in place -- the output of slices 0..s never reaches the input of slice s+1.
// Rows whose slices still overflow (one column carrying more products than the chip holds, ...) are handed to
// k_num_bucket_heavy through a retry queue before anything is written or allocated for them.
// Rows of at most p_lo products are skipped (they are taken by k_num_bucket3 in the same staging area).
// (Measured and dropped: two B rows per warp step in the count and scatter passes, as in k_num_bucket3 -- no change.)
// ---------------------------------------------------------------------------------------------------
constexpr int H2_MAX_LG = 11;   // at most 2048 slices per row (16.7 M products); longer rows -> retry queue

template <typename VT>
constexpr size_t h2_smem_bytes(const int cap, const int nb)
{
    return (size_t)cap * (value_bytes<VT> + 12) + (size_t)(nb + 1) * 4 + (size_t)(CDF_KNOTS + 1) * 4 + (size_t)B3_SCRATCH * 4 +
           (size_t)((1 << H2_MAX_LG) + 1) * 4 + (size_t)cap * 2;
}

template <typename VT, int THREADS>
__global__ void __launch_bounds__(THREADS, 1)
k_num_bucket_heavy2(const int *__restrict__ queue, const int count, const int *__restrict__ rowptrA,
                    const int *__restrict__ colA, const VT *__restrict__ valA, const int *__restrict__ rowptrB,
                    const int *__restrict__ colB, const VT *__restrict__ valB, const ColumnCdf cdf, const int cap,
                    const int nb, int *__restrict__ rc, long long *__restrict__ ct_off, int *__restrict__ ctcol,
                    VT *__restrict__ ctval, const long long ct_base, unsigned long long *__restrict__ cursor,
                    const int *__restrict__ prod, const int p_lo, int *__restrict__ retry_queue, int *__restrict__ retry_cnt)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    VT *v = reinterpret_cast<VT *>(smem_raw);                                 // [cap]
    int *c = reinterpret_cast<int *>(v + cap * vslots<VT>);                   // [cap]
    unsigned *meta = reinterpret_cast<unsigned *>(c + cap);                   // [cap]
    int *key2 = reinterpret_cast<int *>(meta + cap);                          // [cap]
    int *cnt = key2 + cap;                                                    // [nb + 1]
    unsigned *scdf = reinterpret_cast<unsigned *>(cnt + nb + 1);              // [CDF_KNOTS + 1]
    int *scratch = reinterpret_cast<int *>(scdf + CDF_KNOTS + 1);             // [B3_SCRATCH]
    int *hist = scratch + B3_SCRATCH;                                         // [2^H2_MAX_LG + 1] products per slice -> segment ends
    unsigned short *perm = reinterpret_cast<unsigned short *>(hist + (1 << H2_MAX_LG) + 1);   // [cap]
    __shared__ long long s_row_base;
    __shared__ int s_max;
    int *s_next = scratch + 34;
    const int tid = threadIdx.x, lane = tid & 31;

    for (int i = tid; i <= CDF_KNOTS; i += THREADS) scdf[i] = cdf.cdf[i];
    const unsigned fmask = (1u << cdf.shift) - 1u;
    auto feval = [&](const int col) {
        const int i = col >> cdf.shift;
        const unsigned lo = scdf[i], hi = scdf[i + 1];
        return lo + (unsigned)(((unsigned long long)(hi - lo) * ((unsigned)col & fmask)) >> cdf.shift);
    };

    for (int q = blockIdx.x; q < count; q += gridDim.x) {
        const int row = queue[q];
        const int p = prod[row];
        if (p <= p_lo) continue;   // CTA-uniform
        const int a0 = rowptrA[row], a1 = rowptrA[row + 1];
        // slices: 2^lg with 1.5x headroom; one more doubling if the row's own distribution overflows a slice
        int lg = 0;
        while (lg < H2_MAX_LG && ((long long)cap << lg) * 2 < (long long)p * 3) ++lg;
        bool fits = ((long long)cap << lg) >= (long long)p;
        for (int attempt = 0; fits && attempt < 2; ++attempt) {
            const int S = 1 << lg;
            __syncthreads();
            for (int i = tid; i <= S; i += THREADS) hist[i] = 0;
            if (tid == 0) {
                *s_next = 0;
                s_max = 0;
            }
            __syncthreads();
            for (int j = a0 + take_next(s_next, lane); j < a1; j = a0 + take_next(s_next, lane)) {
                const int k = colA[j];
                const int bs = rowptrB[k], be = rowptrB[k + 1];
                for (int e = bs + lane; e < be; e += 32) atomicAdd(&hist[lg ? feval(colB[e]) >> (32 - lg) : 0], 1);
            }
            __syncthreads();
            int mx = 0;
            for (int i = tid; i < S; i += THREADS) mx = max(mx, hist[i]);
            mx = __reduce_max_sync(FULL, mx);
            if (lane == 0 && mx > 0) atomicMax(&s_max, mx);
            __syncthreads();
            if (s_max <= cap) break;
            if (attempt == 0 && lg < H2_MAX_LG) ++lg; else fits = false;
        }
        if (!fits) {   // CTA-uniform: nothing was allocated or written for this row
            if (tid == 0) retry_queue[atomicAdd(retry_cnt, 1)] = row;
            continue;
        }
        const int S = 1 << lg;
        cta_exclusive_scan<THREADS>(hist, S + 1, scratch);   // hist[s] = first entry of slice s, hist[S] = p
        if (tid == 0) {
            s_row_base = ct_base + (long long)atomicAdd(cursor, (unsigned long long)p);
            *s_next = 0;
        }
        __syncthreads();
        const long long o = s_row_base;
        // ---- scatter into the row's staging area, partitioned by slice; afterwards hist[s] = END of slice s ----
        for (int j = a0 + take_next(s_next, lane); j < a1; j = a0 + take_next(s_next, lane)) {
            const int k = colA[j];
            const VT av = valA[j];
            const int bs = rowptrB[k], be = rowptrB[k + 1];
            for (int e = bs + lane; e < be; e += 32) {
                const int col = colB[e];
                const int at = atomicAdd(&hist[lg ? feval(col) >> (32 - lg) : 0], 1);
                ctcol[o + at] = col;
                ctval[o + at] = av * valB[e];
            }
        }
        __syncthreads();   // (the CTA's own global writes are visible to it after the barrier)
        int written = 0;   // CTA-uniform
        for (int s = 0; s < S; ++s) {
            const int first = s ? hist[s - 1] : 0;
            const int n = hist[s] - first;
            if (n == 0) continue;
            for (int i = tid; i <= nb; i += THREADS) cnt[i] = 0;
            __syncthreads();
            const unsigned lo = lg ? (unsigned)s << (32 - lg) : 0u;
            for (int t = tid; t < n; t += THREADS) {
                const int col = ctcol[o + first + t];
                const VT val = ctval[o + first + t];
                const unsigned rel = feval(col) - lo;
                const unsigned b = __umulhi(lg ? rel << lg : rel, (unsigned)nb);
                const unsigned arr = (unsigned)atomicAdd(&cnt[b], 1);
                c[t] = col;
                v[t] = val;
                meta[t] = (b << 16) | arr;
            }
            __syncthreads();
            written += b3_sort_emit<VT, THREADS>(v, c, meta, key2, cnt, perm, scratch, n, nb, ctcol, ctval, o + written);
            __syncthreads();
        }
        if (tid == 0) {
            rc[row] = written;
            ct_off[row] = o;
        }
    }
}

}  // namespace bhb
