// stage_numeric.cuh -- numeric kernels (hash accumulate, sort, write C in place),
// instantiated for float in stage_numeric_f32.cu, double in stage_numeric_f64.cu, complex64 in stage_numeric_c64.cu
// and NoVal in stage_numeric_none.cu.
//
// k_num_group<VT,G,LOG2T,R> : a group of G lanes owns a row: T-slot (column,value) table in
//      shared memory, B rows streamed one per step (columns of one B row are distinct, so the
//      value update needs no atomic -- shared-memory FP atomics are CAS loops on sm_100a).
//      Then: compact the occupied columns, sort them (R>0: register bitonic network over
//      warp shuffles; R==0: bitonic in shared memory), look each sorted column's value up
//      again and store the row at rowptrC[row] with coalesced writes.
//      Covers what ESC_bitonic_scan (bhsparse_cuda.h:1400-1518) and the first rounds of
//      EM_mergepath (:1902-2157) do in the reference; used for nnz(C_i) <= 256.
// k_num_direct<VT,G,LOG2T,R[,FILTER]> : the same kernel as a single pass (no symbolic pass before
//      it): rows are staged `cap` entries apart and copied to their place by k_copy_ct.
// k_num_block<VT,LOG2T,THREADS[,DIRECT]> : one CTA per row, 256 < nnz(C_i) <= 8192, a CTA-wide
//      table (up to 224 KB of shared memory), B rows taken dynamically by the warps, CTA-wide
//      register sort -- the rows the reference sends through EM_mergepath rounds 2..5 and
//      EM_mergepath_global (:2270-2525). DIRECT: single-pass variant for bins that barely compress.
// k_num_large<VT>           : longer rows: rank of a column = popcount prefix of the row's
//      column bitmap (global, L2 resident); products are accumulated straight into the
//      final C row with red.global.add -- no spill, no re-allocation, no sort.
#pragma once
#include "common.cuh"
#include "stage_bucket.cuh"

namespace bhb {

template <typename VT, int G, int LOG2T, int R>
__global__ void __launch_bounds__(256)
k_num_group(const int *__restrict__ queue, const int count, const int *__restrict__ rowptrA,
            const int *__restrict__ colA, const VT *__restrict__ valA, const int *__restrict__ rowptrB,
            const int *__restrict__ colB, const VT *__restrict__ valB, const int64_t *__restrict__ rowoff,
            int *__restrict__ colC, VT *__restrict__ valC)
{
    constexpr int T = 1 << LOG2T;
    constexpr int N = (R > 0) ? G * R : T / 2;   // max nnz(C_i) of the bin (sort capacity); T >= 2N slots
    constexpr size_t PER_GROUP = (size_t)T * value_bytes<VT> + (size_t)T * 4 + (size_t)N * 4;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31;
    const int gl = threadIdx.x & (G - 1);
    const int gib = threadIdx.x / G;
    const int groups_per_block = blockDim.x / G;
    const int gshift = lane & ~(G - 1);
    const unsigned gbits = (G == 32) ? FULL : ((1u << (G & 31)) - 1u);
    unsigned char *mine = smem_raw + (size_t)gib * PER_GROUP;
    VT *vals = reinterpret_cast<VT *>(mine);
    int *keys = reinterpret_cast<int *>(mine + (size_t)T * value_bytes<VT>);
    int *sk = keys + T;

    // All loops are WARP-uniform (trip counts are maxima over the 32/G groups of the warp,
    // groups with less work are predicated off): sub-warp groups with their own loop
    // counters never reconverge on sm_100a and then run at G/32 efficiency.
    for (int q0 = blockIdx.x * groups_per_block + (gib & ~(32 / G - 1)); q0 < count;
         q0 += gridDim.x * groups_per_block) {
        const int q = q0 + (gib & (32 / G - 1));
        const bool active = q < count;
        const int row = active ? queue[q] : 0;
#pragma unroll 4
        for (int s = gl; s < T; s += G) {
            keys[s] = EMPTY_KEY;
            vals[s] = VT(0);
        }
        __syncwarp();
        const int a0 = active ? rowptrA[row] : 0;
        const int na = active ? rowptrA[row + 1] - a0 : 0;
        const int max_na = (G == 32) ? na : __reduce_max_sync(FULL, na);   // uniform already for G == 32
        for (int base = 0; base < max_na; base += G) {
            const int j = base + gl;
            int bs = 0, len = 0;
            VT av = VT(0);
            if (j < na) {
                const int k = colA[a0 + j];
                bs = rowptrB[k];
                len = rowptrB[k + 1] - bs;
                av = valA[a0 + j];
            }
            const int cnt = min(G, max_na - base);
            for (int t = 0; t < cnt; ++t) {
                const int s_bs = __shfl_sync(FULL, bs, t, G);
                const int s_len = __shfl_sync(FULL, len, t, G);
                const VT s_av = __shfl_sync(FULL, av, t, G);
                const int max_len = (G == 32) ? s_len : __reduce_max_sync(FULL, s_len);   // uniform already for G == 32
                for (int off0 = 0; off0 < max_len; off0 += G) {
                    const int off = off0 + gl;
                    if (off < s_len) {
                        const int c = colB[s_bs + off];
                        const VT v = s_av * valB[s_bs + off];
                        bool is_new;
                        const int slot = table_insert<LOG2T>(keys, c, is_new);
                        vals[slot] += v;
                    }
                }
                __syncwarp();   // the next B row may hit the same slots
            }
        }
        // ---- compact the occupied columns into sk[0..cnt) ----
        int cntc = 0;
        for (int s0 = 0; s0 < T; s0 += G) {
            const int k = keys[s0 + gl];
            const bool occ = (k != EMPTY_KEY);
            const unsigned bm = (__ballot_sync(FULL, occ) >> gshift) & gbits;
            if (occ) sk[cntc + __popc(bm & ((1u << gl) - 1u))] = k;
            cntc += __popc(bm);
        }
        __syncwarp();
        // ---- sort ----
        if constexpr (R > 0) {
            constexpr int RR = R;
            static_assert(G * RR == N && T >= 2 * N, "register sort must cover the bin");
            int x[RR];
#pragma unroll
            for (int r = 0; r < RR; ++r) {
                const int i = gl * RR + r;
                x[r] = (i < cntc) ? sk[i] : SORT_PAD;
            }
            if constexpr (RR > 32)   // (rolled variant: measured slower up to R = 32)
                bitonic_sort_regs_rolled<G, RR>(x, gl);
            else
                bitonic_sort_regs<G, RR>(x, gl, FULL);
            __syncwarp();
#pragma unroll
            for (int r = 0; r < RR; ++r) sk[gl * RR + r] = x[r];
            __syncwarp();
        } else {
            // shared-memory bitonic over the largest group size of the warp (uniform stage count)
            const int np = next_pow2(cntc);
            const int np_max = (G == 32) ? np : __reduce_max_sync(FULL, np);   // uniform already for G == 32
            for (int i = cntc + gl; i < np_max; i += G) sk[i] = SORT_PAD;
            __syncwarp();
            bitonic_sort_smem_group<G>(sk, np_max, gl, FULL);
        }
        // ---- emit: sorted columns + their accumulated values, coalesced ----
        const int64_t o = active ? rowoff[row] : 0;
        const int max_c = (G == 32) ? cntc : __reduce_max_sync(FULL, cntc);   // uniform already for G == 32
        for (int i0 = 0; i0 < max_c; i0 += G) {
            const int i = i0 + gl;
            if (i < cntc) {
                const int c = sk[i];
                const int slot = table_find<LOG2T>(keys, c);
                colC[o + i] = c;
                valC[o + i] = vals[slot];
            }
        }
        __syncwarp();
    }
}

// ---------------------------------------------------------------------------------------
// Direct (single-pass) mode, see DirectOut in common.cuh: k_num_group without a symbolic pass
// before it.  The table has T = 2*cap slots for rows that are EXPECTED to have at most
// cap = G*R distinct columns; every step counts the newly inserted columns, a row that
// exceeds cap stops inserting (so probing always terminates), is flagged and queued for the
// two-pass path.  Rows that fit are written sorted to the staging buffer, cap entries apart.
// FILTER (full-warp groups only): take the rows with p_lo < products <= p_hi, stage ct_stride apart.
template <typename VT, int G, int LOG2T, int R, bool FILTER = false>
__global__ void __launch_bounds__(256, (R <= 4) ? 7 : (G == 32 && R == 8) ? 4 : 1)   // CTAs/SM shared memory allows: keep the registers below that
k_num_direct(const int *__restrict__ queue, const int count, const int *__restrict__ rowptrA,
             const int *__restrict__ colA, const VT *__restrict__ valA, const int *__restrict__ rowptrB,
             const int *__restrict__ colB, const VT *__restrict__ valB, int *__restrict__ rc,
             long long *__restrict__ ct_off, int *__restrict__ ctcol, VT *__restrict__ ctval,
             const long long ct_base, int *__restrict__ retry_queue, int *__restrict__ retry_cnt,
             const int *__restrict__ prod = nullptr, const int p_lo = 0, const int p_hi = 0, const int ct_stride = 0)
{
    static_assert(!FILTER || G == 32, "row filter: full-warp groups");
    constexpr int T = 1 << LOG2T;
    constexpr int N = G * R;                 // speculated capacity of a row
    static_assert(T == 2 * N && R > 0, "direct mode uses the register sort and a half-full table");
    constexpr size_t PER_GROUP = (size_t)T * value_bytes<VT> + (size_t)T * 4 + (size_t)N * 4;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31;
    const int gl = threadIdx.x & (G - 1);
    const int gib = threadIdx.x / G;
    const int groups_per_block = blockDim.x / G;
    const int gshift = lane & ~(G - 1);
    const unsigned gbits = (G == 32) ? FULL : ((1u << (G & 31)) - 1u);
    unsigned char *mine = smem_raw + (size_t)gib * PER_GROUP;
    VT *vals = reinterpret_cast<VT *>(mine);
    int *keys = reinterpret_cast<int *>(mine + (size_t)T * value_bytes<VT>);
    int *sk = keys + T;

    for (int q0 = blockIdx.x * groups_per_block + (gib & ~(32 / G - 1)); q0 < count;
         q0 += gridDim.x * groups_per_block) {
        const int q = q0 + (gib & (32 / G - 1));
        const bool active = q < count;
        const int row = active ? queue[q] : 0;
        if constexpr (FILTER) {
            const int p = prod[row];
            if (p <= p_lo || p > p_hi) continue;   // warp-uniform: one row per warp
        }
#pragma unroll 4
        for (int s = gl; s < T; s += G) {
            keys[s] = EMPTY_KEY;
            vals[s] = VT(0);
        }
        __syncwarp();
        const int a0 = active ? rowptrA[row] : 0;
        const int na = active ? rowptrA[row + 1] - a0 : 0;
        const int max_na = (G == 32) ? na : __reduce_max_sync(FULL, na);
        int ndistinct = 0;      // group-uniform
        bool ovf = false;       // group-uniform
        for (int base = 0; base < max_na; base += G) {
            const int j = base + gl;
            int bs = 0, len = 0;
            VT av = VT(0);
            if (j < na) {
                const int k = colA[a0 + j];
                bs = rowptrB[k];
                len = rowptrB[k + 1] - bs;
                av = valA[a0 + j];
            }
            const int cnt = min(G, max_na - base);
            for (int t = 0; t < cnt; ++t) {
                const int s_bs = __shfl_sync(FULL, bs, t, G);
                const int s_len = __shfl_sync(FULL, len, t, G);
                const VT s_av = __shfl_sync(FULL, av, t, G);
                const int max_len = (G == 32) ? s_len : __reduce_max_sync(FULL, s_len);
                for (int off0 = 0; off0 < max_len; off0 += G) {
                    const int off = off0 + gl;
                    bool is_new = false;
                    if (off < s_len && !ovf) {
                        const int c = colB[s_bs + off];
                        const VT v = s_av * valB[s_bs + off];
                        const int slot = table_insert<LOG2T>(keys, c, is_new);
                        vals[slot] += v;
                    }
                    // at most G new columns per sub-step: N + G < T, the table never fills up
                    ndistinct += __popc((__ballot_sync(FULL, is_new) >> gshift) & gbits);
                    ovf = ndistinct > N;
                }
                __syncwarp();
            }
            if (G == 32 && ovf) break;   // (warp-uniform for full-warp groups)
        }
        // ---- compact the occupied columns into sk[0..cnt) ----
        int cntc = 0;
        for (int s0 = 0; s0 < T; s0 += G) {
            const int k = keys[s0 + gl];
            const bool occ = (k != EMPTY_KEY) && !ovf;
            const unsigned bm = (__ballot_sync(FULL, occ) >> gshift) & gbits;
            if (occ) sk[cntc + __popc(bm & ((1u << gl) - 1u))] = k;
            cntc += __popc(bm);
        }
        __syncwarp();
        int x[R];
#pragma unroll
        for (int r = 0; r < R; ++r) {
            const int i = gl * R + r;
            x[r] = (i < cntc) ? sk[i] : SORT_PAD;
        }
        if constexpr (R > 32)
            bitonic_sort_regs_rolled<G, R>(x, gl);
        else
            bitonic_sort_regs<G, R>(x, gl, FULL);
        __syncwarp();
#pragma unroll
        for (int r = 0; r < R; ++r) sk[gl * R + r] = x[r];
        __syncwarp();
        // ---- stage the sorted row (or hand it to the two-pass path) ----
        const long long o = ct_base + (long long)q * (FILTER ? ct_stride : N);
        if (active && gl == 0) {
            if (ovf) {
                ct_off[row] = -1;
                retry_queue[atomicAdd(retry_cnt, 1)] = row;
            } else {
                ct_off[row] = o;
                rc[row] = cntc;
            }
        }
        const int max_c = (G == 32) ? cntc : __reduce_max_sync(FULL, cntc);
        for (int i0 = 0; i0 < max_c; i0 += G) {
            const int i = i0 + gl;
            if (i < cntc) {
                const int c = sk[i];
                const int slot = table_find<LOG2T>(keys, c);
                ctcol[o + i] = c;
                ctval[o + i] = vals[slot];
            }
        }
        __syncwarp();
    }
}

// Staging buffer -> final C (the reference's copyCt2C, bhsparse_cuda.h:2813-2911): G lanes per row,
// coalesced on both sides, four independent loads in flight per lane.
template <typename VT, int G>
__global__ void __launch_bounds__(256)
k_copy_ct(const int *__restrict__ queue, const int count, const int64_t *__restrict__ rowoff,
          const long long *__restrict__ ct_off, const int *__restrict__ ctcol, const VT *__restrict__ ctval,
          int *__restrict__ colC, VT *__restrict__ valC)
{
    const int gl = threadIdx.x & (G - 1);
    const long long q = ((long long)blockIdx.x * blockDim.x + threadIdx.x) / G;
    if (q >= count) return;
    const int row = queue[q];
    const int64_t o = rowoff[row];
    const int n = (int)(rowoff[row + 1] - o);
    const long long src = ct_off[row];
    for (int i0 = 0; i0 < n; i0 += 4 * G) {
        int c[4];
        VT v[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int i = i0 + u * G + gl;
            if (i < n) {
                c[u] = ctcol[src + i];
                v[u] = ctval[src + i];
            }
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int i = i0 + u * G + gl;
            if (i < n) {
                colC[o + i] = c[u];
                valC[o + i] = v[u];
            }
        }
    }
}

// CTAs of k_num_block<VT,LOG2T,THREADS> an SM can hold (threads and shared memory); asking the
// compiler for that many keeps the register count from being the limiter.  Value-free tables are
// counted as f32 ones: at T = 16384 their smaller footprint would ask for two 1024-thread CTAs, i.e.
// 32 registers, and the kernel then spills.
template <typename VT, int LOG2T, int THREADS>
constexpr int num_block_min_ctas()
{
    constexpr int vb = value_bytes<VT> > 4 ? (int)value_bytes<VT> : 4;
    constexpr int smem = (1 << LOG2T) * (vb + 4) + (1 << LOG2T) / 2 * 4 + 1024;
    constexpr int by_smem = (228 * 1024) / smem;   // 228 KB per SM, 1 KB reserved per CTA
    constexpr int by_threads = 2048 / THREADS;
    return by_smem < by_threads ? (by_smem < 1 ? 1 : by_smem) : by_threads;
}

// DIRECT: single-pass mode for the rows of a symbolic bin with p_lo < products <= p_hi <= T/2:
// the row is staged at ct_base + q*ct_stride in the staging buffer (colC/valC then point to
// it), its length and staging offset are recorded for the scan and k_copy_ct; rowoff is not read.
template <typename VT, int LOG2T, int THREADS, bool DIRECT = false>
__global__ void __launch_bounds__(THREADS, (num_block_min_ctas<VT, LOG2T, THREADS>()))
k_num_block(const int *__restrict__ queue, const int count, const int *__restrict__ rowptrA,
            const int *__restrict__ colA, const VT *__restrict__ valA, const int *__restrict__ rowptrB,
            const int *__restrict__ colB, const VT *__restrict__ valB, const int64_t *__restrict__ rowoff,
            int *__restrict__ colC, VT *__restrict__ valC, int *__restrict__ rc = nullptr,
            long long *__restrict__ ct_off = nullptr, const long long ct_base = 0,
            const int *__restrict__ prod = nullptr, const int p_lo = 0, const int p_hi = 0, const int ct_stride = 0)
{
    constexpr int T = 1 << LOG2T;
    constexpr int CHUNKS = T / (4 * THREADS);   // 16-byte key chunks per thread in the compaction
    extern __shared__ __align__(16) unsigned char smem_raw[];
    VT *vals = reinterpret_cast<VT *>(smem_raw);
    int *keys = reinterpret_cast<int *>(smem_raw + (size_t)T * value_bytes<VT>);
    int *sk = keys + T;   // no static shared memory: T=4096 must fit four CTAs per SM to the byte
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    constexpr int nwarps = THREADS / 32;

    for (int q = blockIdx.x; q < count; q += gridDim.x) {
        const int row = queue[q];
        if constexpr (DIRECT) {
            const int p = prod[row];
            if (p <= p_lo || p > p_hi) continue;   // CTA-uniform
        }
        for (int s = threadIdx.x; s < T; s += THREADS) {
            keys[s] = EMPTY_KEY;
            vals[s] = VT(0);
        }
        if (threadIdx.x == 0) sk[0] = 0;   // next B row to take; sk[] is free until the compaction
        __syncthreads();
        // ---- products: the warps take B rows from a shared counter. With a static
        // warp <-> B-row assignment 31 % of the stall samples sat at the barrier below
        // (R-MAT B rows vary from 1 to thousands of elements); taking them dynamically is
        // 7 % faster on the whole R-MAT scale-20 product. Measured and dropped: handing long
        // B rows to the whole CTA, fetching 32 B-row descriptors per warp at once, and
        // keeping two B rows' loads in flight (profiles/r01_notes.md).
        const int a0 = rowptrA[row], a1 = rowptrA[row + 1];
        for (int j = a0 + take_next(&sk[0], lane); j < a1; j = a0 + take_next(&sk[0], lane)) {
            const int k = colA[j];
            const VT av = valA[j];
            const int bs = rowptrB[k], be = rowptrB[k + 1];
            for (int p = bs + lane; p < be; p += 32) {
                const int c = colB[p];
                const VT v = av * valB[p];
                bool is_new;
                const int slot = table_insert<LOG2T>(keys, c, is_new);
                atomicAdd(&vals[slot], v);   // different warps may meet in one slot
            }
        }
        __syncthreads();
        // ---- compact the occupied columns into sk[] (order irrelevant, sorted next):
        // per-thread counts -> warp scan -> warp totals through sk[] -> scatter
        int4 kc[CHUNKS];
        int mine = 0;
#pragma unroll
        for (int r = 0; r < CHUNKS; ++r) {
            kc[r] = reinterpret_cast<const int4 *>(keys)[r * THREADS + threadIdx.x];
            mine += (kc[r].x != EMPTY_KEY) + (kc[r].y != EMPTY_KEY) + (kc[r].z != EMPTY_KEY) + (kc[r].w != EMPTY_KEY);
        }
        int incl = mine;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const int y = __shfl_up_sync(FULL, incl, d);
            if (lane >= d) incl += y;
        }
        if (lane == 31) sk[warp] = incl;
        __syncthreads();
        int wt = (lane < nwarps) ? sk[lane] : 0;
        int wincl = wt;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const int y = __shfl_up_sync(FULL, wincl, d);
            if (lane >= d) wincl += y;
        }
        const int cntc = __shfl_sync(FULL, wincl, nwarps - 1);
        const int wbase = __shfl_sync(FULL, wincl - wt, warp);
        __syncthreads();
        {
            int pos = wbase + incl - mine;
#pragma unroll
            for (int r = 0; r < CHUNKS; ++r) {
                if (kc[r].x != EMPTY_KEY) sk[pos++] = kc[r].x;
                if (kc[r].y != EMPTY_KEY) sk[pos++] = kc[r].y;
                if (kc[r].z != EMPTY_KEY) sk[pos++] = kc[r].z;
                if (kc[r].w != EMPTY_KEY) sk[pos++] = kc[r].w;
            }
        }
        __syncthreads();
        {
            // sort the distinct columns in registers (K per thread), see block_bitonic_sort_regs
            constexpr int K = (T / 2) / THREADS;
            int x[K];
#pragma unroll
            for (int r = 0; r < K; ++r) {
                const int i = (int)threadIdx.x * K + r;
                x[r] = (i < cntc) ? sk[i] : SORT_PAD;
            }
            if constexpr (K <= 4)
                block_bitonic_sort_regs_unrolled<K, THREADS>(x, sk);
            else
                block_bitonic_sort_regs<K, THREADS>(x, sk);
            __syncthreads();
#pragma unroll
            for (int r = 0; r < K; ++r) sk[(int)threadIdx.x * K + r] = x[r];
            __syncthreads();
        }
        int64_t o;
        if constexpr (DIRECT) {
            o = ct_base + (int64_t)q * ct_stride;
            if (threadIdx.x == 0) {
                rc[row] = cntc;
                ct_off[row] = o;
            }
        } else {
            o = rowoff[row];
        }
        for (int i = threadIdx.x; i < cntc; i += blockDim.x) {
            const int c = sk[i];
            const int slot = table_find<LOG2T>(keys, c);
            colC[o + i] = c;
            valC[o + i] = vals[slot];
        }
        __syncthreads();
    }
}

template <typename VT>
__global__ void __launch_bounds__(1024)
k_num_large(const int *__restrict__ queue, const int count, const int *__restrict__ rowptrA,
            const int *__restrict__ colA, const VT *__restrict__ valA, const int *__restrict__ rowptrB,
            const int *__restrict__ colB, const VT *__restrict__ valB, const int64_t *__restrict__ rowoff,
            int *__restrict__ colC, VT *__restrict__ valC, unsigned *__restrict__ bitmap_all,
            int *__restrict__ prefix_all, const int nwords)
{
    __shared__ int s_red[33];
    __shared__ int s_lo, s_hi, s_next[2], s_nlong[2], s_long[2][LONG_CAP];
    unsigned *bm = bitmap_all + (size_t)blockIdx.x * nwords;
    int *prefix = prefix_all + (size_t)blockIdx.x * nwords;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
    for (int q = blockIdx.x; q < count; q += gridDim.x) {
        const int row = queue[q];
        if (threadIdx.x == 0) {
            s_lo = 0x7fffffff;
            s_hi = -1;
            s_next[0] = s_next[1] = 0;
            s_nlong[0] = s_nlong[1] = 0;
        }
        __syncthreads();
        const int a0 = rowptrA[row], a1 = rowptrA[row + 1];
        const int64_t o = rowoff[row];
        const int nout = (int)(rowoff[row + 1] - o);
        // ---- 1. mark the row's columns; zero the row's values ----
        int wlo = 0x7fffffff, whi = -1;
        cta_for_each_b_row(a0, a1, colA, rowptrB, &s_next[0], &s_nlong[0], s_long[0],
                           [&](int, int p0, int pe, int stride) {
                               for (int p = p0; p < pe; p += stride) {
                                   const int c = colB[p];
                                   const int w = c >> 5;
                                   atomicOr(&bm[w], 1u << (c & 31));
                                   wlo = min(wlo, w);
                                   whi = max(whi, w);
                               }
                           });
        if (whi >= 0) {
            atomicMin(&s_lo, wlo);
            atomicMax(&s_hi, whi);
        }
        for (int i = threadIdx.x; i < nout; i += blockDim.x) valC[o + i] = VT(0);
        __threadfence();
        __syncthreads();
        // ---- 2. exclusive popcount prefix over the touched word range ----
        // A warp owns a contiguous chunk of words and walks it 32 words at a time (coalesced;
        // a chunk per THREAD made every load its own 32-byte sector: at n = 4 M columns this
        // phase was most of the kernel's 28.6 ms in config 3).
        // (16-byte loads, the next one issued before the current four words are processed.)
        const int lo = s_lo & ~3, hi = s_hi | 3;   // whole uint4s; the bitmap is padded to 16 bytes
        const int nq = (hi - lo + 1) >> 2;         // uint4s in the touched range
        const uint4 *bq = reinterpret_cast<const uint4 *>(bm + lo);
        const int chunk = (((nq + nwarps - 1) / nwarps) + 31) & ~31;
        const int q0 = warp * chunk;
        const int q1 = min(q0 + chunk, nq);
        int wsum = 0;
#pragma unroll 4
        for (int qi = q0 + lane; qi < q1; qi += 32) {
            const uint4 v = __ldcg(bq + qi);
            wsum += __popc(v.x) + __popc(v.y) + __popc(v.z) + __popc(v.w);
        }
        wsum = warp_sum(wsum);
        if (lane == 0) s_red[warp] = wsum;
        __syncthreads();
        if (warp == 0) {
            int wv = (lane < nwarps) ? s_red[lane] : 0;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const int y = __shfl_up_sync(FULL, wv, d);
                if (lane >= d) wv += y;
            }
            s_red[lane] = wv;
        }
        __syncthreads();
        int run = warp ? s_red[warp - 1] : 0;   // outputs before this warp's chunk
        uint4 nxt = (q0 + lane < q1) ? __ldcg(bq + q0 + lane) : make_uint4(0u, 0u, 0u, 0u);
        for (int qb = q0; qb < q1; qb += 32) {
            const uint4 v = nxt;
            const int qn = qb + 32 + lane;
            nxt = (qn < q1) ? __ldcg(bq + qn) : make_uint4(0u, 0u, 0u, 0u);
            const int pc = __popc(v.x) + __popc(v.y) + __popc(v.z) + __popc(v.w);
            int incl = pc;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const int y = __shfl_up_sync(FULL, incl, d);
                if (lane >= d) incl += y;
            }
            if (pc) {
                int r2 = run + incl - pc;
                const int wbase = lo + ((qb + lane) << 2);
                const unsigned bits4[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    unsigned b = bits4[u];
                    if (b) prefix[wbase + u] = r2;   // (read back only for words that hold a column)
                    // columns of this word are final: write them now, in order
                    while (b) {
                        const int bit = __ffs(b) - 1;
                        b &= b - 1;
                        colC[o + r2] = ((wbase + u) << 5) | bit;
                        ++r2;
                    }
                }
            }
            run += __shfl_sync(FULL, incl, 31);
        }
        __threadfence();
        __syncthreads();
        // ---- 3. accumulate products at their rank ----
        cta_for_each_b_row(a0, a1, colA, rowptrB, &s_next[1], &s_nlong[1], s_long[1],
                           [&](int j, int p0, int pe, int stride) {
                               const VT av = valA[j];
                               // two elements per thread and step: their bitmap/prefix lookups overlap
                               for (int p = p0; p < pe; p += 2 * stride) {
                                   const int pb = p + stride;
                                   const bool two = pb < pe;
                                   const int ca = colB[p];
                                   const int cb = two ? colB[pb] : ca;
                                   const VT va = valB[p];
                                   const VT vb = two ? valB[pb] : VT(0);
                                   const unsigned bita = __ldcg(bm + (ca >> 5)), bitb = __ldcg(bm + (cb >> 5));
                                   const int prea = __ldcg(prefix + (ca >> 5)), preb = __ldcg(prefix + (cb >> 5));
                                   atomicAdd(&valC[o + prea + __popc(bita & ((1u << (ca & 31)) - 1u))], av * va);
                                   if (two) atomicAdd(&valC[o + preb + __popc(bitb & ((1u << (cb & 31)) - 1u))], av * vb);
                               }
                           });
        __syncthreads();
        // ---- 4. restore the all-zero bitmap: only the words of the row's output columns ----
        for (int i = threadIdx.x; i < nout; i += blockDim.x) bm[colC[o + i] >> 5] = 0u;
        __threadfence();
        __syncthreads();
    }
}

// ---- launchers ---------------------------------------------------------------
template <typename VT, int G, int LOG2T, int R>
static cudaError_t launch_num_group_t(const LaunchCtx &lc, const int *queue, int count, Csr A, Csr B,
                                      const int64_t *rowoff, int *colC, void *valC)
{
    constexpr int T = 1 << LOG2T;
    constexpr int N = (R > 0) ? G * R : T / 2;
    constexpr size_t per_group = (size_t)T * value_bytes<VT> + (size_t)T * 4 + (size_t)N * 4;
    int groups = (int)((56 * 1024) / per_group);
    const int max_groups = 256 / G;
    if (groups > max_groups) groups = max_groups;
    const int min_groups = 32 / G;
    groups -= groups % min_groups;   // whole warps only
    if (groups < min_groups) groups = min_groups;
    const int threads = groups * G;
    const size_t smem = per_group * groups;
    if (smem > 48 * 1024) {
        cudaError_t e = cudaFuncSetAttribute(k_num_group<VT, G, LOG2T, R>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
    }
    long long blocks = ((long long)count + groups - 1) / groups;
    const int per_sm = resident_blocks(k_num_group<VT, G, LOG2T, R>, threads, smem);
    const long long cap = (long long)lc.sm_count * per_sm;
    if (blocks > cap) blocks = cap;
    ++*lc.launches;
    k_num_group<VT, G, LOG2T, R><<<(int)blocks, threads, smem, lc.stream>>>(
        queue, count, A.rowptr, A.col, (const VT *)A.val, B.rowptr, B.col, (const VT *)B.val, rowoff, colC, (VT *)valC);
    return cudaGetLastError();
}

template <typename VT, int LOG2T, int THREADS = 512>
static cudaError_t launch_num_block_t(const LaunchCtx &lc, const int *queue, int count, Csr A, Csr B,
                                      const int64_t *rowoff, int *colC, void *valC)
{
    constexpr int T = 1 << LOG2T;
    const size_t smem = (size_t)T * value_bytes<VT> + (size_t)T * 4 + (size_t)(T / 2) * 4;
    static_assert((size_t)T * value_bytes<VT> + (size_t)T * 4 + (size_t)(T / 2) * 4 <= SMEM_BLOCK_MAX, "k_num_block table");
    if (smem > 48 * 1024) {
        cudaError_t e = cudaFuncSetAttribute(k_num_block<VT, LOG2T, THREADS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
    }
    const int per_sm = resident_blocks(k_num_block<VT, LOG2T, THREADS>, THREADS, smem);
    long long blocks = count;
    const long long cap = (long long)lc.sm_count * per_sm;
    if (blocks > cap) blocks = cap;
    ++*lc.launches;
    k_num_block<VT, LOG2T, THREADS><<<(int)blocks, THREADS, smem, lc.stream>>>(
        queue, count, A.rowptr, A.col, (const VT *)A.val, B.rowptr, B.col, (const VT *)B.val, rowoff, colC, (VT *)valC);
    return cudaGetLastError();
}

template <typename VT>
static cudaError_t launch_num_hash_t(const LaunchCtx &lc, int bin, int G, const int *queue, int count, Csr A, Csr B,
                                     const int64_t *rowoff, int *colC, void *valC)
{
    if (count <= 0) return cudaSuccess;
    // register-sort widths: G=32 -> R = N/32; G=8 -> R = N/8 while <= 16, else shared-memory sort
    switch (bin) {
    case NB_G64:
        return G == 8 ? launch_num_group_t<VT, 8, 6, 4>(lc, queue, count, A, B, rowoff, colC, valC)
                      : launch_num_group_t<VT, 32, 6, 1>(lc, queue, count, A, B, rowoff, colC, valC);
    case NB_G128:
        return G == 8 ? launch_num_group_t<VT, 8, 7, 8>(lc, queue, count, A, B, rowoff, colC, valC)
                      : launch_num_group_t<VT, 32, 7, 2>(lc, queue, count, A, B, rowoff, colC, valC);
    case NB_G256:
        return G == 8 ? launch_num_group_t<VT, 8, 8, 16>(lc, queue, count, A, B, rowoff, colC, valC)
                      : launch_num_group_t<VT, 32, 8, 4>(lc, queue, count, A, B, rowoff, colC, valC);
    case NB_G512:
        return G == 8 ? launch_num_group_t<VT, 8, 9, 0>(lc, queue, count, A, B, rowoff, colC, valC)
                      : launch_num_group_t<VT, 32, 9, 8>(lc, queue, count, A, B, rowoff, colC, valC);
    // c > 256: one CTA per row, sized so that an SM holds 2048 threads' worth of rows
    // (R-MAT scale 20: 128/256/512/1024/1024 threads measured best for the five table sizes;
    // a single warp per 1024/2048-slot table was 1.35-1.45x slower, profiles/r01_notes.md).
    case NB_G1024: return launch_num_block_t<VT, 10, 128>(lc, queue, count, A, B, rowoff, colC, valC);
    case NB_G2048: return launch_num_block_t<VT, 11, 256>(lc, queue, count, A, B, rowoff, colC, valC);
    case NB_B4096: return launch_num_block_t<VT, 12, 512>(lc, queue, count, A, B, rowoff, colC, valC);
    case NB_B8192: return launch_num_block_t<VT, 13, 1024>(lc, queue, count, A, B, rowoff, colC, valC);
    case NB_B16384:
        // (16-byte values: no such table, the host runs these rows in k_num_large -- num_hash_last)
        if constexpr (value_bytes<VT> <= 8) return launch_num_block_t<VT, 14, 1024>(lc, queue, count, A, B, rowoff, colC, valC);
        return cudaErrorInvalidValue;
    default: return cudaErrorInvalidValue;
    }
}

template <typename VT>
static cudaError_t launch_num_large_t(const LaunchCtx &lc, const int *queue, int count, int n, Csr A, Csr B,
                                      const int64_t *rowoff, int *colC, void *valC, unsigned *bitmap_scratch,
                                      int *prefix_scratch, int scratch_blocks)
{
    if (count <= 0) return cudaSuccess;
    const int nwords = large_nwords(n);
    const int blocks = count < scratch_blocks ? count : scratch_blocks;
    ++*lc.launches;
    k_num_large<VT><<<blocks, 1024, 0, lc.stream>>>(queue, count, A.rowptr, A.col, (const VT *)A.val, B.rowptr, B.col,
                                                    (const VT *)B.val, rowoff, colC, (VT *)valC, bitmap_scratch,
                                                    prefix_scratch, nwords);
    return cudaGetLastError();
}

template <typename VT, int LOG2T, int R>
static cudaError_t launch_num_direct_filtered(const LaunchCtx &lc, const int *queue, int count, Csr A, Csr B, DirectOut d)
{
    constexpr int T = 1 << LOG2T;
    constexpr size_t per_group = (size_t)T * value_bytes<VT> + (size_t)T * 4 + (size_t)(32 * R) * 4;
    int groups = (int)((56 * 1024) / per_group);
    if (groups > 8) groups = 8;
    if (groups < 1) groups = 1;
    const int threads = groups * 32;
    const size_t smem = per_group * groups;
    auto kern = k_num_direct<VT, 32, LOG2T, R, true>;
    if (smem > 48 * 1024) {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
    }
    long long blocks = ((long long)count + groups - 1) / groups;
    const long long cap = (long long)lc.sm_count * resident_blocks(kern, threads, smem);
    if (blocks > cap) blocks = cap;
    ++*lc.launches;
    kern<<<(int)blocks, threads, smem, lc.stream>>>(queue, count, A.rowptr, A.col, (const VT *)A.val, B.rowptr, B.col,
                                                    (const VT *)B.val, d.rc, d.ct_off, d.ctcol, (VT *)d.ctval, d.ct_base,
                                                    d.retry_queue, d.retry_cnt, d.prod, d.p_lo, d.p_hi,
                                                    d.ct_stride ? d.ct_stride : 32 * R);
    return cudaGetLastError();
}

template <typename VT, int G, int LOG2T, int R>
static cudaError_t launch_num_direct_g(const LaunchCtx &lc, const int *queue, int count, Csr A, Csr B, DirectOut d)
{
    if constexpr (G == 32) {
        if (d.prod) return launch_num_direct_filtered<VT, LOG2T, R>(lc, queue, count, A, B, d);
    }
    constexpr int T = 1 << LOG2T;
    constexpr size_t per_group = (size_t)T * value_bytes<VT> + (size_t)T * 4 + (size_t)(G * R) * 4;
    int groups = (int)((56 * 1024) / per_group);
    const int max_groups = 256 / G;
    if (groups > max_groups) groups = max_groups;
    const int min_groups = 32 / G;
    groups -= groups % min_groups;
    if (groups < min_groups) groups = min_groups;
    const int threads = groups * G;
    const size_t smem = per_group * groups;
    if (smem > 48 * 1024) {
        cudaError_t e = cudaFuncSetAttribute(k_num_direct<VT, G, LOG2T, R>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
    }
    long long blocks = ((long long)count + groups - 1) / groups;
    const long long cap = (long long)lc.sm_count * resident_blocks(k_num_direct<VT, G, LOG2T, R>, threads, smem);
    if (blocks > cap) blocks = cap;
    ++*lc.launches;
    k_num_direct<VT, G, LOG2T, R><<<(int)blocks, threads, smem, lc.stream>>>(
        queue, count, A.rowptr, A.col, (const VT *)A.val, B.rowptr, B.col, (const VT *)B.val, d.rc, d.ct_off, d.ctcol,
        (VT *)d.ctval, d.ct_base, d.retry_queue, d.retry_cnt);
    return cudaGetLastError();
}

template <typename VT, int LOG2T, int THREADS>
static cudaError_t launch_num_block_direct_t(const LaunchCtx &lc, const int *queue, int count, Csr A, Csr B, DirectOut d)
{
    constexpr int T = 1 << LOG2T;
    const size_t smem = (size_t)T * value_bytes<VT> + (size_t)T * 4 + (size_t)(T / 2) * 4;
    static_assert((size_t)T * value_bytes<VT> + (size_t)T * 4 + (size_t)(T / 2) * 4 <= SMEM_BLOCK_MAX, "k_num_block table");
    if (smem > 48 * 1024) {
        cudaError_t e = cudaFuncSetAttribute(k_num_block<VT, LOG2T, THREADS, true>,
                                             cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
    }
    const int per_sm = resident_blocks(k_num_block<VT, LOG2T, THREADS, true>, THREADS, smem);
    long long blocks = count;
    const long long cap = (long long)lc.sm_count * per_sm;
    if (blocks > cap) blocks = cap;
    ++*lc.launches;
    k_num_block<VT, LOG2T, THREADS, true><<<(int)blocks, THREADS, smem, lc.stream>>>(
        queue, count, A.rowptr, A.col, (const VT *)A.val, B.rowptr, B.col, (const VT *)B.val, nullptr, d.ctcol,
        (VT *)d.ctval, d.rc, d.ct_off, d.ct_base, d.prod, d.p_lo, d.p_hi, d.ct_stride ? d.ct_stride : T / 2);
    return cudaGetLastError();
}

template <typename VT>
static cudaError_t launch_num_direct_t(const LaunchCtx &lc, int cap, int G, const int *queue, int count, Csr A, Csr B,
                                       DirectOut d)
{
    if (count <= 0) return cudaSuccess;
    switch (cap) {
    case 256: return launch_num_direct_g<VT, 32, 9, 8>(lc, queue, count, A, B, d);
    case 512: return launch_num_block_direct_t<VT, 10, 128>(lc, queue, count, A, B, d);
    case 1024: return launch_num_block_direct_t<VT, 11, 256>(lc, queue, count, A, B, d);
    case 2048: return launch_num_block_direct_t<VT, 12, 512>(lc, queue, count, A, B, d);
    case 4096: return launch_num_block_direct_t<VT, 13, 1024>(lc, queue, count, A, B, d);
    case 8192:
        // (16-byte values: plan_direct plans no capacity above DirectPlan::table_cap_max)
        if constexpr (value_bytes<VT> <= 8) return launch_num_block_direct_t<VT, 14, 1024>(lc, queue, count, A, B, d);
        return cudaErrorInvalidValue;
    case 32:
        return G == 8 ? launch_num_direct_g<VT, 8, 6, 4>(lc, queue, count, A, B, d)
                      : launch_num_direct_g<VT, 32, 6, 1>(lc, queue, count, A, B, d);
    case 64:
        return G == 8 ? launch_num_direct_g<VT, 8, 7, 8>(lc, queue, count, A, B, d)
                      : launch_num_direct_g<VT, 32, 7, 2>(lc, queue, count, A, B, d);
    case 128:
        return G == 8 ? launch_num_direct_g<VT, 8, 8, 16>(lc, queue, count, A, B, d)
                      : launch_num_direct_g<VT, 32, 8, 4>(lc, queue, count, A, B, d);
    default: return cudaErrorInvalidValue;
    }
}

template <typename VT, int THREADS>
static cudaError_t launch_num_bucket_tt(const LaunchCtx &lc, int cap, const int *queue, int count, Csr A, Csr B, DirectOut d,
                                        ColumnCdf cdf)
{
    // (one bucket per entry for the capacities up to 2048 instead of one per two: measured equal, R-MAT 21 39.46 vs 39.56 ms)
    const int nb = cap / 2;
    // below 1024 threads every fourth knot of the CDF: enough for <= 1024 buckets, and what lets two 4096-entry CTAs share an SM
    constexpr int KB = THREADS < 1024 ? 10 : CDF_BITS;
    const size_t smem = b3_smem_bytes<VT, THREADS>(cap, nb, 1 << KB);
    if (smem > SMEM_BLOCK_MAX) return cudaErrorInvalidValue;   // (16-byte values at cap 8192: plan_direct plans none)
    auto kern = k_num_bucket3<VT, THREADS, KB>;
    if (smem > 48 * 1024) {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
    }
    long long blocks = count;
    const long long lim = (long long)lc.sm_count * resident_blocks(kern, THREADS, smem);
    if (blocks > lim) blocks = lim;
    ++*lc.launches;
    kern<<<(int)blocks, THREADS, smem, lc.stream>>>(queue, count, A.rowptr, A.col, (const VT *)A.val, B.rowptr, B.col,
                                                    (const VT *)B.val, cdf, cap, nb, d.rc, d.ct_off, d.ctcol, (VT *)d.ctval,
                                                    d.ct_base, d.prod, d.p_lo, d.p_hi, d.ct_stride ? d.ct_stride : cap, d.bump);
    return cudaGetLastError();
}

// rows of the queue with p_lo < products <= p_hi <= cap, staged ct_stride apart (wide direct bins)
template <typename VT>
static cudaError_t launch_num_bucket_t(const LaunchCtx &lc, int cap, const int *queue, int count, Csr A, Csr B, DirectOut d,
                                       ColumnCdf cdf)
{
    if (count <= 0) return cudaSuccess;
    // k_num_bucket3: a thread per four entries of the capacity, at most 1024
    switch (cap) {
    case 512: return launch_num_bucket_tt<VT, 128>(lc, cap, queue, count, A, B, d, cdf);
    case 1024: return launch_num_bucket_tt<VT, 256>(lc, cap, queue, count, A, B, d, cdf);
    case 2048: return launch_num_bucket_tt<VT, 512>(lc, cap, queue, count, A, B, d, cdf);
    case 4096: return launch_num_bucket_tt<VT, 768>(lc, cap, queue, count, A, B, d, cdf);   // 2 x 768 threads per SM (109 KB each) beat 1 x 1024
    case 8192: return launch_num_bucket_tt<VT, 1024>(lc, cap, queue, count, A, B, d, cdf);
    default: return cudaErrorInvalidValue;
    }
}

// warp-per-row bucket sort for the bins of at most 96 (capw 128) / 192 (capw 256) products; rows staged `stride` apart
template <typename VT, int CAPW, int SG>
static cudaError_t launch_num_bucket3w_tt(const LaunchCtx &lc, const int *queue, int count, Csr A, Csr B, DirectOut d, ColumnCdf cdf,
                                          int stride)
{
    const size_t smem = ((((size_t)(1 << B3W_KB) + 1) * 4 + 15) & ~(size_t)15) + (size_t)B3W_WARPS * b3w_per_warp<VT, CAPW>();
    auto kern = k_num_bucket3w<VT, CAPW, SG>;
    if (smem > 48 * 1024) {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
    }
    long long blocks = ((long long)count + B3W_WARPS - 1) / B3W_WARPS;
    const long long lim = (long long)lc.sm_count * resident_blocks(kern, B3W_WARPS * 32, smem);
    if (blocks > lim) blocks = lim;
    ++*lc.launches;
    kern<<<(int)blocks, B3W_WARPS * 32, smem, lc.stream>>>(queue, count, A.rowptr, A.col, (const VT *)A.val, B.rowptr, B.col,
                                                          (const VT *)B.val, cdf, d.rc, d.ct_off, d.ctcol, (VT *)d.ctval, d.ct_base,
                                                          stride, d.retry_queue, d.retry_cnt);
    return cudaGetLastError();
}

template <typename VT>
static cudaError_t launch_num_bucket3w_t(const LaunchCtx &lc, int capw, int sg, const int *queue, int count, Csr A, Csr B, DirectOut d,
                                         ColumnCdf cdf, int stride)
{
    if (count <= 0) return cudaSuccess;
    if (capw == 128)
        return sg == 8 ? launch_num_bucket3w_tt<VT, 128, 8>(lc, queue, count, A, B, d, cdf, stride)
                       : launch_num_bucket3w_tt<VT, 128, 32>(lc, queue, count, A, B, d, cdf, stride);
    if (capw == 256)
        return sg == 8 ? launch_num_bucket3w_tt<VT, 256, 8>(lc, queue, count, A, B, d, cdf, stride)
                       : launch_num_bucket3w_tt<VT, 256, 32>(lc, queue, count, A, B, d, cdf, stride);
    return cudaErrorInvalidValue;
}

template <typename VT>
static cudaError_t launch_num_bucket_heavy_t(const LaunchCtx &lc, const int *queue, int count, Csr A, Csr B, DirectOut d,
                                             ColumnCdf cdf, unsigned long long *cursor)
{
    if (count <= 0) return cudaSuccess;
    constexpr int THREADS = 1024;
    // entries of a slice held on chip (16-byte values: 8192, 212 KB)
    constexpr int cap = value_bytes<VT> == 16 ? 8192 : value_bytes<VT> == 8 ? 12288 : 16384;
    // buckets per slice: half the capacity (measured best on R-MAT 24 rank 0: /2 70.3, /4 72.5, /8 72.8 ms)
    constexpr int nb = cap / 2;
    constexpr size_t smem = (size_t)cap * (value_bytes<VT> + 4) + (size_t)(2 * nb + 1 + 34) * 4 + (size_t)(CDF_KNOTS + 1) * 4;
    static_assert(smem <= SMEM_BLOCK_MAX, "k_num_bucket_heavy slice");
    auto kern = k_num_bucket_heavy<VT, THREADS>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    long long blocks = count;
    const long long lim = (long long)lc.sm_count * resident_blocks(kern, THREADS, smem);
    if (blocks > lim) blocks = lim;
    ++*lc.launches;
    kern<<<(int)blocks, THREADS, smem, lc.stream>>>(queue, count, A.rowptr, A.col, (const VT *)A.val, B.rowptr, B.col,
                                                    (const VT *)B.val, cdf, cap, nb, d.rc, d.ct_off, d.ctcol, (VT *)d.ctval,
                                                    d.ct_base, cursor, d.prod, d.count_dev);
    return cudaGetLastError();
}

template <typename VT>
static cudaError_t launch_num_bucket_heavy2_t(const LaunchCtx &lc, const int *queue, int count, Csr A, Csr B, DirectOut d,
                                              ColumnCdf cdf, unsigned long long *cursor)
{
    if (count <= 0) return cudaSuccess;
    constexpr int THREADS = 1024;
    // entries of a slice on chip (22 / 18 bytes each; 16-byte values: 4096 of 30 bytes), buckets per slice
    constexpr int cap = value_bytes<VT> > 8 ? 4096 : 8192, nb = cap / 2;
    constexpr size_t smem = h2_smem_bytes<VT>(cap, nb);
    static_assert(smem <= SMEM_BLOCK_MAX, "k_num_bucket_heavy2 slice");
    auto kern = k_num_bucket_heavy2<VT, THREADS>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    long long blocks = count;
    const long long lim = (long long)lc.sm_count * resident_blocks(kern, THREADS, smem);
    if (blocks > lim) blocks = lim;
    ++*lc.launches;
    kern<<<(int)blocks, THREADS, smem, lc.stream>>>(queue, count, A.rowptr, A.col, (const VT *)A.val, B.rowptr, B.col,
                                                    (const VT *)B.val, cdf, cap, nb, d.rc, d.ct_off, d.ctcol, (VT *)d.ctval,
                                                    d.ct_base, cursor, d.prod, d.p_lo, d.retry_queue, d.retry_cnt);
    return cudaGetLastError();
}

template <typename VT>
static cudaError_t launch_copy_ct_t(const LaunchCtx &lc, const int *queue, int count, const int64_t *rowoff,
                                    const long long *ct_off, const int *ctcol, const void *ctval, int *colC, void *valC,
                                    double avg_row)
{
    if (count <= 0) return cudaSuccess;
    const int threads = 256;
    ++*lc.launches;
    // (measured and dropped: a warp per 32 short rows, their {offset, length, staging offset} read with coalesced loads:
    // config 4's copy 1.50 -> 1.52 ms)
    if (avg_row <= 12.0) {
        const long long blocks = ((long long)count * 8 + threads - 1) / threads;
        k_copy_ct<VT, 8><<<(int)blocks, threads, 0, lc.stream>>>(queue, count, rowoff, ct_off, ctcol, (const VT *)ctval,
                                                                 colC, (VT *)valC);
    } else {
        const long long blocks = ((long long)count * 32 + threads - 1) / threads;
        k_copy_ct<VT, 32><<<(int)blocks, threads, 0, lc.stream>>>(queue, count, rowoff, ct_off, ctcol, (const VT *)ctval,
                                                                  colC, (VT *)valC);
    }
    return cudaGetLastError();
}

}  // namespace bhb
