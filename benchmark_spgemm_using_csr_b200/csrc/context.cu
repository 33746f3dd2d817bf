// context.cu -- the C-ABI (include/bhsparse_b200.h) and the host orchestration of the
// device pipeline.  Counterpart of bhsparse::spgemm_cuda (SpGEMM_cuda/bhsparse.h:297-339)
// and of the memory management in bhsparse_cuda (bhsparse_cuda.h:121-203, 285-301,
// 2783-2811, 3006-3020).  Host <-> device traffic inside one spgemm call: two reads of a
// 300-byte counter block (bin sizes; nnz(C)) -- the reference has >= 8 blocking copies of
// O(m) data plus 3 per merge round (SURVEY.md 3.2).
#include "context.h"
#include "direct_plan.h"
#include "stage_bucket.cuh"

#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>
#include <string>

using namespace bhb;

namespace {

int fail(bhb200_ctx *c, int code, const char *what, cudaError_t e = cudaSuccess)
{
    if (c) {
        c->err = what;
        if (e != cudaSuccess) {
            c->err += ": ";
            c->err += cudaGetErrorString(e);
        }
    }
    return code;
}

#define CU(call, what)                                                            \
    do {                                                                          \
        cudaError_t e__ = (call);                                                 \
        if (e__ != cudaSuccess) {                                                 \
            cudaGetLastError();                                                   \
            return fail(ctx, e__ == cudaErrorMemoryAllocation ? BHB200_ERR_ALLOC  \
                                                              : BHB200_ERR_CUDA,  \
                        what, e__);                                               \
        }                                                                         \
    } while (0)

size_t vsize(int dtype)
{
    return dispatch_value_type(dtype, [](auto v) { return value_bytes<decltype(v)>; });
}

const char *dtype_name(int dtype)
{
    return dtype == BHB200_DTYPE_F64 ? "f64" : dtype == BHB200_DTYPE_C64 ? "c64" : dtype == BHB200_DTYPE_C128 ? "c128" : "f32";
}

int refuse_structure(bhb200_ctx *ctx, const char *what)
{
    std::string msg = what;
    msg += ": the operands are structure-only (BHB200_DTYPE_NONE), C has no values";
    return fail(ctx, BHB200_ERR_INVALID, msg.c_str());
}

// forget the mask (the library's copy stays allocated for the next bhb200_set_mask)
void drop_mask(bhb200_ctx *ctx)
{
    ctx->mask_set = false;
    ctx->M = MaskCsr{nullptr, nullptr, 0};
    ctx->last_masked = false;
}

void release_operands(bhb200_ctx *ctx)
{
    ctx->a_rowptr.release(&ctx->dev_bytes);
    ctx->a_col.release(&ctx->dev_bytes);
    ctx->a_val.release(&ctx->dev_bytes);
    ctx->b_rowptr.release(&ctx->dev_bytes);
    ctx->b_col.release(&ctx->dev_bytes);
    ctx->b_val.release(&ctx->dev_bytes);
    DevBuf *tbufs[] = {&ctx->at_rowptr, &ctx->at_col, &ctx->at_val, &ctx->at_perm,
                       &ctx->bt_rowptr, &ctx->bt_col, &ctx->bt_val, &ctx->bt_perm};
    for (DevBuf *b : tbufs) b->release(&ctx->dev_bytes);
    ctx->A = Csr{nullptr, nullptr, nullptr};
    ctx->B = Csr{nullptr, nullptr, nullptr};
    ctx->As = Csr{nullptr, nullptr, nullptr};
    ctx->Bs = Csr{nullptr, nullptr, nullptr};
    ctx->opA = ctx->opB = BHB200_OP_N;
    ctx->t_pending = ctx->t_shared = false;
    ctx->have_data = false;
    ctx->borrowed = false;
    ctx->aliased = false;
    ctx->slice_e0 = -1;
    ctx->cdf_valid = false;
    ctx->have_C = false;
    ctx->last_pattern = false;
    ctx->nnzC = 0;
    drop_mask(ctx);
}

// (structure-only operands: the values are never read and may be null)
int check_dims(bhb200_ctx *ctx, int dtype, int m, int k, int n, int nnzA, int nnzB, const void *valA, const int32_t *rowptrA,
               const int32_t *colA, const void *valB, const int32_t *rowptrB, const int32_t *colB)
{
    const bool values = dtype != BHB200_DTYPE_NONE;
    if (m < 0 || k < 0 || n < 0 || nnzA < 0 || nnzB < 0) return fail(ctx, BHB200_ERR_INVALID, "negative dimension");
    if (!rowptrA || !rowptrB) return fail(ctx, BHB200_ERR_INVALID, "null row pointer array");
    if (nnzA > 0 && (!colA || (values && !valA))) return fail(ctx, BHB200_ERR_INVALID, "null A arrays");
    if (nnzB > 0 && (!colB || (values && !valB))) return fail(ctx, BHB200_ERR_INVALID, "null B arrays");
    return BHB200_SUCCESS;
}

int check_ops(bhb200_ctx *ctx, int dtype, int opA, int opB)
{
    const bool complex = dtype == BHB200_DTYPE_C64 || dtype == BHB200_DTYPE_C128;
    const int last = complex ? BHB200_OP_C : BHB200_OP_T;
    if (opA < BHB200_OP_N || opA > last || opB < BHB200_OP_N || opB > last)
        return fail(ctx, BHB200_ERR_INVALID,
                    complex ? "op must be BHB200_OP_N, BHB200_OP_T or BHB200_OP_C"
                            : "op must be BHB200_OP_N or BHB200_OP_T (BHB200_OP_C needs complex operands)");
    return BHB200_SUCCESS;
}

// ctx->A / ctx->B from the stored operands: the transposed copies (reserved here, filled by run_transposes) for op = T.
// Structure-only operands have no values to transpose and keep no permutation (nothing is ever re-gathered): the sort
// still writes one, into the transpose scratch (run_transposes).
int set_effective(bhb200_ctx *ctx)
{
    const size_t vs = vsize(ctx->dtype);
    ctx->A = ctx->As;
    ctx->B = ctx->Bs;
    if (ctx->opA) {
        CU(ctx->at_rowptr.reserve(((size_t)ctx->m + 1) * 4, &ctx->dev_bytes), "alloc rowptr of A^T");
        CU(ctx->at_col.reserve((size_t)ctx->nnzA * 4 + 4, &ctx->dev_bytes), "alloc col of A^T");
        if (vs) {
            CU(ctx->at_val.reserve((size_t)ctx->nnzA * vs + 16, &ctx->dev_bytes), "alloc val of A^T");
            CU(ctx->at_perm.reserve((size_t)ctx->nnzA * 4 + 4, &ctx->dev_bytes), "alloc perm of A^T");
        }
        ctx->A = Csr{ctx->at_rowptr.as<int>(), ctx->at_col.as<int>(), vs ? ctx->at_val.p : nullptr};
    }
    if (ctx->opB && ctx->t_shared) {
        ctx->B = ctx->A;
    } else if (ctx->opB) {
        CU(ctx->bt_rowptr.reserve(((size_t)ctx->k + 1) * 4, &ctx->dev_bytes), "alloc rowptr of B^T");
        CU(ctx->bt_col.reserve((size_t)ctx->nnzB * 4 + 4, &ctx->dev_bytes), "alloc col of B^T");
        if (vs) {
            CU(ctx->bt_val.reserve((size_t)ctx->nnzB * vs + 16, &ctx->dev_bytes), "alloc val of B^T");
            CU(ctx->bt_perm.reserve((size_t)ctx->nnzB * 4 + 4, &ctx->dev_bytes), "alloc perm of B^T");
        }
        ctx->B = Csr{ctx->bt_rowptr.as<int>(), ctx->bt_col.as<int>(), vs ? ctx->bt_val.p : nullptr};
    }
    ctx->t_pending = ctx->opA || ctx->opB;
    return BHB200_SUCCESS;
}

// The transposed structure and values of every op = T operand, on the context's stream (no host sync).
// A column of a stored operand outside its range raises a bit of Counters::bad_T, read with the counters.
int run_transposes(bhb200_ctx *ctx, const LaunchCtx &lc)
{
    const bool tb = ctx->opB && !ctx->t_shared;
    const bool keep_perm = ctx->dtype != BHB200_DTYPE_NONE;
    size_t need = 0;
    if (ctx->opA) need = transpose_scratch_bytes(ctx->nnzA, ctx->m);
    if (tb) need = std::max(need, transpose_scratch_bytes(ctx->nnzB, ctx->k));
    const size_t perm_at = need;   // structure only: the sort still produces the permutation, into the scratch after the rest
    if (!keep_perm) need += (size_t)std::max(ctx->opA ? ctx->nnzA : 0, tb ? ctx->nnzB : 0) * 4 + 4;
    if (need) CU(ctx->t_scratch.reserve(need, &ctx->dev_bytes), "alloc transpose scratch");
    int *scratch_perm = reinterpret_cast<int *>(static_cast<unsigned char *>(ctx->t_scratch.p) + perm_at);
    Counters *d_ctr = ctx->counters.as<Counters>();
    CU(cudaMemsetAsync(&d_ctr->bad_T, 0, sizeof(int), lc.stream), "zero transpose flag");
    if (ctx->opA)
        CU(launch_transpose(lc, ctx->dtype, ctx->opA == BHB200_OP_C, ctx->k, ctx->m, ctx->nnzA, ctx->As,
                            TransposeOut{ctx->at_rowptr.as<int>(), ctx->at_col.as<int>(), keep_perm ? ctx->at_val.p : nullptr,
                                         keep_perm ? ctx->at_perm.as<int>() : scratch_perm},
                            ctx->t_scratch.p, &d_ctr->bad_T, 1),
           "transpose A");
    if (tb)
        CU(launch_transpose(lc, ctx->dtype, ctx->opB == BHB200_OP_C, ctx->n, ctx->k, ctx->nnzB, ctx->Bs,
                            TransposeOut{ctx->bt_rowptr.as<int>(), ctx->bt_col.as<int>(), keep_perm ? ctx->bt_val.p : nullptr,
                                         keep_perm ? ctx->bt_perm.as<int>() : scratch_perm},
                            ctx->t_scratch.p, &d_ctr->bad_T, 2),
           "transpose B");
    ctx->t_pending = false;
    return BHB200_SUCCESS;
}

// values of the op = T operands again from the stored values, through the permutation of the last transposition
int run_regathers(bhb200_ctx *ctx, const LaunchCtx &lc)
{
    if (ctx->opA)
        CU(launch_regather(lc, ctx->dtype, ctx->opA == BHB200_OP_C, ctx->nnzA, ctx->As.val, ctx->at_perm.as<int>(), ctx->at_val.p), "re-gather values of A^T");
    if (ctx->opB && !ctx->t_shared)
        CU(launch_regather(lc, ctx->dtype, ctx->opB == BHB200_OP_C, ctx->nnzB, ctx->Bs.val, ctx->bt_perm.as<int>(), ctx->bt_val.p), "re-gather values of B^T");
    return BHB200_SUCCESS;
}

// Counters::bad_T of the transposition of this call's operands (read back with the other counters)
int check_transposed(bhb200_ctx *ctx, int bad_T)
{
    if (!(ctx->opA || ctx->opB) || !bad_T) return BHB200_SUCCESS;
    if (bad_T & 1) return fail(ctx, BHB200_ERR_INVALID, "a column index of the stored A (opA = T) is outside [0, m)");
    return fail(ctx, BHB200_ERR_INVALID, "a column index of the stored B (opB = T) is outside [0, k)");
}

int init_host(bhb200_ctx *ctx, int dtype, int opA, int opB, int m, int k, int n, int nnzA, const void *valA,
              const int32_t *rowptrA, const int32_t *colA, int nnzB, const void *valB, const int32_t *rowptrB,
              const int32_t *colB)
{
    if (!ctx) return BHB200_ERR_INVALID;
    int rc = check_ops(ctx, dtype, opA, opB);
    if (rc) return rc;
    rc = check_dims(ctx, dtype, m, k, n, nnzA, nnzB, valA, rowptrA, colA, valB, rowptrB, colB);
    if (rc) return rc;
    // stored shapes: A is m x k (k x m for opA = T), B is k x n (n x k for opB = T)
    const int ra = opA ? k : m, ca = opA ? m : k, rb = opB ? n : k, cb = opB ? k : n;
    if (rowptrA[0] != 0 || rowptrA[ra] != nnzA) return fail(ctx, BHB200_ERR_INVALID, "rowptrA does not span [0, nnzA]");
    if (rowptrB[0] != 0 || rowptrB[rb] != nnzB) return fail(ctx, BHB200_ERR_INVALID, "rowptrB does not span [0, nnzB]");
    CU(cudaSetDevice(ctx->device), "cudaSetDevice");
    if (ctx->borrowed) release_operands(ctx);
    const size_t vs = vsize(dtype);
    CU(ctx->a_rowptr.reserve((size_t)(ra + 1) * 4, &ctx->dev_bytes), "alloc rowptrA");
    CU(ctx->a_col.reserve((size_t)nnzA * 4 + 4, &ctx->dev_bytes), "alloc colA");
    if (vs) CU(ctx->a_val.reserve((size_t)nnzA * vs + 16, &ctx->dev_bytes), "alloc valA");
    // C = A*A with the SAME host arrays passed twice (the reference driver's stock workloads build
    // A and B identically, main.cu:32-51): one upload, both operands point at it (also A*A^T, A^T*A)
    const bool alias = ra == rb && (!(opA || opB) || ca == cb) && nnzA == nnzB && rowptrA == rowptrB && colA == colB &&
                       valA == valB;
    if (!alias) {
        CU(ctx->b_rowptr.reserve((size_t)(rb + 1) * 4, &ctx->dev_bytes), "alloc rowptrB");
        CU(ctx->b_col.reserve((size_t)nnzB * 4 + 4, &ctx->dev_bytes), "alloc colB");
        if (vs) CU(ctx->b_val.reserve((size_t)nnzB * vs + 16, &ctx->dev_bytes), "alloc valB");
    }
    cudaStream_t s = ctx->stream;
    CU(cudaMemcpyAsync(ctx->a_rowptr.p, rowptrA, (size_t)(ra + 1) * 4, cudaMemcpyHostToDevice, s), "H2D rowptrA");
    if (!alias) CU(cudaMemcpyAsync(ctx->b_rowptr.p, rowptrB, (size_t)(rb + 1) * 4, cudaMemcpyHostToDevice, s), "H2D rowptrB");
    if (nnzA > 0) {
        CU(cudaMemcpyAsync(ctx->a_col.p, colA, (size_t)nnzA * 4, cudaMemcpyHostToDevice, s), "H2D colA");
        if (vs) CU(cudaMemcpyAsync(ctx->a_val.p, valA, (size_t)nnzA * vs, cudaMemcpyHostToDevice, s), "H2D valA");
    }
    if (nnzB > 0 && !alias) {
        CU(cudaMemcpyAsync(ctx->b_col.p, colB, (size_t)nnzB * 4, cudaMemcpyHostToDevice, s), "H2D colB");
        if (vs) CU(cudaMemcpyAsync(ctx->b_val.p, valB, (size_t)nnzB * vs, cudaMemcpyHostToDevice, s), "H2D valB");
    }
    CU(cudaStreamSynchronize(s), "H2D operands");
    ctx->As = Csr{ctx->a_rowptr.as<int>(), ctx->a_col.as<int>(), vs ? ctx->a_val.p : nullptr};
    ctx->Bs = alias ? ctx->As : Csr{ctx->b_rowptr.as<int>(), ctx->b_col.as<int>(), vs ? ctx->b_val.p : nullptr};
    ctx->aliased = alias;
    ctx->dtype = dtype;
    ctx->m = m;
    ctx->k = k;
    ctx->n = n;
    ctx->nnzA = nnzA;
    ctx->nnzB = nnzB;
    ctx->opA = opA;
    ctx->opB = opB;
    ctx->t_shared = alias && opA && opA == opB;   // one transposed copy serves (T, T) and (C, C)
    ctx->have_data = false;
    rc = set_effective(ctx);
    if (rc) return rc;
    ctx->have_data = true;
    ctx->cdf_valid = false;   // new operands: the column CDF of the previous ones is not reused
    ctx->borrowed = false;
    ctx->have_C = false;
    ctx->nnzC = 0;
    drop_mask(ctx);
    return BHB200_SUCCESS;
}

int reserve_workspace(bhb200_ctx *ctx)
{
    const size_t m1 = (size_t)ctx->m + 1;
    CU(ctx->prod.reserve(m1 * 4, &ctx->dev_bytes), "alloc row products");
    CU(ctx->rc.reserve(m1 * 4, &ctx->dev_bytes), "alloc row counts");
    CU(ctx->queue.reserve(m1 * 4, &ctx->dev_bytes), "alloc row queue");
    CU(ctx->rowoff64.reserve(m1 * 8, &ctx->dev_bytes), "alloc rowptrC64");
    CU(ctx->rowptr32.reserve(m1 * 4, &ctx->dev_bytes), "alloc rowptrC");
    CU(ctx->blocksums.reserve((scan_blocksum_count(ctx->m) + 1) * 8, &ctx->dev_bytes), "alloc scan sums");
    CU(ctx->counters.reserve(sizeof(Counters), &ctx->dev_bytes), "alloc counters");
    CU(ctx->brange.reserve(((size_t)ctx->k + 1) * 16, &ctx->dev_bytes), "alloc B row ranges");
    CU(ctx->rlo.reserve(m1 * 4, &ctx->dev_bytes), "alloc row min column");
    CU(ctx->rspan.reserve(m1 * 4, &ctx->dev_bytes), "alloc row span");
    return BHB200_SUCCESS;
}

// scratch of the global-bitmap kernels: one n-bit bitmap (+ one int prefix per word)
// per resident CTA, kept all-zero between uses
int reserve_large_scratch(bhb200_ctx *ctx, bool need_prefix)
{
    const size_t nwords = (size_t)large_nwords(ctx->n);
    const size_t blocks = (size_t)large_scratch_blocks(ctx->sm_count, ctx->n);
    const size_t bytes = nwords * blocks * 4;
    if (bytes > ctx->bitmap.cap) ctx->bitmap_zeroed_bytes = 0;
    CU(ctx->bitmap.reserve(bytes, &ctx->dev_bytes), "alloc bitmap scratch");
    if (ctx->bitmap_zeroed_bytes < bytes) {
        CU(cudaMemsetAsync(ctx->bitmap.p, 0, ctx->bitmap.cap, ctx->stream), "zero bitmap scratch");
        ctx->bitmap_zeroed_bytes = ctx->bitmap.cap;
    }
    if (need_prefix) CU(ctx->prefix.reserve(bytes, &ctx->dev_bytes), "alloc prefix scratch");
    return BHB200_SUCCESS;
}

// profiling: stamp the stream before bin `b` of phase `ph` (b == MAX_BINS: after the last bin)
cudaError_t stamp(bhb200_ctx *ctx, int ph, int b)
{
    if (!ctx->profiling) return cudaSuccess;
    if (!ctx->ev_bin[ph][b]) {
        cudaError_t e = cudaEventCreate(&ctx->ev_bin[ph][b]);
        if (e != cudaSuccess) return e;
    }
    ctx->ev_bin_used[ph][b] = true;
    return cudaEventRecord(ctx->ev_bin[ph][b], ctx->stream);
}

// word-list pool of the range kernels: sized from the product count of the call; if it is
// too small (or cannot be allocated) the numeric kernel marks the affected rows itself
int reserve_word_lists(bhb200_ctx *ctx, int64_t products, WordLists &wl)
{
    const size_t m1 = (size_t)ctx->m + 1;
    CU(ctx->wl_off.reserve(m1 * 8, &ctx->dev_bytes), "alloc word-list offsets");
    CU(ctx->wl_cnt.reserve(m1 * 4, &ctx->dev_bytes), "alloc word-list counts");
    long long cap = products / 4 + (long long)ctx->m + 1024;
    if (cap > (1ll << 31)) cap = 1ll << 31;
    if (ctx->wordlist_cap >= 0) cap = ctx->wordlist_cap;   // tests: force the fallback
    if (ctx->wl_idx.reserve((size_t)cap * 4, &ctx->dev_bytes) != cudaSuccess ||
        ctx->wl_bits.reserve((size_t)cap * 8, &ctx->dev_bytes) != cudaSuccess) {
        cudaGetLastError();
        cap = 0;   // no pool: every row falls back to marking in the numeric kernel
    } else {
        // grow-only buffers may be larger than this call's request: use all of it
        const long long have = (long long)(ctx->wl_idx.cap / 4 < ctx->wl_bits.cap / 8 ? ctx->wl_idx.cap / 4 : ctx->wl_bits.cap / 8);
        if (have > cap && ctx->wordlist_cap < 0) cap = have;
    }
    wl.off = ctx->wl_off.as<long long>();
    wl.cnt = ctx->wl_cnt.as<int>();
    wl.idx = ctx->wl_idx.as<unsigned>();
    wl.bits = ctx->wl_bits.as<unsigned long long>();
    wl.cap = cap;
    return BHB200_SUCCESS;
}

void offsets_from_counts(const int *counts, BinOffsets &o)
{
    int acc = 0;
    for (int b = 0; b < MAX_BINS; ++b) {
        o.off[b] = acc;
        acc += counts[b];
    }
    o.off[MAX_BINS] = acc;
}

// Numeric kernels of every bin except the Ct -> C copy; shared by bhb200_spgemm (stage 4) and
// bhb200_spgemm_numeric (values only, structure of C reused).
int run_numeric_bins(bhb200_ctx *ctx, const LaunchCtx &lc, const int *num_bin, const BinOffsets &no, int G,
                     const WordLists &wl)
{
    int rc = 0;
    const NumericKernels &nk = numeric_kernels(ctx->dtype);
    int *queue = ctx->queue.as<int>();
    int64_t *rowoff = ctx->rowoff64.as<int64_t>();
    int *rlo = ctx->rlo.as<int>();
    int *colC = ctx->colC.as<int>();
    void *valC = ctx->valC.p;
    if (num_bin[NB_ONE] > 0) CU(stamp(ctx, 1, NB_ONE), "event");
    CU(launch_num_single(lc, ctx->dtype, queue + no.off[NB_ONE], num_bin[NB_ONE], ctx->A, ctx->B, rowoff, colC, valC),
       "numeric single");
    if (num_bin[NB_ESC] > 0) CU(stamp(ctx, 1, NB_ESC), "event");
    CU(launch_num_esc(lc, ctx->dtype, queue + no.off[NB_ESC], num_bin[NB_ESC], ctx->n, ctx->A, ctx->B, rowoff, colC, valC),
       "numeric ESC");
    const int last_hash = num_hash_last(vsize(ctx->dtype));
    for (int b = NB_G64; b <= last_hash; ++b) {
        if (num_bin[b] > 0) CU(stamp(ctx, 1, b), "event");
        CU(nk.hash(lc, b, G, queue + no.off[b], num_bin[b], ctx->A, ctx->B, rowoff, colC, valC),
           (std::string("numeric hash ") + dtype_name(ctx->dtype)).c_str());
    }
    // the bins after last_hash and NB_LARGE are consecutive in the queue: one launch of the global-bitmap kernel
    int large_rows = 0;
    for (int b = last_hash + 1; b <= NB_LARGE; ++b) large_rows += num_bin[b];
    if (large_rows > 0) {
        rc = reserve_large_scratch(ctx, true);
        if (rc) return rc;
        const int sb = large_scratch_blocks(ctx->sm_count, ctx->n);
        CU(stamp(ctx, 1, NB_LARGE), "event");
        CU(nk.large(lc, queue + no.off[last_hash + 1], large_rows, ctx->n, ctx->A, ctx->B, rowoff, colC, valC,
                    ctx->bitmap.as<unsigned>(), ctx->prefix.as<int>(), sb),
           (std::string("numeric large ") + dtype_name(ctx->dtype)).c_str());
    }
    {
        const int rb[4] = {NB_RANGE_S128, NB_RANGE_S512, NB_RANGE_L128, NB_RANGE_L512};
        const int rnsum[4] = {NSUM_SMALL, NSUM_SMALL, NSUM_LARGE, NSUM_LARGE};
        const int rnacc[4] = {128, RANGE_NACC_MAX, 128, RANGE_NACC_MAX};
        for (int i = 0; i < 4; ++i) {
            const int b = rb[i];
            if (num_bin[b] <= 0) continue;
            CU(stamp(ctx, 1, b), "event");
            CU(nk.range(lc, rnsum[i], rnacc[i], queue + no.off[b], num_bin[b], ctx->A, ctx->B, rlo, rowoff, colC, valC, wl),
               (std::string("numeric range ") + dtype_name(ctx->dtype)).c_str());
        }
    }
    return BHB200_SUCCESS;
}

// bhb200_stats of the numeric bins as they ran: the rows num_hash_last sends to NB_LARGE are counted there
void report_routed_num_bins(bhb200_stats &st, size_t value_size)
{
    for (int b = num_hash_last(value_size) + 1; b < NB_LARGE; ++b) {
        st.num_bin_rows[NB_LARGE] += st.num_bin_rows[b];
        st.num_bin_products[NB_LARGE] += st.num_bin_products[b];
        st.num_bin_nnzC[NB_LARGE] += st.num_bin_nnzC[b];
        st.num_bin_nnzA[NB_LARGE] += st.num_bin_nnzA[b];
        st.num_bin_rows[b] = st.num_bin_products[b] = st.num_bin_nnzC[b] = st.num_bin_nnzA[b] = 0;
    }
}

void finish_stats(bhb200_ctx *ctx)
{
    bhb200_stats &st = ctx->stats;
    st.kernel_launches = ctx->launches;
    const int64_t v = (int64_t)vsize(ctx->dtype);
    const int64_t m1 = (int64_t)ctx->m + 1;
    st.bytes_algorithmic = (m1 * 4 + (int64_t)ctx->nnzA * (4 + v)) + ((int64_t)ctx->nnzA * 8 + st.products * (4 + v)) +
                           (m1 * 4 + ctx->nnzC * (4 + v));
    // masked: + M read twice (validation, tables) + the staged rows written and read once (DESIGN.md 4.10)
    if (st.masked) st.bytes_algorithmic += (m1 * 4 + 2 * st.nnzM * 4) + 2 * ctx->nnzC * (4 + v);
    st.bytes_compulsory = (m1 * 4 + (int64_t)ctx->nnzA * (4 + v)) + (((int64_t)ctx->k + 1) * 4 + (int64_t)ctx->nnzB * (4 + v)) +
                          (m1 * 4 + ctx->nnzC * (4 + v));
    st.workspace_bytes = (int64_t)ctx->dev_bytes;
}

// per-call state common to bhb200_spgemm and bhb200_spgemm_numeric
int begin_call(bhb200_ctx *ctx)
{
    CU(cudaSetDevice(ctx->device), "cudaSetDevice");
    ctx->timing_valid = false;
    ctx->launches = 0;
    ctx->t_ran = false;
    return BHB200_SUCCESS;
}

int read_counters(bhb200_ctx *ctx, const char *what)
{
    CU(cudaMemcpyAsync(ctx->h_ctr, ctx->counters.p, sizeof(Counters), cudaMemcpyDeviceToHost, ctx->stream), "D2H counters");
    CU(cudaStreamSynchronize(ctx->stream), what);
    return BHB200_SUCCESS;
}

// multi-GPU set-up (bhb200_dist_setup_square): the broadcast of B's values overlapped what ran so far; the rest reads them
int wait_for_values(bhb200_ctx *ctx)
{
    if (ctx->wait_before_values) {
        CU(cudaStreamWaitEvent(ctx->stream, ctx->wait_before_values, 0), "wait for the broadcast of B's values");
        ctx->wait_before_values = nullptr;
    }
    return BHB200_SUCCESS;
}

int64_t spilled_bytes(const DevBuf &b)
{
    return b.host ? (int64_t)b.cap : 0;
}

// colC / valC for nnzC entries, spilled to host memory if the device cannot hold them (structure only: no valC)
int reserve_C(bhb200_ctx *ctx)
{
    const size_t vs = vsize(ctx->dtype);
    CU(ctx->colC.reserve_spillable((size_t)ctx->nnzC * 4 + 16, &ctx->dev_bytes, ctx->device_cap, nullptr), "alloc colC");
    ctx->stats.spill_bytes += spilled_bytes(ctx->colC);
    if (!vs) return BHB200_SUCCESS;
    CU(ctx->valC.reserve_spillable((size_t)ctx->nnzC * vs + 16, &ctx->dev_bytes, ctx->device_cap, nullptr), "alloc valC");
    ctx->stats.spill_bytes += spilled_bytes(ctx->valC);
    return BHB200_SUCCESS;
}

// Diagonal-pattern mode (stage_pattern.cuh).  Called after the stage-1 sync with the offset sets of
// A and B in ctx->h_sets.  Returns PATTERN_NOT_APPLICABLE if the operands do not qualify (the
// caller continues with the general path), otherwise the result of the whole product.
constexpr int PATTERN_NOT_APPLICABLE = 1;
constexpr int PATTERN_PLAN_STALE = 2;   // speculative run on the cached plan: the operands have other offsets now

// speculative: skip the offset-set detection and reuse the plan of the previous product on this context.
// k_pat_codes verifies EVERY entry against the plan's offset lists; a miss is reported with the counters,
// nothing has been written to C by then, and the caller redoes the product with the full detection.
int run_pattern(bhb200_ctx *ctx, const LaunchCtx &lc, bool same_ab, bool speculative)
{
    const size_t vs = vsize(ctx->dtype);
    if (speculative) {
        if (!ctx->plan.valid || ctx->plan.blob.empty() || ctx->plan.value_size != (int)vs) return PATTERN_NOT_APPLICABLE;
        if (same_ab && ctx->plan.DA != ctx->plan.DB) return PATTERN_NOT_APPLICABLE;   // (one code array would serve both lists)
        ctx->plan.reused = true;
    } else {
        const PatSet &sb = ctx->h_sets[1];
        const PatSet &sa = same_ab ? ctx->h_sets[1] : ctx->h_sets[0];
        if (sa.overflow || sb.overflow || sa.count > PAT_MAX_OFFS || sb.count > PAT_MAX_OFFS) return PATTERN_NOT_APPLICABLE;
        const int FILL = PAT_EMPTY;   // what the memset left in unused slots
        int offA[PAT_MAX_OFFS], offB[PAT_MAX_OFFS], nA = 0, nB = 0;
        for (int i = 0; i < PAT_SET_SLOTS; ++i) {
            if (sa.slot[i] != FILL && nA < PAT_MAX_OFFS) offA[nA++] = sa.slot[i];
            if (sb.slot[i] != FILL && nB < PAT_MAX_OFFS) offB[nB++] = sb.slot[i];
        }
        if (nA != sa.count || nB != sb.count) return PATTERN_NOT_APPLICABLE;
        if (!build_pattern_plan(offA, nA, offB, nB, (int)vs, ctx->plan)) return PATTERN_NOT_APPLICABLE;
    }
    const PatternPlan &plan = ctx->plan;
    cudaStream_t s = ctx->stream;
    bhb200_stats &st = ctx->stats;
    // multi-GPU row block of a square product: A's entries are a slice of B's arrays, so the codes of B serve A too
    // (one pass instead of two) as long as both operands index the same offset list
    const bool slice = !same_ab && ctx->slice_e0 >= 0 && ctx->slice_range.p && plan.DA == plan.DB;
    // workspace; any allocation failure falls back to the general path
    const size_t need_tab = plan.blob.size();
    const bool had_tables = ctx->pat_tables.cap >= need_tab && plan.reused;
    if (ctx->pat_tables.reserve(need_tab, &ctx->dev_bytes) != cudaSuccess ||
        ctx->pat_tb.reserve((size_t)ctx->nnzB + 16, &ctx->dev_bytes) != cudaSuccess ||
        (!same_ab && !slice && ctx->pat_ta.reserve((size_t)ctx->nnzA + 16, &ctx->dev_bytes) != cudaSuccess) ||
        ctx->pat_maskB.reserve(((size_t)ctx->k + 1) * 8, &ctx->dev_bytes) != cudaSuccess ||
        ctx->pat_fullbits.reserve(((size_t)ctx->k / 32 + 2) * 4, &ctx->dev_bytes) != cudaSuccess ||
        ctx->pat_outmask.reserve(((size_t)ctx->m + 1) * plan.nw * 4, &ctx->dev_bytes) != cudaSuccess) {
        cudaGetLastError();
        ctx->plan = PatternPlan();
        return PATTERN_NOT_APPLICABLE;
    }
    if (!had_tables)
        CU(cudaMemcpyAsync(ctx->pat_tables.p, plan.blob.data(), need_tab, cudaMemcpyHostToDevice, s), "H2D pattern tables");
    PatTables t = pattern_tables(plan, ctx->pat_tables.as<unsigned char>());
    t.fullbits = ctx->pat_fullbits.as<unsigned>();
    unsigned char *tb = ctx->pat_tb.as<unsigned char>();
    unsigned char *ta = same_ab ? tb : slice ? tb + ctx->slice_e0 : ctx->pat_ta.as<unsigned char>();
    int *rcnt = ctx->rc.as<int>();
    Counters *d_ctr = ctx->counters.as<Counters>();
    const long long spanA = (long long)plan.DA.back() - plan.DA.front() + 1, spanB = (long long)plan.DB.back() - plan.DB.front() + 1;
    // A first (when it is not B itself): its column range tells which rows of B this product reads -- in a
    // multi-GPU row block that is a fraction of B, and only those rows are coded and checked
    if (slice)
        CU(cudaMemcpyAsync(d_ctr->a_col_range, ctx->slice_range.p, 2 * sizeof(int), cudaMemcpyDeviceToDevice, s), "row range of the block");
    else if (!same_ab)
        CU(launch_pat_codes(lc, ctx->m, ctx->k, ctx->A.rowptr, ctx->A.col, t.offsA, t.nDA, spanA, ta, nullptr, &d_ctr->bad_A,
                            &d_ctr->pat_miss, 0ull, nullptr, d_ctr->a_col_range, nullptr),
           "pattern codes of A");
    CU(launch_pat_codes(lc, ctx->k, ctx->n, ctx->B.rowptr, ctx->B.col, t.offsB, t.nDB, spanB, tb, ctx->pat_maskB.as<unsigned long long>(),
                        &d_ctr->bad_B, &d_ctr->pat_miss, t.fullB, ctx->pat_fullbits.as<unsigned>(), nullptr,
                        same_ab ? nullptr : d_ctr->a_col_range),
       "pattern codes of B");
    CU(cudaEventRecord(ctx->ev[1], s), "event");
    // exact nnz(C_i) from the offset masks; also the per-row product counts (compute_nnzCt,
    // bhsparse_cuda.h:210-237) and their total -- the general path's stage-1 kernels are not run
    CU(launch_pat_symbolic(lc, ctx->m, ctx->A, ta, ctx->pat_maskB.as<unsigned long long>(), t, ctx->pat_outmask.as<unsigned>(), rcnt,
                           ctx->prod.as<int>(), d_ctr, ctx->k, (double)ctx->nnzA / (double)ctx->m, ctx->pat_fullbits.as<unsigned>()),
       "pattern symbolic");
    CU(cudaEventRecord(ctx->ev[2], s), "event");
    memset(ctx->ev_bin_used, 0, sizeof(ctx->ev_bin_used));
    CU(launch_scan(lc, ctx->m, ctx->A.rowptr, ctx->prod.as<int>(), rcnt, nullptr, 0u, nullptr,
                   ctx->rowoff64.as<int64_t>(), ctx->rowptr32.as<int>(), ctx->blocksums.as<long long>(), d_ctr),
       "row pointer scan");
    if (int rc = read_counters(ctx, "pattern symbolic / scan")) return rc;
    if (int rc = check_transposed(ctx, ctx->h_ctr->bad_T)) return rc;
    if (ctx->h_ctr->pat_miss) {
        ctx->plan = PatternPlan();   // (speculative or not: these lists do not describe the operands)
        return speculative ? PATTERN_PLAN_STALE : fail(ctx, BHB200_ERR_CUDA, "pattern mode: offset lists inconsistent with the operands");
    }
    if (ctx->h_ctr->bad_B) return fail(ctx, BHB200_ERR_INVALID, "rows of B must be sorted by column, duplicate-free and inside [0, n)");
    if (ctx->h_ctr->bad_A) return fail(ctx, BHB200_ERR_INVALID, "a column index of A is outside [0, k)");
    ctx->nnzC = (int64_t)ctx->h_ctr->nnzC;
    st.nnzC = ctx->nnzC;
    st.products = (int64_t)ctx->h_ctr->products;
    st.max_row_products = ctx->h_ctr->max_row_products;
    if (int rc = reserve_C(ctx)) return rc;
    CU(cudaEventRecord(ctx->ev[3], s), "event");
    CU(launch_pat_numeric(lc, ctx->dtype, ctx->m, ctx->A, ctx->B, ta, tb, t, ctx->pat_outmask.as<unsigned>(),
                          ctx->rowoff64.as<int64_t>(), ctx->colC.as<int>(), ctx->valC.p),
       "pattern numeric");
    CU(cudaEventRecord(ctx->ev[4], s), "event");
    st.pattern_mode = 1;
    st.pattern_nDA = t.nDA;
    st.pattern_nDB = t.nDB;
    st.pattern_nD = t.nD;
    st.pattern_acc_len = t.acc_len;
    finish_stats(ctx);
    ctx->last_pattern = true;
    ctx->last_tables = t;
    ctx->last_ta = ta;
    ctx->last_tb = tb;
    ctx->have_C = true;
    ctx->timing_valid = true;
    return BHB200_SUCCESS;
}


// ---- general mode: the stages of one bhb200_spgemm call ----

// what the stages hand on to each other
struct Product {
    LaunchCtx lc;
    Counters hc{};             // stage-1 counters, then those after the scan
    int G = 32;                // lanes per row group of the hash kernels
    BinOffsets so{}, no{};     // symbolic / numeric bin queues
    DirectPlan plan{};
    int cdf_shift = 0;
    WordLists wl{nullptr, nullptr, nullptr, nullptr, 0};
};

// transposed operands: built once for host copies, on every call for borrowed ones (the caller may have rewritten them)
int transpose_operands(bhb200_ctx *ctx, const LaunchCtx &lc)
{
    if (!ctx->t_pending && !(ctx->borrowed && (ctx->opA || ctx->opB))) return BHB200_SUCCESS;
    const int rc = run_transposes(ctx, lc);
    if (rc) return rc;
    CU(cudaEventRecord(ctx->ev[5], ctx->stream), "event");
    ctx->t_ran = true;
    return BHB200_SUCCESS;
}

// diagonal-pattern mode, speculative on the previous product's plan, then with the exact offset sets of A and B
// (read back by a sync of their own).  PATTERN_NOT_APPLICABLE: the general path follows, on zeroed counters.
int try_pattern(bhb200_ctx *ctx, const LaunchCtx &lc)
{
    cudaStream_t s = ctx->stream;
    Counters *d_ctr = ctx->counters.as<Counters>();
    ctx->last_pattern = false;
    const bool same_ab = ctx->A.rowptr == ctx->B.rowptr && ctx->A.col == ctx->B.col && ctx->m == ctx->k;
    if (!(ctx->pattern_enable && ctx->m > 0 && ctx->nnzA > 0 && ctx->nnzB > 0)) return PATTERN_NOT_APPLICABLE;
    if (ctx->pat_sets.reserve(2 * sizeof(PatSet), &ctx->dev_bytes) != cudaSuccess) {
        cudaGetLastError();
        return PATTERN_NOT_APPLICABLE;
    }
    int rc;
    if (ctx->plan.valid && ctx->pattern_speculate) {
        // the previous product on this context ran in pattern mode: reuse its plan without the detection
        // pass; every entry is verified against it (k_pat_codes), a miss brings us back here
        if ((rc = wait_for_values(ctx))) return rc;
        rc = run_pattern(ctx, lc, same_ab, true);
        if (rc != PATTERN_NOT_APPLICABLE && rc != PATTERN_PLAN_STALE) return rc;
        CU(cudaMemsetAsync(d_ctr, 0, CTR_ZERO_BYTES, s), "zero counters");
    }
    PatSet *sets = ctx->pat_sets.as<PatSet>();
    CU(cudaMemsetAsync(sets, 0x80, 2 * sizeof(PatSet), s), "init offset sets");   // slots = PAT_EMPTY
    CU(cudaMemsetAsync(&sets[0], 0, 8, s), "init offset sets");
    CU(cudaMemsetAsync(&sets[1], 0, 8, s), "init offset sets");
    CU(launch_offset_set(lc, ctx->k, ctx->B.rowptr, ctx->B.col, &sets[1]), "offset set of B");
    if (!same_ab) CU(launch_offset_set(lc, ctx->m, ctx->A.rowptr, ctx->A.col, &sets[0]), "offset set of A");
    CU(cudaMemcpyAsync(ctx->h_sets, ctx->pat_sets.p, 2 * sizeof(PatSet), cudaMemcpyDeviceToHost, s), "D2H offset sets");
    CU(cudaStreamSynchronize(s), "offset sets");
    if ((rc = wait_for_values(ctx))) return rc;
    rc = run_pattern(ctx, lc, same_ab, false);
    if (rc != PATTERN_NOT_APPLICABLE) return rc;
    ctx->plan = PatternPlan();   // these operands are not diagonal-structured: no speculation next time
    CU(cudaMemsetAsync(d_ctr, 0, CTR_ZERO_BYTES, s), "zero counters");
    return PATTERN_NOT_APPLICABLE;
}

// ---- stage 1: upper bound per row + symbolic bins ----
int stage1_counts(bhb200_ctx *ctx, Product &p)
{
    Counters *d_ctr = ctx->counters.as<Counters>();
    bhb200_stats &st = ctx->stats;
    CU(launch_b_row_ranges(p.lc, ctx->k, ctx->n, ctx->B, ctx->brange.as<int4>(), d_ctr), "B row ranges kernel");
    CU(launch_row_products(p.lc, ctx->m, ctx->k, ctx->nnzA, ctx->A, ctx->B, ctx->brange.as<int4>(), ctx->prod.as<int>(),
                           ctx->rc.as<int>(), ctx->rlo.as<int>(), ctx->rspan.as<int>(), d_ctr),
       "row products kernel");
    if (ctx->mask_set) CU(launch_mask_bins(p.lc, ctx->m, ctx->n, ctx->M, ctx->prod.as<int>(), d_ctr), "mask bins kernel");
    int rc = read_counters(ctx, "stage 1");
    if (rc) return rc;
    p.hc = *ctx->h_ctr;
    const Counters &hc = p.hc;
    if ((rc = check_transposed(ctx, hc.bad_T))) return rc;
    if (hc.bad_B) return fail(ctx, BHB200_ERR_INVALID, "rows of B must be sorted by column, duplicate-free and inside [0, n)");
    if (hc.bad_A) return fail(ctx, BHB200_ERR_INVALID, "a column index of A is outside [0, k)");
    if (hc.row_overflow) return fail(ctx, BHB200_ERR_OVERFLOW, "a row has more than INT32_MAX intermediate products");
    st.products = (int64_t)hc.products;
    st.max_row_products = hc.max_row_products;
    for (int b = 0; b < BHB200_NUM_SYM_BINS && b < MAX_BINS; ++b) st.sym_bin_rows[b] = hc.sym_bin[b];
    if ((rc = wait_for_values(ctx))) return rc;
    if (ctx->mask_set) {   // (the masked product bins its rows by the mask: stage_masked)
        if (hc.bad_M & MASK_BAD_ROWPTR)
            return fail(ctx, BHB200_ERR_INVALID, "mask: row pointers must rise from 0 to nnzM");
        if (hc.bad_M & MASK_BAD_COL) return fail(ctx, BHB200_ERR_INVALID, "mask: a column index is outside [0, n)");
        if (hc.bad_M) return fail(ctx, BHB200_ERR_INVALID, "mask: rows must be sorted by column and duplicate-free");
        return BHB200_SUCCESS;
    }
    // lanes per row group: follow the average length of the B rows actually referenced
    const double avg_b = ctx->nnzA > 0 ? (double)hc.products / (double)ctx->nnzA : 0.0;
    p.G = avg_b <= 10.0 ? 8 : 32;
    offsets_from_counts(hc.sym_bin, p.so);
    CU(launch_bin_scatter(p.lc, false, ctx->m, ctx->prod.as<int>(), ctx->rc.as<int>(), ctx->rspan.as<int>(), 0u, nullptr, p.so,
                          d_ctr, ctx->queue.as<int>()),
       "symbolic bin scatter");
    return BHB200_SUCCESS;
}

// ---- direct (single-pass) mode: sample the group-hash bins, plan (direct_plan.cu), staging buffer, column CDF ----
int choose_direct(bhb200_ctx *ctx, Product &p)
{
    Counters *d_ctr = ctx->counters.as<Counters>();
    bhb200_stats &st = ctx->stats;
    const size_t vs = vsize(ctx->dtype);
    const DirectSwitches sw{ctx->direct_mode != 0, ctx->direct_wide != 0, ctx->bucket_warp != 0, ctx->force_cap,
                            ctx->force_heavy};
    const unsigned sampled = direct_sample_bins(p.hc, sw);
    for (int b = SB_G128; b <= SB_G4096; ++b)
        if ((sampled >> b) & 1u)
            CU(launch_sym_hash(p.lc, b, p.G, ctx->queue.as<int>() + p.so.off[b], direct_sample_rows(p.hc.sym_bin[b]), ctx->A,
                               ctx->B, ctx->rc.as<int>(), DIRECT_SAMPLE_STRIDE, &d_ctr->sample_max[b], nullptr,
                               &d_ctr->sample_sum[b]),
               "symbolic sample");
    int rc = sampled ? read_counters(ctx, "direct-mode sampling") : BHB200_SUCCESS;
    if (rc) return rc;
    p.plan = plan_direct(*ctx->h_ctr, sw, vs);   // (*h_ctr: the stage-1 counters, sampled or not)
    DirectPlan &plan = p.plan;
    // the wide staging buffer must not crowd out C itself (at most `products` entries)
    // (only checked when the staging buffer has to grow: cudaMemGetInfo can take milliseconds)
    if (plan.mask() &&
        ((size_t)plan.ct_entries * 4 + 16 > ctx->ct_col.cap || (vs && (size_t)plan.ct_entries * vs + 16 > ctx->ct_val.cap))) {
        size_t free_b = 0, total_b = 0;
        cudaMemGetInfo(&free_b, &total_b);
        const double avail = (double)free_b + (double)ctx->ct_col.cap + (double)ctx->ct_val.cap + (double)ctx->colC.cap +
                             (double)ctx->valC.cap;
        const double need = ((double)plan.ct_entries + (double)st.products) * (4.0 + vs);
        if (need > 0.9 * avail) plan.drop_wide();
    }
    if (plan.mask()) {
        const size_t m1 = (size_t)ctx->m + 1;
        // the staging buffer (the reference's Ct) may spill to host memory like C itself
        if (ctx->ct_off.reserve(m1 * 8, &ctx->dev_bytes) != cudaSuccess ||
            ctx->retry_q.reserve(m1 * 4, &ctx->dev_bytes) != cudaSuccess ||
            ctx->ct_col.reserve_spillable((size_t)plan.ct_entries * 4 + 16, &ctx->dev_bytes, ctx->device_cap, nullptr) != cudaSuccess ||
            (vs && ctx->ct_val.reserve_spillable((size_t)plan.ct_entries * vs + 16, &ctx->dev_bytes, ctx->device_cap, nullptr) !=
                       cudaSuccess)) {
            cudaGetLastError();
            plan.drop_all();   // no room for the staging buffer: two-pass path for everything
        } else {
            st.spill_bytes += spilled_bytes(ctx->ct_col) + (vs ? spilled_bytes(ctx->ct_val) : 0);
        }
    }
    st.direct_ct_bytes = plan.ct_bytes();
    st.direct_bin_mask = (int64_t)plan.mask();
    CU(cudaEventRecord(ctx->ev[1], ctx->stream), "event");
    if (plan.uses_bucket() && (ctx->cdf_colcount.reserve(((size_t)ctx->k + 1) * 4, &ctx->dev_bytes) != cudaSuccess ||
                               ctx->cdf_hist.reserve((size_t)CDF_KNOTS * 8, &ctx->dev_bytes) != cudaSuccess ||
                               ctx->cdf_tab.reserve((size_t)(CDF_KNOTS + 1) * 4, &ctx->dev_bytes) != cudaSuccess)) {
        cudaGetLastError();
        plan.drop_bucket();
    }
    if (plan.uses_bucket() && ctx->cdf_valid) {
        p.cdf_shift = ctx->cdf_shift_cached;
    } else if (plan.uses_bucket()) {
        CU(launch_build_cdf(p.lc, ctx->m, ctx->k, ctx->n, ctx->nnzA, ctx->A, ctx->B, ctx->cdf_colcount.as<int>(),
                            ctx->cdf_hist.as<unsigned long long>(), ctx->cdf_tab.as<unsigned>(), &p.cdf_shift),
           "column CDF");
        ctx->cdf_valid = true;
        ctx->cdf_shift_cached = p.cdf_shift;
    }
    return BHB200_SUCCESS;
}

// the launches DirectPlan::launches lists for direct-mode bin b, in the value type of the operands
int run_direct_bin(bhb200_ctx *ctx, const Product &p, int b)
{
    const NumericKernels &nk = numeric_kernels(ctx->dtype);
    const DirectBin &db = p.plan.bin[b];
    Counters *d_ctr = ctx->counters.as<Counters>();
    const int *queue = ctx->queue.as<int>() + p.so.off[b];
    int *retry_queue = ctx->retry_q.as<int>() + p.so.off[b];
    const ColumnCdf cdf{ctx->cdf_tab.as<unsigned>(), p.cdf_shift};
    const DirectLaunches ls = p.plan.launches(b, p.G);
    for (int i = 0; i < ls.n; ++i) {
        const DirectLaunch &l = ls.at[i];
        DirectOut d{ctx->rc.as<int>(), ctx->ct_off.as<long long>(), ctx->ct_col.as<int>(), ctx->ct_val.p, db.base,
                    retry_queue, &d_ctr->retry_cnt[b]};
        // tight bins take every row of the queue; wide and heavy ones choose and stage rows by their product count
        if (db.mode != DirectMode::TIGHT) d.prod = ctx->prod.as<int>();
        if (db.mode == DirectMode::HEAVY) d.bump = &d_ctr->heavy_cursor;
        d.p_lo = l.p_lo;
        d.p_hi = l.p_hi;
        d.ct_stride = l.stride;
        switch (l.kernel) {
        case DirectKernel::DIRECT:
            CU(nk.direct(p.lc, l.cap, l.sg, queue, db.rows, ctx->A, ctx->B, d), "direct numeric");
            break;
        case DirectKernel::BUCKET:
            CU(nk.bucket(p.lc, l.cap, queue, db.rows, ctx->A, ctx->B, d, cdf), "bucket numeric");
            break;
        case DirectKernel::BUCKET3W:
            CU(nk.bucket3w(p.lc, l.cap, l.sg, queue, db.rows, ctx->A, ctx->B, d, cdf, l.stride), "warp bucket numeric");
            break;
        case DirectKernel::HEAVY:
            CU(nk.heavy2(p.lc, queue, db.rows, ctx->A, ctx->B, d, cdf, &d_ctr->heavy_cursor), "heavy rows");
            d.count_dev = d.retry_cnt;   // what k_num_bucket_heavy2 could not slice
            CU(nk.heavy(p.lc, retry_queue, db.rows, ctx->A, ctx->B, d, cdf, &d_ctr->heavy_cursor), "heavy rows");
            break;
        }
    }
    // rows that did not fit: ordinary symbolic pass, row count read on the device
    if (ls.retry)
        CU(launch_sym_hash(p.lc, b, p.G, retry_queue, db.rows, ctx->A, ctx->B, ctx->rc.as<int>(), 1, nullptr, &d_ctr->retry_cnt[b]),
           "symbolic retry");
    return BHB200_SUCCESS;
}

// ---- stage 2: symbolic, one launch per non-empty bin (direct-mode bins: the numeric kernel itself) ----
int stage2_symbolic(bhb200_ctx *ctx, Product &p)
{
    const Counters &hc = p.hc;
    const int *queue = ctx->queue.as<int>();
    int *rcnt = ctx->rc.as<int>();
    int rc;
    memset(ctx->ev_bin_used, 0, sizeof(ctx->ev_bin_used));
    if (hc.sym_bin[SB_ESC] > 0) CU(stamp(ctx, 0, SB_ESC), "event");
    CU(launch_sym_esc(p.lc, queue + p.so.off[SB_ESC], hc.sym_bin[SB_ESC], ctx->n, ctx->A, ctx->B, rcnt), "symbolic ESC");
    for (int b = SB_G128; b <= SB_LARGE; ++b) {
        const int rows = hc.sym_bin[b];
        if (p.plan.bin[b].mode != DirectMode::TWO_PASS) {
            CU(stamp(ctx, 0, b), "event");
            if ((rc = run_direct_bin(ctx, p, b))) return rc;
            ctx->stats.direct_rows += rows;
        } else if (b < SB_LARGE) {
            if (rows > 0) CU(stamp(ctx, 0, b), "event");
            CU(launch_sym_hash(p.lc, b, p.G, queue + p.so.off[b], rows, ctx->A, ctx->B, rcnt), "symbolic hash");
        } else if (rows > 0) {
            if ((rc = reserve_large_scratch(ctx, false))) return rc;
            CU(stamp(ctx, 0, SB_LARGE), "event");
            CU(launch_sym_large(p.lc, queue + p.so.off[SB_LARGE], rows, ctx->n, ctx->A, ctx->B, rcnt, ctx->bitmap.as<unsigned>(),
                                large_scratch_blocks(ctx->sm_count, ctx->n)),
               "symbolic large");
        }
    }
    if (hc.sym_bin[SB_RANGE_S] + hc.sym_bin[SB_RANGE_L] > 0) {
        if ((rc = reserve_word_lists(ctx, ctx->stats.products, p.wl))) return rc;
        int *rlo = ctx->rlo.as<int>();
        Counters *d_ctr = ctx->counters.as<Counters>();
        if (hc.sym_bin[SB_RANGE_S] > 0) {
            CU(stamp(ctx, 0, SB_RANGE_S), "event");
            CU(launch_sym_range(p.lc, NSUM_SMALL, queue + p.so.off[SB_RANGE_S], hc.sym_bin[SB_RANGE_S], ctx->A, ctx->B, rlo,
                                rcnt, d_ctr, p.wl),
               "symbolic range (small span)");
        }
        if (hc.sym_bin[SB_RANGE_L] > 0) {
            CU(stamp(ctx, 0, SB_RANGE_L), "event");
            CU(launch_sym_range(p.lc, NSUM_LARGE, queue + p.so.off[SB_RANGE_L], hc.sym_bin[SB_RANGE_L], ctx->A, ctx->B, rlo,
                                rcnt, d_ctr, p.wl),
               "symbolic range (large span)");
        }
    }
    CU(stamp(ctx, 0, MAX_BINS), "event");
    CU(cudaEventRecord(ctx->ev[2], ctx->stream), "event");
    return BHB200_SUCCESS;
}

// Row pointers of C, nnz(C) and the numeric bins read back (one host sync), C allocated exactly, rows scattered to
// the numeric bin queues.  spec_mask: symbolic bins whose rows were staged; those with ct_off >= 0 go to NB_COPY.
int scan_and_bin(bhb200_ctx *ctx, Product &p, unsigned spec_mask, const char *what)
{
    Counters *d_ctr = ctx->counters.as<Counters>();
    bhb200_stats &st = ctx->stats;
    CU(launch_scan(p.lc, ctx->m, ctx->A.rowptr, ctx->prod.as<int>(), ctx->rc.as<int>(), ctx->rspan.as<int>(), spec_mask,
                   ctx->ct_off.as<long long>(), ctx->rowoff64.as<int64_t>(), ctx->rowptr32.as<int>(),
                   ctx->blocksums.as<long long>(), d_ctr),
       "row pointer scan");
    int rc = read_counters(ctx, what);
    if (rc) return rc;
    p.hc = *ctx->h_ctr;
    const Counters &hc = p.hc;
    ctx->nnzC = (int64_t)hc.nnzC;
    st.nnzC = ctx->nnzC;
    for (int b = 0; b < BHB200_NUM_NUM_BINS && b < MAX_BINS; ++b) {
        st.num_bin_rows[b] = hc.num_bin[b];
        st.num_bin_products[b] = (int64_t)hc.num_bin_products[b];
        st.num_bin_nnzC[b] = (int64_t)hc.num_bin_nnzc[b];
        st.num_bin_nnzA[b] = (int64_t)hc.num_bin_nnza[b];
    }
    report_routed_num_bins(st, vsize(ctx->dtype));
    if ((rc = reserve_C(ctx))) return rc;
    offsets_from_counts(hc.num_bin, p.no);
    CU(launch_bin_scatter(p.lc, true, ctx->m, ctx->prod.as<int>(), ctx->rc.as<int>(), ctx->rspan.as<int>(), spec_mask,
                          ctx->ct_off.as<long long>(), p.no, d_ctr, ctx->queue.as<int>()),
       "numeric bin scatter");
    for (int b = 0; b < MAX_BINS; ++b) st.direct_retry_rows += hc.retry_cnt[b];   // (zero in a masked product)
    CU(cudaEventRecord(ctx->ev[3], ctx->stream), "event");
    const int copy_rows = hc.num_bin[NB_COPY];
    ctx->last_copy_rows = copy_rows;
    ctx->last_copy_off = p.no.off[NB_COPY];
    ctx->last_copy_avg = copy_rows > 0 ? (double)hc.num_bin_nnzc[NB_COPY] / (double)copy_rows : 0.0;
    return BHB200_SUCCESS;
}

// the k_copy_ct launch of the copy bin that scan_and_bin recorded
int run_copy_bin(bhb200_ctx *ctx, const LaunchCtx &lc)
{
    if (ctx->last_copy_rows <= 0) return BHB200_SUCCESS;
    CU(numeric_kernels(ctx->dtype)
           .copy_ct(lc, ctx->queue.as<int>() + ctx->last_copy_off, ctx->last_copy_rows, ctx->rowoff64.as<int64_t>(),
                    ctx->ct_off.as<long long>(), ctx->ct_col.as<int>(), ctx->ct_val.p, ctx->colC.as<int>(), ctx->valC.p,
                    ctx->last_copy_avg),
       "Ct -> C copy");
    return BHB200_SUCCESS;
}

// ---- stage 3: row pointers, numeric bins, exact allocation of C ----
int stage3_scan_alloc(bhb200_ctx *ctx, Product &p)
{
    return scan_and_bin(ctx, p, p.plan.mask(), "stage 2/3");
}

// ---- stage 4: numeric, C written in place ----
int stage4_numeric(bhb200_ctx *ctx, const Product &p)
{
    int rc = run_numeric_bins(ctx, p.lc, p.hc.num_bin, p.no, p.G, p.wl);
    if (rc) return rc;
    if (ctx->last_copy_rows > 0) CU(stamp(ctx, 1, NB_COPY), "event");
    if ((rc = run_copy_bin(ctx, p.lc))) return rc;
    CU(stamp(ctx, 1, MAX_BINS), "event");
    CU(cudaEventRecord(ctx->ev[4], ctx->stream), "event");
    return BHB200_SUCCESS;
}

// ---- masked product (stage_masked.cu): the masked kernels of every bin, rows staged at their mask offsets ----
// rows per masked kernel: the bins after mask_table_last run in MB_GLOBAL's kernel and are counted there
void routed_mask_bins(const int *bins, size_t value_size, int *rows)
{
    for (int b = 0; b < MB_COUNT; ++b) rows[b] = bins[b];
    for (int b = mask_table_last(value_size) + 1; b < MB_GLOBAL; ++b) {
        rows[MB_GLOBAL] += rows[b];
        rows[b] = 0;
    }
}

int run_mask_bins(bhb200_ctx *ctx, const LaunchCtx &lc)
{
    const MaskOut o{ctx->rc.as<int>(), ctx->ct_off.as<long long>(), ctx->ct_col.as<int>(), ctx->ct_val.p, ctx->mask_acc.p,
                    ctx->mask_hit.as<unsigned char>()};
    memset(ctx->ev_bin_used, 0, sizeof(ctx->ev_bin_used));
    int rows[MB_COUNT];
    routed_mask_bins(ctx->last_mask_bin, vsize(ctx->dtype), rows);
    const int last_table = mask_table_last(vsize(ctx->dtype));
    for (int b = MB_ZERO + 1; b < MB_COUNT; ++b) {
        if (rows[b] <= 0) continue;
        // (MB_GLOBAL starts at the first bin after last_table: the routed bins are its neighbours in the queue)
        const int first = b == MB_GLOBAL ? last_table + 1 : b;
        CU(stamp(ctx, 0, b), "event");
        CU(launch_mask_bin(lc, ctx->dtype, b, ctx->mask_q.as<int>() + ctx->last_mask_off.off[first], rows[b], ctx->A, ctx->B,
                           ctx->brange.as<int4>(), ctx->M, o),
           "masked kernel");
    }
    CU(stamp(ctx, 0, MAX_BINS), "event");
    return BHB200_SUCCESS;
}

// In place of the direct-mode choice and stages 2-4.  Host synchronisations: the one of stage 1 (which
// brought the masked bin sizes and the mask check) and the one after the scan (nnz(C)).
int stage_masked(bhb200_ctx *ctx, Product &p)
{
    Counters *d_ctr = ctx->counters.as<Counters>();
    bhb200_stats &st = ctx->stats;
    cudaStream_t s = ctx->stream;
    const size_t vs = vsize(ctx->dtype);
    const size_t m1 = (size_t)ctx->m + 1, nM = (size_t)ctx->M.nnz;
    const int *prod = ctx->prod.as<int>();
    st.masked = 1;
    st.nnzM = (int64_t)nM;
    int rows[MB_COUNT];
    routed_mask_bins(p.hc.mask_bin, vs, rows);
    for (int b = 0; b < BHB200_NUM_MASK_BINS && b < MB_COUNT; ++b) st.mask_bin_rows[b] = rows[b];
    // staging: exactly nnzM entries, row i at rowptrM[i]; it may spill to host memory like C
    CU(ctx->ct_off.reserve(m1 * 8, &ctx->dev_bytes), "alloc staging offsets");
    CU(ctx->mask_q.reserve(m1 * 4, &ctx->dev_bytes), "alloc masked bin queue");
    CU(ctx->ct_col.reserve_spillable(nM * 4 + 16, &ctx->dev_bytes, ctx->device_cap, nullptr), "alloc staging columns");
    if (vs) CU(ctx->ct_val.reserve_spillable(nM * vs + 16, &ctx->dev_bytes, ctx->device_cap, nullptr), "alloc staging values");
    st.spill_bytes += spilled_bytes(ctx->ct_col) + (vs ? spilled_bytes(ctx->ct_val) : 0);
    if (rows[MB_GLOBAL] > 0) {   // (structure only: hit flags, no accumulator)
        if (vs) CU(ctx->mask_acc.reserve(nM * vs + 16, &ctx->dev_bytes), "alloc masked accumulator");
        CU(ctx->mask_hit.reserve(nM + 16, &ctx->dev_bytes), "alloc masked hit flags");
    }
    memcpy(ctx->last_mask_bin, p.hc.mask_bin, sizeof(ctx->last_mask_bin));
    ctx->last_mask_off = BinOffsets{};
    for (int b = MB_ZERO + 1, acc = 0; b < MB_COUNT; ++b) {   // (MB_ZERO rows are not queued)
        ctx->last_mask_off.off[b] = acc;
        acc += p.hc.mask_bin[b];
    }
    CU(launch_mask_scatter(p.lc, ctx->m, ctx->M, prod, ctx->last_mask_off, d_ctr, ctx->mask_q.as<int>(), ctx->rc.as<int>(),
                           ctx->ct_off.as<long long>()),
       "masked bin scatter");
    CU(cudaEventRecord(ctx->ev[1], s), "event");
    int rc = run_mask_bins(ctx, p.lc);
    if (rc) return rc;
    CU(cudaEventRecord(ctx->ev[2], s), "event");
    // every row with a kernel has ct_off >= 0: with all bins marked direct, the scan and the bin scatter put it in NB_COPY
    if ((rc = scan_and_bin(ctx, p, ~0u, "masked product / scan"))) return rc;
    if ((rc = run_copy_bin(ctx, p.lc))) return rc;
    CU(cudaEventRecord(ctx->ev[4], s), "event");
    ctx->last_masked = true;
    return BHB200_SUCCESS;
}

}  // namespace

// ============================================================================
extern "C" {

const char *bhb200_version(void)
{
    return "bhsparse_b200 0.1.0 sm_100a";
}

int bhb200_create(bhb200_ctx **out, int device)
{
    if (!out) return BHB200_ERR_INVALID;
    *out = nullptr;
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev <= 0) {
        cudaGetLastError();
        return BHB200_ERR_NO_DEVICE;
    }
    if (device < 0 || device >= ndev) return BHB200_ERR_NO_DEVICE;
    bhb200_ctx *ctx = new (std::nothrow) bhb200_ctx();
    if (!ctx) return BHB200_ERR_ALLOC;
    ctx->device = device;
    memset(&ctx->stats, 0, sizeof(ctx->stats));
    cudaDeviceProp prop;
    if (cudaSetDevice(device) != cudaSuccess || cudaGetDeviceProperties(&prop, device) != cudaSuccess) {
        cudaGetLastError();
        delete ctx;
        return BHB200_ERR_NO_DEVICE;
    }
    if (prop.major < 10) {
        // the kernels are built for sm_100a only; there is no fallback path
        delete ctx;
        return BHB200_ERR_NO_DEVICE;
    }
    ctx->sm_count = prop.multiProcessorCount;
    snprintf(ctx->name, sizeof(ctx->name), "%s", prop.name);
    if (cudaStreamCreateWithFlags(&ctx->own_stream, cudaStreamNonBlocking) != cudaSuccess ||
        cudaHostAlloc((void **)&ctx->h_ctr, sizeof(Counters), cudaHostAllocDefault) != cudaSuccess) {
        cudaGetLastError();
        delete ctx;
        return BHB200_ERR_CUDA;
    }
    ctx->stream = ctx->own_stream;
    if (cudaHostAlloc((void **)&ctx->h_sets, 2 * sizeof(PatSet), cudaHostAllocDefault) != cudaSuccess) {
        cudaGetLastError();
        delete ctx;
        return BHB200_ERR_CUDA;
    }
    if (const char *pm = getenv("BHB200_PATTERN")) {
        ctx->pattern_enable = strcmp(pm, "off") != 0;
        ctx->pattern_speculate = strcmp(pm, "detect") != 0;   // "detect": run the offset-set pass on every call
    }
    if (const char *bw = getenv("BHB200_BUCKET_W")) ctx->bucket_warp = strcmp(bw, "off") != 0;
    if (const char *dm = getenv("BHB200_DIRECT")) {
        ctx->direct_mode = strcmp(dm, "off") != 0;
        ctx->direct_wide = strcmp(dm, "tight") != 0;
    }
    if (const char *rm = getenv("BHB200_RANGE")) {
        if (!strcmp(rm, "off")) ctx->max_span = -1;
        else if (!strcmp(rm, "small")) ctx->max_span = SPAN_SMALL;
        else if (!strcmp(rm, "all")) ctx->max_span = SPAN_LARGE;
    }
    if (const char *dc = getenv("BHB200_DEBUG_DEVICE_CAP")) ctx->device_cap = (size_t)atoll(dc);
    if (const char *fc = getenv("BHB200_DEBUG_FORCE_CAP")) ctx->force_cap = atoi(fc) > 0 ? atoi(fc) : 0;
    ctx->force_heavy = getenv("BHB200_DEBUG_FORCE_HEAVY") != nullptr;
    if (const char *wc = getenv("BHB200_DEBUG_WORDLIST_CAP")) ctx->wordlist_cap = atoll(wc) > 0 ? atoll(wc) : 0;
    for (auto &ev : ctx->ev) {
        if (cudaEventCreate(&ev) != cudaSuccess) {
            cudaGetLastError();
            delete ctx;
            return BHB200_ERR_CUDA;
        }
    }
    *out = ctx;
    return BHB200_SUCCESS;
}

int bhb200_free_mem(bhb200_ctx *ctx)
{
    if (!ctx) return BHB200_ERR_INVALID;
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    release_operands(ctx);
    ctx->plan = PatternPlan();
    ctx->last_pattern = false;
    DevBuf *bufs[] = {&ctx->pat_sets, &ctx->pat_ta, &ctx->pat_tb, &ctx->pat_maskB, &ctx->pat_outmask, &ctx->pat_tables, &ctx->pat_fullbits,
                      &ctx->cdf_colcount, &ctx->cdf_hist, &ctx->cdf_tab, &ctx->ct_off, &ctx->ct_col, &ctx->ct_val, &ctx->retry_q,
                      &ctx->brange, &ctx->rlo, &ctx->rspan, &ctx->wl_off, &ctx->wl_cnt, &ctx->wl_idx, &ctx->wl_bits,
                      &ctx->prod, &ctx->rc, &ctx->queue, &ctx->rowoff64, &ctx->rowptr32, &ctx->blocksums,
                      &ctx->counters, &ctx->bitmap, &ctx->prefix, &ctx->colC, &ctx->valC, &ctx->slice_range, &ctx->t_scratch,
                      &ctx->mask_rowptr, &ctx->mask_col, &ctx->mask_q, &ctx->mask_acc, &ctx->mask_hit};
    for (DevBuf *b : bufs) b->release(&ctx->dev_bytes);
    ctx->bitmap_zeroed_bytes = 0;
    cudaGetLastError();
    return BHB200_SUCCESS;
}

int bhb200_destroy(bhb200_ctx *ctx)
{
    if (!ctx) return BHB200_ERR_INVALID;
    bhb200_dist_finalize(ctx);
    bhb200_free_mem(ctx);
    for (auto &ev : ctx->ev)
        if (ev) cudaEventDestroy(ev);
    for (auto &row : ctx->ev_bin)
        for (auto &ev : row)
            if (ev) cudaEventDestroy(ev);
    if (ctx->own_stream) cudaStreamDestroy(ctx->own_stream);
    if (ctx->h_ctr) cudaFreeHost(ctx->h_ctr);
    if (ctx->h_sets) cudaFreeHost(ctx->h_sets);
    cudaGetLastError();
    delete ctx;
    return BHB200_SUCCESS;
}

int bhb200_set_stream(bhb200_ctx *ctx, void *cuda_stream)
{
    if (!ctx) return BHB200_ERR_INVALID;
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    ctx->stream = cuda_stream ? (cudaStream_t)cuda_stream : ctx->own_stream;
    return BHB200_SUCCESS;
}

const char *bhb200_last_error(const bhb200_ctx *ctx)
{
    return ctx ? ctx->err.c_str() : "null context";
}
const char *bhb200_device_name(const bhb200_ctx *ctx)
{
    return ctx ? ctx->name : "";
}
int bhb200_sm_count(const bhb200_ctx *ctx)
{
    return ctx ? ctx->sm_count : 0;
}

int bhb200_init_data_f64(bhb200_ctx *ctx, int m, int k, int n, int nnzA, const double *valA, const int32_t *rowptrA,
                         const int32_t *colA, int nnzB, const double *valB, const int32_t *rowptrB,
                         const int32_t *colB)
{
    return init_host(ctx, BHB200_DTYPE_F64, BHB200_OP_N, BHB200_OP_N, m, k, n, nnzA, valA, rowptrA, colA, nnzB, valB,
                     rowptrB, colB);
}
int bhb200_init_data_f32(bhb200_ctx *ctx, int m, int k, int n, int nnzA, const float *valA, const int32_t *rowptrA,
                         const int32_t *colA, int nnzB, const float *valB, const int32_t *rowptrB,
                         const int32_t *colB)
{
    return init_host(ctx, BHB200_DTYPE_F32, BHB200_OP_N, BHB200_OP_N, m, k, n, nnzA, valA, rowptrA, colA, nnzB, valB,
                     rowptrB, colB);
}
int bhb200_init_data_op_f64(bhb200_ctx *ctx, int opA, int opB, int m, int k, int n, int nnzA, const double *valA,
                            const int32_t *rowptrA, const int32_t *colA, int nnzB, const double *valB, const int32_t *rowptrB,
                            const int32_t *colB)
{
    return init_host(ctx, BHB200_DTYPE_F64, opA, opB, m, k, n, nnzA, valA, rowptrA, colA, nnzB, valB, rowptrB, colB);
}
int bhb200_init_data_op_f32(bhb200_ctx *ctx, int opA, int opB, int m, int k, int n, int nnzA, const float *valA,
                            const int32_t *rowptrA, const int32_t *colA, int nnzB, const float *valB, const int32_t *rowptrB,
                            const int32_t *colB)
{
    return init_host(ctx, BHB200_DTYPE_F32, opA, opB, m, k, n, nnzA, valA, rowptrA, colA, nnzB, valB, rowptrB, colB);
}

int bhb200_init_data_op_c64(bhb200_ctx *ctx, int opA, int opB, int m, int k, int n, int nnzA, const float *valA,
                            const int32_t *rowptrA, const int32_t *colA, int nnzB, const float *valB, const int32_t *rowptrB,
                            const int32_t *colB)
{
    return init_host(ctx, BHB200_DTYPE_C64, opA, opB, m, k, n, nnzA, valA, rowptrA, colA, nnzB, valB, rowptrB, colB);
}

int bhb200_init_data_op_c128(bhb200_ctx *ctx, int opA, int opB, int m, int k, int n, int nnzA, const double *valA,
                             const int32_t *rowptrA, const int32_t *colA, int nnzB, const double *valB,
                             const int32_t *rowptrB, const int32_t *colB)
{
    return init_host(ctx, BHB200_DTYPE_C128, opA, opB, m, k, n, nnzA, valA, rowptrA, colA, nnzB, valB, rowptrB, colB);
}

int bhb200_init_data_structure(bhb200_ctx *ctx, int opA, int opB, int m, int k, int n, int nnzA, const int32_t *rowptrA,
                               const int32_t *colA, int nnzB, const int32_t *rowptrB, const int32_t *colB)
{
    return init_host(ctx, BHB200_DTYPE_NONE, opA, opB, m, k, n, nnzA, nullptr, rowptrA, colA, nnzB, nullptr, rowptrB, colB);
}

int bhb200_init_data_device(bhb200_ctx *ctx, int dtype, int m, int k, int n, int nnzA, const void *valA,
                            const int32_t *rowptrA, const int32_t *colA, int nnzB, const void *valB,
                            const int32_t *rowptrB, const int32_t *colB)
{
    return bhb200_init_data_device_op(ctx, dtype, BHB200_OP_N, BHB200_OP_N, m, k, n, nnzA, valA, rowptrA, colA, nnzB, valB,
                                      rowptrB, colB);
}

int bhb200_init_data_device_op(bhb200_ctx *ctx, int dtype, int opA, int opB, int m, int k, int n, int nnzA,
                               const void *valA, const int32_t *rowptrA, const int32_t *colA, int nnzB, const void *valB,
                               const int32_t *rowptrB, const int32_t *colB)
{
    if (!ctx) return BHB200_ERR_INVALID;
    if (dtype != BHB200_DTYPE_F32 && dtype != BHB200_DTYPE_F64 && dtype != BHB200_DTYPE_NONE && dtype != BHB200_DTYPE_C64 &&
        dtype != BHB200_DTYPE_C128)
        return fail(ctx, BHB200_ERR_INVALID, "bad dtype");
    int rc = check_ops(ctx, dtype, opA, opB);
    if (rc) return rc;
    rc = check_dims(ctx, dtype, m, k, n, nnzA, nnzB, valA, rowptrA, colA, valB, rowptrB, colB);
    if (rc) return rc;
    // (checked here, before any kernel reads them: the kernels load complex64 values as 8-byte words)
    if (dtype == BHB200_DTYPE_C64 && (((uintptr_t)valA | (uintptr_t)valB) & 7u))
        return fail(ctx, BHB200_ERR_INVALID, "complex64 value arrays must be 8-byte aligned");
    // (complex128: 128-bit loads)
    if (dtype == BHB200_DTYPE_C128 && (((uintptr_t)valA | (uintptr_t)valB) & 15u))
        return fail(ctx, BHB200_ERR_INVALID, "complex128 value arrays must be 16-byte aligned");
    CU(cudaSetDevice(ctx->device), "cudaSetDevice");
    release_operands(ctx);
    const bool values = dtype != BHB200_DTYPE_NONE;   // (structure only: the caller's value pointers are never read)
    ctx->As = Csr{rowptrA, colA, values ? valA : nullptr};
    ctx->Bs = Csr{rowptrB, colB, values ? valB : nullptr};
    ctx->dtype = dtype;
    ctx->m = m;
    ctx->k = k;
    ctx->n = n;
    ctx->nnzA = nnzA;
    ctx->nnzB = nnzB;
    ctx->opA = opA;
    ctx->opB = opB;
    rc = set_effective(ctx);
    if (rc) return rc;
    ctx->have_data = true;
    ctx->cdf_valid = false;   // new operands: the column CDF of the previous ones is not reused
    ctx->borrowed = true;
    return BHB200_SUCCESS;
}

static int set_mask_any(bhb200_ctx *ctx, bool device, int nnzM, const int32_t *rowptrM, const int32_t *colM)
{
    if (!ctx) return BHB200_ERR_INVALID;
    if (!ctx->have_data) return fail(ctx, BHB200_ERR_INVALID, "mask: set_mask needs operands (initData) for its shape");
    if (ctx->dist) return fail(ctx, BHB200_ERR_INVALID, "mask: masked products are not available on a multi-GPU context");
    if (nnzM < 0 || !rowptrM || (nnzM > 0 && !colM)) return fail(ctx, BHB200_ERR_INVALID, "mask: null array or negative nnzM");
    ctx->mask_changed = true;
    drop_mask(ctx);
    if (device) {
        ctx->M = MaskCsr{rowptrM, colM, nnzM};
    } else {
        CU(cudaSetDevice(ctx->device), "cudaSetDevice");
        const size_t m1 = (size_t)ctx->m + 1;
        CU(ctx->mask_rowptr.reserve(m1 * 4, &ctx->dev_bytes), "alloc mask row pointers");
        CU(ctx->mask_col.reserve((size_t)nnzM * 4 + 4, &ctx->dev_bytes), "alloc mask columns");
        // (the stream may still be reading the previous mask: the copies are ordered after it)
        CU(cudaMemcpyAsync(ctx->mask_rowptr.p, rowptrM, m1 * 4, cudaMemcpyHostToDevice, ctx->stream), "H2D mask row pointers");
        if (nnzM > 0)
            CU(cudaMemcpyAsync(ctx->mask_col.p, colM, (size_t)nnzM * 4, cudaMemcpyHostToDevice, ctx->stream), "H2D mask columns");
        CU(cudaStreamSynchronize(ctx->stream), "H2D mask");
        ctx->M = MaskCsr{ctx->mask_rowptr.as<int>(), ctx->mask_col.as<int>(), nnzM};
    }
    ctx->mask_set = true;
    return BHB200_SUCCESS;
}

int bhb200_set_mask(bhb200_ctx *ctx, int nnzM, const int32_t *rowptrM, const int32_t *colM)
{
    return set_mask_any(ctx, false, nnzM, rowptrM, colM);
}

int bhb200_set_mask_device(bhb200_ctx *ctx, int nnzM, const int32_t *rowptrM, const int32_t *colM)
{
    return set_mask_any(ctx, true, nnzM, rowptrM, colM);
}

int bhb200_clear_mask(bhb200_ctx *ctx)
{
    if (!ctx) return BHB200_ERR_INVALID;
    if (ctx->mask_set) ctx->mask_changed = true;
    drop_mask(ctx);
    return BHB200_SUCCESS;
}

int bhb200_warmup(bhb200_ctx *ctx)
{
    if (!ctx || !ctx->have_data) return fail(ctx, BHB200_ERR_INVALID, "warmup before initData");
    CU(cudaSetDevice(ctx->device), "cudaSetDevice");
    if (ctx->m == 0) return BHB200_SUCCESS;
    int rc = reserve_workspace(ctx);
    if (rc) return rc;
    LaunchCtx lc{ctx->stream, ctx->sm_count, &ctx->launches, ctx->max_span};
    if (ctx->t_pending) {   // (its column check is reported by the next spgemm)
        rc = run_transposes(ctx, lc);
        if (rc) return rc;
    }
    CU(launch_b_row_ranges(lc, ctx->k, ctx->n, ctx->B, ctx->brange.as<int4>(), ctx->counters.as<Counters>()), "B row ranges kernel");
    // like the reference's warm-up (bhsparse.h:341-363: compute_nnzCt only) this must leave an existing
    // result intact: k_row_products rewrites rc[] and the counters, so it is skipped once C exists
    if (ctx->have_C) return BHB200_SUCCESS;
    CU(cudaMemsetAsync(ctx->counters.p, 0, CTR_ZERO_BYTES, ctx->stream), "zero counters");
    CU(launch_row_products(lc, ctx->m, ctx->k, ctx->nnzA, ctx->A, ctx->B, ctx->brange.as<int4>(), ctx->prod.as<int>(),
                           ctx->rc.as<int>(), ctx->rlo.as<int>(), ctx->rspan.as<int>(), ctx->counters.as<Counters>()),
       "row products kernel");
    return BHB200_SUCCESS;
}

int bhb200_spgemm(bhb200_ctx *ctx)
{
    if (!ctx || !ctx->have_data) return fail(ctx, BHB200_ERR_INVALID, "spgemm before initData");
    int rc = begin_call(ctx);
    if (rc) return rc;
    ctx->have_C = false;
    ctx->reuse_bins_valid = false;
    ctx->last_masked = false;
    ctx->mask_changed = false;
    bhb200_stats &st = ctx->stats;
    memset(&st, 0, sizeof(st));
    st.transposed_ops = (ctx->opA ? 1 : 0) | (ctx->opB ? 2 : 0);
    st.m = ctx->m;
    st.k = ctx->k;
    st.n = ctx->n;
    st.nnzA = ctx->nnzA;
    st.nnzB = ctx->nnzB;
    st.dtype = ctx->dtype;
    if ((rc = reserve_workspace(ctx))) return rc;
    Product p{LaunchCtx{ctx->stream, ctx->sm_count, &ctx->launches, ctx->max_span}};
    CU(cudaEventRecord(ctx->ev[0], ctx->stream), "event");
    if ((rc = transpose_operands(ctx, p.lc))) return rc;
    CU(cudaMemsetAsync(ctx->counters.p, 0, CTR_ZERO_BYTES, ctx->stream), "zero counters");
    if (ctx->mask_set) {
        ctx->last_pattern = false;   // (a masked product never takes the diagonal-pattern mode)
        if ((rc = stage1_counts(ctx, p))) return rc;
        if ((rc = stage_masked(ctx, p))) return rc;
    } else {
        rc = try_pattern(ctx, p.lc);
        if (rc != PATTERN_NOT_APPLICABLE) return rc;
        if ((rc = stage1_counts(ctx, p))) return rc;
        if ((rc = choose_direct(ctx, p))) return rc;
        if ((rc = stage2_symbolic(ctx, p))) return rc;
        if ((rc = stage3_scan_alloc(ctx, p))) return rc;
        if ((rc = stage4_numeric(ctx, p))) return rc;
    }
    finish_stats(ctx);
    ctx->last_G = p.G;
    ctx->last_wl = p.wl;
    ctx->have_C = true;
    ctx->timing_valid = true;
    return BHB200_SUCCESS;
}

// Values of C for new values of A and/or B with the SAME sparsity patterns as the last
// bhb200_spgemm: stage 1, the symbolic pass, the scan and the allocation are skipped; the
// numeric kernels run on the known row sizes and overwrite C in place (SURVEY.md 8f-3: AMG
// set-up phases multiply the same patterns many times).
int bhb200_spgemm_numeric(bhb200_ctx *ctx)
{
    if (!ctx || !ctx->have_data || !ctx->have_C)
        return fail(ctx, BHB200_ERR_INVALID, "spgemm_numeric needs a completed spgemm on the same operands");
    if (ctx->mask_changed) return fail(ctx, BHB200_ERR_INVALID, "spgemm_numeric: the mask changed since the last spgemm");
    if (ctx->dtype == BHB200_DTYPE_NONE) return refuse_structure(ctx, "spgemm_numeric");
    int rc = begin_call(ctx);
    if (rc) return rc;
    bhb200_stats &st = ctx->stats;
    cudaStream_t s = ctx->stream;
    LaunchCtx lc{s, ctx->sm_count, &ctx->launches, ctx->max_span};
    Counters *d_ctr = ctx->counters.as<Counters>();
    CU(cudaEventRecord(ctx->ev[0], s), "event");
    if (ctx->borrowed && (ctx->opA || ctx->opB)) {
        // borrowed operands are rewritten in place by the caller: their values again through perm
        if ((rc = run_regathers(ctx, lc))) return rc;
        CU(cudaEventRecord(ctx->ev[5], s), "event");
        ctx->t_ran = true;
    }
    CU(cudaEventRecord(ctx->ev[1], s), "event");
    if (ctx->last_masked) {
        // masked product: the masked kernels on the cached bin queues, then the copy of the cached copy bin
        if ((rc = run_mask_bins(ctx, lc))) return rc;
        CU(cudaEventRecord(ctx->ev[2], s), "event");
        CU(cudaEventRecord(ctx->ev[3], s), "event");
        if ((rc = run_copy_bin(ctx, lc))) return rc;
        CU(cudaEventRecord(ctx->ev[4], s), "event");
        st.kernel_launches = ctx->launches;
        ctx->timing_valid = true;
        return BHB200_SUCCESS;
    }
    CU(cudaEventRecord(ctx->ev[2], s), "event");
    memset(ctx->ev_bin_used, 0, sizeof(ctx->ev_bin_used));
    if (ctx->last_pattern) {
        // pattern mode: codes, masks, tables and row pointers are still valid -- one kernel
        CU(cudaEventRecord(ctx->ev[3], s), "event");
        CU(launch_pat_numeric(lc, ctx->dtype, ctx->m, ctx->A, ctx->B, ctx->last_ta, ctx->last_tb, ctx->last_tables,
                              ctx->pat_outmask.as<unsigned>(), ctx->rowoff64.as<int64_t>(), ctx->colC.as<int>(), ctx->valC.p),
           "pattern numeric");
        CU(cudaEventRecord(ctx->ev[4], s), "event");
        st.kernel_launches = ctx->launches;
        ctx->timing_valid = true;
        return BHB200_SUCCESS;
    }
    if (!ctx->reuse_bins_valid) {
        // numeric bins of ALL rows (the direct-mode rows of the full product sit in the copy bin)
        CU(cudaMemsetAsync(d_ctr, 0, CTR_ZERO_BYTES, s), "zero counters");
        CU(launch_scan(lc, ctx->m, ctx->A.rowptr, ctx->prod.as<int>(), ctx->rc.as<int>(), ctx->rspan.as<int>(), 0u, nullptr,
                       ctx->rowoff64.as<int64_t>(), ctx->rowptr32.as<int>(), ctx->blocksums.as<long long>(), d_ctr),
           "row pointer scan");
        if ((rc = read_counters(ctx, "numeric-only binning"))) return rc;
        if ((int64_t)ctx->h_ctr->nnzC != ctx->nnzC) return fail(ctx, BHB200_ERR_INVALID, "structure of C changed");
        memcpy(ctx->reuse_num_bin, ctx->h_ctr->num_bin, sizeof(ctx->reuse_num_bin));
        BinOffsets no0;
        offsets_from_counts(ctx->reuse_num_bin, no0);
        CU(launch_bin_scatter(lc, true, ctx->m, ctx->prod.as<int>(), ctx->rc.as<int>(), ctx->rspan.as<int>(), 0u, nullptr, no0,
                              d_ctr, ctx->queue.as<int>()),
           "numeric bin scatter");
        ctx->reuse_bins_valid = true;
    }
    BinOffsets no;
    offsets_from_counts(ctx->reuse_num_bin, no);
    CU(cudaEventRecord(ctx->ev[3], s), "event");
    if ((rc = run_numeric_bins(ctx, lc, ctx->reuse_num_bin, no, ctx->last_G, ctx->last_wl))) return rc;
    CU(stamp(ctx, 1, MAX_BINS), "event");
    CU(cudaEventRecord(ctx->ev[4], s), "event");
    for (int b = 0; b < BHB200_NUM_NUM_BINS && b < MAX_BINS; ++b) st.num_bin_rows[b] = ctx->reuse_num_bin[b];
    report_routed_num_bins(st, vsize(ctx->dtype));
    st.kernel_launches = ctx->launches;
    st.direct_rows = 0;
    st.direct_retry_rows = 0;
    ctx->timing_valid = true;
    return BHB200_SUCCESS;
}

static int update_values_any(bhb200_ctx *ctx, int dtype, const void *valA, const void *valB)
{
    if (!ctx || !ctx->have_data) return fail(ctx, BHB200_ERR_INVALID, "update_values before initData");
    if (ctx->dtype == BHB200_DTYPE_NONE) return refuse_structure(ctx, "update_values");
    if (ctx->borrowed) return fail(ctx, BHB200_ERR_INVALID, "operands are caller-owned device arrays: update them in place");
    if (dtype != ctx->dtype) return fail(ctx, BHB200_ERR_INVALID, "value type differs from initData");
    CU(cudaSetDevice(ctx->device), "cudaSetDevice");
    const size_t vs = vsize(ctx->dtype);
    if (ctx->aliased && (valA || valB) && valA != valB) {
        // A and B share one device copy (same host arrays in initData) but now get different values:
        // give B its own copy (patterns unchanged, so every cached structure stays valid)
        const int rb = ctx->opB ? ctx->n : ctx->k;   // rows of B as stored
        CU(ctx->b_rowptr.reserve((size_t)(rb + 1) * 4, &ctx->dev_bytes), "alloc rowptrB");
        CU(ctx->b_col.reserve((size_t)ctx->nnzB * 4 + 4, &ctx->dev_bytes), "alloc colB");
        CU(ctx->b_val.reserve((size_t)ctx->nnzB * vs + 8, &ctx->dev_bytes), "alloc valB");
        CU(cudaMemcpyAsync(ctx->b_rowptr.p, ctx->a_rowptr.p, (size_t)(rb + 1) * 4, cudaMemcpyDeviceToDevice, ctx->stream), "D2D rowptrB");
        if (ctx->nnzB > 0) {
            CU(cudaMemcpyAsync(ctx->b_col.p, ctx->a_col.p, (size_t)ctx->nnzB * 4, cudaMemcpyDeviceToDevice, ctx->stream), "D2D colB");
            CU(cudaMemcpyAsync(ctx->b_val.p, ctx->a_val.p, (size_t)ctx->nnzB * vs, cudaMemcpyDeviceToDevice, ctx->stream), "D2D valB");
        }
        ctx->Bs = Csr{ctx->b_rowptr.as<int>(), ctx->b_col.as<int>(), ctx->b_val.p};
        if (!ctx->opB) {
            ctx->B = ctx->Bs;
        } else if (ctx->t_shared) {
            // op(B) shared op(A)'s transposed copy: B gets its own (same structure and permutation)
            const bool pending = ctx->t_pending;
            ctx->t_shared = false;
            int rc = set_effective(ctx);
            if (rc) return rc;
            ctx->t_pending = pending;
            cudaStream_t s = ctx->stream;
            if (!pending)
                CU(cudaMemcpyAsync(ctx->bt_rowptr.p, ctx->at_rowptr.p, (size_t)(ctx->k + 1) * 4, cudaMemcpyDeviceToDevice, s),
                   "D2D rowptr of B^T");
            if (!pending && ctx->nnzB > 0) {
                CU(cudaMemcpyAsync(ctx->bt_col.p, ctx->at_col.p, (size_t)ctx->nnzB * 4, cudaMemcpyDeviceToDevice, s), "D2D col of B^T");
                CU(cudaMemcpyAsync(ctx->bt_perm.p, ctx->at_perm.p, (size_t)ctx->nnzB * 4, cudaMemcpyDeviceToDevice, s), "D2D perm of B^T");
            }
        }
        ctx->aliased = false;
    }
    if (valA && ctx->nnzA > 0)
        CU(cudaMemcpyAsync(ctx->a_val.p, valA, (size_t)ctx->nnzA * vs, cudaMemcpyHostToDevice, ctx->stream), "H2D valA");
    if (valB && ctx->nnzB > 0 && !ctx->aliased)   // (still aliased: valB == valA, the shared copy has just been written)
        CU(cudaMemcpyAsync(ctx->b_val.p, valB, (size_t)ctx->nnzB * vs, cudaMemcpyHostToDevice, ctx->stream), "H2D valB");
    if (!ctx->t_pending && (ctx->opA || ctx->opB)) {
        // transposed operands: their values through the permutation of the transposition
        LaunchCtx lc{ctx->stream, ctx->sm_count, &ctx->launches, ctx->max_span};
        int rc = run_regathers(ctx, lc);
        if (rc) return rc;
    }
    CU(cudaStreamSynchronize(ctx->stream), "update values");
    return BHB200_SUCCESS;
}

int bhb200_update_values_f64(bhb200_ctx *ctx, const double *valA, const double *valB)
{
    return update_values_any(ctx, BHB200_DTYPE_F64, valA, valB);
}

int bhb200_update_values_f32(bhb200_ctx *ctx, const float *valA, const float *valB)
{
    return update_values_any(ctx, BHB200_DTYPE_F32, valA, valB);
}

int bhb200_update_values_c64(bhb200_ctx *ctx, const float *valA, const float *valB)
{
    return update_values_any(ctx, BHB200_DTYPE_C64, valA, valB);
}

int bhb200_update_values_c128(bhb200_ctx *ctx, const double *valA, const double *valB)
{
    return update_values_any(ctx, BHB200_DTYPE_C128, valA, valB);
}

int bhb200_set_profiling(bhb200_ctx *ctx, int enabled)
{
    if (!ctx) return BHB200_ERR_INVALID;
    ctx->profiling = enabled != 0;
    return BHB200_SUCCESS;
}

int bhb200_synchronize(bhb200_ctx *ctx)
{
    if (!ctx) return BHB200_ERR_INVALID;
    CU(cudaSetDevice(ctx->device), "cudaSetDevice");
    CU(cudaStreamSynchronize(ctx->stream), "synchronize");
    return BHB200_SUCCESS;
}

int bhb200_get_operands_device(const bhb200_ctx *ctx, int32_t *dims, const int32_t **rowptrA, const int32_t **colA,
                               const void **valA, const int32_t **rowptrB, const int32_t **colB, const void **valB)
{
    if (!ctx || !ctx->have_data) return BHB200_ERR_INVALID;
    if (dims) {
        dims[0] = ctx->m;
        dims[1] = ctx->k;
        dims[2] = ctx->n;
        dims[3] = ctx->nnzA;
        dims[4] = ctx->nnzB;
        dims[5] = ctx->dtype;
    }
    if (rowptrA) *rowptrA = ctx->A.rowptr;
    if (colA) *colA = ctx->A.col;
    if (valA) *valA = ctx->A.val;
    if (rowptrB) *rowptrB = ctx->B.rowptr;
    if (colB) *colB = ctx->B.col;
    if (valB) *valB = ctx->B.val;
    return BHB200_SUCCESS;
}

int bhb200_pattern_plan_probe(const int32_t *offsA, int nA, const int32_t *offsB, int nB, int value_size, int32_t *info,
                              uint8_t *position, int32_t *offsC)
{
    // host-only: the plan the diagonal-pattern mode would build for these offset sets (tests, tools)
    if (!offsA || !offsB || !info || (value_size != 4 && value_size != 8 && value_size != 16)) return BHB200_ERR_INVALID;
    PatternPlan plan;
    if (!build_pattern_plan(offsA, nA, offsB, nB, value_size, plan)) {
        info[0] = 0;
        return BHB200_SUCCESS;
    }
    const int nb = pattern_lane_group(value_size);
    const unsigned char *mphys = plan.blob.data() + plan.off_mphys;
    int cost = 0, groups = 0;
    for (int ja = 0; ja < nA; ++ja)
        for (int j0 = 0; j0 < nB; j0 += nb) {
            int cnt[32] = {0}, mx = 0;
            for (int jb = j0; jb < nB && jb < j0 + nb; ++jb) mx = std::max(mx, ++cnt[mphys[(size_t)ja * nB + jb] % nb]);
            cost += mx;
            ++groups;
        }
    info[0] = 1;
    info[1] = plan.nD;
    info[2] = plan.nw;
    info[3] = plan.acc_len;
    info[4] = cost;      // shared-memory wavefronts of one accumulate pass over all (A offset, lane group) pairs
    info[5] = groups;    // ... and its conflict-free minimum
    if (position) memcpy(position, mphys, (size_t)nA * nB);
    if (offsC) memcpy(offsC, plan.blob.data() + plan.off_dcol, (size_t)plan.nD * 4);
    return BHB200_SUCCESS;
}

int bhb200_operands_aliased(const bhb200_ctx *ctx)
{
    return (ctx && ctx->have_data && ctx->aliased) ? 1 : 0;
}

int64_t bhb200_get_nnzC(const bhb200_ctx *ctx)
{
    return (ctx && ctx->have_C) ? ctx->nnzC : -1;
}

// dtype BHB200_DTYPE_NONE: the structure of C (any product), valC is null
static int get_C_any(bhb200_ctx *ctx, int dtype, int32_t *rowptrC, int32_t *colC, void *valC)
{
    if (!ctx || !ctx->have_C) return fail(ctx, BHB200_ERR_INVALID, "get_C before spgemm");
    if (dtype != BHB200_DTYPE_NONE && ctx->dtype == BHB200_DTYPE_NONE) return refuse_structure(ctx, "get_C");
    if (dtype != BHB200_DTYPE_NONE && dtype != ctx->dtype) return fail(ctx, BHB200_ERR_INVALID, "get_C dtype differs from initData dtype");
    if (ctx->nnzC > 0x7fffffffLL) return fail(ctx, BHB200_ERR_OVERFLOW, "nnz(C) exceeds INT32_MAX; use the int64 row pointers");
    CU(cudaSetDevice(ctx->device), "cudaSetDevice");
    cudaStream_t s = ctx->stream;
    if (rowptrC)
        CU(cudaMemcpyAsync(rowptrC, ctx->rowptr32.p, ((size_t)ctx->m + 1) * 4, cudaMemcpyDeviceToHost, s), "D2H rowptrC");
    if (colC && ctx->nnzC > 0)
        CU(cudaMemcpyAsync(colC, ctx->colC.p, (size_t)ctx->nnzC * 4, cudaMemcpyDefault, s), "D2H colC");
    if (valC && ctx->nnzC > 0)
        CU(cudaMemcpyAsync(valC, ctx->valC.p, (size_t)ctx->nnzC * vsize(dtype), cudaMemcpyDefault, s), "D2H valC");
    CU(cudaStreamSynchronize(s), "D2H C");
    return BHB200_SUCCESS;
}

int bhb200_get_C_f64(bhb200_ctx *ctx, int32_t *rowptrC, int32_t *colC, double *valC)
{
    return get_C_any(ctx, BHB200_DTYPE_F64, rowptrC, colC, valC);
}
int bhb200_get_C_f32(bhb200_ctx *ctx, int32_t *rowptrC, int32_t *colC, float *valC)
{
    return get_C_any(ctx, BHB200_DTYPE_F32, rowptrC, colC, valC);
}
int bhb200_get_C_c64(bhb200_ctx *ctx, int32_t *rowptrC, int32_t *colC, float *valC)
{
    return get_C_any(ctx, BHB200_DTYPE_C64, rowptrC, colC, valC);
}

int bhb200_get_C_c128(bhb200_ctx *ctx, int32_t *rowptrC, int32_t *colC, double *valC)
{
    return get_C_any(ctx, BHB200_DTYPE_C128, rowptrC, colC, valC);
}

int bhb200_get_C_structure(bhb200_ctx *ctx, int32_t *rowptrC, int32_t *colC)
{
    return get_C_any(ctx, BHB200_DTYPE_NONE, rowptrC, colC, nullptr);
}

int bhb200_get_C_range(bhb200_ctx *ctx, int64_t first, int64_t count, int32_t *colC, void *valC)
{
    if (!ctx || !ctx->have_C) return fail(ctx, BHB200_ERR_INVALID, "get_C_range before spgemm");
    if (first < 0 || count < 0 || first + count > ctx->nnzC) return fail(ctx, BHB200_ERR_INVALID, "range outside [0, nnzC]");
    if (valC && ctx->dtype == BHB200_DTYPE_NONE) return refuse_structure(ctx, "get_C_range with valC");
    CU(cudaSetDevice(ctx->device), "cudaSetDevice");
    cudaStream_t s = ctx->stream;
    const size_t vs = vsize(ctx->dtype);
    if (colC && count > 0)
        CU(cudaMemcpyAsync(colC, ctx->colC.as<int>() + first, (size_t)count * 4, cudaMemcpyDefault, s), "D2H colC range");
    if (valC && count > 0)
        CU(cudaMemcpyAsync(valC, (const char *)ctx->valC.p + (size_t)first * vs, (size_t)count * vs, cudaMemcpyDefault, s),
           "D2H valC range");
    CU(cudaStreamSynchronize(s), "D2H C range");
    return BHB200_SUCCESS;
}

int bhb200_get_rowptrC_i64(bhb200_ctx *ctx, int64_t *rowptrC64)
{
    if (!ctx || !ctx->have_C) return fail(ctx, BHB200_ERR_INVALID, "get_rowptrC before spgemm");
    if (!rowptrC64) return fail(ctx, BHB200_ERR_INVALID, "null pointer");
    CU(cudaSetDevice(ctx->device), "cudaSetDevice");
    CU(cudaMemcpyAsync(rowptrC64, ctx->rowoff64.p, ((size_t)ctx->m + 1) * 8, cudaMemcpyDeviceToHost, ctx->stream), "D2H rowptrC64");
    CU(cudaStreamSynchronize(ctx->stream), "D2H rowptrC64");
    return BHB200_SUCCESS;
}

int bhb200_get_C_device(bhb200_ctx *ctx, const int32_t **rowptr32, const int64_t **rowptr64, const int32_t **colC,
                        const void **valC)
{
    if (!ctx || !ctx->have_C) return fail(ctx, BHB200_ERR_INVALID, "get_C_device before spgemm");
    if (rowptr32) *rowptr32 = ctx->nnzC > 0x7fffffffLL ? nullptr : ctx->rowptr32.as<int32_t>();
    if (rowptr64) *rowptr64 = ctx->rowoff64.as<int64_t>();
    if (colC) *colC = ctx->colC.as<int32_t>();
    if (valC) *valC = ctx->dtype == BHB200_DTYPE_NONE ? nullptr : ctx->valC.p;
    return BHB200_SUCCESS;
}

int bhb200_copy_C_to_device(bhb200_ctx *ctx, int64_t *rowptrC64, int32_t *colC, void *valC)
{
    if (!ctx || !ctx->have_C) return fail(ctx, BHB200_ERR_INVALID, "copy_C_to_device before spgemm");
    if (valC && ctx->dtype == BHB200_DTYPE_NONE) return refuse_structure(ctx, "copy_C_to_device with valC");
    CU(cudaSetDevice(ctx->device), "cudaSetDevice");
    cudaStream_t s = ctx->stream;
    if (rowptrC64)
        CU(cudaMemcpyAsync(rowptrC64, ctx->rowoff64.p, ((size_t)ctx->m + 1) * 8, cudaMemcpyDeviceToDevice, s), "D2D rowptrC64");
    if (colC && ctx->nnzC > 0)
        CU(cudaMemcpyAsync(colC, ctx->colC.p, (size_t)ctx->nnzC * 4, cudaMemcpyDefault, s), "D2D colC");
    if (valC && ctx->nnzC > 0)
        CU(cudaMemcpyAsync(valC, ctx->valC.p, (size_t)ctx->nnzC * vsize(ctx->dtype), cudaMemcpyDefault, s), "D2D valC");
    CU(cudaStreamSynchronize(s), "D2D C");
    return BHB200_SUCCESS;
}

int bhb200_get_row_products(bhb200_ctx *ctx, int32_t *row_products)
{
    if (!ctx || !ctx->have_data || !ctx->prod.p) return fail(ctx, BHB200_ERR_INVALID, "no row products yet");
    if (!row_products) return fail(ctx, BHB200_ERR_INVALID, "null pointer");
    CU(cudaSetDevice(ctx->device), "cudaSetDevice");
    if (ctx->m > 0)
        CU(cudaMemcpyAsync(row_products, ctx->prod.p, (size_t)ctx->m * 4, cudaMemcpyDeviceToHost, ctx->stream), "D2H row products");
    CU(cudaStreamSynchronize(ctx->stream), "D2H row products");
    return BHB200_SUCCESS;
}

int bhb200_get_stats(const bhb200_ctx *cctx, bhb200_stats *out)
{
    bhb200_ctx *ctx = const_cast<bhb200_ctx *>(cctx);
    if (!ctx || !out) return BHB200_ERR_INVALID;
    if (ctx->timing_valid) {
        CU(cudaSetDevice(ctx->device), "cudaSetDevice");
        CU(cudaEventSynchronize(ctx->ev[4]), "event sync");
        bhb200_stats &st = ctx->stats;
        cudaEventElapsedTime(&st.ms_total, ctx->ev[0], ctx->ev[4]);
        cudaEventElapsedTime(&st.ms_count, ctx->ev[0], ctx->ev[1]);
        st.ms_transpose = 0.f;
        if (ctx->t_ran) {   // (ms_count then starts after the transposition)
            cudaEventElapsedTime(&st.ms_transpose, ctx->ev[0], ctx->ev[5]);
            cudaEventElapsedTime(&st.ms_count, ctx->ev[5], ctx->ev[1]);
        }
        cudaEventElapsedTime(&st.ms_symbolic, ctx->ev[1], ctx->ev[2]);
        cudaEventElapsedTime(&st.ms_scan, ctx->ev[2], ctx->ev[3]);
        cudaEventElapsedTime(&st.ms_numeric, ctx->ev[3], ctx->ev[4]);
        if (ctx->profiling) {
            // time of bin b = next stamped event - its own (launches are serial on one stream)
            for (int ph = 0; ph < 2; ++ph) {
                float *dst = ph ? st.ms_num_bin : st.ms_sym_bin;
                for (int b = 0; b < MAX_BINS; ++b) {
                    dst[b] = 0.f;
                    if (!ctx->ev_bin_used[ph][b]) continue;
                    int nx = b + 1;
                    while (nx < MAX_BINS && !ctx->ev_bin_used[ph][nx]) ++nx;
                    if (ctx->ev_bin_used[ph][nx]) cudaEventElapsedTime(&dst[b], ctx->ev_bin[ph][b], ctx->ev_bin[ph][nx]);
                }
            }
        }
    }
    *out = ctx->stats;
    return BHB200_SUCCESS;
}

}  // extern "C"
