// dist_nccl.cu -- multi-GPU SpGEMM behind the C-ABI (bhb200_dist_*), NCCL called directly.
//
// One process per GPU, one context per process.  Scheme (SURVEY.md 8e; the reference is
// single-GPU, bhsparse_cuda.h:100-101):
//   * rows of A are split into contiguous blocks on the prefix sum of the per-row intermediate
//     products (computed on the root's device with the stage-1 kernels, never on the host);
//   * B is broadcast from the root with ncclBroadcast -- the small partition record first, then
//     rowptr and col on the context's stream, then val on a second stream, so that the value
//     transfer overlaps stage 1 (compute_nnzCt + binning need only rowptr and col); the compute
//     stream waits for the values right before the first kernel that reads them;
//   * every rank runs the single-GPU pipeline on its block (A's block is a slice of its copy of B
//     for C = B*B, with rebased row pointers);
//   * per step one ncclAllGather of the int64 nnz(C) of every rank, consumed by a device kernel that
//     turns the local row pointers into global ones -- no host round trip per step.
// NCCL is opened with dlopen at the first bhb200_dist_* call: the single-GPU library has no link
// dependency on it.
#include <algorithm>
#include "context.h"

#include <dlfcn.h>

#include <cstring>

using namespace bhb;

namespace {

// the few NCCL declarations used (ABI-stable since NCCL 2.0; nccl.h is not needed to build)
typedef struct ncclComm *ncclComm_t;
struct ncclUniqueId {
    char internal[128];
};
static_assert(sizeof(ncclUniqueId) == BHB200_DIST_ID_BYTES, "NCCL unique id size");
enum { ncclInt8 = 0, ncclInt32 = 2, ncclInt64 = 4, ncclFloat32 = 7, ncclFloat64 = 8 };

struct NcclApi {
    void *handle = nullptr;
    int (*GetUniqueId)(ncclUniqueId *) = nullptr;
    int (*CommInitRank)(ncclComm_t *, int, ncclUniqueId, int) = nullptr;
    int (*CommDestroy)(ncclComm_t) = nullptr;
    int (*Broadcast)(const void *, void *, size_t, int, int, ncclComm_t, cudaStream_t) = nullptr;
    int (*AllGather)(const void *, void *, size_t, int, ncclComm_t, cudaStream_t) = nullptr;
    const char *(*GetErrorString)(int) = nullptr;
    bool ok = false;
};

NcclApi &nccl()
{
    static NcclApi api;
    if (api.handle || api.ok) return api;
    // a copy already loaded into the process (e.g. the one bundled with PyTorch) is reused
    const char *names[] = {"libnccl.so.2", "libnccl.so"};
    for (const char *nm : names) {
        api.handle = dlopen(nm, RTLD_NOW | RTLD_GLOBAL);
        if (api.handle) break;
    }
    if (!api.handle) return api;
    auto sym = [&](const char *n) { return dlsym(api.handle, n); };
    api.GetUniqueId = (int (*)(ncclUniqueId *))sym("ncclGetUniqueId");
    api.CommInitRank = (int (*)(ncclComm_t *, int, ncclUniqueId, int))sym("ncclCommInitRank");
    api.CommDestroy = (int (*)(ncclComm_t))sym("ncclCommDestroy");
    api.Broadcast = (int (*)(const void *, void *, size_t, int, int, ncclComm_t, cudaStream_t))sym("ncclBroadcast");
    api.AllGather = (int (*)(const void *, void *, size_t, int, ncclComm_t, cudaStream_t))sym("ncclAllGather");
    api.GetErrorString = (const char *(*)(int))sym("ncclGetErrorString");
    api.ok = api.GetUniqueId && api.CommInitRank && api.CommDestroy && api.Broadcast && api.AllGather;
    return api;
}

constexpr int MAX_RANKS = 64;
// partition record, broadcast from the root: bounds[0..nranks], nnz_bounds[0..nranks], products
struct Partition {
    long long bounds[MAX_RANKS + 1];
    long long nnz_bounds[MAX_RANKS + 1];
    long long products;
    long long block_products[MAX_RANKS];
};

}  // namespace

namespace bhb {
struct DistState {
    ncclComm_t comm = nullptr;
    int rank = 0, nranks = 1;
    cudaStream_t val_stream = nullptr;
    cudaEvent_t ev_ready = nullptr, ev_val = nullptr, ev_t0 = nullptr, ev_t1 = nullptr;
    DevBuf d_part, d_counts, d_global_rowptr, d_cprefix;
    Partition part{};
    Partition *h_part = nullptr;   // pinned
    long long *h_counts = nullptr;   // pinned [nranks]
    int n = 0;
    bool have_layout = false;
    float broadcast_ms = 0.f;
};
}  // namespace bhb

namespace {

int dfail(bhb200_ctx *c, int code, const char *what, const char *detail = nullptr)
{
    if (c) {
        c->err = what;
        if (detail) {
            c->err += ": ";
            c->err += detail;
        }
    }
    return code;
}

#define DCU(call, what)                                                                                   \
    do {                                                                                                  \
        cudaError_t e__ = (call);                                                                         \
        if (e__ != cudaSuccess) {                                                                         \
            cudaGetLastError();                                                                           \
            return dfail(ctx, e__ == cudaErrorMemoryAllocation ? BHB200_ERR_ALLOC : BHB200_ERR_CUDA, what, \
                         cudaGetErrorString(e__));                                                        \
        }                                                                                                 \
    } while (0)
#define DNC(call, what)                                                                                  \
    do {                                                                                                 \
        int r__ = (call);                                                                                \
        if (r__ != 0) return dfail(ctx, BHB200_ERR_CUDA, what, nccl().GetErrorString ? nccl().GetErrorString(r__) : "NCCL error"); \
    } while (0)

// Cost of a row for the partition: its intermediate products, times 11/8 beyond 12288 products -- rows that
// leave the on-chip tables are sliced through global memory (k_num_bucket_heavy2) and cost about that much more per
// product (R-MAT 24 / 8 blocks: 24.4 products/ns in block 0, which holds the hub rows, 26.1 in block 3;
// profiles/r02_notes.md section 5.  The factor was 2.5 for the first heavy-row kernel; with 1.25 block 0 was still the slowest by 3 % at 8 GPUs).  dist.py::row_cost is the same function.
constexpr int COST_HEAVY_ROW = 12288;
__global__ void k_row_cost(const int n, const int *__restrict__ prod, int *__restrict__ cost)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const long long p = prod[i];
    const long long c = p > COST_HEAVY_ROW ? (p * 11) / 8 : p;
    cost[i] = (int)(c > 0x7fffffffLL ? 0x7fffffffLL : c);
}

// first row i with cprefix[i] >= total * r / nranks  (cprefix = exclusive scan of the per-row costs, n+1 entries;
// prefix = the same for the products, for the report)
__global__ void k_partition_bounds(const int n, const int nranks, const int64_t *__restrict__ cprefix,
                                   const int64_t *__restrict__ prefix, const int *__restrict__ rowptr,
                                   Partition *__restrict__ out)
{
    const int r = threadIdx.x;
    if (r > nranks) return;
    const long long total = cprefix[n];
    long long b;
    if (r == 0) b = 0;
    else if (r == nranks) b = n;
    else {
        const long long target = (long long)(((__int128)total * r) / nranks);
        int lo = 0, hi = n;   // first index with prefix[idx] >= target
        while (lo < hi) {
            const int mid = lo + ((hi - lo) >> 1);
            if (cprefix[mid] < target) lo = mid + 1;
            else hi = mid;
        }
        b = lo;
    }
    out->bounds[r] = b;
    out->nnz_bounds[r] = rowptr[b];
    if (r == 0) out->products = prefix[n];
    __syncthreads();
    if (r < nranks) out->block_products[r] = prefix[out->bounds[r + 1]] - prefix[out->bounds[r]];
}

__global__ void k_rebase_rowptr(const int rows, const int *__restrict__ rowptr, const int first, int *__restrict__ out)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i <= rows) out[i] = rowptr[first + i] - rowptr[first];
}

// {max, INT_MAX - min} over the columns of a block of A and the block's own rows [r0, r1): the rows of B a
// diagonal-pattern product has to code when A's entries are a slice of B's (context.cu::run_pattern)
__global__ void k_slice_range(const long long nnz, const int *__restrict__ col, const int r0, const int r1, int *__restrict__ out)
{
    int mx = r1 - 1, mn = r0;
    for (long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x; j < nnz; j += (long long)gridDim.x * blockDim.x) {
        const int c = col[j];
        mx = max(mx, c);
        mn = min(mn, c);
    }
    mx = __reduce_max_sync(0xffffffffu, mx);
    mn = __reduce_min_sync(0xffffffffu, mn);
    if ((threadIdx.x & 31) == 0) {
        atomicMax(&out[0], mx);
        atomicMax(&out[1], 0x7fffffff - mn);
    }
}

__global__ void k_put_count(const Counters *__restrict__ ctr, long long *__restrict__ slot)
{
    *slot = (long long)ctr->nnzC;
}

__global__ void k_global_rowptr(const int rows, const int rank, const long long *__restrict__ counts,
                                const int64_t *__restrict__ local, int64_t *__restrict__ global)
{
    long long off = 0;
    for (int r = 0; r < rank; ++r) off += counts[r];
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i <= rows) global[i] = local[i] + off;
}

}  // namespace

extern "C" {

int bhb200_dist_unique_id(void *id)
{
    if (!id) return BHB200_ERR_INVALID;
    if (!nccl().ok) return BHB200_ERR_NO_DEVICE;
    return nccl().GetUniqueId((ncclUniqueId *)id) == 0 ? BHB200_SUCCESS : BHB200_ERR_CUDA;
}

int bhb200_dist_init(bhb200_ctx *ctx, int rank, int nranks, const void *id)
{
    if (!ctx || !id || nranks < 1 || nranks > MAX_RANKS || rank < 0 || rank >= nranks)
        return dfail(ctx, BHB200_ERR_INVALID, "bad rank / communicator size");
    if (!nccl().ok) return dfail(ctx, BHB200_ERR_NO_DEVICE, "libnccl.so.2 could not be loaded");
    if (ctx->dist) return dfail(ctx, BHB200_ERR_INVALID, "communicator already initialised");
    DCU(cudaSetDevice(ctx->device), "cudaSetDevice");
    DistState *d = new (std::nothrow) DistState();
    if (!d) return dfail(ctx, BHB200_ERR_ALLOC, "host allocation");
    d->rank = rank;
    d->nranks = nranks;
    ncclUniqueId uid;
    memcpy(&uid, id, sizeof(uid));
    int r = nccl().CommInitRank(&d->comm, nranks, uid, rank);
    if (r != 0) {
        delete d;
        return dfail(ctx, BHB200_ERR_CUDA, "ncclCommInitRank", nccl().GetErrorString ? nccl().GetErrorString(r) : nullptr);
    }
    ctx->dist = d;
    DCU(cudaStreamCreateWithFlags(&d->val_stream, cudaStreamNonBlocking), "stream");
    DCU(cudaEventCreateWithFlags(&d->ev_ready, cudaEventDisableTiming), "event");
    DCU(cudaEventCreateWithFlags(&d->ev_val, cudaEventDisableTiming), "event");
    DCU(cudaEventCreate(&d->ev_t0), "event");
    DCU(cudaEventCreate(&d->ev_t1), "event");
    DCU(cudaHostAlloc((void **)&d->h_part, sizeof(Partition), cudaHostAllocDefault), "pinned");
    DCU(cudaHostAlloc((void **)&d->h_counts, sizeof(long long) * MAX_RANKS, cudaHostAllocDefault), "pinned");
    DCU(d->d_part.reserve(sizeof(Partition), &ctx->dev_bytes), "alloc partition record");
    DCU(d->d_counts.reserve(sizeof(long long) * (MAX_RANKS + 1), &ctx->dev_bytes), "alloc counts");
    // NCCL builds its rings / NVLS trees at the first collective of each kind on a communicator (hundreds
    // of milliseconds): do that here, on both streams that will carry traffic, not inside the first set-up
    long long *counts = d->d_counts.as<long long>();
    DCU(cudaMemsetAsync(counts, 0, sizeof(long long) * (MAX_RANKS + 1), ctx->stream), "zero counts");
    DNC(nccl().AllGather(counts + MAX_RANKS, counts, 1, ncclInt64, d->comm, ctx->stream), "ncclAllGather(warm-up)");
    DNC(nccl().Broadcast(d->d_part.p, d->d_part.p, sizeof(Partition), ncclInt8, 0, d->comm, ctx->stream), "ncclBroadcast(warm-up)");
    DCU(cudaStreamSynchronize(ctx->stream), "NCCL warm-up");
    DNC(nccl().Broadcast(d->d_part.p, d->d_part.p, sizeof(Partition), ncclInt8, 0, d->comm, d->val_stream), "ncclBroadcast(warm-up)");
    DCU(cudaStreamSynchronize(d->val_stream), "NCCL warm-up");
    return BHB200_SUCCESS;
}

int bhb200_dist_finalize(bhb200_ctx *ctx)
{
    if (!ctx || !ctx->dist) return BHB200_SUCCESS;
    DistState *d = ctx->dist;
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    if (d->val_stream) cudaStreamSynchronize(d->val_stream);
    if (d->comm) nccl().CommDestroy(d->comm);
    d->d_part.release(&ctx->dev_bytes);
    d->d_counts.release(&ctx->dev_bytes);
    d->d_global_rowptr.release(&ctx->dev_bytes);
    d->d_cprefix.release(&ctx->dev_bytes);
    if (d->val_stream) cudaStreamDestroy(d->val_stream);
    for (cudaEvent_t e : {d->ev_ready, d->ev_val, d->ev_t0, d->ev_t1})
        if (e) cudaEventDestroy(e);
    if (d->h_part) cudaFreeHost(d->h_part);
    if (d->h_counts) cudaFreeHost(d->h_counts);
    cudaGetLastError();
    delete d;
    ctx->dist = nullptr;
    ctx->wait_before_values = nullptr;
    return BHB200_SUCCESS;
}

int bhb200_dist_setup_square(bhb200_ctx *ctx, int root, int dtype, int n, int64_t nnz, const int32_t *rowptr,
                             const int32_t *col, const void *val)
{
    if (!ctx || !ctx->dist) return dfail(ctx, BHB200_ERR_INVALID, "bhb200_dist_init first");
    DistState *d = ctx->dist;
    if (root < 0 || root >= d->nranks || n < 0 || nnz < 0 || nnz > 0x7fffffffLL) return dfail(ctx, BHB200_ERR_INVALID, "bad argument");
    if (dtype != BHB200_DTYPE_F32 && dtype != BHB200_DTYPE_F64 && dtype != BHB200_DTYPE_C64 && dtype != BHB200_DTYPE_C128)
        return dfail(ctx, BHB200_ERR_INVALID, "bad dtype");
    const bool is_root = d->rank == root;
    if (is_root && (!rowptr || (nnz > 0 && (!col || !val)))) return dfail(ctx, BHB200_ERR_INVALID, "null B on the root");
    DCU(cudaSetDevice(ctx->device), "cudaSetDevice");
    cudaStream_t s = ctx->stream;
    const size_t vs = dispatch_value_type(dtype, [](auto v) { return value_bytes<decltype(v)>; });
    if (is_root && vs == 8 && ((uintptr_t)val & 7u)) return dfail(ctx, BHB200_ERR_INVALID, "valB is not 8-byte aligned");
    if (is_root && vs == 16 && ((uintptr_t)val & 15u)) return dfail(ctx, BHB200_ERR_INVALID, "valB is not 16-byte aligned");
    // forget the previous operands (library-owned buffers are reused by reserve())
    ctx->have_data = false;
    ctx->have_C = false;
    ctx->last_pattern = false;
    ctx->reuse_bins_valid = false;
    ctx->mask_set = false;   // (a mask set before bhb200_dist_init: masked products are single-GPU)
    ctx->M = MaskCsr{nullptr, nullptr, 0};
    ctx->last_masked = false;
    d->have_layout = false;
    Partition *dp = d->d_part.as<Partition>();
    DCU(cudaEventRecord(d->ev_t0, s), "event");

    // ---- root: per-row products of B*B, their prefix, the block boundaries (all on the device) ----
    if (is_root) {
        ctx->m = ctx->k = ctx->n = n;
        ctx->nnzA = ctx->nnzB = (int)nnz;
        ctx->dtype = dtype;
        ctx->A = ctx->B = Csr{rowptr, col, val};
        int rc = BHB200_SUCCESS;
        {
            const size_t m1 = (size_t)n + 1;
            DCU(ctx->prod.reserve(m1 * 4, &ctx->dev_bytes), "alloc");
            DCU(ctx->rc.reserve(m1 * 4, &ctx->dev_bytes), "alloc");
            DCU(ctx->rlo.reserve(m1 * 4, &ctx->dev_bytes), "alloc");
            DCU(ctx->rspan.reserve(m1 * 4, &ctx->dev_bytes), "alloc");
            DCU(ctx->rowoff64.reserve(m1 * 8, &ctx->dev_bytes), "alloc");
            DCU(ctx->rowptr32.reserve(m1 * 4, &ctx->dev_bytes), "alloc");
            DCU(ctx->blocksums.reserve((scan_blocksum_count(n) + 1) * 8, &ctx->dev_bytes), "alloc");
            DCU(ctx->counters.reserve(sizeof(Counters), &ctx->dev_bytes), "alloc");
            DCU(ctx->brange.reserve(m1 * 16, &ctx->dev_bytes), "alloc");
        }
        (void)rc;
        LaunchCtx lc{s, ctx->sm_count, &ctx->launches, ctx->max_span};
        Counters *d_ctr = ctx->counters.as<Counters>();
        DCU(cudaMemsetAsync(d_ctr, 0, sizeof(Counters), s), "zero counters");
        DCU(launch_b_row_ranges(lc, n, n, ctx->B, ctx->brange.as<int4>(), d_ctr), "B row ranges");
        DCU(launch_row_products(lc, n, n, (int)nnz, ctx->A, ctx->B, ctx->brange.as<int4>(), ctx->prod.as<int>(),
                                ctx->rc.as<int>(), ctx->rlo.as<int>(), ctx->rspan.as<int>(), d_ctr),
            "row products");
        // exclusive scan of the products (the scan kernels take the per-row counts as `rc`)
        DCU(launch_scan(lc, n, rowptr, ctx->prod.as<int>(), ctx->prod.as<int>(), nullptr, 0u, nullptr,
                        ctx->rowoff64.as<int64_t>(), ctx->rowptr32.as<int>(), ctx->blocksums.as<long long>(), d_ctr),
            "product prefix");
        // ... and of the per-row costs (rc[] and a second prefix buffer are free at this point)
        DCU(d->d_cprefix.reserve(((size_t)n + 1) * 8, &ctx->dev_bytes), "alloc");
        k_row_cost<<<(n + 255) / 256, 256, 0, s>>>(n, ctx->prod.as<int>(), ctx->rc.as<int>());
        DCU(cudaGetLastError(), "row cost kernel");
        DCU(launch_scan(lc, n, rowptr, ctx->prod.as<int>(), ctx->rc.as<int>(), nullptr, 0u, nullptr, d->d_cprefix.as<int64_t>(),
                        ctx->rowptr32.as<int>(), ctx->blocksums.as<long long>(), d_ctr),
            "cost prefix");
        k_partition_bounds<<<1, MAX_RANKS + 1, 0, s>>>(n, d->nranks, d->d_cprefix.as<int64_t>(), ctx->rowoff64.as<int64_t>(), rowptr, dp);
        DCU(cudaGetLastError(), "partition kernel");
    }
    // ---- broadcast: partition record, rowptr, col on the compute stream; val on its own stream ----
    DNC(nccl().Broadcast(dp, dp, sizeof(Partition), ncclInt8, root, d->comm, s), "ncclBroadcast(partition)");
    DCU(cudaMemcpyAsync(d->h_part, dp, sizeof(Partition), cudaMemcpyDeviceToHost, s), "D2H partition");
    int32_t *b_rowptr;
    int32_t *b_col;
    void *b_val;
    if (is_root) {
        b_rowptr = const_cast<int32_t *>(rowptr);
        b_col = const_cast<int32_t *>(col);
        b_val = const_cast<void *>(val);
    } else {
        DCU(ctx->b_rowptr.reserve(((size_t)n + 1) * 4, &ctx->dev_bytes), "alloc rowptrB");
        DCU(ctx->b_col.reserve((size_t)nnz * 4 + 16, &ctx->dev_bytes), "alloc colB");
        DCU(ctx->b_val.reserve((size_t)nnz * vs + 16, &ctx->dev_bytes), "alloc valB");
        b_rowptr = ctx->b_rowptr.as<int32_t>();
        b_col = ctx->b_col.as<int32_t>();
        b_val = ctx->b_val.p;
    }
    DCU(cudaEventRecord(d->ev_ready, s), "event");
    DCU(cudaStreamWaitEvent(d->val_stream, d->ev_ready, 0), "wait");
    DNC(nccl().Broadcast(b_rowptr, b_rowptr, (size_t)n + 1, ncclInt32, root, d->comm, s), "ncclBroadcast(rowptrB)");
    if (nnz > 0) DNC(nccl().Broadcast(b_col, b_col, (size_t)nnz, ncclInt32, root, d->comm, s), "ncclBroadcast(colB)");
    DCU(cudaEventRecord(d->ev_ready, s), "event");
    DCU(cudaStreamWaitEvent(d->val_stream, d->ev_ready, 0), "wait");
    if (nnz > 0)
        // (values only move: complex64 as one 8-byte word, complex128 as two)
        DNC(nccl().Broadcast(b_val, b_val, (size_t)nnz * (vs == 16 ? 2 : 1), vs == 4 ? ncclFloat32 : ncclFloat64, root,
                             d->comm, d->val_stream),
            "ncclBroadcast(valB)");
    DCU(cudaEventRecord(d->ev_val, d->val_stream), "event");
    DCU(cudaStreamSynchronize(s), "partition record");
    d->part = *d->h_part;
    d->n = n;
    // ---- this rank's block of A: a slice of B with rebased row pointers ----
    const long long r0 = d->part.bounds[d->rank], r1 = d->part.bounds[d->rank + 1];
    const long long e0 = d->part.nnz_bounds[d->rank], e1 = d->part.nnz_bounds[d->rank + 1];
    const int rows = (int)(r1 - r0);
    ctx->B = Csr{b_rowptr, b_col, b_val};
    if (d->nranks == 1) {
        ctx->A = ctx->B;   // one rank: A IS B
    } else {
        DCU(ctx->a_rowptr.reserve(((size_t)rows + 1) * 4, &ctx->dev_bytes), "alloc rowptrA");
        k_rebase_rowptr<<<(rows + 256) / 256, 256, 0, s>>>(rows, b_rowptr, (int)r0, ctx->a_rowptr.as<int>());
        DCU(cudaGetLastError(), "rebase kernel");
        ctx->A = Csr{ctx->a_rowptr.as<int>(), b_col + e0, (const char *)b_val + (size_t)e0 * vs};
    }
    ctx->slice_e0 = -1;
    if (d->nranks > 1 && rows > 0 && ctx->slice_range.reserve(2 * sizeof(int), &ctx->dev_bytes) == cudaSuccess) {
        DCU(cudaMemsetAsync(ctx->slice_range.p, 0, 2 * sizeof(int), s), "memset");
        const long long na = e1 - e0;
        const int blocks = (int)std::min<long long>((na + 255) / 256 + 1, 1184);
        k_slice_range<<<blocks, 256, 0, s>>>(na, b_col + e0, (int)r0, (int)r1, ctx->slice_range.as<int>());
        DCU(cudaGetLastError(), "slice range kernel");
        ctx->slice_e0 = e0;
    }
    ctx->dtype = dtype;
    ctx->m = rows;
    ctx->k = n;
    ctx->n = n;
    ctx->nnzA = (int)(e1 - e0);
    ctx->nnzB = (int)nnz;
    ctx->have_data = true;
    ctx->cdf_valid = false;   // new operands: the column CDF of the previous ones is not reused
    ctx->borrowed = true;    // (update_values does not apply; the b_* buffers stay library-owned)
    ctx->aliased = false;
    ctx->opA = ctx->opB = BHB200_OP_N;   // (no transposed operands in the multi-GPU driver)
    ctx->t_pending = ctx->t_shared = false;
    ctx->wait_before_values = d->ev_val;   // the first spgemm waits for the values after its stage 1
    DCU(cudaEventRecord(d->ev_t1, d->val_stream), "event");
    return BHB200_SUCCESS;
}

int bhb200_dist_spgemm(bhb200_ctx *ctx)
{
    if (!ctx || !ctx->dist) return dfail(ctx, BHB200_ERR_INVALID, "bhb200_dist_init first");
    DistState *d = ctx->dist;
    int rc = bhb200_spgemm(ctx);
    if (rc != BHB200_SUCCESS) return rc;
    cudaStream_t s = ctx->stream;
    long long *counts = d->d_counts.as<long long>();
    k_put_count<<<1, 1, 0, s>>>(ctx->counters.as<Counters>(), counts + MAX_RANKS);
    DNC(nccl().AllGather(counts + MAX_RANKS, counts, 1, ncclInt64, d->comm, s), "ncclAllGather(nnzC)");
    DCU(d->d_global_rowptr.reserve(((size_t)ctx->m + 1) * 8, &ctx->dev_bytes), "alloc global row pointers");
    k_global_rowptr<<<(ctx->m + 256) / 256, 256, 0, s>>>(ctx->m, d->rank, counts, ctx->rowoff64.as<int64_t>(),
                                                        d->d_global_rowptr.as<int64_t>());
    DCU(cudaGetLastError(), "global row pointer kernel");
    d->have_layout = true;
    return BHB200_SUCCESS;
}

int bhb200_dist_get_layout(bhb200_ctx *ctx, int64_t *row_begin, int64_t *row_end, int64_t *nnz_offset, int64_t *nnz_total,
                           int64_t *products_total)
{
    if (!ctx || !ctx->dist || !ctx->have_data) return dfail(ctx, BHB200_ERR_INVALID, "no distributed operands");
    DistState *d = ctx->dist;
    if (row_begin) *row_begin = d->part.bounds[d->rank];
    if (row_end) *row_end = d->part.bounds[d->rank + 1];
    if (products_total) *products_total = d->part.products;
    if (nnz_offset || nnz_total) {
        if (!d->have_layout) return dfail(ctx, BHB200_ERR_INVALID, "bhb200_dist_spgemm first");
        DCU(cudaSetDevice(ctx->device), "cudaSetDevice");
        DCU(cudaMemcpyAsync(d->h_counts, d->d_counts.p, sizeof(long long) * d->nranks, cudaMemcpyDeviceToHost, ctx->stream), "D2H counts");
        DCU(cudaStreamSynchronize(ctx->stream), "D2H counts");
        long long off = 0, total = 0;
        for (int r = 0; r < d->nranks; ++r) {
            if (r < d->rank) off += d->h_counts[r];
            total += d->h_counts[r];
        }
        if (nnz_offset) *nnz_offset = off;
        if (nnz_total) *nnz_total = total;
    }
    return BHB200_SUCCESS;
}

int bhb200_dist_get_block_products(bhb200_ctx *ctx, int64_t *block_products)
{
    if (!ctx || !ctx->dist || !ctx->have_data || !block_products) return dfail(ctx, BHB200_ERR_INVALID, "no distributed operands");
    for (int r = 0; r < ctx->dist->nranks; ++r) block_products[r] = ctx->dist->part.block_products[r];
    return BHB200_SUCCESS;
}

int bhb200_dist_get_global_rowptr_device(bhb200_ctx *ctx, const int64_t **rowptr_global)
{
    if (!ctx || !ctx->dist || !ctx->dist->have_layout || !rowptr_global) return dfail(ctx, BHB200_ERR_INVALID, "bhb200_dist_spgemm first");
    *rowptr_global = ctx->dist->d_global_rowptr.as<int64_t>();
    return BHB200_SUCCESS;
}

int bhb200_dist_broadcast_ms(bhb200_ctx *ctx, float *ms)
{
    if (!ctx || !ctx->dist || !ms) return BHB200_ERR_INVALID;
    DistState *d = ctx->dist;
    DCU(cudaSetDevice(ctx->device), "cudaSetDevice");
    DCU(cudaEventSynchronize(d->ev_t1), "event sync");
    DCU(cudaEventElapsedTime(ms, d->ev_t0, d->ev_t1), "event time");
    return BHB200_SUCCESS;
}

}  // extern "C"
