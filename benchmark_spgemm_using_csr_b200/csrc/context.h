// context.h -- the library's context object (private to csrc/): operands, grow-only workspace,
// results, cached plans.  include/bhsparse_b200.h exposes it as the opaque bhb200_ctx.
#pragma once
#include "../../include/bhsparse_b200.h"
#include "common.cuh"
#include "pattern_plan.h"

#include <string>

namespace bhb {

struct DevBuf {
    void *p = nullptr;
    size_t cap = 0;
    bool host = false;   // spilled: pinned, device-mapped HOST memory (see reserve_spillable)
    void drop(size_t *total)
    {
        if (p) {
            if (host) cudaFreeHost(p);
            else cudaFree(p);
            *total -= cap;
        }
        p = nullptr;
        cap = 0;
        host = false;
    }
    cudaError_t reserve(size_t bytes, size_t *total)
    {
        if (bytes <= cap) return cudaSuccess;
        drop(total);
        // round up to 256 B; grow-only cache, released by free_mem
        size_t want = (bytes + 255) & ~(size_t)255;
        cudaError_t e = cudaMalloc(&p, want);
        if (e != cudaSuccess) {
            p = nullptr;
            return e;
        }
        cap = want;
        *total += cap;
        return cudaSuccess;
    }
    // Host-memory spill (SURVEY.md 8f-4; the reference's OpenCL build keeps Ct in host-coherent
    // "re-allocatable" memory for the same reason, SpGEMM_opencl/bhsparse_opencl.cpp:219-227,
    // 441-454, 832-863): if the device cannot hold the buffer -- cudaMalloc fails, or the request
    // exceeds `device_cap` (BHB200_DEBUG_DEVICE_CAP, tests) -- it is placed in pinned host memory
    // mapped into the device address space; kernels then write it across NVLink-C2C / PCIe.
    cudaError_t reserve_spillable(size_t bytes, size_t *total, size_t device_cap, bool *spilled)
    {
        if (bytes <= cap) return cudaSuccess;
        cudaError_t e = cudaErrorMemoryAllocation;
        if (bytes <= device_cap) e = reserve(bytes, total);
        if (e == cudaSuccess) return e;
        cudaGetLastError();
        drop(total);
        size_t want = (bytes + 4095) & ~(size_t)4095;
        e = cudaHostAlloc(&p, want, cudaHostAllocMapped | cudaHostAllocPortable);
        if (e != cudaSuccess) {
            p = nullptr;
            return e;
        }
        cap = want;
        host = true;
        *total += cap;
        if (spilled) *spilled = true;
        return cudaSuccess;
    }
    void release(size_t *total) { drop(total); }
    template <typename T>
    T *as() const
    {
        return reinterpret_cast<T *>(p);
    }
};


struct DistState;   // dist_nccl.cu

}  // namespace bhb

struct bhb200_ctx {
    int device = 0;
    int sm_count = 0;
    char name[256] = {0};
    cudaStream_t own_stream = nullptr;
    cudaStream_t stream = nullptr;
    std::string err;

    // operands
    bool have_data = false;
    bool borrowed = false;
    bool aliased = false;   // host API: A and B were the same host arrays, uploaded once
    // multi-GPU row block: A's entries ARE entries slice_e0 .. of B's arrays (bhb200_dist_setup_square), -1 otherwise;
    // slice_range = {max, INT_MAX - min} over A's columns and A's own rows: the rows of B whose codes the product needs
    long long slice_e0 = -1;
    bhb::DevBuf slice_range;
    int dtype = BHB200_DTYPE_F64;
    int m = 0, k = 0, n = 0, nnzA = 0, nnzB = 0;
    bhb::DevBuf a_rowptr, a_col, a_val, b_rowptr, b_col, b_val;
    bhb::Csr A{nullptr, nullptr, nullptr}, B{nullptr, nullptr, nullptr};   // the effective operands op(A), op(B)
    // transposed operands (stage_transpose.cu): As / Bs are the operands as stored (host copies or borrowed);
    // with op = BHB200_OP_T, A / B point at the library's transposed copy at_* / bt_* (grow-only)
    int opA = BHB200_OP_N, opB = BHB200_OP_N;
    bhb::Csr As{nullptr, nullptr, nullptr}, Bs{nullptr, nullptr, nullptr};
    bhb::DevBuf at_rowptr, at_col, at_val, at_perm, bt_rowptr, bt_col, bt_val, bt_perm, t_scratch;
    bool t_pending = false;   // the transposed structure is not built yet (host operands: once after init_data)
    bool t_shared = false;    // same host arrays and both ops T: op(B) IS op(A) (one transposed copy)
    bool t_ran = false;       // the last call transposed or re-gathered: ev[5] marks its end

    // workspace (grow-only, reused across calls)
    bhb::DevBuf prod, rc, queue, rowoff64, rowptr32, blocksums, counters, bitmap, prefix;
    bhb::DevBuf brange, rlo, rspan, wl_off, wl_cnt, wl_idx, wl_bits;   // span info + word-list pool (range kernels)
    bhb::DevBuf cdf_colcount, cdf_hist, cdf_tab;                          // bucket-sort kernels: column CDF of the products
    // the table of the previous product on these operands is kept: it only balances the buckets (any monotone table gives
    // the same C), and it depends on the patterns alone; reset whenever operands are (re)initialised
    bool cdf_valid = false;
    int cdf_shift_cached = 0;
    int bucket_warp = 1;                                                  // BHB200_BUCKET_W=off: hash kernels instead of k_num_bucket3w
    bhb::DevBuf ct_off, ct_col, ct_val, retry_q;                       // direct mode: staging buffer (Ct) + retry queues
    // diagonal-pattern mode (stage_pattern.cuh): offset sets, per-entry codes, masks, tables
    bhb::DevBuf pat_sets, pat_ta, pat_tb, pat_maskB, pat_outmask, pat_tables, pat_fullbits;
    bhb::PatSet *h_sets = nullptr;    // pinned, [2]
    bhb::PatternPlan plan;
    size_t device_cap = ~(size_t)0;   // BHB200_DEBUG_DEVICE_CAP: largest single buffer the device may hold (tests)
    int pattern_enable = 1;      // BHB200_PATTERN=off disables
    int pattern_speculate = 1;   // reuse the previous plan without the detection pass (verified; BHB200_PATTERN=detect disables)
    bool last_pattern = false;   // the last product ran in pattern mode
    bhb::PatTables last_tables{};
    const unsigned char *last_ta = nullptr, *last_tb = nullptr;
    int direct_mode = 1;                                          // BHB200_DIRECT=off disables
    int direct_wide = 1;                                          // BHB200_DIRECT=tight: speculated capacities <= 128 only
    int force_cap = -1;            // BHB200_DEBUG_FORCE_CAP (tests): speculate this capacity whatever the sample says; -1: off
    bool force_heavy = false;      // BHB200_DEBUG_FORCE_HEAVY (tests): rows beyond the on-chip tables take the sliced bucket sort
    long long wordlist_cap = -1;   // BHB200_DEBUG_WORDLIST_CAP (tests): size of the range kernels' word-list pool; -1: by product count
    size_t bitmap_zeroed_bytes = 0;
    // masked product (stage_masked.cu): M is the library's copy (bhb200_set_mask) or the caller's arrays
    // (bhb200_set_mask_device); mask_q holds the masked bin queues of the last masked product
    bool mask_set = false;
    bool mask_changed = false;   // set / cleared since the last bhb200_spgemm: no bhb200_spgemm_numeric
    bhb::MaskCsr M{nullptr, nullptr, 0};
    bhb::DevBuf mask_rowptr, mask_col, mask_q, mask_acc, mask_hit;
    bool last_masked = false;
    int last_mask_bin[bhb::MB_COUNT] = {0};
    bhb::BinOffsets last_mask_off{};   // where each masked bin's queue starts in mask_q
    // copy bin (NB_COPY) of the last scan: rows, their place in `queue`, staged entries per row
    int last_copy_rows = 0, last_copy_off = 0;
    double last_copy_avg = 0.0;
    bhb::DevBuf colC, valC;
    bhb::Counters *h_ctr = nullptr;   // pinned
    size_t dev_bytes = 0;

    bool have_C = false;
    int64_t nnzC = 0;
    // structure reuse (bhb200_spgemm_numeric): what the last full product left behind
    int last_G = 32;
    bhb::WordLists last_wl{nullptr, nullptr, nullptr, nullptr, 0};
    bool reuse_bins_valid = false;   // queue holds the numeric bins without the copy bin
    int reuse_num_bin[bhb::MAX_BINS] = {0};
    cudaEvent_t ev[6] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};   // [5]: after the transposition
    bool timing_valid = false;
    bool profiling = false;
    int max_span = bhb::SPAN_SMALL;   // BHB200_RANGE=off|small|all overrides (experiments)
    // per-launch events: [0] symbolic, [1] numeric; one before each bin + one after the last
    cudaEvent_t ev_bin[2][bhb::MAX_BINS + 1] = {};
    bool ev_bin_used[2][bhb::MAX_BINS + 1] = {};
    int launches = 0;
    bhb200_stats stats;
    cudaEvent_t wait_before_values = nullptr;   // set by bhb200_dist_setup_square: B's values are still in flight
    bhb::DistState *dist = nullptr;   // multi-GPU state (dist_nccl.cu), created by bhb200_dist_init
};

