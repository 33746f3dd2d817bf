// direct_plan.h -- host-side plan of the direct (single-pass) mode: which symbolic bins skip the symbolic pass,
// at which staging capacity and base, and which numeric kernels run them (DirectOut in common.cuh).
#pragma once
#include "common.cuh"

namespace bhb {

// the library's switches that shape the plan (fields of bhb200_ctx, read at bhb200_create)
struct DirectSwitches {
    bool direct_mode;   // BHB200_DIRECT=off: false
    bool direct_wide;   // BHB200_DIRECT=tight: false
    bool bucket_warp;   // BHB200_BUCKET_W=off: false
    int force_cap;      // BHB200_DEBUG_FORCE_CAP, -1: off
    bool force_heavy;   // BHB200_DEBUG_FORCE_HEAVY
};

// every DIRECT_SAMPLE_STRIDE-th row of a group-hash bin is counted by the symbolic kernel before the plan is made
constexpr int DIRECT_SAMPLE_STRIDE = 64;
inline int direct_sample_rows(int rows)
{
    return (rows + DIRECT_SAMPLE_STRIDE - 1) / DIRECT_SAMPLE_STRIDE;
}
// bit b set: bin b is sampled (before the counters are read back a second time)
unsigned direct_sample_bins(const Counters &hc, const DirectSwitches &sw);

enum class DirectMode {
    TWO_PASS,   // symbolic + numeric kernels (not in the mask)
    TIGHT,      // speculated capacity 32 / 64 / 128, rows that overflow are retried through the two-pass path
    WIDE,       // rows that barely compress: capacity of the product bound, nothing can overflow
    HEAVY,      // rows beyond the on-chip tables: sliced bucket sort, staged at their product count
};

enum class DirectKernel {
    DIRECT,     // k_num_direct / k_num_block (NumericKernels::direct)
    BUCKET,     // k_num_bucket3 (NumericKernels::bucket); in a heavy bin staged by atomic bump
    BUCKET3W,   // k_num_bucket3w (NumericKernels::bucket3w)
    HEAVY,      // k_num_bucket_heavy2, then k_num_bucket_heavy on the rows it could not slice
};

constexpr int DIRECT_P_MAX = 0x7fffffff;

// The largest staging capacity of one row on chip (k_num_block, k_num_bucket3).  At 8192 entries their tables hold
// 8-byte values (224 / 221 KB) but not 16-byte ones (352 / 289 KB of the 227 KB a CTA may have): with complex128
// values SB_B8192 rows that would be WIDE at 8192 run as HEAVY, and HEAVY bins hand k_num_bucket3 the rows of at
// most 4096 products instead of 8192.
inline int direct_cap_max(size_t value_size)
{
    return value_size > 8 ? 4096 : 8192;
}

struct DirectLaunch {
    DirectKernel kernel;
    int cap;          // table capacity (BUCKET3W: capw); 0 for HEAVY
    int sg;           // lanes per B row (DIRECT, BUCKET3W); 0 otherwise
    int p_lo, p_hi;   // the launch takes the rows with p_lo < products <= p_hi
    int stride;       // staging entries between rows (DirectOut::ct_stride; BUCKET3W: its stride argument); 0: the kernel's capacity
};

struct DirectLaunches {
    int n = 0;
    DirectLaunch at[2];
    bool retry = false;   // a symbolic retry over the bin's retry queue follows
};

struct DirectBin {
    DirectMode mode = DirectMode::TWO_PASS;
    int rows = 0;
    int cap = 0;             // staging entries per row (TIGHT, WIDE)
    bool warp = false;       // SB_G128 / SB_G256 in the mask: warp-per-row bucket sort (k_num_bucket3w)
    long long base = 0;      // first staging entry of the bin (HEAVY: heavy_base)
};

struct DirectPlan {
    DirectBin bin[MAX_BINS];
    long long heavy_base = 0;   // the heavy rows' staging area (atomic bump from here)
    long long ct_entries = 0;   // staging entries of all bins
    size_t value_size = 0;
    bool bucket_ok = true;      // false after drop_bucket

    unsigned mask() const;      // bit b set: bin b runs in direct mode (launch_bin_scatter / launch_scan)
    bool uses_bucket() const;   // the bucket kernels run: the column CDF is needed
    long long ct_bytes() const { return ct_entries * (4 + (long long)value_size); }
    DirectLaunches launches(int b, int G) const;   // G: lanes per row group of the hash kernels

    // demotions to the two-pass path
    void drop_wide();     // the staging would crowd out C: wide and heavy bins leave, tight bins are packed again
    void drop_all();      // the staging buffer could not be allocated
    void drop_bucket();   // the column CDF could not be allocated: heavy bins leave, no bucket kernels
};

// hc: the counters after the sampling of direct_sample_bins (if it sampled any bin)
DirectPlan plan_direct(const Counters &hc, const DirectSwitches &sw, size_t value_size);

}  // namespace bhb
