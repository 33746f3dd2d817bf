// direct_plan.cu -- host-only: the direct-mode plan of a product from its stage-1 counters and the sampled
// nnz(C_i) of its group-hash bins (DESIGN.md 4.7).  Two cases per sampled bin:
//  * tight: every sampled row has nnz(C_i) <= 128 -> speculate 32/64/128 entries per row,
//    rows that overflow go through the two-pass path (stencils: 1728 products -> 125);
//  * wide: the sampled rows barely compress (mean nnz(C_i) >= a quarter of the bin's table
//    capacity, R-MAT: nnz(C_i) ~ products) -> the numeric kernel would use the table the
//    product bound dictates anyway, so it runs once, staged, and the symbolic pass is
//    skipped; the bound is below the capacity, nothing can overflow.
#include "direct_plan.h"

namespace bhb {

namespace {

int min_sampled_rows(const DirectSwitches &sw)
{
    return sw.force_cap >= 0 ? 1 : 4096;
}

// wide bins with 512+ entries per row run the bucket-sort kernels, which need the column CDF of the products
// (k_num_bucket3 beats the hash kernels from a capacity of 512 up, profiles/r02_notes.md section 5)
constexpr int BUCKET_MIN_CAP = 512;

}  // namespace

unsigned direct_sample_bins(const Counters &hc, const DirectSwitches &sw)
{
    unsigned bins = 0;
    if (!sw.direct_mode) return 0;
    for (int b = SB_G128; b <= SB_G4096; ++b)
        if (hc.sym_bin[b] >= min_sampled_rows(sw)) bins |= 1u << b;
    return bins;
}

DirectPlan plan_direct(const Counters &hc, const DirectSwitches &sw, size_t value_size)
{
    DirectPlan p;
    p.value_size = value_size;
    for (int b = 0; b < MAX_BINS; ++b) p.bin[b].rows = hc.sym_bin[b];
    if (!sw.direct_mode) return p;
    const bool force = sw.force_cap >= 0;
    bool wide_above = false;
    bool heavy8192 = false;   // SB_B8192 follows a wide neighbour but its capacity does not fit on chip: HEAVY below
    for (int b = SB_G128; b <= SB_B8192; ++b) {
        DirectBin &d = p.bin[b];
        if (d.rows <= 0) continue;   // (an empty bin leaves wide_above as it is)
        if (b == SB_B8192) {
            // not sampled (the group kernels stop at 4096 slots): follows its neighbour
            if (!wide_above) continue;
            if (8192 > direct_cap_max(value_size)) {
                heavy8192 = true;
                continue;
            }
            d.mode = DirectMode::WIDE;
            d.cap = 8192;
        } else {
            wide_above = false;
            const int smax = force ? sw.force_cap : hc.sample_max[b];
            if (d.rows < min_sampled_rows(sw) || smax < 1) continue;
            const double mean = (double)hc.sample_sum[b] / direct_sample_rows(d.rows);
            const int wcap = 128 << (b - SB_G128);
            if (smax <= 128) {
                d.mode = DirectMode::TIGHT;
                d.cap = smax <= 32 ? 32 : smax <= 64 ? 64 : 128;
            } else if (sw.direct_wide && !force && mean * 4.0 >= wcap) {
                d.mode = DirectMode::WIDE;
                d.cap = wcap;
                wide_above = true;
            } else {
                continue;
            }
            // bins of at most 96 / 192 products whose sampled rows keep at least half of their products as outputs:
            // sorting the products (k_num_bucket3w) beats hashing them (BHB200_BUCKET_W=off: hash kernels)
            d.warp = sw.bucket_warp && b <= SB_G256 && !force &&
                     mean * 2.0 * (double)d.rows >= (double)hc.sym_bin_products[b];
        }
        d.base = p.ct_entries;
        p.ct_entries += (long long)d.rows * d.cap;
    }
    // rows with more products than the on-chip tables hold follow the largest sampled bin: if that one
    // does not compress they run once through the sliced bucket sort, staged at their product count
    // (BHB200_DEBUG_FORCE_HEAVY: tests send them there whatever the sample says)
    bool top_wide = sw.force_heavy || heavy8192;
    for (int b = SB_B8192; b >= SB_G128 && !top_wide; --b)
        if (p.bin[b].rows > 0) {
            top_wide = p.bin[b].mode == DirectMode::WIDE;
            break;
        }
    // (k_num_bucket_heavy2, measured on R-MAT 21, n = 2 M columns: 4.0 ms for these rows against 7.0 ms through the
    // two-pass tables + global column bitmap, whose cost also grows with n -- profiles/r02_notes.md section 5)
    if (top_wide && sw.direct_wide) {
        p.heavy_base = p.ct_entries;
        for (int b = heavy8192 ? SB_B8192 : SB_B16384; b <= SB_LARGE; ++b) {
            if (p.bin[b].rows <= 0) continue;
            p.bin[b].mode = DirectMode::HEAVY;
            p.bin[b].base = p.heavy_base;
            p.ct_entries += (long long)hc.sym_bin_products[b];
        }
    }
    return p;
}

unsigned DirectPlan::mask() const
{
    unsigned m = 0;
    for (int b = 0; b < MAX_BINS; ++b)
        if (bin[b].mode != DirectMode::TWO_PASS) m |= 1u << b;
    return m;
}

bool DirectPlan::uses_bucket() const
{
    if (!bucket_ok) return false;
    for (const DirectBin &d : bin)
        if (d.warp || d.mode == DirectMode::HEAVY || (d.mode == DirectMode::WIDE && d.cap >= BUCKET_MIN_CAP)) return true;
    return false;
}

void DirectPlan::drop_wide()
{
    ct_entries = 0;   // (heavy_base keeps its value: no launch reads it any more)
    for (DirectBin &d : bin) {
        if (d.mode == DirectMode::WIDE || d.mode == DirectMode::HEAVY) d = DirectBin{DirectMode::TWO_PASS, d.rows};
        if (d.mode != DirectMode::TIGHT) continue;
        d.base = ct_entries;
        ct_entries += (long long)d.rows * d.cap;
    }
}

void DirectPlan::drop_all()
{
    for (DirectBin &d : bin) d = DirectBin{DirectMode::TWO_PASS, d.rows};
    heavy_base = ct_entries = 0;
}

void DirectPlan::drop_bucket()
{
    bucket_ok = false;   // (the heavy rows' staging stays allocated but unused)
    for (DirectBin &d : bin)
        if (d.mode == DirectMode::HEAVY) d = DirectBin{DirectMode::TWO_PASS, d.rows};
}

DirectLaunches DirectPlan::launches(int b, int G) const
{
    DirectLaunches ls;
    const DirectBin &d = bin[b];
    auto add = [&ls](DirectKernel k, int cap, int sg, int p_lo, int p_hi, int stride) {
        ls.at[ls.n++] = DirectLaunch{k, cap, sg, p_lo, p_hi, stride};
    };
    if (d.mode == DirectMode::HEAVY) {
        // rows of at most cap products by k_num_bucket3 itself when the bin has such rows (8-byte values: SB_B16384,
        // 6144 < products <= 12288, cap 8192; 16-byte values: SB_B8192, 3072 < products <= 6144, cap 4096), the rest
        // by k_num_bucket_heavy2, partitioned by slice through the row's own staging area
        const int cap = direct_cap_max(value_size);
        const int p_floor = 96 << (b - SB_G256);   // the bin's rows have more products than this (sym_bin_of)
        const int p_bucket = p_floor < cap ? cap : 0;
        if (p_bucket) add(DirectKernel::BUCKET, cap, 0, 0, cap, 0);
        add(DirectKernel::HEAVY, 0, 0, p_bucket, DIRECT_P_MAX, 0);
    } else if (d.warp && bucket_ok) {
        add(DirectKernel::BUCKET3W, b == SB_G128 ? 128 : 256, G, 0, DIRECT_P_MAX, d.cap);
    } else if (d.mode == DirectMode::TIGHT) {
        add(DirectKernel::DIRECT, d.cap, G, 0, DIRECT_P_MAX, 0);
    } else if (d.mode == DirectMode::WIDE) {
        // the rows up to half the capacity run with the half-size table
        for (int pass = 0; pass < 2; ++pass) {
            const int cap = pass ? d.cap : d.cap / 2;
            const bool bucket = bucket_ok && cap >= BUCKET_MIN_CAP;
            add(bucket ? DirectKernel::BUCKET : DirectKernel::DIRECT, cap, bucket ? 0 : 32, pass ? d.cap / 2 : 0,
                pass ? DIRECT_P_MAX : d.cap / 2, d.cap);
        }
    }
    ls.retry = d.mode == DirectMode::TIGHT;
    return ls;
}

}  // namespace bhb
