"""Host side of the direct (single-pass) mode (csrc/direct_plan.cu) -- no GPU needed: which symbolic bins are
sampled, the mode, capacity, staging base and warp-bucket choice of every bin, the demotions, and the numeric
launches each bin gets.  The planner is compiled with a small extern "C" harness into a throwaway library.

The expected plans are worked out by hand from the selection code as it stood inline in bhb200_spgemm
(csrc/context.cu) before it moved into the planner; the planner must keep every one of them."""
import ctypes
import math
import os
import subprocess

import numpy as np
import pytest

from benchmark_spgemm_using_csr_b200 import build as libbuild

SB_G128, SB_G256, SB_G512, SB_G1024, SB_G2048, SB_G4096, SB_B8192, SB_B16384, SB_B32768, SB_LARGE = range(3, 13)
SB_RANGE_S, SB_COUNT = 13, 15
P_MAX = 0x7FFFFFFF
MODES = ["two_pass", "tight", "wide", "heavy"]
KERNELS = ["direct", "bucket", "bucket3w", "heavy"]
PER_BIN = 6 + 2 * 6

HARNESS = r'''
#include "direct_plan.h"
using namespace bhb;

extern "C" __attribute__((visibility("default")))
void direct_plan_probe(const int *rows, const long long *products, const int *sample_max, const long long *sample_sum,
                       const int *sw, int value_size, const char *drops, int G, long long *out)
{
    Counters hc{};
    for (int b = 0; b < SB_COUNT; ++b) {
        hc.sym_bin[b] = rows[b];
        hc.sym_bin_products[b] = products[b];
        hc.sample_max[b] = sample_max[b];
        hc.sample_sum[b] = sample_sum[b];
    }
    const DirectSwitches s{sw[0] != 0, sw[1] != 0, sw[2] != 0, sw[3], sw[4] != 0};
    *out++ = direct_sample_bins(hc, s);
    DirectPlan p = plan_direct(hc, s, (size_t)value_size);
    for (; *drops; ++drops) {
        if (*drops == 'w') p.drop_wide();
        if (*drops == 'a') p.drop_all();
        if (*drops == 'b') p.drop_bucket();
    }
    *out++ = p.mask();
    *out++ = p.uses_bucket();
    *out++ = p.heavy_base;
    *out++ = p.ct_entries;
    *out++ = p.ct_bytes();
    for (int b = 0; b < SB_COUNT; ++b) {
        const DirectBin &d = p.bin[b];
        const DirectLaunches ls = p.launches(b, G);
        *out++ = (int)d.mode;
        *out++ = d.cap;
        *out++ = d.warp;
        *out++ = d.base;
        *out++ = ls.retry;
        *out++ = ls.n;
        for (int i = 0; i < 2; ++i) {
            const DirectLaunch l = i < ls.n ? ls.at[i] : DirectLaunch{};
            *out++ = (int)l.kernel;
            *out++ = l.cap;
            *out++ = l.sg;
            *out++ = l.p_lo;
            *out++ = l.p_hi;
            *out++ = l.stride;
        }
    }
}
'''


@pytest.fixture(scope="module")
def probe(tmp_path_factory):
    try:
        nvcc = libbuild.nvcc()
    except RuntimeError:
        pytest.skip("nvcc not found")
    tmp = tmp_path_factory.mktemp("direct_plan")
    src = tmp / "harness.cu"
    src.write_text(HARNESS)
    lib = tmp / "libdirect_plan_probe.so"
    cmd = ([nvcc] + libbuild.ccbin() + libbuild.NVCC_FLAGS + ["-I", libbuild.CSRC, "-shared",
           os.path.join(libbuild.CSRC, "direct_plan.cu"), str(src), "-o", str(lib)])
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    fn = ctypes.CDLL(str(lib)).direct_plan_probe
    fn.restype = None
    return fn


def plan(probe, bins, *, direct=True, wide=True, warp=True, force_cap=-1, force_heavy=False, vs=8, G=8, drops=""):
    """bins: {bin: (rows, products, sampled max nnz(C_i), sampled mean nnz(C_i))}.  The sampled sum is the mean
    times the number of sampled rows (every 64th row), as the symbolic kernel leaves it."""
    rows, prods, smax, ssum = (np.zeros(SB_COUNT, dtype=t) for t in (np.int32, np.int64, np.int32, np.int64))
    for b, (r, p, mx, mean) in bins.items():
        rows[b], prods[b], smax[b], ssum[b] = r, p, mx, round(mean * math.ceil(r / 64))
    out = np.zeros(6 + SB_COUNT * PER_BIN, dtype=np.int64)
    sw = np.array([direct, wide, warp, force_cap, force_heavy], dtype=np.int32)
    ptr = lambda a: ctypes.c_void_p(a.ctypes.data)
    probe(ptr(rows), ptr(prods), ptr(smax), ptr(ssum), ptr(sw), vs, drops.encode(), G, ptr(out))
    res = dict(sampled={b for b in range(SB_COUNT) if (int(out[0]) >> b) & 1}, mask={b for b in range(SB_COUNT) if (int(out[1]) >> b) & 1},
               uses_bucket=bool(out[2]), heavy_base=int(out[3]), ct_entries=int(out[4]), ct_bytes=int(out[5]), bins={})
    for b in range(SB_COUNT):
        v = [int(x) for x in out[6 + b * PER_BIN:6 + (b + 1) * PER_BIN]]
        mode, cap, warp_, base, retry, n = v[:6]
        launches = [(KERNELS[k], *rest) for k, *rest in (v[6 + 6 * i:12 + 6 * i] for i in range(n))]
        if mode == 0:
            assert (cap, warp_, base, retry, n) == (0, 0, 0, 0, 0), f"bin {b} outside the mask carries a plan"
            continue
        res["bins"][b] = dict(mode=MODES[mode], cap=cap, warp=bool(warp_), base=base, retry=bool(retry), launches=launches)
    assert res["mask"] == set(res["bins"])
    return res


def tight(cap, base, G, warp=False):
    launch = ("bucket3w", 128, G, 0, P_MAX, cap) if warp else ("direct", cap, G, 0, P_MAX, 0)
    return dict(mode="tight", cap=cap, warp=warp, base=base, retry=True, launches=[launch])


def wide(cap, base, bucket=True):
    def one(c, lo, hi):
        if bucket and c >= 512:
            return ("bucket", c, 0, lo, hi, cap)
        return ("direct", c, 32, lo, hi, cap)
    return dict(mode="wide", cap=cap, warp=False, base=base, retry=False,
                launches=[one(cap // 2, 0, cap // 2), one(cap, cap // 2, P_MAX)])


def heavy(b, base):
    launches = [("heavy", 0, 0, 8192 if b == SB_B16384 else 0, P_MAX, 0)]
    if b == SB_B16384:
        launches.insert(0, ("bucket", 8192, 0, 0, 8192, 0))
    return dict(mode="heavy", cap=0, warp=False, base=base, retry=False, launches=launches)


# R-MAT-like: every group-hash bin from G512 up barely compresses; G512 sits exactly on the wide threshold
# (mean * 4 == capacity); G128 compresses (tight, 32 entries)
RMAT = {SB_G128: (8000, 8000 * 60, 30, 10.0),
        SB_G512: (5000, 5000 * 300, 384, 128.0), SB_G1024: (5000, 5000 * 600, 700, 300.0),
        SB_G2048: (5000, 5000 * 1200, 1400, 600.0), SB_G4096: (5000, 5000 * 2500, 3000, 1100.0)}
HEAVY_ROWS = {SB_B16384: (50, 50 * 10000, 0, 0.0), SB_B32768: (20, 20 * 20000, 0, 0.0), SB_LARGE: (5, 5 * 100000, 0, 0.0)}
RMAT_TOP = 8000 * 32 + 5000 * (512 + 1024 + 2048 + 4096)   # staging entries of the sampled bins


def test_direct_off_and_tight_switch(probe):
    bins = {**RMAT, **HEAVY_ROWS}
    p = plan(probe, bins, direct=False, force_heavy=True)
    assert p["sampled"] == set() and p["mask"] == set() and p["ct_entries"] == 0 and p["ct_bytes"] == 0
    assert not p["uses_bucket"]
    # BHB200_DIRECT=tight: only the bins that compress; no wide and no heavy bins, not even with force_heavy
    p = plan(probe, bins, wide=False, force_heavy=True)
    assert p["sampled"] == {SB_G128, SB_G512, SB_G1024, SB_G2048, SB_G4096}
    assert p["bins"] == {SB_G128: tight(32, 0, 8)}
    assert p["ct_entries"] == 8000 * 32 and p["heavy_base"] == 0 and not p["uses_bucket"]


def test_stencil_like_tight_capacities(probe):
    bins = {SB_G128: (8000, 8000 * 90, 20, 20.0), SB_G256: (10000, 10000 * 150, 50, 50.0),
            SB_G512: (6000, 6000 * 300, 125, 100.0), SB_RANGE_S: (99999, 99999 * 40, 0, 0.0)}
    for G in (8, 32):
        p = plan(probe, bins, G=G, vs=8)
        assert p["sampled"] == {SB_G128, SB_G256, SB_G512}
        assert p["bins"] == {SB_G128: tight(32, 0, G), SB_G256: tight(64, 8000 * 32, G),
                             SB_G512: tight(128, 8000 * 32 + 10000 * 64, G)}
        assert p["ct_entries"] == 8000 * 32 + 10000 * 64 + 6000 * 128
        assert p["ct_bytes"] == p["ct_entries"] * 12 and not p["uses_bucket"]
    assert plan(probe, bins, vs=4)["ct_bytes"] == (8000 * 32 + 10000 * 64 + 6000 * 128) * 8
    # the speculated capacity is the smallest of 32 / 64 / 128 that holds the largest sampled row
    for smax, cap in ((1, 32), (32, 32), (33, 64), (64, 64), (65, 128), (128, 128), (129, None)):
        p = plan(probe, {SB_G256: (5000, 5000 * 150, smax, 20.0)})
        assert p["bins"] == ({SB_G256: tight(cap, 0, 8)} if cap else {})


def test_small_bins_are_not_sampled_unless_forced(probe):
    bins = {SB_G256: (4095, 4095 * 150, 50, 50.0), SB_G512: (4096, 4096 * 300, 100, 90.0)}
    p = plan(probe, bins)
    assert p["sampled"] == {SB_G512} and p["bins"] == {SB_G512: tight(128, 0, 8)}
    # forced capacity: one row is enough, the sample is ignored, no wide and no warp-bucket bins
    bins = {SB_G128: (1, 90, 0, 90.0), SB_G256: (3, 3 * 150, 0, 150.0), SB_G1024: (5000, 5000 * 700, 700, 700.0)}
    p = plan(probe, bins, force_cap=64)
    assert p["sampled"] == {SB_G128, SB_G256, SB_G1024}
    assert p["bins"] == {SB_G128: tight(64, 0, 8), SB_G256: tight(64, 64, 8), SB_G1024: tight(64, 4 * 64, 8)}
    p = plan(probe, bins, force_cap=256)            # beyond the speculated capacities, and wide is off when forced
    assert p["sampled"] == {SB_G128, SB_G256, SB_G1024} and p["mask"] == set()
    p = plan(probe, bins, force_cap=0)
    assert p["mask"] == set()


def test_rmat_chain_of_wide_bins(probe):
    p = plan(probe, RMAT, G=32)
    assert p["bins"] == {SB_G128: tight(32, 0, 32), SB_G512: wide(512, 8000 * 32),
                         SB_G1024: wide(1024, 8000 * 32 + 5000 * 512), SB_G2048: wide(2048, 8000 * 32 + 5000 * 1536),
                         SB_G4096: wide(4096, 8000 * 32 + 5000 * 3584)}
    # G512: half-size table with the direct kernel (32 lanes per row), full size with the bucket kernel
    assert p["bins"][SB_G512]["launches"] == [("direct", 256, 32, 0, 256, 512), ("bucket", 512, 0, 256, P_MAX, 512)]
    assert p["ct_entries"] == RMAT_TOP and p["uses_bucket"]
    # just below the threshold (mean * 4 < capacity) the bin is neither wide nor tight
    below = dict(RMAT)
    below[SB_G512] = (5000, 5000 * 300, 384, 127.0)
    assert SB_G512 not in plan(probe, below)["mask"]


def test_b8192_follows_the_nearest_sampled_bin_below(probe):
    b8 = {SB_B8192: (5000, 5000 * 5000, 0, 0.0)}
    p = plan(probe, {**RMAT, **b8})
    assert SB_B8192 not in p["sampled"] and p["bins"][SB_B8192] == wide(8192, RMAT_TOP)
    assert p["bins"][SB_B8192]["launches"] == [("bucket", 4096, 0, 0, 4096, 8192), ("bucket", 8192, 0, 4096, P_MAX, 8192)]
    # an empty SB_G4096 keeps the decision of SB_G2048
    no4096 = {b: v for b, v in RMAT.items() if b != SB_G4096}
    p = plan(probe, {**no4096, **b8})
    assert p["bins"][SB_B8192] == wide(8192, RMAT_TOP - 5000 * 4096)
    # a non-empty SB_G4096 that is not sampled (below 4096 rows) clears it
    p = plan(probe, {**no4096, SB_G4096: (100, 100 * 2500, 0, 0.0), **b8})
    assert SB_B8192 not in p["mask"] and SB_G4096 not in p["mask"] and SB_G2048 in p["mask"]
    # and so does a tight SB_G4096
    p = plan(probe, {**no4096, SB_G4096: (5000, 5000 * 2500, 100, 90.0), **b8})
    assert SB_B8192 not in p["mask"] and p["bins"][SB_G4096] == tight(128, RMAT_TOP - 5000 * 4096, 8)


def test_warp_bucket_threshold(probe):
    # SB_G128, 8000 rows, sampled mean 40: warp bucket sort iff 40 * 2 * 8000 = 640000 >= products
    for products, want in ((640000, True), (640001, False)):
        p = plan(probe, {SB_G128: (8000, products, 60, 40.0)}, G=32)
        assert p["bins"] == {SB_G128: tight(64, 0, 32, warp=want)} and p["uses_bucket"] == want
    p = plan(probe, {SB_G128: (8000, 640000, 60, 40.0)}, warp=False)
    assert p["bins"] == {SB_G128: tight(64, 0, 8)} and not p["uses_bucket"]
    # a wide SB_G256 (sampled max > 128, mean >= 64) that keeps most of its products: warp bucket sort, staged
    # 256 apart, no retry
    g256 = {SB_G256: (5000, 5000 * 180, 192, 150.0)}
    p = plan(probe, g256, G=8)
    assert p["bins"] == {SB_G256: dict(mode="wide", cap=256, warp=True, base=0, retry=False,
                                       launches=[("bucket3w", 256, 8, 0, P_MAX, 256)])}
    assert p["uses_bucket"]
    p = plan(probe, g256, warp=False)
    assert p["bins"] == {SB_G256: wide(256, 0)} and not p["uses_bucket"]
    assert p["bins"][SB_G256]["launches"] == [("direct", 128, 32, 0, 128, 256), ("direct", 256, 32, 128, P_MAX, 256)]


def test_heavy_bins(probe):
    # the top sampled bin is wide: the heavy bins share one staging area after everything else
    p = plan(probe, {**RMAT, **HEAVY_ROWS})
    assert p["heavy_base"] == RMAT_TOP
    for b in (SB_B16384, SB_B32768, SB_LARGE):
        assert p["bins"][b] == heavy(b, RMAT_TOP)
    assert p["ct_entries"] == RMAT_TOP + 50 * 10000 + 20 * 20000 + 5 * 100000
    # the top bin compresses: no heavy bins
    top_tight = {**RMAT, SB_G4096: (5000, 5000 * 2500, 100, 90.0), **HEAVY_ROWS}
    p = plan(probe, top_tight)
    assert p["mask"] & {SB_B16384, SB_B32768, SB_LARGE} == set() and p["heavy_base"] == 0
    # BHB200_DEBUG_FORCE_HEAVY: heavy whatever the sample says, also without any sampled bin
    p = plan(probe, top_tight, force_heavy=True)
    assert p["bins"][SB_LARGE] == heavy(SB_LARGE, p["heavy_base"]) and p["uses_bucket"]
    p = plan(probe, {SB_G128: (10, 10 * 50, 0, 0.0), **HEAVY_ROWS}, force_heavy=True)
    assert p["sampled"] == set() and p["heavy_base"] == 0
    assert p["bins"] == {b: heavy(b, 0) for b in (SB_B16384, SB_B32768, SB_LARGE)}
    assert plan(probe, HEAVY_ROWS, force_heavy=True, direct=False)["mask"] == set()


def test_demotions(probe):
    bins = {**RMAT, SB_G1024: (5000, 5000 * 700, 120, 100.0), **HEAVY_ROWS}     # G1024 tight amid wide bins
    p = plan(probe, bins)
    assert p["bins"][SB_G1024] == tight(128, 8000 * 32 + 5000 * 512, 8)
    heavy_base = p["heavy_base"]
    assert heavy_base == 8000 * 32 + 5000 * (512 + 128 + 2048 + 4096)
    # staging budget: the wide and heavy bins leave, the tight ones are packed from 0 again;
    # heavy_base keeps its value (no launch reads it any more)
    d = plan(probe, bins, drops="w")
    assert d["bins"] == {SB_G128: tight(32, 0, 8), SB_G1024: tight(128, 8000 * 32, 8)}
    assert d["ct_entries"] == 8000 * 32 + 5000 * 128 and d["heavy_base"] == heavy_base and not d["uses_bucket"]
    # no staging buffer: nothing is left
    d = plan(probe, bins, drops="a")
    assert d["mask"] == set() and d["ct_entries"] == 0 and d["ct_bytes"] == 0 and not d["uses_bucket"]
    # no column CDF: heavy bins leave (their staging stays counted), the bucket kernels fall back to the direct ones
    bins = {**RMAT, SB_G128: (8000, 640000, 60, 40.0), SB_G256: (5000, 5000 * 180, 192, 150.0), **HEAVY_ROWS}
    p = plan(probe, bins)
    assert p["bins"][SB_G128]["warp"] and p["bins"][SB_G256]["warp"] and SB_LARGE in p["mask"]
    d = plan(probe, bins, drops="b")
    assert d["ct_entries"] == p["ct_entries"] and not d["uses_bucket"]
    assert d["mask"] == {SB_G128, SB_G256, SB_G512, SB_G1024, SB_G2048, SB_G4096}
    assert d["bins"][SB_G128] == dict(tight(64, 0, 8), warp=True)
    assert d["bins"][SB_G128]["launches"] == [("direct", 64, 8, 0, P_MAX, 0)]
    assert d["bins"][SB_G256] == dict(wide(256, 8000 * 64), warp=True)
    for b, cap in ((SB_G512, 512), (SB_G1024, 1024), (SB_G2048, 2048), (SB_G4096, 4096)):
        assert d["bins"][b]["launches"] == [("direct", cap // 2, 32, 0, cap // 2, cap), ("direct", cap, 32, cap // 2, P_MAX, cap)]
