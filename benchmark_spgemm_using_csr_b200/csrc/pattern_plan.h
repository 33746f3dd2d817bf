// pattern_plan.h -- host-side plan of the diagonal-pattern mode (stage_pattern.cuh).
#pragma once
#include <vector>

#include "stage_pattern.cuh"

namespace bhb {

struct PatternPlan {
    bool valid = false;
    bool reused = false;            // same offset sets as the previous call (tables already uploaded)
    int value_size = 0;
    std::vector<int> DA, DB;        // sorted offsets of A and B
    int nD = 0, nw = 0, acc_len = 0;
    std::vector<unsigned char> blob;   // all device tables, uploaded as one copy
    size_t off_mphys = 0, off_mlog = 0, off_pos = 0, off_pfull = 0, off_dcol = 0, off_offsA = 0, off_offsB = 0;
};

// Lanes whose accumulator slots one shared-memory wavefront (128 bytes) serves: 32 for 4-byte values, 16 for 8-byte
// and 8 for 16-byte ones (complex128).  The accumulator layout colours the products of such lane groups into
// distinct banks (choose_layout).
inline int pattern_lane_group(int value_size)
{
    return 128 / value_size;
}

// offs*: the distinct offsets (any order).  False if the product has more than PAT_MAX_OUT diagonals.
bool build_pattern_plan(const int *offsA, int nA, const int *offsB, int nB, int value_size, PatternPlan &plan);
PatTables pattern_tables(const PatternPlan &plan, const unsigned char *dev_blob);

}  // namespace bhb
