// stage_numeric_c128.cu -- complex128 instantiation of the numeric kernels (stage_numeric.cuh): VT = c128, two
// doubles in 16 bytes.  The launchers leave out the layouts that hold at most 8-byte values (the host routes
// those rows elsewhere: num_hash_last, plan_direct) and the 128-bit range-vec kernel.
#include "stage_numeric.cuh"
#include "stage_range_vec.cuh"

namespace bhb {

const NumericKernels NUMERIC_C128{&launch_num_hash_t<c128>,         &launch_num_large_t<c128>,
                                  &launch_num_range_pick_t<c128>,   &launch_num_direct_t<c128>,
                                  &launch_num_bucket_t<c128>,       &launch_num_bucket3w_t<c128>,
                                  &launch_num_bucket_heavy_t<c128>, &launch_num_bucket_heavy2_t<c128>,
                                  &launch_copy_ct_t<c128>};

}  // namespace bhb
