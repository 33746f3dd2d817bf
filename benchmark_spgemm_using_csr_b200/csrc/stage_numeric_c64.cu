// stage_numeric_c64.cu -- complex64 instantiation of the numeric kernels (stage_numeric.cuh): VT = c64, two floats
// in the 8 bytes a double takes, so every kernel runs with the tables, bins and launch shapes of f64.
#include "stage_numeric.cuh"
#include "stage_range_vec.cuh"

namespace bhb {

const NumericKernels NUMERIC_C64{&launch_num_hash_t<c64>,        &launch_num_large_t<c64>,
                                 &launch_num_range_pick_t<c64>,  &launch_num_direct_t<c64>,
                                 &launch_num_bucket_t<c64>,      &launch_num_bucket3w_t<c64>,
                                 &launch_num_bucket_heavy_t<c64>, &launch_num_bucket_heavy2_t<c64>,
                                 &launch_copy_ct_t<c64>};

}  // namespace bhb
