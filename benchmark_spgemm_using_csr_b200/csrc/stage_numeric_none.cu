// stage_numeric_none.cu -- structure-only instantiation of the numeric kernels (stage_numeric.cuh): VT = NoVal,
// so the kernels write the columns of C and no value is loaded, accumulated, staged or stored.
#include "stage_numeric.cuh"
#include "stage_range_vec.cuh"

namespace bhb {

const NumericKernels NUMERIC_NONE{&launch_num_hash_t<NoVal>,        &launch_num_large_t<NoVal>,
                                  &launch_num_range_pick_t<NoVal>,  &launch_num_direct_t<NoVal>,
                                  &launch_num_bucket_t<NoVal>,      &launch_num_bucket3w_t<NoVal>,
                                  &launch_num_bucket_heavy_t<NoVal>, &launch_num_bucket_heavy2_t<NoVal>,
                                  &launch_copy_ct_t<NoVal>};

}  // namespace bhb
