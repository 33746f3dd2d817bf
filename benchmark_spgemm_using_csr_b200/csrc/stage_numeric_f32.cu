// stage_numeric_f32.cu -- float instantiation of the numeric kernels (stage_numeric.cuh).
#include "stage_numeric.cuh"
#include "stage_range_vec.cuh"

namespace bhb {

const NumericKernels NUMERIC_F32{&launch_num_hash_t<float>,        &launch_num_large_t<float>,
                                 &launch_num_range_pick_t<float>,  &launch_num_direct_t<float>,
                                 &launch_num_bucket_t<float>,      &launch_num_bucket3w_t<float>,
                                 &launch_num_bucket_heavy_t<float>, &launch_num_bucket_heavy2_t<float>,
                                 &launch_copy_ct_t<float>};

}  // namespace bhb
