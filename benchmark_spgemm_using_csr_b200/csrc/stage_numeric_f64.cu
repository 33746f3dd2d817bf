// stage_numeric_f64.cu -- double instantiation of the numeric kernels (stage_numeric.cuh).
#include "stage_numeric.cuh"
#include "stage_range_vec.cuh"

namespace bhb {

const NumericKernels NUMERIC_F64{&launch_num_hash_t<double>,        &launch_num_large_t<double>,
                                 &launch_num_range_pick_t<double>,  &launch_num_direct_t<double>,
                                 &launch_num_bucket_t<double>,      &launch_num_bucket3w_t<double>,
                                 &launch_num_bucket_heavy_t<double>, &launch_num_bucket_heavy2_t<double>,
                                 &launch_copy_ct_t<double>};

}  // namespace bhb
