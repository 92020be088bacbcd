/* tl/nvl reduction kernels instantiated for float32_complex (nvl_c64) */
#include "nvl_reduce_impl.cuh"
NVL_INSTANTIATE_REDUCE(nvl_c64, c64)
