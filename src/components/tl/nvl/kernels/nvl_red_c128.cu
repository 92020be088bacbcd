/* tl/nvl reduction kernels instantiated for float64_complex (nvl_c128) */
#include "nvl_reduce_impl.cuh"
NVL_INSTANTIATE_REDUCE(nvl_c128, c128)
