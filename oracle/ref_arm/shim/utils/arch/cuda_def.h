/* Build shim for the reference arm (oracle/ref_arm/build.sh): the UNMODIFIED reference kernels include
 * "utils/arch/cuda_def.h" for CUDA_CHECK; the real header drags in the UCS logger (the arm is built without UCX),
 * so this stand-in supplies the same macros on top of stdio.  Not part of the product. */
#ifndef REF_ARM_CUDA_DEF_H
#define REF_ARM_CUDA_DEF_H
#include <cuda_runtime.h>
#include <cuda.h>
#include <stdio.h>
#include <assert.h>
#include "ucc/api/ucc.h"

#define ucc_unlikely(x) __builtin_expect(!!(x), 0)
#define ucc_likely(x)   __builtin_expect(!!(x), 1)
#define ucc_assert(x)   assert(x)
#define ucc_error(...)  do { fprintf(stderr, "[ref_arm] " __VA_ARGS__); fprintf(stderr, "\n"); } while (0)

static inline ucc_status_t cuda_error_to_ucc_status(cudaError_t e)
{
    return e == cudaSuccess ? UCC_OK : e == cudaErrorNotReady ? UCC_INPROGRESS
         : e == cudaErrorInvalidValue ? UCC_ERR_INVALID_PARAM : UCC_ERR_NO_MESSAGE;
}
#define CUDA_FUNC(_func) ({ cudaError_t _r = (_func); if (_r != cudaSuccess) ucc_error("%s failed: %s", #_func, cudaGetErrorString(_r)); cuda_error_to_ucc_status(_r); })
#define CUDA_CHECK(_cmd) do { ucc_status_t _s = CUDA_FUNC(_cmd); if (_s != UCC_OK) return _s; } while (0)
#endif
