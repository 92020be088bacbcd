#include "ec_cuda_kernels.h"
#include "components/tl/nvl/kernels/nvl_device.cuh"
#include <cuComplex.h>

/* ------------------------------------------------------------------ */
/* element-wise reduction of n sources                                 */
/* ------------------------------------------------------------------ */
template <int OP, typename A> struct EcOp { static __device__ __forceinline__ A f(A a, A b) { return OpFn<OP, A>::f(a, b); } };
/* complex numbers: sum is component wise, prod is the complex product */
template <> struct EcOp<EC_OP_SUM, cuFloatComplex> { static __device__ __forceinline__ cuFloatComplex f(cuFloatComplex a, cuFloatComplex b) { return cuCaddf(a, b); } };
template <> struct EcOp<EC_OP_PROD, cuFloatComplex> { static __device__ __forceinline__ cuFloatComplex f(cuFloatComplex a, cuFloatComplex b) { return cuCmulf(a, b); } };
template <> struct EcOp<EC_OP_SUM, cuDoubleComplex> { static __device__ __forceinline__ cuDoubleComplex f(cuDoubleComplex a, cuDoubleComplex b) { return cuCadd(a, b); } };
template <> struct EcOp<EC_OP_PROD, cuDoubleComplex> { static __device__ __forceinline__ cuDoubleComplex f(cuDoubleComplex a, cuDoubleComplex b) { return cuCmul(a, b); } };

static_assert((int)EC_OP_SUM == (int)NVL_OP_SUM && (int)EC_OP_BXOR == (int)NVL_OP_BXOR, "operator enums must line up");

/* x * alpha: integer accumulators are scaled in double precision and truncated (reference ec_cuda_reduce_ops.h: d[i] * alpha),
 * casting alpha (1/N for AVG) to the integer type first would make it 0 */
template <typename T> __device__ __forceinline__ T scale(T x, double alpha)
{
    if constexpr (IsIntAcc<T>::v) return (T)((double)x * alpha);
    else return (T)(x * (T)alpha);
}
template <> __device__ __forceinline__ cuFloatComplex scale(cuFloatComplex x, double a) { return make_cuFloatComplex(x.x * (float)a, x.y * (float)a); }
template <> __device__ __forceinline__ cuDoubleComplex scale(cuDoubleComplex x, double a) { return make_cuDoubleComplex(x.x * a, x.y * a); }

static __device__ __forceinline__ const void *src_k(const ec_reduce_args_t &a, int k)
{ return (!a.strided || k == 0) ? a.srcs[a.strided ? 0 : k] : (const char *)a.src2 + (size_t)(k - 1) * a.stride; }

/* scalar path: any alignment, any type */
template <typename T, typename A, int OP, typename LD, typename ST>
static __device__ __forceinline__ void reduce_scalar(const ec_reduce_args_t &a, size_t begin, size_t end, LD ld, ST st, size_t tid, size_t nt)
{
    for (size_t i = begin + tid; i < end; i += nt) {
        A acc = ld(((const T *)src_k(a, 0))[i]);
        for (int k = 1; k < a.n_srcs; k++) acc = EcOp<OP, A>::f(acc, ld(((const T *)src_k(a, k))[i]));
        if (a.with_alpha) acc = scale<A>(acc, a.alpha);
        ((T *)a.dst)[i] = st(acc);
    }
}

/* tid / nt = index of the calling thread among the threads that share this task: the whole grid for the one-shot kernels,
 * one worker block inside the persistent executor */
template <typename T, int OP> static __device__ __forceinline__ void reduce_body(const ec_reduce_args_t &a, size_t tid, size_t nt)
{
    typedef typename AccOf<T>::type A;
    constexpr int E = 16 / sizeof(T);
    bool aligned = ((uintptr_t)a.dst & 15) == 0;
    for (int k = 0; k < a.n_srcs; k++) aligned = aligned && (((uintptr_t)src_k(a, k) & 15) == 0);
    size_t nvec = aligned ? a.count / E : 0;
    for (size_t v = tid; v < nvec; v += nt) { /* 128-bit path */
        VecAcc<T, OP> acc;
        acc.set(ld_src_v4((const char *)src_k(a, 0) + v * 16));
        for (int k = 1; k < a.n_srcs; k++) acc.add(ld_src_v4((const char *)src_k(a, k) + v * 16));
        if (a.with_alpha) {
#pragma unroll
            for (int i = 0; i < E; i++) acc.a[i] = scale<A>(acc.a[i], a.alpha);
        }
        st_v4((char *)a.dst + v * 16, acc.get(1));
    }
    reduce_scalar<T, A, OP>(a, nvec * E, a.count, [](T x) { return to_acc<T>(x); }, [](A x) { return from_acc<T>(x); }, tid, nt);
}
template <typename T, int OP> static __device__ __forceinline__ void reduce_body_cplx(const ec_reduce_args_t &a, size_t tid, size_t nt)
{ reduce_scalar<T, T, OP>(a, 0, a.count, [](T x) { return x; }, [](T x) { return x; }, tid, nt); }

template <typename T> static __device__ __forceinline__ void reduce_dispatch(const ec_reduce_args_t &a, size_t tid, size_t nt)
{
#define CALL_EC_REDUCE(_T, _OP) reduce_body<_T, _OP>(a, tid, nt)
    int op = a.op;
    NVL_DISPATCH_OP(T, op, CALL_EC_REDUCE);
}
static __device__ __noinline__ void reduce_any(const ec_reduce_args_t &a, size_t tid, size_t nt)
{
    switch (a.dt) {
    case EC_DT_I8: reduce_dispatch<int8_t>(a, tid, nt); break; case EC_DT_I16: reduce_dispatch<int16_t>(a, tid, nt); break;
    case EC_DT_I32: reduce_dispatch<int32_t>(a, tid, nt); break; case EC_DT_I64: reduce_dispatch<int64_t>(a, tid, nt); break;
    case EC_DT_U8: reduce_dispatch<uint8_t>(a, tid, nt); break; case EC_DT_U16: reduce_dispatch<uint16_t>(a, tid, nt); break;
    case EC_DT_U32: reduce_dispatch<uint32_t>(a, tid, nt); break; case EC_DT_U64: reduce_dispatch<uint64_t>(a, tid, nt); break;
    case EC_DT_F16: reduce_dispatch<__half>(a, tid, nt); break; case EC_DT_BF16: reduce_dispatch<__nv_bfloat16>(a, tid, nt); break;
    case EC_DT_F32: reduce_dispatch<float>(a, tid, nt); break; case EC_DT_F64: reduce_dispatch<double>(a, tid, nt); break;
    case EC_DT_C64: if (a.op == EC_OP_SUM) reduce_body_cplx<cuFloatComplex, EC_OP_SUM>(a, tid, nt); else if (a.op == EC_OP_PROD) reduce_body_cplx<cuFloatComplex, EC_OP_PROD>(a, tid, nt); break;
    case EC_DT_C128: if (a.op == EC_OP_SUM) reduce_body_cplx<cuDoubleComplex, EC_OP_SUM>(a, tid, nt); else if (a.op == EC_OP_PROD) reduce_body_cplx<cuDoubleComplex, EC_OP_PROD>(a, tid, nt); break;
    default: break;
    }
}
#define EC_GRID_TID ((size_t)blockIdx.x * blockDim.x + threadIdx.x)
#define EC_GRID_NT ((size_t)gridDim.x * blockDim.x)
/* one-shot reduce: (datatype, operator) picked on the HOST at launch - one body per kernel; the persistent executor below has to
 * switch at run time (reduce_any) because its tasks arrive while it is running */
template <typename T, int OP> __global__ void __launch_bounds__(1024) ec_reduce_kernel_t(const __grid_constant__ ec_reduce_args_t a) { reduce_body<T, OP>(a, EC_GRID_TID, EC_GRID_NT); }
template <typename T, int OP> __global__ void __launch_bounds__(1024) ec_reduce_cplx_kernel_t(const __grid_constant__ ec_reduce_args_t a) { reduce_body_cplx<T, OP>(a, EC_GRID_TID, EC_GRID_NT); }
template <typename T> static cudaError_t ec_launch_reduce_t(const ec_reduce_args_t *a, int nb, int nt, cudaStream_t s)
{
#define CALL_EC_LAUNCH(_T, _OP) ec_reduce_kernel_t<_T, _OP><<<nb, nt, 0, s>>>(*a)
    NVL_DISPATCH_OP(T, a->op, CALL_EC_LAUNCH);
    return cudaGetLastError();
}

/* up to 7 independent dst[j] = src1[j] op src2[j]; blockIdx.y selects the buffer */
__global__ void __launch_bounds__(1024) ec_reduce_multi_dst_kernel(ec_reduce_multi_dst_args_t m)
{
    int j = blockIdx.y;
    if (j >= m.n_bufs) return;
    ec_reduce_args_t a; a.dst = m.dst[j]; a.srcs[0] = m.src1[j]; a.srcs[1] = m.src2[j]; a.n_srcs = 2; a.strided = 0; a.src2 = nullptr; a.stride = 0;
    a.count = m.counts[j]; a.dt = m.dt; a.op = m.op; a.with_alpha = 0; a.alpha = 1.0;
    reduce_any(a, EC_GRID_TID, EC_GRID_NT);
}

/* ------------------------------------------------------------------ */
/* copies                                                              */
/* ------------------------------------------------------------------ */
static __device__ __forceinline__ void copy_grid(char *dst, const char *src, size_t n, size_t tid, size_t nt)
{
    if ((((uintptr_t)dst | (uintptr_t)src) & 15) == 0) {
        size_t nv = n / 16;
        for (size_t v = tid; v < nv; v += nt) st_v4(dst + v * 16, ld_src_v4(src + v * 16));
        for (size_t i = nv * 16 + tid; i < n; i += nt) dst[i] = src[i];
    } else for (size_t i = tid; i < n; i += nt) dst[i] = src[i];
}
__global__ void __launch_bounds__(1024) ec_copy_multi_kernel(ec_copy_multi_args_t c)
{
    int j = blockIdx.y;
    if (j >= c.n) return;
    copy_grid((char *)c.dst[j], (const char *)c.src[j], c.bytes[j], (size_t)blockIdx.x * blockDim.x + threadIdx.x, (size_t)gridDim.x * blockDim.x);
}

/* ------------------------------------------------------------------ */
/* persistent executor: worker blocks pop tasks from a host-pinned ring */
/* (reference ec/cuda/kernel/ec_cuda_executor.cu:125-188: num_workers blocks share one task ring).  Worker block w serves  */
/* slots w, w + W, w + 2W, ... - the host fills the ring in order, so consecutive tasks land on different workers and     */
/* run concurrently; inside a task only the worker's own threads take part (tid = threadIdx.x, nt = blockDim.x).        */
/* ------------------------------------------------------------------ */
__global__ void __launch_bounds__(1024) ec_persistent_kernel(ec_ring_t *ring)
{
    __shared__ uint32_t s_cmd; /* 0 = run slot, 1 = shutdown */
    uint32_t idx = blockIdx.x;
    const uint32_t W = gridDim.x;
    const size_t tid = threadIdx.x, nt = blockDim.x;
    if (blockIdx.x == 0 && threadIdx.x == 0) { ring->started = 1; __threadfence_system(); }
    for (;;) {
        ec_ring_slot_t *slot = &ring->slots[idx % ring->n_slots];
        if (threadIdx.x == 0) {
            uint32_t cmd;
            for (;;) {
                if (ring->shutdown) { cmd = 1; break; }
                if (slot->state == EC_SLOT_POSTED) { cmd = 0; break; }
            }
            __threadfence_system(); /* arguments written by the host before the state flip are visible now */
            s_cmd = cmd;
        }
        __syncthreads();
        if (s_cmd == 1) return;
        switch (slot->kind) {
        case EC_TASK_REDUCE: {
            ec_reduce_args_t a = slot->u.reduce;
            reduce_any(a, tid, nt);
            break; }
        case EC_TASK_REDUCE_MULTI_DST: {
            ec_reduce_multi_dst_args_t m = slot->u.rmd;
            for (int j = 0; j < m.n_bufs; j++) {
                ec_reduce_args_t a; a.dst = m.dst[j]; a.srcs[0] = m.src1[j]; a.srcs[1] = m.src2[j]; a.n_srcs = 2; a.strided = 0; a.src2 = nullptr; a.stride = 0;
                a.count = m.counts[j]; a.dt = m.dt; a.op = m.op; a.with_alpha = 0; a.alpha = 1.0;
                reduce_any(a, tid, nt);
            }
            break; }
        case EC_TASK_COPY: case EC_TASK_COPY_MULTI: {
            ec_copy_multi_args_t c = slot->u.copy;
            for (int j = 0; j < c.n; j++) copy_grid((char *)c.dst[j], (const char *)c.src[j], c.bytes[j], tid, nt);
            break; }
        default: break;
        }
        __syncthreads();
        if (threadIdx.x == 0) { __threadfence_system(); slot->state = EC_SLOT_DONE; }
        idx += W;
    }
}

__global__ void ec_wait_kernel(volatile uint32_t *state) { while (*state == 0) { } }

/* ------------------------------------------------------------------ */
extern "C" size_t ec_dt_size(int dt)
{ static const size_t s[EC_DT_LAST] = {1, 2, 4, 8, 1, 2, 4, 8, 2, 4, 8, 2, 8, 16}; return dt >= 0 && dt < EC_DT_LAST ? s[dt] : 0; }
extern "C" int ec_dt_supports_op(int dt, int op)
{
    if (dt < 0 || dt >= EC_DT_LAST || op < 0 || op >= EC_OP_LAST) return 0;
    if (dt == EC_DT_C64 || dt == EC_DT_C128) return op == EC_OP_SUM || op == EC_OP_PROD;
    if (dt == EC_DT_F16 || dt == EC_DT_F32 || dt == EC_DT_F64 || dt == EC_DT_BF16) return op <= EC_OP_MIN;
    return 1;
}
extern "C" cudaError_t ec_launch_reduce(const ec_reduce_args_t *a, int nblocks, int nthreads, cudaStream_t s)
{
    switch (a->dt) {
    case EC_DT_I8: return ec_launch_reduce_t<int8_t>(a, nblocks, nthreads, s); case EC_DT_I16: return ec_launch_reduce_t<int16_t>(a, nblocks, nthreads, s);
    case EC_DT_I32: return ec_launch_reduce_t<int32_t>(a, nblocks, nthreads, s); case EC_DT_I64: return ec_launch_reduce_t<int64_t>(a, nblocks, nthreads, s);
    case EC_DT_U8: return ec_launch_reduce_t<uint8_t>(a, nblocks, nthreads, s); case EC_DT_U16: return ec_launch_reduce_t<uint16_t>(a, nblocks, nthreads, s);
    case EC_DT_U32: return ec_launch_reduce_t<uint32_t>(a, nblocks, nthreads, s); case EC_DT_U64: return ec_launch_reduce_t<uint64_t>(a, nblocks, nthreads, s);
    case EC_DT_F16: return ec_launch_reduce_t<__half>(a, nblocks, nthreads, s); case EC_DT_BF16: return ec_launch_reduce_t<__nv_bfloat16>(a, nblocks, nthreads, s);
    case EC_DT_F32: return ec_launch_reduce_t<float>(a, nblocks, nthreads, s); case EC_DT_F64: return ec_launch_reduce_t<double>(a, nblocks, nthreads, s);
    case EC_DT_C64:
        if (a->op == EC_OP_SUM) ec_reduce_cplx_kernel_t<cuFloatComplex, EC_OP_SUM><<<nblocks, nthreads, 0, s>>>(*a);
        else if (a->op == EC_OP_PROD) ec_reduce_cplx_kernel_t<cuFloatComplex, EC_OP_PROD><<<nblocks, nthreads, 0, s>>>(*a);
        else return cudaErrorInvalidValue;
        return cudaGetLastError();
    case EC_DT_C128:
        if (a->op == EC_OP_SUM) ec_reduce_cplx_kernel_t<cuDoubleComplex, EC_OP_SUM><<<nblocks, nthreads, 0, s>>>(*a);
        else if (a->op == EC_OP_PROD) ec_reduce_cplx_kernel_t<cuDoubleComplex, EC_OP_PROD><<<nblocks, nthreads, 0, s>>>(*a);
        else return cudaErrorInvalidValue;
        return cudaGetLastError();
    default: return cudaErrorInvalidValue;
    }
}
extern "C" cudaError_t ec_launch_reduce_multi_dst(const ec_reduce_multi_dst_args_t *a, int nthreads, cudaStream_t s)
{ ec_reduce_multi_dst_kernel<<<dim3(4, a->n_bufs), nthreads, 0, s>>>(*a); return cudaGetLastError(); }
extern "C" cudaError_t ec_launch_copy_multi(const ec_copy_multi_args_t *a, int nthreads, cudaStream_t s)
{ ec_copy_multi_kernel<<<dim3(4, a->n), nthreads, 0, s>>>(*a); return cudaGetLastError(); }
extern "C" cudaError_t ec_launch_persistent(ec_ring_t *ring_dev, int nworkers, int nthreads, int cooperative, cudaStream_t s)
{
    /* the workers spin on their slots, so all of them must be resident at once: at most one per SM here (they are long-lived
     * and should leave room for everything else); the cooperative launch makes the runtime verify co-residency */
    if (nworkers < 1) nworkers = 1;
    if (cooperative) {
        void *args[] = {&ring_dev};
        return cudaLaunchCooperativeKernel((void *)ec_persistent_kernel, dim3((unsigned)nworkers), dim3((unsigned)nthreads), args, 0, s);
    }
    ec_persistent_kernel<<<nworkers, nthreads, 0, s>>>(ring_dev);
    return cudaGetLastError();
}
extern "C" cudaError_t ec_launch_wait(volatile uint32_t *state_dev, cudaStream_t s) { ec_wait_kernel<<<1, 1, 0, s>>>(state_dev); return cudaGetLastError(); }
