// Launchers of the tl/nvl kernels for the host-emulated build of the plugin that also serves the complex datatypes
// (tests/emu/build_hostemu_complex.sh, tests/test_nvl_complex.py): the launchers of nvl_emu_launch.cpp with float32_complex and
// float64_complex added to the datatypes it builds.  Same C interface as kernels/nvl_kernels.h; a launch enqueues a closure on the
// emulated stream (cudart_emu.cpp) that runs the grid with one OS thread per CUDA thread.
#include <cstdio>
#include <cstdlib>
#include <cstdint>
#include <cstring>
#include <functional>
#include <thread>
#include <vector>
#include <pthread.h>
#include <cuda_runtime_api.h>
#include <vector_types.h>
#include <vector_functions.h>
#define NVL_HOST_EMU 1
#ifndef __launch_bounds__
#define __launch_bounds__(...)
#endif
struct emu_dim3 { unsigned x, y, z; };
static thread_local emu_dim3 threadIdx, blockIdx, blockDim, gridDim;
static thread_local pthread_barrier_t *emu_cta_barrier;
static inline void __syncthreads() { pthread_barrier_wait(emu_cta_barrier); }
static inline void __threadfence() { __atomic_thread_fence(__ATOMIC_SEQ_CST); }
static inline unsigned atomicAdd(unsigned *p, unsigned v) { return __atomic_fetch_add(p, v, __ATOMIC_ACQ_REL); }

#include "nvl_reduce_impl.cuh"
nvl_emu_world g_emu;   /* no multicast in this build: teams never get an mc_heap */
#include "nvl_kernels.cu"
#include "nvl_pipe.cu"
#include "nvl_symm.cu"
#include "nvl_push.cu"
#include "nvl_oneshot_rs.cu"
#include "nvl_p2p.cu"

extern "C" void emu_stream_enqueue(cudaStream_t s, std::function<void()> *f);

template <typename F> static cudaError_t enqueue_grid(cudaStream_t s, int nb, int nt, F body)
{
    if (nb < 1 || nt < 1) return cudaErrorInvalidValue;
    std::function<void()> f = [nb, nt, body]() {
        std::vector<pthread_barrier_t> bars((size_t)nb);
        for (auto &b : bars) pthread_barrier_init(&b, nullptr, (unsigned)nt);
        std::vector<std::thread> th;
        th.reserve((size_t)nb * nt);
        for (int b = 0; b < nb; b++) for (int t = 0; t < nt; t++)
            th.emplace_back([=, &bars]() {
                threadIdx = {(unsigned)t, 0, 0}; blockIdx = {(unsigned)b, 0, 0}; blockDim = {(unsigned)nt, 1, 1}; gridDim = {(unsigned)nb, 1, 1};
                emu_cta_barrier = &bars[(size_t)b];
                body();
            });
        for (auto &x : th) x.join();
        for (auto &b : bars) pthread_barrier_destroy(&b);
    };
    emu_stream_enqueue(s, &f);
    return cudaSuccess;
}

/* a representative subset of the real datatypes plus both complex ones keeps the build of this test-only plugin short */
#define BY_DT(_a, _K)                                                                 \
    switch ((_a).dt) {                                                                \
    case NVL_DT_I32: return enqueue_grid(s, nb, nt, [a]() { _K<int32_t>(a); });       \
    case NVL_DT_I64: return enqueue_grid(s, nb, nt, [a]() { _K<int64_t>(a); });       \
    case NVL_DT_U8: return enqueue_grid(s, nb, nt, [a]() { _K<uint8_t>(a); });        \
    case NVL_DT_F32: return enqueue_grid(s, nb, nt, [a]() { _K<float>(a); });         \
    case NVL_DT_F64: return enqueue_grid(s, nb, nt, [a]() { _K<double>(a); });        \
    case NVL_DT_BF16: return enqueue_grid(s, nb, nt, [a]() { _K<__nv_bfloat16>(a); }); \
    case NVL_DT_C64: return enqueue_grid(s, nb, nt, [a]() { _K<nvl_c64>(a); });       \
    case NVL_DT_C128: return enqueue_grid(s, nb, nt, [a]() { _K<nvl_c128>(a); });     \
    default: return cudaErrorInvalidValue;                                            \
    }

template <typename T> static void direct_any(nvl_red_args_t a) { nvl_reduce_direct_kernel<T>(a); }

extern "C" {
size_t nvl_dt_size(int dt) { static const size_t sz[NVL_DT_LAST] = {1, 2, 4, 8, 1, 2, 4, 8, 2, 4, 8, 2, 8, 16}; return dt >= 0 && dt < NVL_DT_LAST ? sz[dt] : 0; }
int nvl_dt_supports_op(int dt, int op)
{
    if (dt < 0 || dt >= NVL_DT_LAST || op < 0 || op >= NVL_OP_LAST) return 0;
    if (dt != NVL_DT_I32 && dt != NVL_DT_I64 && dt != NVL_DT_U8 && dt != NVL_DT_F32 && dt != NVL_DT_F64 && dt != NVL_DT_BF16 && dt != NVL_DT_C64 && dt != NVL_DT_C128) return 0; /* not built here: falls back to the next TL */
    if (dt == NVL_DT_F16 || dt == NVL_DT_F32 || dt == NVL_DT_F64 || dt == NVL_DT_BF16) return op == NVL_OP_SUM || op == NVL_OP_PROD || op == NVL_OP_MAX || op == NVL_OP_MIN || op == NVL_OP_AVG;
    if (dt == NVL_DT_C64 || dt == NVL_DT_C128) return op == NVL_OP_SUM || op == NVL_OP_PROD || op == NVL_OP_AVG;
    return 1;
}
int nvl_nvls_supports(int, int) { return 0; }
cudaError_t nvl_launch_allreduce_oneshot(const nvl_red_args_t *ap, int nb, int nt, cudaStream_t s) { nvl_red_args_t a = *ap; BY_DT(a, nvl_allreduce_oneshot_kernel) }
cudaError_t nvl_launch_reduce_staged(const nvl_red_args_t *ap, int nb, int nt, cudaStream_t s) { nvl_red_args_t a = *ap; BY_DT(a, nvl_reduce_staged_kernel) }
cudaError_t nvl_launch_reduce_direct(const nvl_red_args_t *ap, int nb, int nt, cudaStream_t s) { nvl_red_args_t a = *ap; BY_DT(a, direct_any) }
cudaError_t nvl_launch_reduce_steps(const nvl_red_args_t *ap, int nb, int nt, cudaStream_t s) { nvl_red_args_t a = *ap; BY_DT(a, nvl_reduce_steps_kernel) }
cudaError_t nvl_launch_reduce_scatter_oneshot(const nvl_red_args_t *ap, int nb, int nt, cudaStream_t s) { nvl_red_args_t a = *ap; BY_DT(a, nvl_reduce_scatter_oneshot_kernel) }
cudaError_t nvl_launch_reduce_pipe(const nvl_red_args_t *, int, int, cudaStream_t) { return cudaErrorInvalidValue; }   /* NVLS only */
cudaError_t nvl_launch_reduce_symm(const nvl_red_args_t *, int, int, cudaStream_t) { return cudaErrorInvalidValue; }
cudaError_t nvl_launch_allgather_symm(const nvl_xchg_args_t *, int, int, cudaStream_t) { return cudaErrorInvalidValue; }
cudaError_t nvl_launch_exchange(const nvl_xchg_args_t *ap, int nb, int nt, cudaStream_t s) { nvl_xchg_args_t a = *ap; return enqueue_grid(s, nb, nt, [a]() { nvl_exchange_kernel(a); }); }
cudaError_t nvl_launch_exchange_push(const nvl_push_args_t *ap, int nb, int nt, cudaStream_t s) { nvl_push_args_t a = *ap; return enqueue_grid(s, nb, nt, [a]() { nvl_exchange_push_kernel(a); }); }
int nvl_p2p_lanes(size_t bytes) { size_t n = (bytes + NVL_P2P_LANE_BYTES - 1) / NVL_P2P_LANE_BYTES; return n < 1 ? 1 : (n > NVL_P2P_MAX_CTAS ? NVL_P2P_MAX_CTAS : (int)n); }
int nvl_p2p_push_ctas(size_t bytes) { size_t n = bytes / (64 * 1024); return n < 1 ? 1 : (n > 4 ? 4 : (int)n); }
cudaError_t nvl_launch_p2p(const nvl_p2p_args_t *ap, int nt, cudaStream_t s)
{
    nvl_p2p_args_t a = *ap;
    if (a.mode == NVL_P2P_PUSH) return enqueue_grid(s, nvl_p2p_push_ctas(a.bytes), nt > 64 ? 64 : nt, [a]() { nvl_p2p_push_kernel(a); });
    if (a.mode == NVL_P2P_WAIT) return enqueue_grid(s, 1, 32, [a]() { nvl_p2p_wait_kernel(a); });
    return enqueue_grid(s, nvl_p2p_lanes(a.bytes), nt > 64 ? 64 : nt, [a]() { nvl_p2p_kernel(a); });
}
cudaError_t nvl_launch_exchange_push_bulk(const nvl_push_args_t *ap, int nb, cudaStream_t s) { return nvl_launch_exchange_push(ap, nb, 32, s); }   /* no TMA here: the thread-copy kernel */
cudaError_t nvl_launch_barrier(const nvl_team_dev_t *tp, cudaStream_t s) { nvl_team_dev_t t = *tp; return enqueue_grid(s, 1, 32, [t]() { nvl_barrier_kernel(t); }); }
cudaError_t nvl_launch_self_copy(void *dst, const void *src, size_t bytes, int, int, cudaStream_t s)
{ return enqueue_grid(s, 1, 1, [=]() { memmove(dst, src, bytes); }); }
cudaError_t nvl_launch_self_copy_bulk(void *dst, const void *src, size_t bytes, int nb, cudaStream_t s) { return nvl_launch_self_copy(dst, src, bytes, nb, 32, s); }
cudaError_t nvl_launch_ctrl_init(void *heap_base, cudaStream_t s) { return enqueue_grid(s, 1, 1, [=]() { memset(heap_base, 0, sizeof(nvl_ctrl_t)); }); }
}
