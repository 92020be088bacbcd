// Host emulation harness of the tl/nvl reduction kernels, shared by the drivers that check their numbers
// (nvl_emu_complex.cpp, nvl_emu_numerics.cpp): the kernel sources compiled as plain C++ (NVL_HOST_EMU), one OS thread per CUDA
// thread, every "GPU" a heap in this address space and the NVSwitch multicast window a fake address range (nvl_device_emu.h).
#ifndef NVL_EMU_WORLD_H_
#define NVL_EMU_WORLD_H_
#include <cstdio>
#include <cstdlib>
#include <cstdint>
#include <cstring>
#include <cmath>
#include <vector>
#include <thread>
#include <string>
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
nvl_emu_world g_emu;
#include "nvl_kernels.cu"
#include "nvl_pipe.cu"
#include "nvl_oneshot_rs.cu"
#include "nvl_symm.cu"

#define CHECK(c) do { if (!(c)) { printf("EMU FAIL line %d: %s\n", __LINE__, #c); exit(1); } } while (0)

struct World {
    int N; size_t data_size, user_size, heap_size;
    std::vector<char *> heaps; uint32_t host_err = 0;
    World(int n, size_t data, size_t user) : N(n), data_size(data), user_size(user)
    {
        heap_size = NVL_DATA_OFFSET + data + user;
        for (int p = 0; p < n; p++) { char *h = (char *)calloc(1, heap_size + 64); CHECK(h); heaps.push_back((char *)(((uintptr_t)h + 63) & ~(uintptr_t)63)); }
        g_emu.n = n; g_emu.heap_size = heap_size; g_emu.mc_base = (char *)(uintptr_t)0x500000000000ull;
        for (int p = 0; p < n; p++) g_emu.heaps[p] = heaps[p];
    }
    nvl_team_dev_t team(int r, bool nvls) const
    {
        nvl_team_dev_t t; memset(&t, 0, sizeof(t));
        t.rank = r; t.size = N; for (int p = 0; p < N; p++) t.heap[p] = heaps[p];
        t.mc_heap = nvls ? g_emu.mc_base : nullptr; t.data_size = data_size; t.timeout_ns = 60ull * 1000000000ull; t.host_err = const_cast<uint32_t *>(&host_err);
        return t;
    }
    char *user(int r) const { return heaps[r] + NVL_DATA_OFFSET + data_size; }
};

// run fn(rank) as a grid of nb x nt threads on every rank concurrently
template <typename F> static void launch_all(int N, int nb, int nt, F fn)
{
    std::vector<pthread_barrier_t> bars((size_t)N * nb);
    for (auto &b : bars) pthread_barrier_init(&b, nullptr, (unsigned)nt);
    std::vector<std::thread> th;
    th.reserve((size_t)N * nb * nt);
    for (int r = 0; r < N; r++) for (int b = 0; b < nb; b++) for (int t = 0; t < nt; t++)
        th.emplace_back([=, &bars]() {
            threadIdx = {(unsigned)t, 0, 0}; blockIdx = {(unsigned)b, 0, 0}; blockDim = {(unsigned)nt, 1, 1}; gridDim = {(unsigned)nb, 1, 1};
            emu_cta_barrier = &bars[(size_t)r * nb + b];
            fn(r);
        });
    for (auto &x : th) x.join();
    for (auto &b : bars) pthread_barrier_destroy(&b);
}

enum Kern { K_ONESHOT, K_ONESHOT_RS, K_STAGED, K_STAGED_NVLS, K_DIRECT, K_RING, K_RHD, K_PIPE, K_SYMM, K_LAST };
static const char *kname[K_LAST] = {"oneshot", "oneshot_rs", "staged p2p", "staged nvls", "direct", "ring", "rhd", "nvls_pipe", "symm"};
static inline bool kern_nvls(int k) { return k == K_STAGED_NVLS || k == K_PIPE || k == K_SYMM; }

template <typename T> static void run_kernel(int k, nvl_red_args_t a)
{
    switch (k) {
    case K_ONESHOT: nvl_allreduce_oneshot_kernel<T>(a); break;
    case K_ONESHOT_RS: nvl_reduce_scatter_oneshot_kernel<T>(a); break;
    case K_STAGED: case K_STAGED_NVLS: nvl_reduce_staged_kernel<T>(a); break;
    case K_DIRECT: nvl_reduce_direct_kernel<T>(a); break;
    case K_RING: a.sched = 1; nvl_reduce_steps_kernel<T>(a); break;
    case K_RHD: a.sched = 2; nvl_reduce_steps_kernel<T>(a); break;
    case K_PIPE: nvl_allreduce_nvls_pipe_kernel<T>(a); break;
    case K_SYMM: nvl_allreduce_symm_kernel<T>(a); break;
    }
}

/* one collective of kernel k on every rank, arguments built the way tl_nvl_coll.c builds them: src[r] / dst[r] are element
 * pointers of type T (REDUCE: dst only at the root; REDUCE_SCATTER: dst[r] = rank r's block).  REDUCE_SCATTER uses equal blocks
 * unless `rs` gives the count of every block (reduce_scatterv). */
template <typename T> static void launch(World &w, int k, int kind, int op, size_t count, const std::vector<T *> &src, const std::vector<T *> &dst,
                                         int root = 0, const std::vector<size_t> *rs = nullptr)
{
    const int N = w.N;
    const bool nvls = kern_nvls(k);
    const int nb = k == K_PIPE ? 1 : 2, nt = k == K_PIPE ? 128 : 32;
    launch_all(N, nb, nt, [&](int r) {
        nvl_red_args_t a; memset(&a, 0, sizeof(a));
        a.team = w.team(r, nvls); a.src = src[r]; a.dst = dst[r]; a.count = count; a.op = op; a.kind = kind; a.root = root; a.use_nvls = nvls;
        if (kind == NVL_RED_REDUCE_SCATTER) {
            size_t off = 0;
            for (int p = 0; p < N; p++) { a.rs_offset[p] = off; a.rs_count[p] = rs ? (*rs)[p] : count / N; off += a.rs_count[p]; }
        }
        if (k == K_DIRECT) { a.direct = NVL_DIRECT_FULL; for (int p = 0; p < N; p++) { a.d.src[p] = (const char *)src[p]; a.d.dst[p] = (char *)dst[p]; } }
        if (k == K_SYMM) { a.d.src[0] = (const char *)src[r]; a.d.dst[0] = (char *)dst[r]; }
        run_kernel<T>(k, a);
    });
    CHECK(w.host_err == 0);
}
#endif
