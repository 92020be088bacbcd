/* Reduction kernels of tl/nvl (templates).  Each datatype is instantiated in its own translation unit
 * (nvl_red_<type>.cu) so the build parallelises; see nvl_kernels.cu for the design notes. */
#ifndef UCC_TL_NVL_REDUCE_IMPL_CUH_
#define UCC_TL_NVL_REDUCE_IMPL_CUH_
#include "nvl_device.cuh"

#define NVL_THREADS_MAX 512
/* bandwidth kernels: threads per CTA the register allocation is sized for (2 CTAs per SM: 512 -> 64 registers, 256 -> 128) and
 * the matching depth of the copy / in-switch reduction loops (16-byte transactions in flight per thread) */
#ifndef NVL_BW_THREADS
#define NVL_BW_THREADS 512
#endif
#define NVL_BW_U (NVL_BW_THREADS <= 256 ? 8 : 4)

/* Kernels are templates over (datatype, operator): the operator is chosen on the HOST at launch time, so each instantiation
 * carries exactly one reduction body (an operator switch inside the kernel made every kernel 11 bodies long and cost registers).
 *   GPU build : <name>_launch<T>(args, grid, block, stream) switches on args->op and launches <name>_t<T, OP>
 *   host emulation (tests/emu, kernels compiled as C++ functions): <name><T>(args) does the same switch and calls the body */
#ifdef NVL_HOST_EMU
#ifndef __grid_constant__
#define __grid_constant__
#endif
#define NVL_DEFINE_ENTRY(_name, _args_t)                                                                       \
    template <typename T> static void _name(_args_t a)                                                          \
    {                                                                                                          \
        NVL_DISPATCH_OP(T, a.op, NVL_ENTRY_CALL_##_name);                                                      \
    }
#define NVL_ENTRY_CALL_nvl_allreduce_oneshot_kernel(_T, _OP) nvl_allreduce_oneshot_kernel_t<_T, _OP>(a)
#define NVL_ENTRY_CALL_nvl_reduce_steps_kernel(_T, _OP) nvl_reduce_steps_kernel_t<_T, _OP>(a)
#define NVL_ENTRY_CALL_nvl_allreduce_nvls_pipe_kernel(_T, _OP) nvl_allreduce_nvls_pipe_kernel_t<_T, _OP>(a)
#define NVL_ENTRY_CALL_nvl_allreduce_symm_kernel(_T, _OP) nvl_allreduce_symm_kernel_t<_T, _OP>(a)
#define NVL_ENTRY_CALL_nvl_reduce_scatter_oneshot_kernel(_T, _OP) nvl_reduce_scatter_oneshot_kernel_t<_T, _OP>(a)
#else
#define NVL_DEFINE_ENTRY(_name, _args_t)                                                                       \
    template <typename T> static cudaError_t _name##_launch(const _args_t *ap, int nb, int nt, cudaStream_t s)  \
    {                                                                                                          \
        NVL_DISPATCH_OP(T, ap->op, NVL_ENTRY_CALL_##_name);                                                    \
        return cudaGetLastError();                                                                             \
    }
#define NVL_ENTRY_CALL_nvl_allreduce_oneshot_kernel(_T, _OP) nvl_allreduce_oneshot_kernel_t<_T, _OP><<<nb, nt, 0, s>>>(*ap)
#define NVL_ENTRY_CALL_nvl_reduce_steps_kernel(_T, _OP) nvl_reduce_steps_kernel_t<_T, _OP><<<nb, nt, 0, s>>>(*ap)
#define NVL_ENTRY_CALL_nvl_allreduce_nvls_pipe_kernel(_T, _OP) nvl_allreduce_nvls_pipe_kernel_t<_T, _OP><<<nb, nt, 0, s>>>(*ap)
#define NVL_ENTRY_CALL_nvl_allreduce_symm_kernel(_T, _OP) nvl_allreduce_symm_kernel_t<_T, _OP><<<nb, nt, 0, s>>>(*ap)
#define NVL_ENTRY_CALL_nvl_reduce_scatter_oneshot_kernel(_T, _OP) nvl_reduce_scatter_oneshot_kernel_t<_T, _OP><<<nb, nt, 0, s>>>(*ap)
#endif

/* ------------------------------------------------------------------ */
/* small helpers                                                       */
/* ------------------------------------------------------------------ */
static __device__ __forceinline__ size_t dmin(size_t a, size_t b) { return a < b ? a : b; }
static __device__ __forceinline__ char *data_of(const nvl_team_dev_t &t, int p) { return t.heap[p] + NVL_DATA_OFFSET; }

/* block-strided copy of 16-byte vectors [v0,v1): U loads in flight per thread */
template <int U, bool PEER> static __device__ __forceinline__ void copy_vecs(char *dst, const char *src, size_t v0, size_t v1)
{
    const size_t nt = blockDim.x;
    size_t v = v0 + threadIdx.x;
    for (; v + (U - 1) * nt < v1; v += U * nt) {
        uint4 x[U];
#pragma unroll
        for (int u = 0; u < U; u++) x[u] = PEER ? ld_peer_v4(src + (v + u * nt) * 16) : ld_src_v4(src + (v + u * nt) * 16);
#pragma unroll
        for (int u = 0; u < U; u++) st_v4(dst + (v + u * nt) * 16, x[u]);
    }
    for (; v < v1; v += nt) st_v4(dst + v * 16, PEER ? ld_peer_v4(src + v * 16) : ld_src_v4(src + v * 16));
}

/* ------------------------------------------------------------------ */
/* one-shot push allreduce (latency path)                              */
/*   every rank stores its vector into a private slot of every peer's  */
/*   heap, raises a flag, then reduces the N vectors it received.      */
/*   Two slot sets alternate so no trailing barrier is needed.         */
/* ------------------------------------------------------------------ */
template <typename T, int OP>
static __device__ __forceinline__ void oneshot_body(const nvl_red_args_t &a, nvl_ctrl_t *mine, uint32_t seq)
{
    constexpr int E = 16 / sizeof(T);
    const nvl_team_dev_t &t = a.team;
    const int N = t.size, me = t.rank;
    const T *src = static_cast<const T *>(a.src);
    T *dst = static_cast<T *>(a.dst);
    const size_t n = a.count, nvec = (n + E - 1) / E;
    const size_t per = (nvec + gridDim.x - 1) / gridDim.x, v0 = dmin((size_t)blockIdx.x * per, nvec), v1 = dmin(v0 + per, nvec);
    const bool sal = ((uintptr_t)src & 15) == 0, dal = ((uintptr_t)dst & 15) == 0;
    const size_t slot = (size_t)((seq & 1) * NVL_MAX_PEERS) * NVL_LL_MAX;

    for (size_t v = v0 + threadIdx.x; v < v1; v += blockDim.x) {
        uint4 x = load_src_vec<T>(src, v * E, n, sal);
        for (int i = 1; i < N; i++) { /* start at my right neighbour so the N senders do not hit one peer at once */
            int p = me + i; if (p >= N) p -= N;
            st_v4(t.heap[p] + NVL_LL_OFFSET + slot + (size_t)me * NVL_LL_MAX + v * 16, x);
        }
    }
    __syncthreads();
    if ((int)threadIdx.x < N && (int)threadIdx.x != me) {
        fence_sys();
        st_relaxed_sys_u32(&reinterpret_cast<nvl_ctrl_t *>(t.heap[threadIdx.x])->ll_flags[blockIdx.x][me], seq);
        BlockSync bs; bs.mine = mine;
        bs.spin(t, &mine->ll_flags[blockIdx.x][threadIdx.x], seq);
    }
    __syncthreads();
    /* reduce in rank order 0..N-1 on every rank (vector p: my own source for p == me, slot p of my heap otherwise), so that
     * every rank stores the same bits - floating-point addition is not associative, and replicas of a data-parallel model
     * drift apart when their gradients differ in the last bit.  The reads hit my own heap, so their order costs nothing.
     * x[] is only indexed with unrolled constants: no local-memory stack. */
    const char *mybase = t.heap[me] + NVL_LL_OFFSET + slot;
    for (size_t v = v0 + threadIdx.x; v < v1; v += blockDim.x) {
        uint4 x[NVL_MAX_PEERS];
#pragma unroll
        for (int p = 0; p < NVL_MAX_PEERS; p++)
            if (p < N) x[p] = p == me ? load_src_vec<T>(src, v * E, n, sal) : ld_peer_v4(mybase + (size_t)p * NVL_LL_MAX + v * 16);
        VecAcc<T, OP> acc; acc.set(x[0]);
#pragma unroll
        for (int p = 1; p < NVL_MAX_PEERS; p++) if (p < N) acc.add(x[p]);
        store_dst_vec<T>(dst, v * E, n, dal, acc.get(N));
    }
}

/* One sequence number per TEAM (ctrl.ll_seq[0]; ll_seq[1] counts the finished blocks of the running kernel): every block of a
 * launch reads the same value - it only advances when the LAST block of a kernel retires - so the slot parity is the same for
 * all blocks whatever the grid size of this launch and of the previous ones.  (A per-block sequence let two consecutive launches
 * with different grids pick the same slot set for overlapping vector ranges.)  Shared by the one-shot allreduce and the one-shot
 * reduce_scatter; it lives on the device, so captured (CUDA graph) launches replay correctly. */
static __device__ __forceinline__ uint32_t ll_seq_begin(nvl_ctrl_t *mine) { return ld_volatile_u32(&mine->ll_seq[0]) + 1; }
static __device__ __forceinline__ void ll_seq_end(nvl_ctrl_t *mine, uint32_t seq)
{
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        if (atomicAdd(&mine->ll_seq[1], 1u) == gridDim.x - 1) { mine->ll_seq[1] = 0; __threadfence(); mine->ll_seq[0] = seq; }
    }
}

template <typename T, int OP> __global__ void __launch_bounds__(NVL_THREADS_MAX) nvl_allreduce_oneshot_kernel_t(const __grid_constant__ nvl_red_args_t a)
{
    nvl_ctrl_t *mine = reinterpret_cast<nvl_ctrl_t *>(a.team.heap[a.team.rank]);
    const uint32_t seq = ll_seq_begin(mine);
    oneshot_body<T, OP>(a, mine, seq);
    ll_seq_end(mine, seq);
}
NVL_DEFINE_ENTRY(nvl_allreduce_oneshot_kernel, nvl_red_args_t)

/* ------------------------------------------------------------------ */
/* staged two-shot reduction: allreduce / reduce_scatter(v) / reduce   */
/* ------------------------------------------------------------------ */
/* (datatype, operator) pairs the NVSwitch can reduce; must mirror nvl_nvls_supports() in nvl_kernels.cu */
template <typename T, int OP> struct McRed { static __device__ __forceinline__ uint4 ld(const void *) { return make_uint4(0, 0, 0, 0); } };
#define NVL_MCRED(_T, _OP, _fn) template <> struct McRed<_T, _OP> { static __device__ __forceinline__ uint4 ld(const void *p) { return _fn(p); } };
NVL_MCRED(float, NVL_OP_SUM, mc_ld_reduce_f32) NVL_MCRED(float, NVL_OP_AVG, mc_ld_reduce_f32)
NVL_MCRED(__half, NVL_OP_SUM, mc_ld_reduce_f16) NVL_MCRED(__half, NVL_OP_AVG, mc_ld_reduce_f16)
NVL_MCRED(__nv_bfloat16, NVL_OP_SUM, mc_ld_reduce_bf16) NVL_MCRED(__nv_bfloat16, NVL_OP_AVG, mc_ld_reduce_bf16)
/* c64 SUM / AVG are f32 adds part by part; c128 would need the scalar f64 form, which would also move f64 onto this path */
NVL_MCRED(nvl_c64, NVL_OP_SUM, mc_ld_reduce_f32) NVL_MCRED(nvl_c64, NVL_OP_AVG, mc_ld_reduce_f32)
NVL_MCRED(int32_t, NVL_OP_SUM, mc_red_add_s32) NVL_MCRED(int32_t, NVL_OP_MIN, mc_red_min_s32) NVL_MCRED(int32_t, NVL_OP_MAX, mc_red_max_s32)
NVL_MCRED(int32_t, NVL_OP_BAND, mc_red_and_b32) NVL_MCRED(int32_t, NVL_OP_BOR, mc_red_or_b32) NVL_MCRED(int32_t, NVL_OP_BXOR, mc_red_xor_b32)
NVL_MCRED(uint32_t, NVL_OP_SUM, mc_red_add_u32) NVL_MCRED(uint32_t, NVL_OP_MIN, mc_red_min_u32) NVL_MCRED(uint32_t, NVL_OP_MAX, mc_red_max_u32)
NVL_MCRED(uint32_t, NVL_OP_BAND, mc_red_and_b32) NVL_MCRED(uint32_t, NVL_OP_BOR, mc_red_or_b32) NVL_MCRED(uint32_t, NVL_OP_BXOR, mc_red_xor_b32)
NVL_MCRED(int64_t, NVL_OP_SUM, mc_red_add_u64) NVL_MCRED(int64_t, NVL_OP_MIN, mc_red_min_s64) NVL_MCRED(int64_t, NVL_OP_MAX, mc_red_max_s64)
NVL_MCRED(int64_t, NVL_OP_BAND, mc_red_and_b64) NVL_MCRED(int64_t, NVL_OP_BOR, mc_red_or_b64) NVL_MCRED(int64_t, NVL_OP_BXOR, mc_red_xor_b64)
NVL_MCRED(uint64_t, NVL_OP_SUM, mc_red_add_u64) NVL_MCRED(uint64_t, NVL_OP_MIN, mc_red_min_u64) NVL_MCRED(uint64_t, NVL_OP_MAX, mc_red_max_u64)
NVL_MCRED(uint64_t, NVL_OP_BAND, mc_red_and_b64) NVL_MCRED(uint64_t, NVL_OP_BOR, mc_red_or_b64) NVL_MCRED(uint64_t, NVL_OP_BXOR, mc_red_xor_b64)

/* Slice geometry.  Deliberately scalar: per-slice offsets / counts are recomputed from the kernel parameters (constant bank,
 * dynamically indexable) instead of living in a per-thread array, which the compiler would have to put on the local-memory stack. */
struct SlicePlan {
    size_t slice_max, cap_e;   /* longest slice; elements of one slice per round */
    size_t se;                 /* allreduce / reduce: elements per slice (multiple of a vector) */
    int    rounds;
};
static __device__ __forceinline__ size_t slice_off(const nvl_red_args_t &a, const SlicePlan &pl, int s)
{ return a.kind == NVL_RED_REDUCE_SCATTER ? a.rs_offset[s] : dmin((size_t)s * pl.se, a.count); }
static __device__ __forceinline__ size_t slice_cnt(const nvl_red_args_t &a, const SlicePlan &pl, int s)
{ if (a.kind == NVL_RED_REDUCE_SCATTER) return a.rs_count[s]; const size_t o = dmin((size_t)s * pl.se, a.count); return dmin(pl.se, a.count - o); }

template <typename T> static __device__ __forceinline__ void make_plan(const nvl_red_args_t &a, SlicePlan &pl)
{
    constexpr int E = 16 / sizeof(T);
    const int N = a.team.size;
    pl.slice_max = 0; pl.se = 0;
    if (a.kind == NVL_RED_REDUCE_SCATTER) {
        for (int s = 0; s < N; s++) if (a.rs_count[s] > pl.slice_max) pl.slice_max = a.rs_count[s];
    } else {
        size_t se = (a.count + N - 1) / N; se = (se + E - 1) / E * E;
        pl.se = se; pl.slice_max = se;
    }
    pl.cap_e = (a.team.data_size / N / 16) * E;
    pl.rounds = (int)((pl.slice_max + pl.cap_e - 1) / pl.cap_e);
}

/* The reduction loop shared by the staged and the zero-copy kernels: vectors [j0,jend) of my slice.  src_of(i) = base address of
 * the i-th source (i = 0: my own copy, then my right neighbours), store(jj, r) disposes of the reduced vector jj.
 * Sources are consumed in groups of NP with U vectors per thread in flight (U x NP 16-byte loads outstanding; the NVLink
 * bandwidth-delay product needs ~20 bytes per resident thread, so NP <= 4 keeps the loop inside the 64-register budget of
 * 2 x 512 threads per SM).  CN = team size when it is one of the common ones (2, 4, 8): every bound below is then a
 * compile-time constant and the loop carries no predicates; CN = 0 is the generic team size. */
template <typename T, int OP, int CN, int NP, int U, typename SRC, typename ST>
static __device__ __forceinline__ void reduce_core(int n_rt, size_t j0, size_t jend, SRC src_of, ST store)
{
    const int N = CN ? CN : n_rt;
    const size_t nt = blockDim.x;
    for (size_t j = j0 + threadIdx.x; j < jend; j += U * nt) {
        VecAcc<T, OP> acc[U];
        {
            uint4 x[U][NP];
#pragma unroll
            for (int u = 0; u < U; u++) {
                const size_t jj = j + u * nt;
                if (jj < jend) {
#pragma unroll
                    for (int i = 0; i < NP; i++) if (i < N) x[u][i] = ld_peer_v4(src_of(i) + jj * 16);
                }
            }
#pragma unroll
            for (int u = 0; u < U; u++) {
                if (j + u * nt < jend) {
                    acc[u].set(x[u][0]);
#pragma unroll
                    for (int i = 1; i < NP; i++) if (i < N) acc[u].add(x[u][i]);
                }
            }
        }
#pragma unroll 2
        for (int g = NP; g < N; g += NP) {
            uint4 x[U][NP];
#pragma unroll
            for (int u = 0; u < U; u++) {
                const size_t jj = j + u * nt;
                if (jj < jend) {
#pragma unroll
                    for (int i = 0; i < NP; i++) if (g + i < N) x[u][i] = ld_peer_v4(src_of(g + i) + jj * 16);
                }
            }
#pragma unroll
            for (int u = 0; u < U; u++) {
                if (j + u * nt < jend) {
#pragma unroll
                    for (int i = 0; i < NP; i++) if (g + i < N) acc[u].add(x[u][i]);
                }
            }
        }
#pragma unroll
        for (int u = 0; u < U; u++) {
            const size_t jj = j + u * nt;
            if (jj < jend) store(jj, acc[u].get(N));
        }
    }
}
/* team size -> kernel class */
static inline int nvl_size_class(int n) { return (n == 2 || n == 4 || n == 8) ? n : 0; }
template <int CN> struct RedShape { static constexpr int NP = CN == 2 ? 2 : 4, U = (CN == 2 ? 2 : 1) * (NVL_BW_THREADS <= 256 ? 2 : 1); };

/* phase B of the staged kernel over P2P: sources = the members' staging areas, result -> every member's staging area
 * (allreduce), the root's (reduce) or straight into my destination block (reduce_scatter) */
template <typename T, int OP, int CN>
static __device__ __forceinline__ void reduce_p2p(const nvl_red_args_t &a, size_t base, size_t j0, size_t jend, T *db, size_t rc, bool dal)
{
    constexpr int E = 16 / sizeof(T);
    const int N = CN ? CN : a.team.size, me = a.team.rank;
    auto src_of = [&](int i) -> char * { int p = me + i; if (p >= N) p -= N; return data_of(a.team, p) + base; };
    auto store = [&](size_t jj, uint4 r) {
        if (a.kind == NVL_RED_ALLREDUCE) {
#pragma unroll 4
            for (int i = 0; i < N; i++) st_v4(src_of(i) + jj * 16, r);
        } else if (a.kind == NVL_RED_REDUCE) st_v4(data_of(a.team, a.root) + base + jj * 16, r);
        else store_dst_vec<T>(db, jj * E, rc, dal, r);
    };
    reduce_core<T, OP, CN, RedShape<CN>::NP, RedShape<CN>::U>(N, j0, jend, src_of, store);
}

template <typename T, int OP, int U>
static __device__ __forceinline__ void reduce_nvls(const nvl_red_args_t &a, size_t base, size_t j0, size_t jend, T *db, size_t rc, bool dal)
{
    constexpr int E = 16 / sizeof(T);
    const size_t nt = blockDim.x;
    char *mc = a.team.mc_heap + NVL_DATA_OFFSET + base;
    for (size_t j = j0 + threadIdx.x; j < jend; j += U * nt) {
        uint4 r[U];
#pragma unroll
        for (int u = 0; u < U; u++) if (j + u * nt < jend) r[u] = McRed<T, OP>::ld(mc + (j + u * nt) * 16);
#pragma unroll
        for (int u = 0; u < U; u++) {
            const size_t jj = j + u * nt;
            if (jj < jend) {
                uint4 v = r[u];
                if (OP == NVL_OP_AVG) { VecAcc<T, OP> acc; acc.set(v); v = acc.get(a.team.size); }
                if (a.kind == NVL_RED_ALLREDUCE) mc_st_v4(mc + jj * 16, v);
                else if (a.kind == NVL_RED_REDUCE) st_v4(data_of(a.team, a.root) + base + jj * 16, v);
                else store_dst_vec<T>(db, jj * E, rc, dal, v);
            }
        }
    }
}

/* MODE: -1 = reduce in the switch (NVLS), otherwise the P2P team-size class CN (2, 4, 8; 0 = any other size) */
template <typename T, int OP, int MODE>
static __device__ __forceinline__ void staged_body(const nvl_red_args_t &a, BlockSync &bs, const SlicePlan &pl)
{
    constexpr int E = 16 / sizeof(T);
    const nvl_team_dev_t &t = a.team;
    const int N = t.size, me = t.rank, nb = gridDim.x, b = blockIdx.x;
    const T *src = static_cast<const T *>(a.src);
    T *dst = static_cast<T *>(a.dst);
    const size_t cap_bytes = pl.cap_e * sizeof(T);
    char *mydata = data_of(t, me);

    for (int k = 0; k < pl.rounds; k++) {
        const size_t e0 = (size_t)k * pl.cap_e;                       /* first element of every slice in this round */
        const size_t rmax = dmin(pl.cap_e, pl.slice_max - e0);        /* longest slice part in this round */
        /* Blocks only synchronise with the SAME block of the peers, so block b may be a round ahead of block b' of its own rank:
         * the vector range a block owns must not move between rounds.  With several rounds it is cut from the full round
         * capacity (a shorter last round leaves the upper blocks idle) - cutting it from the round's own length let block b's
         * staging of the last round overwrite heap vectors block b' had not copied out yet (found in the host emulation). */
        const size_t nvmax = (rmax + E - 1) / E, nvsplit = pl.rounds > 1 ? pl.cap_e / E : nvmax, per = (nvsplit + nb - 1) / nb;
        const size_t j0 = dmin((size_t)b * per, nvmax), j1 = dmin(j0 + per, nvmax); /* my vector range inside every slice */

        /* phase A: stage vector range [j0,j1) of EVERY slice into my heap */
        for (int s = 0; s < N; s++) {
            const size_t rc = slice_cnt(a, pl, s) > e0 ? dmin(pl.cap_e, slice_cnt(a, pl, s) - e0) : 0;
            const size_t nfull = rc / E, jend = dmin(j1, (rc + E - 1) / E);
            const T *sb = src + slice_off(a, pl, s) + e0;
            char *hb = mydata + (size_t)s * cap_bytes;
            if (((uintptr_t)sb & 15) == 0) {
                copy_vecs<NVL_BW_U, false>(hb, reinterpret_cast<const char *>(sb), j0, dmin(jend, nfull));
                /* ragged tail: by the thread that owns this vector index in copy_vecs (v = j0 + tid mod blockDim) - the same thread
                 * copied the vector out of the heap in the previous round's phase C, and there is no block barrier in between */
                if (nfull >= j0 && nfull < jend && threadIdx.x == (unsigned)((nfull - j0) % blockDim.x)) st_v4(hb + nfull * 16, load_src_vec<T>(sb, nfull * E, rc, false));
            } else {
                for (size_t j = j0 + threadIdx.x; j < jend; j += blockDim.x) st_v4(hb + j * 16, load_src_vec<T>(sb, j * E, rc, false));
            }
        }
        bs.barrier(t, 2 * k + 1);

        /* phase B: reduce my slice from every member's staging area (over NVLink or in the switch) and publish it */
        {
            const size_t rc = slice_cnt(a, pl, me) > e0 ? dmin(pl.cap_e, slice_cnt(a, pl, me) - e0) : 0;
            const size_t jend = dmin(j1, (rc + E - 1) / E), base = (size_t)me * cap_bytes;
            T *db = dst + (a.kind == NVL_RED_REDUCE_SCATTER ? 0 : slice_off(a, pl, me)) + e0;
            const bool dal = ((uintptr_t)db & 15) == 0;
            if constexpr (MODE < 0) reduce_nvls<T, OP, NVL_BW_U>(a, base, j0, jend, db, rc, dal);
            else reduce_p2p<T, OP, MODE>(a, base, j0, jend, db, rc, dal);
        }
        bs.barrier(t, 2 * k + 2);

        /* phase C: my heap now holds vector range [j0,j1) of every reduced slice */
        if (a.kind == NVL_RED_ALLREDUCE || (a.kind == NVL_RED_REDUCE && me == a.root)) {
            for (int s = 0; s < N; s++) {
                const size_t rc = slice_cnt(a, pl, s) > e0 ? dmin(pl.cap_e, slice_cnt(a, pl, s) - e0) : 0;
                const size_t nfull = rc / E, jend = dmin(j1, (rc + E - 1) / E);
                T *db = dst + slice_off(a, pl, s) + e0;
                const char *hb = mydata + (size_t)s * cap_bytes;
                if (((uintptr_t)db & 15) == 0) {
                    copy_vecs<NVL_BW_U, true>(reinterpret_cast<char *>(db), hb, j0, dmin(jend, nfull));
                    if (nfull >= j0 && nfull < jend && threadIdx.x == (unsigned)((nfull - j0) % blockDim.x)) store_dst_vec<T>(db, nfull * E, rc, false, ld_peer_v4(hb + nfull * 16));
                } else {
                    for (size_t j = j0 + threadIdx.x; j < jend; j += blockDim.x) store_dst_vec<T>(db, j * E, rc, false, ld_peer_v4(hb + j * 16));
                }
            }
        }
    }
}

template <typename T, int OP, int MODE> __global__ void __launch_bounds__(NVL_BW_THREADS, 2) nvl_reduce_staged_kernel_t(const __grid_constant__ nvl_red_args_t a)
{
    BlockSync bs; bs.init(a.team);
    SlicePlan pl; make_plan<T>(a, pl);
    staged_body<T, OP, MODE>(a, bs, pl);
    bs.finish(2 * (uint32_t)pl.rounds);
}
static inline int nvl_staged_mode(const nvl_red_args_t &a) { return (a.use_nvls && a.team.mc_heap) ? -1 : nvl_size_class(a.team.size); }
#ifdef NVL_HOST_EMU
#define NVL_STAGED_GO(_T, _OP, _M) nvl_reduce_staged_kernel_t<_T, _OP, _M>(a)
#define NVL_STAGED_ARGS a
#else
#define NVL_STAGED_GO(_T, _OP, _M) nvl_reduce_staged_kernel_t<_T, _OP, _M><<<nb, nt, 0, s>>>(*ap)
#define NVL_STAGED_ARGS (*ap)
#endif
#define NVL_CALL_STAGED(_T, _OP) do { switch (nvl_staged_mode(NVL_STAGED_ARGS)) { case -1: NVL_STAGED_GO(_T, _OP, -1); break; case 2: NVL_STAGED_GO(_T, _OP, 2); break; \
    case 4: NVL_STAGED_GO(_T, _OP, 4); break; case 8: NVL_STAGED_GO(_T, _OP, 8); break; default: NVL_STAGED_GO(_T, _OP, 0); break; } } while (0)
#ifdef NVL_HOST_EMU
template <typename T> static void nvl_reduce_staged_kernel(nvl_red_args_t a) { NVL_DISPATCH_OP(T, a.op, NVL_CALL_STAGED); }
#else
template <typename T> static cudaError_t nvl_reduce_staged_kernel_launch(const nvl_red_args_t *ap, int nb, int nt, cudaStream_t s)
{ NVL_DISPATCH_OP(T, ap->op, NVL_CALL_STAGED); return cudaGetLastError(); }
#endif


/* ------------------------------------------------------------------ */
/* zero-copy two-shot: no staging, no copy-out                         */
/*   barrier (every member's kernel is running => its src is final and */
/*   its dst may be written) -> reduce my slice straight from the N    */
/*   src buffers -> store into every member's dst -> barrier.          */
/*   Each byte crosses NVLink exactly once per direction and HBM is    */
/*   touched only for the payload itself.                              */
/* ------------------------------------------------------------------ */
/* The host ROTATES the pointer tables before the launch (nvl_direct_rotate): a.d.src[i] / a.d.dst[i] belong to my i-th right
 * neighbour (i = 0: myself).  Inside the unrolled loops every index is a compile-time constant, so the addresses are formed
 * straight from the constant bank that holds the kernel parameters - no pointer table in registers, nothing on the stack. */
template <typename T, int OP, int CN>
static __device__ __forceinline__ void direct_p2p(const nvl_red_args_t &a, size_t so, size_t j0, size_t jend)
{
    const int N = CN ? CN : a.team.size;
    const int rooti = a.kind == NVL_RED_REDUCE ? (a.root - a.team.rank + N) % N : 0;
    char *const single = a.kind == NVL_RED_REDUCE ? a.d.dst[rooti] + so : static_cast<char *>(a.dst); /* REDUCE: the root's dst; REDUCE_SCATTER: my block */
    auto src_of = [&](int i) -> const char * { return a.d.src[i] + so; };
    auto store = [&](size_t jj, uint4 r) {
        if (a.kind == NVL_RED_ALLREDUCE) {
#pragma unroll 8
            for (int i = 0; i < N; i++) st_v4(a.d.dst[i] + so + jj * 16, r);
        } else st_v4(single + jj * 16, r);
    };
    reduce_core<T, OP, CN, RedShape<CN>::NP, RedShape<CN>::U>(N, j0, jend, src_of, store);
}

template <typename T, int OP, int CN>
static __device__ __forceinline__ void direct_body(const nvl_red_args_t &a, const SlicePlan &pl)
{
    constexpr int E = 16 / sizeof(T);
    typedef typename AccOf<T>::type A;
    const nvl_team_dev_t &t = a.team;
    const int N = CN ? CN : t.size, me = t.rank, nb = gridDim.x, b = blockIdx.x;
    const size_t cnt = slice_cnt(a, pl, me), nfull = cnt / E, per = (nfull + nb - 1) / nb;
    const size_t j0 = dmin((size_t)b * per, nfull), j1 = dmin(j0 + per, nfull);
    const size_t so = slice_off(a, pl, me) * sizeof(T);
    /* in flight per thread: U x NP 16-byte loads; 2 CTAs x 512 threads per SM keep > 64 KB outstanding per SM, far above
     * the NVLink bandwidth-delay product */
    direct_p2p<T, OP, CN>(a, so, j0, j1); /* the team size class is a kernel template parameter: each class gets its own register allocation */
    /* ragged tail of the slice (fewer than E elements): one thread, element by element (cold; dynamic constant-bank indexing) */
    if (b == nb - 1 && threadIdx.x == 0 && nfull * E < cnt) {
        const int rooti = a.kind == NVL_RED_REDUCE ? (a.root - me + N) % N : 0;
        for (size_t e = nfull * E; e < cnt; e++) {
            A acc = to_acc<T>(reinterpret_cast<const T *>(a.d.src[0] + so)[e]);
            for (int i = 1; i < N; i++) acc = OpFn<OP, A>::f(acc, to_acc<T>(reinterpret_cast<const T *>(a.d.src[i] + so)[e]));
            acc = avg_scale<OP, A>(acc, N);
            if (a.kind == NVL_RED_ALLREDUCE) { for (int i = 0; i < N; i++) reinterpret_cast<T *>(a.d.dst[i] + so)[e] = from_acc<T>(acc); }
            else if (a.kind == NVL_RED_REDUCE) reinterpret_cast<T *>(a.d.dst[rooti] + so)[e] = from_acc<T>(acc);
            else static_cast<T *>(a.dst)[e] = from_acc<T>(acc); /* reduce_scatter(v): my block, already a local pointer */
        }
    }
}

template <typename T, int OP, int CN> __global__ void __launch_bounds__(NVL_BW_THREADS, 2) nvl_reduce_direct_kernel_t(const __grid_constant__ nvl_red_args_t a)
{
    BlockSync bs; bs.init(a.team);
    SlicePlan pl; make_plan<T>(a, pl);
    bs.barrier(a.team, 1);
    direct_body<T, OP, CN>(a, pl);
    bs.barrier(a.team, 2);
    bs.finish(2);
}
/* team-size class -> instantiation */
template <typename T, int OP> struct nvl_reduce_direct_by_size {
#ifdef NVL_HOST_EMU
    static void run(const nvl_red_args_t &a)
    {
        switch (nvl_size_class(a.team.size)) {
        case 2: nvl_reduce_direct_kernel_t<T, OP, 2>(a); break;
        case 4: nvl_reduce_direct_kernel_t<T, OP, 4>(a); break;
        case 8: nvl_reduce_direct_kernel_t<T, OP, 8>(a); break;
        default: nvl_reduce_direct_kernel_t<T, OP, 0>(a); break;
        }
    }
#else
    static void launch(const nvl_red_args_t &a, int nb, int nt, cudaStream_t s)
    {
        switch (nvl_size_class(a.team.size)) {
        case 2: nvl_reduce_direct_kernel_t<T, OP, 2><<<nb, nt, 0, s>>>(a); break;
        case 4: nvl_reduce_direct_kernel_t<T, OP, 4><<<nb, nt, 0, s>>>(a); break;
        case 8: nvl_reduce_direct_kernel_t<T, OP, 8><<<nb, nt, 0, s>>>(a); break;
        default: nvl_reduce_direct_kernel_t<T, OP, 0><<<nb, nt, 0, s>>>(a); break;
        }
    }
#endif
};
#ifdef NVL_HOST_EMU
template <typename T> static void nvl_reduce_direct_kernel(nvl_red_args_t a)
{
    nvl_direct_rotate(&a);
#define NVL_CALL_DIRECT(_T, _OP) nvl_reduce_direct_by_size<_T, _OP>::run(a)
    NVL_DISPATCH_OP(T, a.op, NVL_CALL_DIRECT);
}
#else
template <typename T> static cudaError_t nvl_reduce_direct_kernel_launch(const nvl_red_args_t *ap, int nb, int nt, cudaStream_t s)
{
    nvl_red_args_t a = *ap;
    nvl_direct_rotate(&a);
#define NVL_CALL_DIRECT(_T, _OP) nvl_reduce_direct_by_size<_T, _OP>::launch(a, nb, nt, s)
    NVL_DISPATCH_OP(T, a.op, NVL_CALL_DIRECT);
    return cudaGetLastError();
}
#endif

/* ------------------------------------------------------------------ */
/* step-structured allreduce / reduce_scatter through the heaps:       */
/*   sched 1: ring (N-1 reduce-scatter steps + N-1 allgather steps,    */
/*            neighbour links only)                                    */
/*   sched 2: recursive halving + recursive doubling (log2 N + log2 N  */
/*            pairwise steps; "SRA" with radix 2, power-of-two teams)  */
/* Both keep every slice at the same heap slot on every rank and give  */
/* block b the same vector range of every slice, so one per-block flag */
/* wait per step is all the synchronisation needed.  Single round: the */
/* vector has to fit the heap (larger ones use the two-shot kernels).  */
/* ------------------------------------------------------------------ */
/* acc[j] = op(peer[j], mine[j]) for my block's vectors of one slice; optionally scaled (AVG) and mirrored into dst */
template <typename T, int OP>
static __device__ __forceinline__ void step_reduce(const char *peer, char *mine, size_t j0, size_t jend, bool last, int N, T *db, size_t rc, bool dal)
{
    constexpr int E = 16 / sizeof(T);
    const size_t nt = blockDim.x;
    for (size_t j = j0 + threadIdx.x; j < jend; j += 4 * nt) {
        uint4 x[4], y[4];
#pragma unroll
        for (int u = 0; u < 4; u++) if (j + u * nt < jend) { x[u] = ld_peer_v4(peer + (j + u * nt) * 16); y[u] = ld_peer_v4(mine + (j + u * nt) * 16); }
#pragma unroll
        for (int u = 0; u < 4; u++) if (j + u * nt < jend) {
            VecAcc<T, OP> acc; acc.set(y[u]); acc.add(x[u]);
            const uint4 r = acc.get(last ? N : 1); /* get() scales for AVG only; partial sums must stay unscaled */
            st_v4(mine + (j + u * nt) * 16, r);
            if (db) store_dst_vec<T>(db, (j + u * nt) * E, rc, dal, r);
        }
    }
}
/* mine[j] = peer[j] (+ dst) for my block's vectors of one slice */
template <typename T>
static __device__ __forceinline__ void step_copy(const char *peer, char *mine, size_t j0, size_t jend, bool keep, T *db, size_t rc, bool dal)
{
    constexpr int E = 16 / sizeof(T);
    const size_t nt = blockDim.x;
    for (size_t j = j0 + threadIdx.x; j < jend; j += 4 * nt) {
        uint4 x[4];
#pragma unroll
        for (int u = 0; u < 4; u++) if (j + u * nt < jend) x[u] = ld_peer_v4(peer + (j + u * nt) * 16);
#pragma unroll
        for (int u = 0; u < 4; u++) if (j + u * nt < jend) {
            if (keep) st_v4(mine + (j + u * nt) * 16, x[u]);
            store_dst_vec<T>(db, (j + u * nt) * E, rc, dal, x[u]);
        }
    }
}

template <typename T, int OP>
static __device__ __forceinline__ void steps_body(const nvl_red_args_t &a, BlockSync &bs, const SlicePlan &pl, uint32_t &phase)
{
    constexpr int E = 16 / sizeof(T);
    const nvl_team_dev_t &t = a.team;
    const int N = t.size, me = t.rank, nb = gridDim.x, b = blockIdx.x;
    const T *src = static_cast<const T *>(a.src);
    T *dst = static_cast<T *>(a.dst);
    const size_t cap_bytes = pl.cap_e * sizeof(T);
    const size_t nvmax = (pl.slice_max + E - 1) / E, per = (nvmax + nb - 1) / nb;
    const size_t j0 = dmin((size_t)b * per, nvmax), j1 = dmin(j0 + per, nvmax);
    char *mydata = data_of(t, me);
    const bool allred = a.kind == NVL_RED_ALLREDUCE;
#define SLICE_JEND(_s) dmin(j1, (slice_cnt(a, pl, _s) + E - 1) / E)
#define SLICE_DST(_s) (dst + (allred ? slice_off(a, pl, _s) : 0))
    /* stage every slice of my vector (same loop as phase A of the two-shot kernel) */
    for (int s = 0; s < N; s++) {
        const size_t rc = slice_cnt(a, pl, s), nfull = rc / E, jend = SLICE_JEND(s);
        const T *sb = src + slice_off(a, pl, s);
        char *hb = mydata + (size_t)s * cap_bytes;
        if (((uintptr_t)sb & 15) == 0) {
            copy_vecs<NVL_BW_U, false>(hb, reinterpret_cast<const char *>(sb), j0, dmin(jend, nfull));
            if (nfull >= j0 && nfull < jend && threadIdx.x == 0) st_v4(hb + nfull * 16, load_src_vec<T>(sb, nfull * E, rc, false));
        } else {
            for (size_t j = j0 + threadIdx.x; j < jend; j += blockDim.x) st_v4(hb + j * 16, load_src_vec<T>(sb, j * E, rc, false));
        }
    }
    bs.barrier(t, ++phase);
    if (a.sched == 1) {
        /* ---- ring ---- slice j starts at rank j+1 and ends, complete, at rank j */
        const int L = (me + N - 1) % N;
        char *left = data_of(t, L);
        for (int s = 0; s + 1 < N; s++) {
            const int c = (me - 2 - s + 3 * N) % N;
            const bool last = s + 2 == N;
            T *db = last ? SLICE_DST(c) : nullptr; /* c == me in the last step */
            step_reduce<T, OP>(left + (size_t)c * cap_bytes, mydata + (size_t)c * cap_bytes, j0, SLICE_JEND(c), last, N, db, slice_cnt(a, pl, c), db && ((uintptr_t)db & 15) == 0);
            bs.barrier(t, ++phase);
        }
        if (allred) for (int s = 0; s + 1 < N; s++) {
            const int c = (me - 1 - s + 2 * N) % N;
            T *db = SLICE_DST(c);
            step_copy<T>(left + (size_t)c * cap_bytes, mydata + (size_t)c * cap_bytes, j0, SLICE_JEND(c), s + 2 < N, db, slice_cnt(a, pl, c), ((uintptr_t)db & 15) == 0);
            bs.barrier(t, ++phase);
        }
    } else {
        /* ---- recursive halving (reduce-scatter) ... ---- */
        int lo = 0, hi = N; /* slices [lo,hi) are still mine to reduce */
        for (int d = N >> 1; d >= 1; d >>= 1) {
            const int partner = me ^ d, mid = lo + (hi - lo) / 2;
            const int klo = (me & d) ? mid : lo, khi = (me & d) ? hi : mid; /* the half I keep */
            const bool last = d == 1;
            char *pd = data_of(t, partner);
            for (int c = klo; c < khi; c++) {
                T *db = last ? SLICE_DST(c) : nullptr;
                step_reduce<T, OP>(pd + (size_t)c * cap_bytes, mydata + (size_t)c * cap_bytes, j0, SLICE_JEND(c), last, N, db, slice_cnt(a, pl, c), db && ((uintptr_t)db & 15) == 0);
            }
            lo = klo; hi = khi;
            bs.barrier(t, ++phase);
        }
        /* ---- ... recursive doubling (allgather) ---- */
        if (allred) for (int d = 1; d < N; d <<= 1) {
            const int partner = me ^ d, span = hi - lo;
            const int plo = (me & d) ? lo - span : hi; /* the partner's complete range sits next to mine */
            char *pd = data_of(t, partner);
            for (int c = plo; c < plo + span; c++) {
                T *db = SLICE_DST(c);
                step_copy<T>(pd + (size_t)c * cap_bytes, mydata + (size_t)c * cap_bytes, j0, SLICE_JEND(c), (d << 1) < N, db, slice_cnt(a, pl, c), ((uintptr_t)db & 15) == 0);
            }
            if (me & d) lo -= span; else hi += span;
            bs.barrier(t, ++phase);
        }
    }
#undef SLICE_JEND
#undef SLICE_DST
}

template <typename T, int OP> __global__ void __launch_bounds__(NVL_BW_THREADS, 2) nvl_reduce_steps_kernel_t(const __grid_constant__ nvl_red_args_t a)
{
    BlockSync bs; bs.init(a.team);
    SlicePlan pl; make_plan<T>(a, pl);
    uint32_t phase = 0;
    steps_body<T, OP>(a, bs, pl, phase);
    bs.finish(phase);
}
NVL_DEFINE_ENTRY(nvl_reduce_steps_kernel, nvl_red_args_t)

/* one translation unit per datatype defines these launchers */
#define NVL_INSTANTIATE_REDUCE(_T, _suffix)                                                                              \
    extern "C" cudaError_t nvl_launch_oneshot_##_suffix(const nvl_red_args_t *a, int nblocks, int nthreads, cudaStream_t s) \
    { return nvl_allreduce_oneshot_kernel_launch<_T>(a, nblocks, nthreads, s); }                                          \
    extern "C" cudaError_t nvl_launch_staged_##_suffix(const nvl_red_args_t *a, int nblocks, int nthreads, cudaStream_t s)  \
    { return nvl_reduce_staged_kernel_launch<_T>(a, nblocks, nthreads, s); }                                              \
    extern "C" cudaError_t nvl_launch_direct_##_suffix(const nvl_red_args_t *a, int nblocks, int nthreads, cudaStream_t s)  \
    { return nvl_reduce_direct_kernel_launch<_T>(a, nblocks, nthreads, s); }                                              \
    extern "C" cudaError_t nvl_launch_steps_##_suffix(const nvl_red_args_t *a, int nblocks, int nthreads, cudaStream_t s)   \
    { return nvl_reduce_steps_kernel_launch<_T>(a, nblocks, nthreads, s); }
#endif
