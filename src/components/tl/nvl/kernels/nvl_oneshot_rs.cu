/* One-shot reduce_scatter(v) (algorithm "oneshot", opt-in): the latency path of reduce_scatter, built like the one-shot
 * allreduce (nvl_reduce_impl.cuh: oneshot_body).  Every rank stores block p of its vector into a private slot of member p's
 * heap (latency region, 1 MB per source, two slot sets alternating by launch parity so that no trailing barrier is needed),
 * raises a flag, and reduces the N-1 blocks it received with its own.  One flag exchange instead of the two barriers of the
 * staged kernel; every block of the vector crosses NVLink once.  Blocks of at most NVL_LL_MAX bytes.
 *
 * The slot sets and per-block sequence numbers (ll_flags / ll_seq) are shared with the one-shot allreduce: both kernels bump
 * ll_seq[block] once per launch on every rank, so they can be mixed freely.
 *
 * Status: written after the round-1 GPU budget was spent; logic checked in the host emulation (tests/emu), not yet run on GPUs. */
#include "nvl_reduce_impl.cuh"

template <typename T, int OP>
static __device__ __forceinline__ void oneshot_rs_body(const nvl_red_args_t &a, nvl_ctrl_t *mine, uint32_t seq)
{
    constexpr int E = 16 / sizeof(T);
    const nvl_team_dev_t &t = a.team;
    const int N = t.size, me = t.rank, nb = gridDim.x, b = blockIdx.x;
    const T *src = static_cast<const T *>(a.src);
    T *dst = static_cast<T *>(a.dst);
    const size_t slot = (size_t)((seq & 1) * NVL_MAX_PEERS) * NVL_LL_MAX;

    /* push: block p of my vector -> slot `me` of member p; CTA b handles the same vector range of a block on both sides */
    for (int i = 1; i < N; i++) {
        int p = me + i; if (p >= N) p -= N;
        const T *sb = src + a.rs_offset[p];
        const size_t cnt = a.rs_count[p], nvec = (cnt + E - 1) / E, per = (nvec + nb - 1) / nb;
        const size_t v0 = dmin((size_t)b * per, nvec), v1 = dmin(v0 + per, nvec);
        const bool sal = ((uintptr_t)sb & 15) == 0;
        char *out = t.heap[p] + NVL_LL_OFFSET + slot + (size_t)me * NVL_LL_MAX;
        for (size_t v = v0 + threadIdx.x; v < v1; v += blockDim.x) st_v4(out + v * 16, load_src_vec<T>(sb, v * E, cnt, sal));
    }
    __syncthreads();
    if ((int)threadIdx.x < N && (int)threadIdx.x != me) {
        fence_sys();
        st_relaxed_sys_u32(&reinterpret_cast<nvl_ctrl_t *>(t.heap[threadIdx.x])->ll_flags[b][me], seq);
        BlockSync bs; bs.mine = mine;
        bs.spin(t, &mine->ll_flags[b][threadIdx.x], seq);
    }
    __syncthreads();
    /* reduce my block: own contribution straight from src, the others from my slots */
    {
        const T *sb = src + a.rs_offset[me];
        const size_t cnt = a.rs_count[me], nvec = (cnt + E - 1) / E, per = (nvec + nb - 1) / nb;
        const size_t v0 = dmin((size_t)b * per, nvec), v1 = dmin(v0 + per, nvec);
        const bool sal = ((uintptr_t)sb & 15) == 0, dal = ((uintptr_t)dst & 15) == 0;
        const char *mybase = t.heap[me] + NVL_LL_OFFSET + slot;
        for (size_t v = v0 + threadIdx.x; v < v1; v += blockDim.x) {
            uint4 x[NVL_MAX_PEERS];
            x[0] = load_src_vec<T>(sb, v * E, cnt, sal);
#pragma unroll
            for (int i = 1; i < NVL_MAX_PEERS; i++) if (i < N) { int p = me + i; if (p >= N) p -= N; x[i] = ld_peer_v4(mybase + (size_t)p * NVL_LL_MAX + v * 16); }
            VecAcc<T, OP> acc; acc.set(x[0]);
#pragma unroll
            for (int i = 1; i < NVL_MAX_PEERS; i++) if (i < N) acc.add(x[i]);
            store_dst_vec<T>(dst, v * E, cnt, dal, acc.get(N));
        }
    }
}

template <typename T, int OP> __global__ void __launch_bounds__(NVL_THREADS_MAX) nvl_reduce_scatter_oneshot_kernel_t(const __grid_constant__ nvl_red_args_t a)
{
    nvl_ctrl_t *mine = reinterpret_cast<nvl_ctrl_t *>(a.team.heap[a.team.rank]);
    const uint32_t seq = ll_seq_begin(mine);   /* team-wide sequence shared with the one-shot allreduce */
    oneshot_rs_body<T, OP>(a, mine, seq);
    ll_seq_end(mine, seq);
}
NVL_DEFINE_ENTRY(nvl_reduce_scatter_oneshot_kernel, nvl_red_args_t)

#ifndef NVL_HOST_EMU /* the host emulation calls the kernels directly */
extern "C" cudaError_t nvl_launch_reduce_scatter_oneshot(const nvl_red_args_t *a, int nblocks, int nthreads, cudaStream_t s)
{
    if (nthreads > NVL_THREADS_MAX) nthreads = NVL_THREADS_MAX;
    if (a->kind != NVL_RED_REDUCE_SCATTER) return cudaErrorInvalidValue;
    switch (a->dt) {
    case NVL_DT_I8: return nvl_reduce_scatter_oneshot_kernel_launch<int8_t>(a, nblocks, nthreads, s);
    case NVL_DT_I16: return nvl_reduce_scatter_oneshot_kernel_launch<int16_t>(a, nblocks, nthreads, s);
    case NVL_DT_I32: return nvl_reduce_scatter_oneshot_kernel_launch<int32_t>(a, nblocks, nthreads, s);
    case NVL_DT_I64: return nvl_reduce_scatter_oneshot_kernel_launch<int64_t>(a, nblocks, nthreads, s);
    case NVL_DT_U8: return nvl_reduce_scatter_oneshot_kernel_launch<uint8_t>(a, nblocks, nthreads, s);
    case NVL_DT_U16: return nvl_reduce_scatter_oneshot_kernel_launch<uint16_t>(a, nblocks, nthreads, s);
    case NVL_DT_U32: return nvl_reduce_scatter_oneshot_kernel_launch<uint32_t>(a, nblocks, nthreads, s);
    case NVL_DT_U64: return nvl_reduce_scatter_oneshot_kernel_launch<uint64_t>(a, nblocks, nthreads, s);
    case NVL_DT_F16: return nvl_reduce_scatter_oneshot_kernel_launch<__half>(a, nblocks, nthreads, s);
    case NVL_DT_F32: return nvl_reduce_scatter_oneshot_kernel_launch<float>(a, nblocks, nthreads, s);
    case NVL_DT_F64: return nvl_reduce_scatter_oneshot_kernel_launch<double>(a, nblocks, nthreads, s);
    case NVL_DT_BF16: return nvl_reduce_scatter_oneshot_kernel_launch<__nv_bfloat16>(a, nblocks, nthreads, s);
    case NVL_DT_C64: return nvl_reduce_scatter_oneshot_kernel_launch<nvl_c64>(a, nblocks, nthreads, s);
    case NVL_DT_C128: return nvl_reduce_scatter_oneshot_kernel_launch<nvl_c128>(a, nblocks, nthreads, s);
    default: return cudaErrorInvalidValue;
    }
    return cudaGetLastError();
}
#endif
