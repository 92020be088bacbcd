/* In-place NVLS allreduce (and reduce_scatter(v) out of a symmetric source) on SYMMETRIC USER MEMORY (UCC_TL_NVL_USER_SIZE > 0).
 *
 * When src and dst live in the user region of the team heap (allocated through ucc_tl_nvl_symm_region(), same offsets on every
 * member - the NVSHMEM / ncclMemAlloc+register contract), they are already bound to the team's multicast object.  Nothing is
 * staged and nothing is copied out:
 *     barrier   (every member's kernel runs => its src is final, its dst may be written)
 *     my slice: multimem.ld_reduce of src through the switch -> multimem.st into every member's dst
 *     barrier   (every slice has landed)
 * Each GPU injects count/N (stores) + answers count*(N-1)/N (loads of the others) and receives the same: one vector's worth
 * of bytes per direction, the minimum an allreduce can move, and HBM is touched once for reading and once for writing.
 *
 * d.src[0] / d.dst[0] carry the LOCAL addresses of src / dst inside my heap mapping; the multicast address is the same offset
 * in team.mc_heap.  Requires 16-byte aligned offsets (the allocator hands out 256-byte aligned blocks).
 *
 * Status: written at the end of round 1 without GPU time left; compiled for sm_100a, NOT yet run (tools/gpu_experimental.sh). */
#include "nvl_reduce_impl.cuh"

template <typename T, int OP>
static __device__ __forceinline__ void symm_body(const nvl_red_args_t &a, BlockSync &bs, const SlicePlan &pl)
{
    constexpr int E = 16 / sizeof(T);
    constexpr int U = NVL_BW_U;
    const nvl_team_dev_t &t = a.team;
    const int N = t.size, me = t.rank;
    const bool rs = a.kind == NVL_RED_REDUCE_SCATTER;   /* reduce_scatter(v): only src is symmetric, my block goes to the local a.dst */
    const size_t so = (size_t)(a.d.src[0] - t.heap[me]), dof = rs ? 0 : (size_t)(a.d.dst[0] - t.heap[me]);
    const size_t nt = blockDim.x;

    bs.barrier(t, 1);
    if (rs) {
        const size_t cnt = slice_cnt(a, pl, me), nv = (cnt + E - 1) / E;
        const size_t per = (nv + gridDim.x - 1) / gridDim.x, j0 = dmin((size_t)blockIdx.x * per, nv), j1 = dmin(j0 + per, nv);
        const char *mcs = t.mc_heap + so + slice_off(a, pl, me) * sizeof(T);
        T *db = static_cast<T *>(a.dst);
        const bool dal = ((uintptr_t)db & 15) == 0;
        size_t j = j0 + threadIdx.x;
        for (; j + (size_t)(U - 1) * nt < j1; j += (size_t)U * nt) {
            uint4 r[U];
#pragma unroll
            for (int u = 0; u < U; u++) r[u] = McRed<T, OP>::ld(mcs + (j + (size_t)u * nt) * 16);
#pragma unroll
            for (int u = 0; u < U; u++) {
                uint4 v = r[u];
                if (OP == NVL_OP_AVG) { VecAcc<T, OP> acc; acc.set(v); v = acc.get(N); }
                store_dst_vec<T>(db, (j + (size_t)u * nt) * E, cnt, dal, v);   /* bounds-checked: the ragged last vector is cut at cnt */
            }
        }
        for (; j < j1; j += nt) {
            uint4 v = McRed<T, OP>::ld(mcs + j * 16);
            if (OP == NVL_OP_AVG) { VecAcc<T, OP> acc; acc.set(v); v = acc.get(N); }
            store_dst_vec<T>(db, j * E, cnt, dal, v);
        }
    } else {
        const size_t cnt = slice_cnt(a, pl, me), nfull = cnt / E, nv = (cnt + E - 1) / E;
        const size_t per = (nv + gridDim.x - 1) / gridDim.x, j0 = dmin((size_t)blockIdx.x * per, nv), j1 = dmin(j0 + per, nv);
        const size_t jfull = dmin(j1, nfull);                               /* whole vectors of my range */
        const char *mcs = t.mc_heap + so + slice_off(a, pl, me) * sizeof(T);
        char *mcd = t.mc_heap + dof + slice_off(a, pl, me) * sizeof(T);
        size_t j = j0 + threadIdx.x;
        for (; j + (size_t)(U - 1) * nt < jfull; j += (size_t)U * nt) {
            uint4 r[U];
#pragma unroll
            for (int u = 0; u < U; u++) r[u] = McRed<T, OP>::ld(mcs + (j + (size_t)u * nt) * 16);
#pragma unroll
            for (int u = 0; u < U; u++) {
                uint4 v = r[u];
                if (OP == NVL_OP_AVG) { VecAcc<T, OP> acc; acc.set(v); v = acc.get(N); }
                mc_st_v4(mcd + (j + (size_t)u * nt) * 16, v);
            }
        }
        for (; j < jfull; j += nt) {
            uint4 v = McRed<T, OP>::ld(mcs + j * 16);
            if (OP == NVL_OP_AVG) { VecAcc<T, OP> acc; acc.set(v); v = acc.get(N); }
            mc_st_v4(mcd + j * 16, v);
        }
        /* ragged end of the vector (only the last non-empty slice can have one): the 16-byte load stays inside the 256-byte
         * aligned allocation, but the store must not touch bytes behind dst's last element - write the valid elements to every
         * member's unicast mapping instead */
        if (nfull < nv && nfull >= j0 && nfull < j1 && threadIdx.x == 0) {
            uint4 v = McRed<T, OP>::ld(mcs + nfull * 16);
            if (OP == NVL_OP_AVG) { VecAcc<T, OP> acc; acc.set(v); v = acc.get(N); }
            for (int p = 0; p < N; p++)
                store_dst_vec<T>(reinterpret_cast<T *>(t.heap[p] + dof) + slice_off(a, pl, me), nfull * E, cnt, false, v);
        }
    }
    bs.barrier(t, 2);
}

template <typename T, int OP> __global__ void __launch_bounds__(NVL_THREADS_MAX, 2) nvl_allreduce_symm_kernel_t(const __grid_constant__ nvl_red_args_t a)
{
    BlockSync bs; bs.init(a.team);
    SlicePlan pl; make_plan<T>(a, pl);
    symm_body<T, OP>(a, bs, pl);
    bs.finish(2);
}
NVL_DEFINE_ENTRY(nvl_allreduce_symm_kernel, nvl_red_args_t)

#ifndef NVL_HOST_EMU /* the host emulation calls the kernels directly */
extern "C" cudaError_t nvl_launch_reduce_symm(const nvl_red_args_t *a, int nblocks, int nthreads, cudaStream_t s)
{
    if (nthreads > NVL_THREADS_MAX) nthreads = NVL_THREADS_MAX;
    if ((a->kind != NVL_RED_ALLREDUCE && a->kind != NVL_RED_REDUCE_SCATTER) || !a->team.mc_heap || !nvl_nvls_supports(a->dt, a->op) || !a->d.src[0]) return cudaErrorInvalidValue;
    if (a->kind == NVL_RED_ALLREDUCE && !a->d.dst[0]) return cudaErrorInvalidValue;
    switch (a->dt) {
    case NVL_DT_F32: return nvl_allreduce_symm_kernel_launch<float>(a, nblocks, nthreads, s);
    case NVL_DT_F16: return nvl_allreduce_symm_kernel_launch<__half>(a, nblocks, nthreads, s);
    case NVL_DT_BF16: return nvl_allreduce_symm_kernel_launch<__nv_bfloat16>(a, nblocks, nthreads, s);
    case NVL_DT_I32: return nvl_allreduce_symm_kernel_launch<int32_t>(a, nblocks, nthreads, s);
    case NVL_DT_U32: return nvl_allreduce_symm_kernel_launch<uint32_t>(a, nblocks, nthreads, s);
    case NVL_DT_I64: return nvl_allreduce_symm_kernel_launch<int64_t>(a, nblocks, nthreads, s);
    case NVL_DT_U64: return nvl_allreduce_symm_kernel_launch<uint64_t>(a, nblocks, nthreads, s);
    case NVL_DT_C64: return nvl_allreduce_symm_kernel_launch<nvl_c64>(a, nblocks, nthreads, s);
    default: return cudaErrorInvalidValue;
    }
    return cudaGetLastError();
}
#endif

/* ------------------------------------------------------------------ */
/* allgather INTO a symmetric destination: every member multicasts its */
/* block to the same offset of everybody's dst with multimem.st - no   */
/* staging, no pull, no copy-out; the block is read once from local    */
/* memory and crosses each link once.                                  */
/*   a.src / a.src_bytes = my block (any local memory, 16-byte aligned)*/
/*   a.dst = LOCAL address of the gathered buffer inside my heap       */
/*   a.push_off = byte offset of my block inside it (multiple of 16)   */
/* ------------------------------------------------------------------ */
__global__ void __launch_bounds__(NVL_THREADS_MAX, 2) nvl_allgather_symm_kernel(const __grid_constant__ nvl_xchg_args_t a)
{
    const nvl_team_dev_t &t = a.team;
    const int N = t.size, me = t.rank;
    BlockSync bs; bs.init(t);
    const size_t dof = (size_t)(static_cast<char *>(a.dst) - t.heap[me]) + a.push_off;
    const char *src = static_cast<const char *>(a.src);
    char *mc = t.mc_heap + dof;
    const size_t nfull = a.src_bytes / 16, per = (nfull + gridDim.x - 1) / gridDim.x;
    const size_t j0 = dmin((size_t)blockIdx.x * per, nfull), j1 = dmin(j0 + per, nfull), nt = blockDim.x;
    constexpr int U = 8;

    bs.barrier(t, 1);                       /* every member's kernel runs: its dst may be written */
    size_t j = j0 + threadIdx.x;
    for (; j + (size_t)(U - 1) * nt < j1; j += (size_t)U * nt) {
        uint4 x[U];
#pragma unroll
        for (int u = 0; u < U; u++) x[u] = ld_src_v4(src + (j + (size_t)u * nt) * 16);
#pragma unroll
        for (int u = 0; u < U; u++) mc_st_v4(mc + (j + (size_t)u * nt) * 16, x[u]);
    }
    for (; j < j1; j += nt) mc_st_v4(mc + j * 16, ld_src_v4(src + j * 16));
    /* trailing bytes (block size not a multiple of 16): plain byte stores to every member's unicast mapping */
    if (blockIdx.x == 0 && threadIdx.x < (a.src_bytes & 15))
        for (int p = 0; p < N; p++) t.heap[p][dof + nfull * 16 + threadIdx.x] = src[nfull * 16 + threadIdx.x];
    bs.barrier(t, 2);                       /* every block has landed everywhere */
    bs.finish(2);
}

#ifndef NVL_HOST_EMU /* the host emulation calls the kernels directly */
extern "C" cudaError_t nvl_launch_allgather_symm(const nvl_xchg_args_t *a, int nblocks, int nthreads, cudaStream_t s)
{
    if (nthreads > NVL_THREADS_MAX) nthreads = NVL_THREADS_MAX;
    if (!a->team.mc_heap || !a->dst || !a->src || (a->push_off & 15) || ((uintptr_t)a->src & 15) || ((uintptr_t)a->dst & 15)) return cudaErrorInvalidValue;
    nvl_allgather_symm_kernel<<<nblocks, nthreads, 0, s>>>(*a);
    return cudaGetLastError();
}
#endif
