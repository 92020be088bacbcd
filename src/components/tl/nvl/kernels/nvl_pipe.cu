/* Pipelined staged NVLS allreduce (algorithm "nvls_pipe", opt-in through UCC_TL_NVL_TUNE=allreduce:...:@nvls_pipe).
 *
 * The plain staged kernel (nvl_reduce_impl.cuh: staged_body) runs, per heap round,
 *     A: stage my part of every slice into my heap   (local HBM copy)
 *     -- inter-GPU barrier --
 *     B: multimem.ld_reduce my slice + multimem.st   (NVLink / NVSwitch)
 *     -- inter-GPU barrier --
 *     C: copy every reduced slice out of my heap     (local HBM copy)
 * strictly one after the other, so the NVLink sits idle during A and C (about a third of a round at 8 GPUs) and every round
 * pays two barriers.  Here the data region is cut into THREE buffers and the warps of every CTA are split into three roles
 * that work on three consecutive chunks at the same time:
 *     iteration i:   A-warps stage chunk i   -> buffer  i    % 3
 *                    B-warps reduce chunk i-1 in buffer (i-1) % 3
 *                    C-warps copy out chunk i-2 from buffer (i-2) % 3
 *                    -- ONE inter-GPU barrier --
 * Hazards: B(k) needs A(k) of every member (iteration k, then a barrier); C(k) needs B(k) of every member (iteration k+1,
 * then a barrier); A(k+3) reuses the buffer of chunk k, whose C(k) ran in iteration k+2 and whose peers' B(k) loads ended
 * before the barrier of iteration k+1.  The HBM copies hide behind the switch traffic and the barrier count per chunk drops
 * from two to one.  CTA b of every member owns the same vector range of every chunk, exactly like the staged kernel, so the
 * per-block flag barrier (BlockSync) is reused unchanged.
 *
 * Status: written at the end of round 1 without GPU time left; compiled for sm_100a, NOT yet run.  It is therefore not in
 * the default score table; tests/test_nvl_gpu.py::test_allreduce_nvls_pipe and tools/gpu_bench.sh exercise it. */
#include "nvl_reduce_impl.cuh"

template <int U, bool PEER>
static __device__ __forceinline__ void role_copy_vecs(char *dst, const char *src, size_t v0, size_t v1, int rtid, int rnt)
{
    size_t v = v0 + rtid;
    for (; v + (size_t)(U - 1) * rnt < v1; v += (size_t)U * rnt) {
        uint4 x[U];
#pragma unroll
        for (int u = 0; u < U; u++) x[u] = PEER ? ld_peer_v4(src + (v + (size_t)u * rnt) * 16) : ld_src_v4(src + (v + (size_t)u * rnt) * 16);
#pragma unroll
        for (int u = 0; u < U; u++) st_v4(dst + (v + (size_t)u * rnt) * 16, x[u]);
    }
    for (; v < v1; v += rnt) st_v4(dst + v * 16, PEER ? ld_peer_v4(src + v * 16) : ld_src_v4(src + v * 16));
}

struct PipeGeom {
    size_t cap_e, cap_bytes, buf_bytes; /* elements / bytes of one slice per chunk; bytes of one of the three buffers */
    int    chunks;
};

template <typename T> static __device__ __forceinline__ void pipe_geom(const nvl_red_args_t &a, const SlicePlan &pl, PipeGeom &g)
{
    const size_t N = (size_t)a.team.size;
    g.cap_bytes = (a.team.data_size / 3 / N / 16) * 16;
    g.cap_e = g.cap_bytes / sizeof(T);
    g.buf_bytes = g.cap_bytes * N;
    g.chunks = (int)((pl.slice_max + g.cap_e - 1) / g.cap_e);
}

/* vector range [j0,j1) of chunk k that CTA b owns inside every slice (same formula on every member) */
template <typename T> static __device__ __forceinline__ void chunk_range(const SlicePlan &pl, const PipeGeom &g, int k, size_t &e0, size_t &j0, size_t &j1)
{
    constexpr int E = 16 / sizeof(T);
    e0 = (size_t)k * g.cap_e;
    /* the range a block owns must not move between chunks (blocks of one rank are not synchronised with each other and the
     * roles work on three chunks at once): cut it from the full chunk capacity, a shorter last chunk leaves upper blocks idle */
    const size_t rmax = dmin(g.cap_e, pl.slice_max - e0), nvmax = (rmax + E - 1) / E;
    const size_t nvsplit = g.chunks > 1 ? g.cap_e / E : nvmax, per = (nvsplit + gridDim.x - 1) / gridDim.x;
    j0 = dmin((size_t)blockIdx.x * per, nvmax); j1 = dmin(j0 + per, nvmax);
}

template <typename T> static __device__ __forceinline__ void pipe_stage(const nvl_red_args_t &a, const SlicePlan &pl, const PipeGeom &g, int k, int rtid, int rnt)
{
    constexpr int E = 16 / sizeof(T);
    const int N = a.team.size;
    const T *src = static_cast<const T *>(a.src);
    char *buf = data_of(a.team, a.team.rank) + (size_t)(k % 3) * g.buf_bytes;
    size_t e0, j0, j1; chunk_range<T>(pl, g, k, e0, j0, j1);
    for (int s = 0; s < N; s++) {
        const size_t rc = slice_cnt(a, pl, s) > e0 ? dmin(g.cap_e, slice_cnt(a, pl, s) - e0) : 0;
        const size_t nfull = rc / E, jend = dmin(j1, (rc + E - 1) / E);
        const T *sb = src + slice_off(a, pl, s) + e0;
        char *hb = buf + (size_t)s * g.cap_bytes;
        if (((uintptr_t)sb & 15) == 0) {
            role_copy_vecs<4, false>(hb, reinterpret_cast<const char *>(sb), j0, dmin(jend, nfull), rtid, rnt);
            if (nfull >= j0 && nfull < jend && rtid == 0) st_v4(hb + nfull * 16, load_src_vec<T>(sb, nfull * E, rc, false)); /* ragged tail */
        } else {
            for (size_t j = j0 + rtid; j < jend; j += rnt) st_v4(hb + j * 16, load_src_vec<T>(sb, j * E, rc, false));
        }
    }
}

template <typename T, int OP> static __device__ __forceinline__ void pipe_reduce(const nvl_red_args_t &a, const SlicePlan &pl, const PipeGeom &g, int k, int rtid, int rnt)
{
    constexpr int E = 16 / sizeof(T);
    constexpr int U = NVL_BW_U;
    const int me = a.team.rank;
    size_t e0, j0, j1; chunk_range<T>(pl, g, k, e0, j0, j1);
    const size_t rc = slice_cnt(a, pl, me) > e0 ? dmin(g.cap_e, slice_cnt(a, pl, me) - e0) : 0;
    const size_t jend = dmin(j1, (rc + E - 1) / E);
    char *mc = a.team.mc_heap + NVL_DATA_OFFSET + (size_t)(k % 3) * g.buf_bytes + (size_t)me * g.cap_bytes;
    size_t j = j0 + rtid;
    /* full groups: U in-switch reductions in flight per thread, no per-lane bounds checks */
    for (; j + (size_t)(U - 1) * rnt < jend; j += (size_t)U * rnt) {
        uint4 r[U];
#pragma unroll
        for (int u = 0; u < U; u++) r[u] = McRed<T, OP>::ld(mc + (j + (size_t)u * rnt) * 16);
#pragma unroll
        for (int u = 0; u < U; u++) {
            uint4 v = r[u];
            if (OP == NVL_OP_AVG) { VecAcc<T, OP> acc; acc.set(v); v = acc.get(a.team.size); }
            mc_st_v4(mc + (j + (size_t)u * rnt) * 16, v); /* the padding lanes of a ragged last vector are reduced and stored too: they stay inside the slot */
        }
    }
    for (; j < jend; j += rnt) {
        uint4 v = McRed<T, OP>::ld(mc + j * 16);
        if (OP == NVL_OP_AVG) { VecAcc<T, OP> acc; acc.set(v); v = acc.get(a.team.size); }
        mc_st_v4(mc + j * 16, v);
    }
}

template <typename T> static __device__ __forceinline__ void pipe_copy_out(const nvl_red_args_t &a, const SlicePlan &pl, const PipeGeom &g, int k, int rtid, int rnt)
{
    constexpr int E = 16 / sizeof(T);
    const int N = a.team.size;
    T *dst = static_cast<T *>(a.dst);
    const char *buf = data_of(a.team, a.team.rank) + (size_t)(k % 3) * g.buf_bytes;
    size_t e0, j0, j1; chunk_range<T>(pl, g, k, e0, j0, j1);
    for (int s = 0; s < N; s++) {
        const size_t rc = slice_cnt(a, pl, s) > e0 ? dmin(g.cap_e, slice_cnt(a, pl, s) - e0) : 0;
        const size_t nfull = rc / E, jend = dmin(j1, (rc + E - 1) / E);
        T *db = dst + slice_off(a, pl, s) + e0;
        const char *hb = buf + (size_t)s * g.cap_bytes;
        if (((uintptr_t)db & 15) == 0) {
            role_copy_vecs<4, true>(reinterpret_cast<char *>(db), hb, j0, dmin(jend, nfull), rtid, rnt);
            if (nfull >= j0 && nfull < jend && rtid == 0) store_dst_vec<T>(db, nfull * E, rc, false, ld_peer_v4(hb + nfull * 16));
        } else {
            for (size_t j = j0 + rtid; j < jend; j += rnt) store_dst_vec<T>(db, j * E, rc, false, ld_peer_v4(hb + j * 16));
        }
    }
}

template <typename T, int OP>
static __device__ __forceinline__ void pipe_body(const nvl_red_args_t &a, BlockSync &bs, const SlicePlan &pl, const PipeGeom &g)
{
    /* roles by warp: a quarter stages, half reduces (the NVLink-bound part), a quarter copies out */
    const int W = (int)blockDim.x / 32, WA = W / 4, WB = W / 2, w = (int)threadIdx.x / 32;
    const int role = w < WA ? 0 : (w < WA + WB ? 1 : 2);
    const int rnt = (role == 0 ? WA : (role == 1 ? WB : W - WA - WB)) * 32;
    const int rtid = (int)threadIdx.x - (role == 0 ? 0 : (role == 1 ? WA : WA + WB)) * 32;
    const int R = g.chunks;
    for (int it = 0; it < R + 2; it++) {
        if (role == 0) { if (it < R) pipe_stage<T>(a, pl, g, it, rtid, rnt); }
        else if (role == 1) { if (it >= 1 && it - 1 < R) pipe_reduce<T, OP>(a, pl, g, it - 1, rtid, rnt); }
        else { if (it >= 2) pipe_copy_out<T>(a, pl, g, it - 2, rtid, rnt); }
        if (it < R + 1) bs.barrier(a.team, (uint32_t)it + 1);
    }
}

template <typename T, int OP> __global__ void __launch_bounds__(NVL_THREADS_MAX, 2) nvl_allreduce_nvls_pipe_kernel_t(const __grid_constant__ nvl_red_args_t a)
{
    BlockSync bs; bs.init(a.team);
    SlicePlan pl; make_plan<T>(a, pl);
    PipeGeom g; pipe_geom<T>(a, pl, g);
    pipe_body<T, OP>(a, bs, pl, g);
    bs.finish((uint32_t)g.chunks + 1);
}
NVL_DEFINE_ENTRY(nvl_allreduce_nvls_pipe_kernel, nvl_red_args_t)

#ifndef NVL_HOST_EMU /* the host emulation calls the kernels directly */
extern "C" cudaError_t nvl_launch_reduce_pipe(const nvl_red_args_t *a, int nblocks, int nthreads, cudaStream_t s)
{
    if (nthreads > NVL_THREADS_MAX) nthreads = NVL_THREADS_MAX;
    if (nthreads < 128 || (nthreads & 127)) return cudaErrorInvalidValue; /* three roles need at least four warps */
    if (a->kind != NVL_RED_ALLREDUCE || !a->use_nvls || !a->team.mc_heap || !nvl_nvls_supports(a->dt, a->op)) return cudaErrorInvalidValue;
    switch (a->dt) {
    case NVL_DT_F32: return nvl_allreduce_nvls_pipe_kernel_launch<float>(a, nblocks, nthreads, s);
    case NVL_DT_F16: return nvl_allreduce_nvls_pipe_kernel_launch<__half>(a, nblocks, nthreads, s);
    case NVL_DT_BF16: return nvl_allreduce_nvls_pipe_kernel_launch<__nv_bfloat16>(a, nblocks, nthreads, s);
    case NVL_DT_I32: return nvl_allreduce_nvls_pipe_kernel_launch<int32_t>(a, nblocks, nthreads, s);
    case NVL_DT_U32: return nvl_allreduce_nvls_pipe_kernel_launch<uint32_t>(a, nblocks, nthreads, s);
    case NVL_DT_I64: return nvl_allreduce_nvls_pipe_kernel_launch<int64_t>(a, nblocks, nthreads, s);
    case NVL_DT_U64: return nvl_allreduce_nvls_pipe_kernel_launch<uint64_t>(a, nblocks, nthreads, s);
    case NVL_DT_C64: return nvl_allreduce_nvls_pipe_kernel_launch<nvl_c64>(a, nblocks, nthreads, s);
    default: return cudaErrorInvalidValue;
    }
    return cudaGetLastError();
}
#endif
