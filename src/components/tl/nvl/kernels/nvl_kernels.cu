/* tl/nvl collective kernels for sm_100a.  See nvl_kernels.h for the contract.
 *
 * Reference parity (what each kernel replaces):
 *   allreduce_oneshot  - no reference equivalent below NVLS; tl_cuda has no P2P allreduce (tl/cuda/tl_cuda.h:40-44)
 *   reduce_staged      - tl_cuda reduce_scatterv_linear (copy to peer scratch via executor + separate
 *                        REDUCE_STRIDED kernel + CPU polled step counters, reduce_scatterv_linear.c:229-328)
 *                        and the NVLS kernels K1/K2/K4 with their two staging cudaMemcpyAsync
 *                        (kernels/allreduce_kernel.cu:21-141, allreduce_nvls.c:81-116) fused into one launch
 *   exchange           - allgatherv_linear / alltoallv_ce / bcast_linear state machines (host driven
 *                        copy-engine or executor copies) as one pull kernel with device-side flags
 *
 * Performance notes: every data loop keeps several independent 16-byte transactions per thread in
 * flight (loads are issued in batches before the dependent stores) because a single NVLink round trip is
 * ~2 us; with 512 threads x 8 x 16 B per CTA a few dozen CTAs cover the bandwidth-delay product.
 */
#include "nvl_reduce_impl.cuh"

static_assert(sizeof(nvl_ctrl_t) <= NVL_CTRL_SIZE, "control block outgrew its heap region");

__global__ void nvl_ctrl_init_kernel(nvl_ctrl_t *c)
{
    uint32_t *w = reinterpret_cast<uint32_t *>(c);
    for (size_t i = threadIdx.x + (size_t)blockIdx.x * blockDim.x; i < sizeof(nvl_ctrl_t) / 4; i += (size_t)gridDim.x * blockDim.x) w[i] = 0;
}

__global__ void nvl_barrier_kernel(nvl_team_dev_t t)
{
    BlockSync bs; bs.init(t);
    bs.barrier(t, 1);
    bs.finish(1);
}

/* ------------------------------------------------------------------ */
/* staged exchange (pull): allgather(v) alltoall(v) bcast gather(v) scatter(v) */
/* ------------------------------------------------------------------ */
template <bool PEER> static __device__ __forceinline__ void copy_bytes_grid(char *dst, const char *src, size_t n)
{
    const size_t tid = (size_t)blockIdx.x * blockDim.x + threadIdx.x, nt = (size_t)gridDim.x * blockDim.x;
    const uintptr_t mis = ((uintptr_t)dst | (uintptr_t)src);
    if ((mis & 15) == 0) {
        const size_t nv = n / 16;
        size_t v = tid;
        for (; v + 7 * nt < nv; v += 8 * nt) {
            uint4 x[8];
#pragma unroll
            for (int u = 0; u < 8; u++) x[u] = PEER ? ld_peer_v4(src + (v + u * nt) * 16) : ld_src_v4(src + (v + u * nt) * 16);
#pragma unroll
            for (int u = 0; u < 8; u++) st_v4(dst + (v + u * nt) * 16, x[u]);
        }
        for (; v < nv; v += nt) st_v4(dst + v * 16, PEER ? ld_peer_v4(src + v * 16) : ld_src_v4(src + v * 16));
        for (size_t i = nv * 16 + tid; i < n; i += nt) dst[i] = *(volatile const char *)(src + i);
    } else if ((mis & 3) == 0) {
        const size_t nw = n / 4;
        for (size_t v = tid; v < nw; v += nt) ((uint32_t *)dst)[v] = ((volatile const uint32_t *)src)[v];
        for (size_t i = nw * 4 + tid; i < n; i += nt) dst[i] = *(volatile const char *)(src + i);
    } else {
        for (size_t i = tid; i < n; i += nt) dst[i] = *(volatile const char *)(src + i);
    }
}

/* store up to 16 bytes of x at an arbitrarily aligned address */
static __device__ __forceinline__ void store_any16(char *d, uint4 x, size_t nbytes)
{
    if (nbytes >= 16 && ((uintptr_t)d & 15) == 0) { st_v4(d, x); return; }
    const unsigned w[4] = {x.x, x.y, x.z, x.w};
    if (((uintptr_t)d & 3) == 0 && (nbytes & 3) == 0) { for (size_t i = 0; i < nbytes / 4 && i < 4; i++) reinterpret_cast<unsigned *>(d)[i] = w[i]; return; }
    for (size_t i = 0; i < nbytes && i < 16; i++) d[i] = (char)(w[i >> 2] >> (8 * (i & 3)));
}

/* ring allgather(v) (reference tl/cuda allgatherv_ring.c: host-driven multi-ring pipeline through scratch): N-1 steps, at
 * step s every rank pulls block (me-1-s) from its LEFT neighbour's heap into its own heap and into dst.  Only
 * neighbour links are used, so it also serves topologies without an all-to-all NVLink fabric.  All heaps use the
 * same 16-byte aligned block layout (pull_off[]), which makes block b of a rank depend only on block b of its
 * neighbour: one per-block flag wait per step. */
static __device__ void exchange_ring(const nvl_xchg_args_t &a, BlockSync &bs)
{
    const nvl_team_dev_t &t = a.team;
    const int N = t.size, me = t.rank, pos = a.ring_pos, L = a.ring_order[(pos + N - 1) % N];   /* my left neighbour ON THE RING (link-aware order) */
    const size_t tid = (size_t)blockIdx.x * blockDim.x + threadIdx.x, nt = (size_t)gridDim.x * blockDim.x;
    char *mine = data_of(t, me) + NVL_XCHG_TABLE_BYTES;
    const char *left = data_of(t, L) + NVL_XCHG_TABLE_BYTES;
    /* step -1: my own block into my heap (vector granularity, identical thread->vector mapping as the steps below) and into dst */
    {
        const size_t n = a.pull_bytes[me], nv = (n + 15) / 16;
        const char *s = static_cast<const char *>(a.src);
        char *d = static_cast<char *>(a.dst) + a.dst_off[me];
        for (size_t v = tid; v < nv; v += nt) {
            const size_t nb = n - v * 16 < 16 ? n - v * 16 : 16;
            uint4 x = make_uint4(0, 0, 0, 0);
            if (nb == 16 && ((uintptr_t)s & 15) == 0) x = ld_src_v4(s + v * 16);
            else { unsigned w[4] = {0, 0, 0, 0}; for (size_t i = 0; i < nb; i++) w[i >> 2] |= (unsigned)(unsigned char)s[v * 16 + i] << (8 * (i & 3)); x = make_uint4(w[0], w[1], w[2], w[3]); }
            st_v4(mine + a.pull_off[me] + v * 16, x);
            if (d != s) store_any16(d + v * 16, x, nb);
        }
    }
    for (int s = 0; s + 1 < N; s++) {
        const int c = a.ring_order[(pos - 1 - s + 2 * N) % N];   /* the block that has travelled s + 1 hops towards me */
        const size_t n = a.pull_bytes[c], nv = (n + 15) / 16;
        char *d = static_cast<char *>(a.dst) + a.dst_off[c];
        bs.barrier(t, (uint32_t)s + 1);
        for (size_t v = tid; v < nv; v += 4 * nt) {
            uint4 x[4];
#pragma unroll
            for (int u = 0; u < 4; u++) if (v + u * nt < nv) x[u] = ld_peer_v4(left + a.pull_off[c] + (v + u * nt) * 16);
#pragma unroll
            for (int u = 0; u < 4; u++) if (v + u * nt < nv) {
                const size_t vv = v + u * nt, nb = n - vv * 16 < 16 ? n - vv * 16 : 16;
                if (s + 2 < N) st_v4(mine + a.pull_off[c] + vv * 16, x[u]); /* the last step's block is not forwarded */
                store_any16(d + vv * 16, x[u], nb);
            }
        }
    }
    bs.barrier(t, (uint32_t)N); /* nobody leaves while its right neighbour may still be reading its heap */
    bs.finish((uint32_t)N);
}

/* 2 CTAs per SM like the reduce kernels: wait_all_blocks() needs every block of every rank resident, and the host caps
 * the grid at 2 x SM count */
__global__ void __launch_bounds__(NVL_THREADS_MAX, 2) nvl_exchange_kernel(nvl_xchg_args_t a)
{
    const nvl_team_dev_t &t = a.team;
    const int N = t.size, me = t.rank;
    BlockSync bs; bs.init(t);
    char *mydata = data_of(t, me);
    if (a.ring) { exchange_ring(a, bs); return; }
    /* phase A: publish my bytes (and the offset table peers use to find their block) */
    if (a.publish_table && blockIdx.x == 0 && (int)threadIdx.x < N) reinterpret_cast<uint64_t *>(mydata)[threadIdx.x] = (uint64_t)a.stage_off[threadIdx.x];
    if (a.use_mc) {
        /* NVLS push (reference kernel K5, tl/cuda/kernels/allgatherv_kernel.cu:19-51, there followed by a cudaMemcpyAsync):
         * one multimem.st per vector lands my block in EVERY member's heap; phase B then is a local copy */
        if (a.src_bytes) {
            char *mc = t.mc_heap + NVL_DATA_OFFSET + NVL_XCHG_TABLE_BYTES + a.push_off;
            const char *s = static_cast<const char *>(a.src);
            /* a misaligned source (only its owner knows) cannot feed 16-byte multicast stores: it goes the slow per-byte way */
            const size_t tid = (size_t)blockIdx.x * blockDim.x + threadIdx.x, nt = (size_t)gridDim.x * blockDim.x, nv = ((uintptr_t)s & 15) ? 0 : a.src_bytes / 16;
            size_t v = tid;
            for (; v + 3 * nt < nv; v += 4 * nt) {
                uint4 x[4];
#pragma unroll
                for (int u = 0; u < 4; u++) x[u] = ld_src_v4(s + (v + u * nt) * 16);
#pragma unroll
                for (int u = 0; u < 4; u++) mc_st_v4(mc + (v + u * nt) * 16, x[u]);
            }
            for (; v < nv; v += nt) mc_st_v4(mc + v * 16, ld_src_v4(s + v * 16));
            /* ragged tail (< 16 bytes): plain stores into each member's heap */
            for (size_t i = nv * 16 + tid; i < a.src_bytes; i += nt)
                for (int p = 0; p < N; p++) data_of(t, p)[NVL_XCHG_TABLE_BYTES + a.push_off + i] = s[i];
        }
    } else if (a.src_bytes && !a.direct) {
        /* (zero-copy mode: the peers read my user buffer in place, nothing to stage) */
        copy_bytes_grid<false>(mydata + NVL_XCHG_TABLE_BYTES, static_cast<const char *>(a.src), a.src_bytes);
    }
    bs.signal(t, 1);
    bs.wait_all_blocks(t, 1);
    /* phase B: pull.  Resolve every remote block first; when all of them are 16-byte aligned the vectors of up to eight
     * peers are requested together (one NVLink round trip instead of one per peer - what matters for the 1..64 MB range
     * where a thread owns only a few vectors of each block) */
    /* the per-peer source / destination / length tables live in shared memory (built by one thread): they are indexed with
     * run-time values in the batched loop below, which would put per-thread copies on the local-memory stack */
#ifdef NVL_HOST_EMU   /* host emulation: no shared memory, every (OS) thread builds its own copy */
    const char *sp[NVL_MAX_PEERS]; char *dp[NVL_MAX_PEERS]; size_t nb[NVL_MAX_PEERS]; int s_np; int s_vec; size_t s_nvmax;
    const bool fill = true;
#else
    __shared__ const char *sp[NVL_MAX_PEERS]; __shared__ char *dp[NVL_MAX_PEERS]; __shared__ size_t nb[NVL_MAX_PEERS];
    __shared__ int s_np; __shared__ int s_vec; __shared__ size_t s_nvmax;
    const bool fill = threadIdx.x == 0;
#endif
    if (fill) {
        int np_ = 0; int vec_ = 1; size_t nvmax_ = 0;
        for (int i = 1; i < N; i++) {
            int p = me + i; if (p >= N) p -= N;
            const size_t n = a.pull_bytes[p];
            if (!n) continue;
            size_t off = a.pull_off[p];
            if (off == NVL_XCHG_LOOKUP) off = (size_t) * reinterpret_cast<volatile const uint64_t *>(data_of(t, p) + (size_t)me * 8);
            sp[np_] = (a.direct ? a.d.src[p] : (a.use_mc ? mydata : data_of(t, p)) + NVL_XCHG_TABLE_BYTES) + off;
            dp[np_] = static_cast<char *>(a.dst) + a.dst_off[p]; nb[np_] = n;
            if (((uintptr_t)sp[np_] | (uintptr_t)dp[np_]) & 15) vec_ = 0;
            if (n / 16 > nvmax_) nvmax_ = n / 16;
            np_++;
        }
        s_np = np_; s_vec = vec_; s_nvmax = nvmax_;
    }
    __syncthreads();
    const int np = s_np; const bool vec = s_vec != 0; const size_t nvmax = s_nvmax;
    if (a.pull_bytes[me]) { /* own block: a local copy */
        char *d = static_cast<char *>(a.dst) + a.dst_off[me];
        if (d != static_cast<const char *>(a.src) + a.self_off) copy_bytes_grid<false>(d, static_cast<const char *>(a.src) + a.self_off, a.pull_bytes[me]);
    }
    if (vec && np > 1) {
        const size_t tid = (size_t)blockIdx.x * blockDim.x + threadIdx.x, nt = (size_t)gridDim.x * blockDim.x;
        for (int g = 0; g < np; g += 8) {
            for (size_t v = tid; v < nvmax; v += nt) {
                uint4 x[8];
#pragma unroll
                for (int k = 0; k < 8; k++) if (g + k < np && v < nb[g + k] / 16) x[k] = ld_peer_v4(sp[g + k] + v * 16);
#pragma unroll
                for (int k = 0; k < 8; k++) if (g + k < np && v < nb[g + k] / 16) st_v4(dp[g + k] + v * 16, x[k]);
            }
        }
        for (int q = 0; q < np; q++) /* ragged tails (< 16 bytes per block) */
            for (size_t i = (nb[q] / 16) * 16 + tid; i < nb[q]; i += nt) dp[q][i] = *(volatile const char *)(sp[q] + i);
    } else {
        for (int q = 0; q < np; q++) copy_bytes_grid<true>(dp[q], sp[q], nb[q]);
    }
    bs.signal(t, 2);
    bs.wait_all_blocks(t, 2);
    bs.finish(2);
}

/* ------------------------------------------------------------------ */
/* host-side launchers                                                 */
/* ------------------------------------------------------------------ */
/* the datatype / operator tables are also compiled into the host emulation that checks every supported pair
 * (tests/emu/nvl_emu_numerics.cpp defines NVL_EMU_SUPPORT_TABLES) */
#if !defined(NVL_HOST_EMU) || defined(NVL_EMU_SUPPORT_TABLES)
extern "C" int nvl_dt_supports_op(int dt, int op)
{
    if (dt < 0 || dt >= NVL_DT_LAST || op < 0 || op >= NVL_OP_LAST) return 0;
    if (dt == NVL_DT_F16 || dt == NVL_DT_F32 || dt == NVL_DT_F64 || dt == NVL_DT_BF16)
        return op == NVL_OP_SUM || op == NVL_OP_PROD || op == NVL_OP_MAX || op == NVL_OP_MIN || op == NVL_OP_AVG;
    if (dt == NVL_DT_C64 || dt == NVL_DT_C128) return op == NVL_OP_SUM || op == NVL_OP_PROD || op == NVL_OP_AVG;
    return 1;
}
extern "C" int nvl_nvls_supports(int dt, int op)
{
    /* mirrors the McRed<T,OP> specialisations: what multimem.ld_reduce can do for 16-byte vectors of that type */
    if (dt == NVL_DT_F32 || dt == NVL_DT_BF16 || dt == NVL_DT_F16 || dt == NVL_DT_C64) return op == NVL_OP_SUM || op == NVL_OP_AVG;
    if (dt == NVL_DT_I32 || dt == NVL_DT_U32 || dt == NVL_DT_I64 || dt == NVL_DT_U64)
        return op == NVL_OP_SUM || op == NVL_OP_MIN || op == NVL_OP_MAX || op == NVL_OP_BAND || op == NVL_OP_BOR || op == NVL_OP_BXOR;
    return 0;
}
#endif

#ifndef NVL_HOST_EMU /* tests/emu includes the kernels above and calls them directly */
extern "C" size_t nvl_dt_size(int dt)
{
    static const size_t s[NVL_DT_LAST] = {1, 2, 4, 8, 1, 2, 4, 8, 2, 4, 8, 2, 8, 16};
    return dt >= 0 && dt < NVL_DT_LAST ? s[dt] : 0;
}

typedef cudaError_t (*nvl_red_launch_fn)(const nvl_red_args_t *, int, int, cudaStream_t);
#define DECL(_s) extern "C" cudaError_t nvl_launch_oneshot_##_s(const nvl_red_args_t *, int, int, cudaStream_t); \
                 extern "C" cudaError_t nvl_launch_staged_##_s(const nvl_red_args_t *, int, int, cudaStream_t);
DECL(i8) DECL(i16) DECL(i32) DECL(i64) DECL(u8) DECL(u16) DECL(u32) DECL(u64) DECL(f16) DECL(f32) DECL(f64) DECL(bf16) DECL(c64) DECL(c128)
static const nvl_red_launch_fn oneshot_fns[NVL_DT_LAST] = {nvl_launch_oneshot_i8, nvl_launch_oneshot_i16, nvl_launch_oneshot_i32, nvl_launch_oneshot_i64, nvl_launch_oneshot_u8, nvl_launch_oneshot_u16,
    nvl_launch_oneshot_u32, nvl_launch_oneshot_u64, nvl_launch_oneshot_f16, nvl_launch_oneshot_f32, nvl_launch_oneshot_f64, nvl_launch_oneshot_bf16,
    nvl_launch_oneshot_c64, nvl_launch_oneshot_c128};
static const nvl_red_launch_fn staged_fns[NVL_DT_LAST] = {nvl_launch_staged_i8, nvl_launch_staged_i16, nvl_launch_staged_i32, nvl_launch_staged_i64, nvl_launch_staged_u8, nvl_launch_staged_u16,
    nvl_launch_staged_u32, nvl_launch_staged_u64, nvl_launch_staged_f16, nvl_launch_staged_f32, nvl_launch_staged_f64, nvl_launch_staged_bf16,
    nvl_launch_staged_c64, nvl_launch_staged_c128};

extern "C" cudaError_t nvl_launch_allreduce_oneshot(const nvl_red_args_t *a, int nblocks, int nthreads, cudaStream_t s)
{
    if (nthreads > NVL_THREADS_MAX) nthreads = NVL_THREADS_MAX;
    if (a->dt < 0 || a->dt >= NVL_DT_LAST) return cudaErrorInvalidValue;
    return oneshot_fns[a->dt](a, nblocks, nthreads, s);
}
extern "C" cudaError_t nvl_launch_reduce_staged(const nvl_red_args_t *a, int nblocks, int nthreads, cudaStream_t s)
{
    if (nthreads > NVL_THREADS_MAX) nthreads = NVL_THREADS_MAX;
    if (a->dt < 0 || a->dt >= NVL_DT_LAST) return cudaErrorInvalidValue;
    return staged_fns[a->dt](a, nblocks, nthreads, s);
}
#define DECLD(_s) extern "C" cudaError_t nvl_launch_direct_##_s(const nvl_red_args_t *, int, int, cudaStream_t);
DECLD(i8) DECLD(i16) DECLD(i32) DECLD(i64) DECLD(u8) DECLD(u16) DECLD(u32) DECLD(u64) DECLD(f16) DECLD(f32) DECLD(f64) DECLD(bf16) DECLD(c64) DECLD(c128)
static const nvl_red_launch_fn direct_fns[NVL_DT_LAST] = {nvl_launch_direct_i8, nvl_launch_direct_i16, nvl_launch_direct_i32, nvl_launch_direct_i64, nvl_launch_direct_u8, nvl_launch_direct_u16,
    nvl_launch_direct_u32, nvl_launch_direct_u64, nvl_launch_direct_f16, nvl_launch_direct_f32, nvl_launch_direct_f64, nvl_launch_direct_bf16,
    nvl_launch_direct_c64, nvl_launch_direct_c128};
extern "C" cudaError_t nvl_launch_reduce_direct(const nvl_red_args_t *a, int nblocks, int nthreads, cudaStream_t s)
{
    if (nthreads > NVL_THREADS_MAX) nthreads = NVL_THREADS_MAX;
    if (a->dt < 0 || a->dt >= NVL_DT_LAST) return cudaErrorInvalidValue;
    return direct_fns[a->dt](a, nblocks, nthreads, s);
}
#define DECLS(_s) extern "C" cudaError_t nvl_launch_steps_##_s(const nvl_red_args_t *, int, int, cudaStream_t);
DECLS(i8) DECLS(i16) DECLS(i32) DECLS(i64) DECLS(u8) DECLS(u16) DECLS(u32) DECLS(u64) DECLS(f16) DECLS(f32) DECLS(f64) DECLS(bf16) DECLS(c64) DECLS(c128)
static const nvl_red_launch_fn steps_fns[NVL_DT_LAST] = {nvl_launch_steps_i8, nvl_launch_steps_i16, nvl_launch_steps_i32, nvl_launch_steps_i64, nvl_launch_steps_u8, nvl_launch_steps_u16,
    nvl_launch_steps_u32, nvl_launch_steps_u64, nvl_launch_steps_f16, nvl_launch_steps_f32, nvl_launch_steps_f64, nvl_launch_steps_bf16,
    nvl_launch_steps_c64, nvl_launch_steps_c128};
extern "C" cudaError_t nvl_launch_reduce_steps(const nvl_red_args_t *a, int nblocks, int nthreads, cudaStream_t s)
{
    if (nthreads > NVL_THREADS_MAX) nthreads = NVL_THREADS_MAX;
    if (a->dt < 0 || a->dt >= NVL_DT_LAST) return cudaErrorInvalidValue;
    return steps_fns[a->dt](a, nblocks, nthreads, s);
}
extern "C" cudaError_t nvl_launch_exchange(const nvl_xchg_args_t *a, int nblocks, int nthreads, cudaStream_t s)
{
    if (nthreads > NVL_THREADS_MAX) nthreads = NVL_THREADS_MAX;
    nvl_exchange_kernel<<<nblocks, nthreads, 0, s>>>(*a);
    return cudaGetLastError();
}
/* single-member team: every collective degenerates to (at most) one device copy; this is that copy, at HBM speed */
__global__ void __launch_bounds__(NVL_THREADS_MAX, 2) nvl_self_copy_kernel(char *dst, const char *src, size_t n)
{ copy_bytes_grid<false>(dst, src, n); }
extern "C" cudaError_t nvl_launch_self_copy(void *dst, const void *src, size_t bytes, int nblocks, int nthreads, cudaStream_t s)
{
    if (nthreads > NVL_THREADS_MAX) nthreads = NVL_THREADS_MAX;
    nvl_self_copy_kernel<<<nblocks, nthreads, 0, s>>>(static_cast<char *>(dst), static_cast<const char *>(src), bytes);
    return cudaGetLastError();
}
extern "C" cudaError_t nvl_launch_barrier(const nvl_team_dev_t *t, cudaStream_t s)
{
    nvl_barrier_kernel<<<1, 32, 0, s>>>(*t);
    return cudaGetLastError();
}
extern "C" cudaError_t nvl_launch_ctrl_init(void *heap_base, cudaStream_t s)
{
    nvl_ctrl_init_kernel<<<4, 256, 0, s>>>(static_cast<nvl_ctrl_t *>(heap_base));
    return cudaGetLastError();
}
#endif /* NVL_HOST_EMU */
