/* Device-side building blocks of tl/nvl (sm_100a):
 *   - system-scope flag signalling between GPUs (st.release.sys / ld.acquire.sys)
 *   - per-block barriers with monotonically increasing epochs and a spin budget
 *   - 16-byte vector load/store helpers (aligned fast path, guarded element path)
 *   - datatype x operator reduction templates (the inlined "executor")
 *   - NVLS multimem.ld_reduce / multimem.st wrappers
 */
#ifndef UCC_TL_NVL_DEVICE_CUH_
#define UCC_TL_NVL_DEVICE_CUH_
#include "nvl_kernels.h"
#include <cuda_fp16.h>
#include <cuda_bf16.h>

#define NVL_DEV __device__ __forceinline__

/* ------------------------------------------------------------------ */
/* memory-model primitives                                             */
/* ------------------------------------------------------------------ */
#ifdef NVL_HOST_EMU
/* tests/emu: the kernels compiled as host C++ (one OS thread per CUDA thread); the PTX below is replaced by C++ equivalents */
#include "nvl_device_emu.h"
#else
NVL_DEV void st_release_sys_u32(uint32_t *p, uint32_t v) { asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory"); }
NVL_DEV void st_relaxed_sys_u32(uint32_t *p, uint32_t v) { asm volatile("st.relaxed.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory"); }
NVL_DEV uint32_t ld_acquire_sys_u32(const uint32_t *p) { uint32_t v; asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory"); return v; }
NVL_DEV uint64_t ld_acquire_sys_u64(const uint64_t *p) { uint64_t v; asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory"); return v; }
NVL_DEV uint32_t ld_volatile_u32(const uint32_t *p) { uint32_t v; asm volatile("ld.volatile.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory"); return v; }
NVL_DEV void fence_sys() { asm volatile("fence.acq_rel.sys;" ::: "memory"); }
NVL_DEV uint64_t globaltimer_ns() { uint64_t t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); return t; }

/* data loads of memory other GPUs write during the kernel: never served from a stale L1 line */
NVL_DEV uint4 ld_peer_v4(const void *p)
{ uint4 v; asm volatile("ld.volatile.global.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p) : "memory"); return v; }
/* streaming load of the user's (read-only) source buffer */
NVL_DEV uint4 ld_src_v4(const void *p)
{ uint4 v; asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p)); return v; }
NVL_DEV void st_v4(void *p, uint4 v)
{ asm volatile("st.global.v4.u32 [%0], {%1,%2,%3,%4};" ::"l"(p), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory"); }

/* NVLS: the address is inside the multicast mapping; the switch performs the add / the replication */
NVL_DEV uint4 mc_ld_reduce_f32(const void *mc) { uint4 v; asm volatile("multimem.ld_reduce.relaxed.sys.global.add.v4.f32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(mc) : "memory"); return v; }
NVL_DEV uint4 mc_ld_reduce_bf16(const void *mc) { uint4 v; asm volatile("multimem.ld_reduce.relaxed.sys.global.add.acc::f32.v4.bf16x2 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(mc) : "memory"); return v; }
NVL_DEV uint4 mc_ld_reduce_f16(const void *mc) { uint4 v; asm volatile("multimem.ld_reduce.relaxed.sys.global.add.acc::f32.v4.f16x2 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(mc) : "memory"); return v; }
/* integer / bitwise in-switch reductions are scalar (32 or 64 bit per instruction): 4 resp. 2 of them make one 16-byte vector
 * (reference kernels K2: tl/cuda/kernels/allreduce_kernel.cu:59-141 do the same for add) */
#define NVL_MC_RED32(_name, _op)                                                                                         \
    NVL_DEV uint4 _name(const void *mc) { uint4 v; const char *p = static_cast<const char *>(mc);                          \
        asm volatile("multimem.ld_reduce.relaxed.sys.global." _op " %0, [%1];" : "=r"(v.x) : "l"(p) : "memory");        \
        asm volatile("multimem.ld_reduce.relaxed.sys.global." _op " %0, [%1];" : "=r"(v.y) : "l"(p + 4) : "memory");    \
        asm volatile("multimem.ld_reduce.relaxed.sys.global." _op " %0, [%1];" : "=r"(v.z) : "l"(p + 8) : "memory");    \
        asm volatile("multimem.ld_reduce.relaxed.sys.global." _op " %0, [%1];" : "=r"(v.w) : "l"(p + 12) : "memory");   \
        return v; }
#define NVL_MC_RED64(_name, _op)                                                                                         \
    NVL_DEV uint4 _name(const void *mc) { unsigned long long a, b; const char *p = static_cast<const char *>(mc);         \
        asm volatile("multimem.ld_reduce.relaxed.sys.global." _op " %0, [%1];" : "=l"(a) : "l"(p) : "memory");          \
        asm volatile("multimem.ld_reduce.relaxed.sys.global." _op " %0, [%1];" : "=l"(b) : "l"(p + 8) : "memory");      \
        return make_uint4((unsigned)a, (unsigned)(a >> 32), (unsigned)b, (unsigned)(b >> 32)); }
NVL_MC_RED32(mc_red_add_s32, "add.s32") NVL_MC_RED32(mc_red_add_u32, "add.u32") NVL_MC_RED32(mc_red_min_s32, "min.s32") NVL_MC_RED32(mc_red_max_s32, "max.s32")
NVL_MC_RED32(mc_red_min_u32, "min.u32") NVL_MC_RED32(mc_red_max_u32, "max.u32") NVL_MC_RED32(mc_red_and_b32, "and.b32") NVL_MC_RED32(mc_red_or_b32, "or.b32")
NVL_MC_RED32(mc_red_xor_b32, "xor.b32")
NVL_MC_RED64(mc_red_add_u64, "add.u64") NVL_MC_RED64(mc_red_min_s64, "min.s64") NVL_MC_RED64(mc_red_max_s64, "max.s64") NVL_MC_RED64(mc_red_min_u64, "min.u64")
NVL_MC_RED64(mc_red_max_u64, "max.u64") NVL_MC_RED64(mc_red_and_b64, "and.b64") NVL_MC_RED64(mc_red_or_b64, "or.b64") NVL_MC_RED64(mc_red_xor_b64, "xor.b64")
NVL_DEV void mc_st_v4(void *mc, uint4 v) { asm volatile("multimem.st.relaxed.sys.global.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(mc), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory"); }
#endif /* NVL_HOST_EMU */

/* ------------------------------------------------------------------ */
/* per-block inter-GPU barrier                                         */
/* ------------------------------------------------------------------ */
struct BlockSync {
    nvl_ctrl_t *mine;
    uint32_t    epoch;
    int         blk;
    bool        timed_out;

    NVL_DEV void init(const nvl_team_dev_t &t)
    {
        mine = reinterpret_cast<nvl_ctrl_t *>(t.heap[t.rank]);
        blk = blockIdx.x;
        /* one epoch per rank; it only changes when the LAST block of a kernel retires, so every
         * block of this kernel reads the same value no matter when it starts */
        epoch = ld_volatile_u32(&mine->epoch);
        timed_out = false;
    }
    NVL_DEV void spin(const nvl_team_dev_t &t, const uint32_t *f, uint32_t target)
    {
        uint64_t t0 = 0; uint32_t spins = 0;
        while ((int32_t)(ld_acquire_sys_u32(f) - target) < 0) {
            if ((++spins & 0x3ff) == 0) {
                uint64_t now = globaltimer_ns();
                if (!t0) t0 = now;
                else if (now - t0 > t.timeout_ns) { if (t.host_err) *t.host_err = 1; mine->error = 1; break; }
            }
        }
    }
    /* wait until EVERY block of every peer signalled `phase` (for kernels whose blocks read
     * data staged by arbitrary peer blocks) */
    NVL_DEV void wait_all_blocks(const nvl_team_dev_t &t, uint32_t phase)
    {
        int nb = gridDim.x;
        for (int i = threadIdx.x; i < nb * t.size; i += blockDim.x) {
            int p = i / nb, b = i % nb;
            if (p != t.rank) spin(t, &mine->flags[b][p], epoch + phase);
        }
        __syncthreads();
    }
    /* everything this block wrote so far becomes visible to the peers before they see the flag */
    NVL_DEV void signal(const nvl_team_dev_t &t, uint32_t phase)
    {
        __syncthreads();
        int p = threadIdx.x;
        if (p < t.size && p != t.rank) {
            fence_sys();
            st_relaxed_sys_u32(&reinterpret_cast<nvl_ctrl_t *>(t.heap[p])->flags[blk][t.rank], epoch + phase);
        }
    }
    NVL_DEV void wait(const nvl_team_dev_t &t, uint32_t phase)
    {
        int p = threadIdx.x;
        if (p < t.size && p != t.rank) spin(t, &mine->flags[blk][p], epoch + phase);
        __syncthreads();
    }
    NVL_DEV void barrier(const nvl_team_dev_t &t, uint32_t phase) { signal(t, phase); wait(t, phase); }
    NVL_DEV void finish(uint32_t nphases)
    {
        __syncthreads();
        if (threadIdx.x == 0) {
            __threadfence();
            if (atomicAdd(&mine->done_blocks, 1u) == gridDim.x - 1) { mine->done_blocks = 0; __threadfence(); mine->epoch = epoch + nphases; }
        }
    }
};

/* ------------------------------------------------------------------ */
/* vectors of 16 bytes                                                 */
/* ------------------------------------------------------------------ */
template <typename T> struct Vec { static constexpr int E = 16 / sizeof(T); union { uint4 v; T e[16 / sizeof(T)]; }; };

template <typename T> NVL_DEV uint4 load_src_vec(const T *base, size_t idx, size_t n, bool aligned)
{
    constexpr int E = 16 / sizeof(T);
    if (aligned && idx + E <= n) return ld_src_v4(base + idx);
    Vec<T> u; u.v = make_uint4(0, 0, 0, 0);
#pragma unroll
    for (int i = 0; i < E; i++) if (idx + i < n) u.e[i] = base[idx + i];
    return u.v;
}
template <typename T> NVL_DEV void store_dst_vec(T *base, size_t idx, size_t n, bool aligned, uint4 x)
{
    constexpr int E = 16 / sizeof(T);
    if (aligned && idx + E <= n) { st_v4(base + idx, x); return; }
    Vec<T> u; u.v = x;
#pragma unroll
    for (int i = 0; i < E; i++) if (idx + i < n) base[idx + i] = u.e[i];
}

/* ------------------------------------------------------------------ */
/* reduction templates                                                 */
/* ------------------------------------------------------------------ */
/* complex elements (UCC_DT_FLOAT32_COMPLEX / FLOAT64_COMPLEX): plain pairs aligned like their component (4 / 8 bytes, not 16),
 * so the guarded element path (base[idx + i]) never issues an access wider than the alignment the caller's buffer has */
struct nvl_c64 { float re, im; };
struct nvl_c128 { double re, im; };
template <typename T> struct IsComplex { static constexpr bool v = false; };
template <> struct IsComplex<nvl_c64> { static constexpr bool v = true; };
template <> struct IsComplex<nvl_c128> { static constexpr bool v = true; };

template <typename T> struct AccOf { typedef T type; };
template <> struct AccOf<__half> { typedef float type; };
template <> struct AccOf<__nv_bfloat16> { typedef float type; };

template <typename T> NVL_DEV typename AccOf<T>::type to_acc(T x) { return x; }
template <> NVL_DEV float to_acc<__half>(__half x) { return __half2float(x); }
template <> NVL_DEV float to_acc<__nv_bfloat16>(__nv_bfloat16 x) { return __bfloat162float(x); }
template <typename T> NVL_DEV T from_acc(typename AccOf<T>::type x) { return (T)x; }
template <> NVL_DEV __half from_acc<__half>(float x) { return __float2half_rn(x); }
template <> NVL_DEV __nv_bfloat16 from_acc<__nv_bfloat16>(float x) { return __float2bfloat16_rn(x); }

template <int OP, typename A> struct OpFn;
template <typename A> struct OpFn<NVL_OP_SUM, A> { static NVL_DEV A f(A a, A b) { return a + b; } };
template <typename A> struct OpFn<NVL_OP_AVG, A> { static NVL_DEV A f(A a, A b) { return a + b; } };
template <typename A> struct OpFn<NVL_OP_PROD, A> { static NVL_DEV A f(A a, A b) { return a * b; } };
template <typename A> struct OpFn<NVL_OP_MAX, A> { static NVL_DEV A f(A a, A b) { return a > b ? a : b; } };
template <typename A> struct OpFn<NVL_OP_MIN, A> { static NVL_DEV A f(A a, A b) { return a < b ? a : b; } };
template <typename A> struct OpFn<NVL_OP_LAND, A> { static NVL_DEV A f(A a, A b) { return (A)(a && b); } };
template <typename A> struct OpFn<NVL_OP_LOR, A> { static NVL_DEV A f(A a, A b) { return (A)(a || b); } };
template <typename A> struct OpFn<NVL_OP_LXOR, A> { static NVL_DEV A f(A a, A b) { return (A)((!a) != (!b)); } };
template <typename A> struct OpFn<NVL_OP_BAND, A> { static NVL_DEV A f(A a, A b) { return (A)(a & b); } };
template <typename A> struct OpFn<NVL_OP_BOR, A> { static NVL_DEV A f(A a, A b) { return (A)(a | b); } };
template <typename A> struct OpFn<NVL_OP_BXOR, A> { static NVL_DEV A f(A a, A b) { return (A)(a ^ b); } };
/* complex: SUM / AVG part by part, PROD = (ac - bd) + (ad + bc)i as cuCmul computes it (no Annex G inf / nan recovery);
 * accumulation stays in the component precision */
#define NVL_COMPLEX_OPS(_C)                                                                                                  \
    template <> struct OpFn<NVL_OP_SUM, _C> { static NVL_DEV _C f(_C a, _C b) { return {a.re + b.re, a.im + b.im}; } };     \
    template <> struct OpFn<NVL_OP_AVG, _C> { static NVL_DEV _C f(_C a, _C b) { return {a.re + b.re, a.im + b.im}; } };     \
    template <> struct OpFn<NVL_OP_PROD, _C> {                                                                              \
        static NVL_DEV _C f(_C a, _C b) { return {a.re * b.re - a.im * b.im, a.re * b.im + a.im * b.re}; } };
NVL_COMPLEX_OPS(nvl_c64)
NVL_COMPLEX_OPS(nvl_c128)
#undef NVL_COMPLEX_OPS

/* AVG = SUM scaled by 1/N at the very end.  Floating types multiply by 1/N computed in the accumulator's precision (float for
 * f16 / bf16 / f32, double for f64; a float 1/N would cost f64 about 1e-8 relative for N = 3); integer types divide by N
 * (truncating, i.e. what the reference's d[i] * (1/N) in double precision yields for every sum a double represents exactly) -
 * casting 1/N to an integer accumulator would be 0 */
template <typename A> struct IsIntAcc { static constexpr bool v = true; };
template <> struct IsIntAcc<float> { static constexpr bool v = false; };
template <> struct IsIntAcc<double> { static constexpr bool v = false; };
template <int OP, typename A> NVL_DEV A avg_scale(A x, int n)
{
    if (OP != NVL_OP_AVG) return x;
    if constexpr (IsComplex<A>::v) { typedef decltype(x.re) R; const R s = (R)1 / (R)n; return {x.re * s, x.im * s}; } /* 1/N in the component precision (IsIntAcc is true for it) */
    else if constexpr (IsIntAcc<A>::v) return n > 1 ? (A)(x / (A)n) : x;
    else return (A)(x * ((A)1 / (A)n));
}

/* accumulator for one 16-byte vector of T */
template <typename T, int OP> struct VecAcc {
    typedef typename AccOf<T>::type A;
    static constexpr int E = 16 / sizeof(T);
    A a[E];
    NVL_DEV void set(uint4 x) { Vec<T> u; u.v = x;
#pragma unroll
        for (int i = 0; i < E; i++) a[i] = to_acc<T>(u.e[i]); }
    NVL_DEV void add(uint4 x) { Vec<T> u; u.v = x;
#pragma unroll
        for (int i = 0; i < E; i++) a[i] = OpFn<OP, A>::f(a[i], to_acc<T>(u.e[i])); }
    NVL_DEV uint4 get(int n) { Vec<T> u;
#pragma unroll
        for (int i = 0; i < E; i++) u.e[i] = from_acc<T>(avg_scale<OP, A>(a[i], n));
        return u.v; }
};

template <typename T> struct IsFloatLike { static constexpr bool v = false; };
template <> struct IsFloatLike<float> { static constexpr bool v = true; };
template <> struct IsFloatLike<double> { static constexpr bool v = true; };
template <> struct IsFloatLike<__half> { static constexpr bool v = true; };
template <> struct IsFloatLike<__nv_bfloat16> { static constexpr bool v = true; };

/* run F<T,OP>::run(args...) for the runtime operator; MAX / MIN do not exist for complex types, bit/logic operators only for
 * integer types */
#define NVL_DISPATCH_OP(_T, _op, _CALL)                                                         \
    do {                                                                                        \
        switch (_op) {                                                                          \
        case NVL_OP_SUM: _CALL(_T, NVL_OP_SUM); break;                                          \
        case NVL_OP_AVG: _CALL(_T, NVL_OP_AVG); break;                                          \
        case NVL_OP_PROD: _CALL(_T, NVL_OP_PROD); break;                                        \
        default:                                                                                \
            if constexpr (!IsComplex<_T>::v) {                                                  \
                switch (_op) {                                                                  \
                case NVL_OP_MAX: _CALL(_T, NVL_OP_MAX); break;                                  \
                case NVL_OP_MIN: _CALL(_T, NVL_OP_MIN); break;                                  \
                default:                                                                        \
                    if constexpr (!IsFloatLike<_T>::v) {                                        \
                        switch (_op) {                                                          \
                        case NVL_OP_LAND: _CALL(_T, NVL_OP_LAND); break;                        \
                        case NVL_OP_LOR: _CALL(_T, NVL_OP_LOR); break;                          \
                        case NVL_OP_LXOR: _CALL(_T, NVL_OP_LXOR); break;                        \
                        case NVL_OP_BAND: _CALL(_T, NVL_OP_BAND); break;                        \
                        case NVL_OP_BOR: _CALL(_T, NVL_OP_BOR); break;                          \
                        case NVL_OP_BXOR: _CALL(_T, NVL_OP_BXOR); break;                        \
                        default: break;                                                         \
                        }                                                                       \
                    }                                                                           \
                    break;                                                                      \
                }                                                                               \
            }                                                                                   \
            break;                                                                              \
        }                                                                                       \
    } while (0)
#endif
