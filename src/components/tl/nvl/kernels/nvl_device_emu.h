/* Host emulation of the PTX primitives of nvl_device.cuh (NVL_HOST_EMU): lets tests/test_nvl_emu.py compile the collective
 * kernels as ordinary C++ and run them with one OS thread per CUDA thread - N "GPUs" are N heaps in one address space, the
 * NVSwitch multicast mapping is a reserved fake address range whose offsets are applied to every heap.  Only the logic of the
 * kernels (indexing, phases, flag protocol) is exercised this way; memory-model subtleties of the real hardware are not. */
#ifndef UCC_TL_NVL_DEVICE_EMU_H_
#define UCC_TL_NVL_DEVICE_EMU_H_
#include <string.h>
#include <time.h>
#include <sched.h>

struct nvl_emu_world {
    char  *heaps[NVL_MAX_PEERS];
    int    n;
    char  *mc_base;      /* fake base of the multicast mapping (never dereferenced) */
    size_t heap_size;
};
extern nvl_emu_world g_emu;

static inline void st_release_sys_u32(uint32_t *p, uint32_t v) { __atomic_store_n(p, v, __ATOMIC_RELEASE); }
static inline void st_relaxed_sys_u32(uint32_t *p, uint32_t v) { __atomic_store_n(p, v, __ATOMIC_RELEASE); }
static inline uint32_t ld_acquire_sys_u32(const uint32_t *p) { uint32_t v = __atomic_load_n(p, __ATOMIC_ACQUIRE); sched_yield(); return v; }
static inline uint64_t ld_acquire_sys_u64(const uint64_t *p) { return __atomic_load_n(p, __ATOMIC_ACQUIRE); }
static inline uint32_t ld_volatile_u32(const uint32_t *p) { return __atomic_load_n(p, __ATOMIC_ACQUIRE); }
static inline void fence_sys() { __atomic_thread_fence(__ATOMIC_SEQ_CST); }
static inline uint64_t globaltimer_ns() { timespec ts; clock_gettime(CLOCK_MONOTONIC, &ts); return (uint64_t)ts.tv_sec * 1000000000ull + (uint64_t)ts.tv_nsec; }
static inline uint4 ld_peer_v4(const void *p) { uint4 v; memcpy(&v, p, 16); return v; }
static inline uint4 ld_src_v4(const void *p) { uint4 v; memcpy(&v, p, 16); return v; }
static inline void st_v4(void *p, uint4 v) { memcpy(p, &v, 16); }

/* multicast helpers: offset inside the fake mapping -> the same offset of every heap */
static inline size_t emu_mc_off(const void *mc)
{
    size_t off = (size_t)(static_cast<const char *>(mc) - g_emu.mc_base);
    if (off + 16 > g_emu.heap_size) { fprintf(stderr, "EMU: multicast access outside the heap (offset %zu)\n", off); abort(); }
    if (off & 15) { fprintf(stderr, "EMU: unaligned multicast access (offset %zu)\n", off); abort(); }
    return off;
}
template <typename E, typename F> static inline uint4 emu_mc_reduce(const void *mc, F f)
{
    const size_t off = emu_mc_off(mc);
    constexpr int n = 16 / sizeof(E);
    E acc[n], cur[n];
    memcpy(acc, g_emu.heaps[0] + off, 16);
    for (int p = 1; p < g_emu.n; p++) { memcpy(cur, g_emu.heaps[p] + off, 16); for (int i = 0; i < n; i++) acc[i] = f(acc[i], cur[i]); }
    uint4 v; memcpy(&v, acc, 16); return v;
}
static inline uint4 mc_ld_reduce_f32(const void *mc) { return emu_mc_reduce<float>(mc, [](float a, float b) { return a + b; }); }
/* .acc::f32: the switch adds the 16-bit values in float and rounds the sum once to the storage type */
template <typename H, typename TO, typename FROM> static inline uint4 emu_mc_reduce_acc_f32(const void *mc, TO to_f, FROM from_f)
{
    const size_t off = emu_mc_off(mc);
    H cur[8]; float acc[8];
    for (int p = 0; p < g_emu.n; p++) { memcpy(cur, g_emu.heaps[p] + off, 16); for (int i = 0; i < 8; i++) acc[i] = p ? acc[i] + to_f(cur[i]) : to_f(cur[i]); }
    for (int i = 0; i < 8; i++) cur[i] = from_f(acc[i]);
    uint4 v; memcpy(&v, cur, 16); return v;
}
static inline uint4 mc_ld_reduce_bf16(const void *mc)
{ return emu_mc_reduce_acc_f32<__nv_bfloat16>(mc, [](__nv_bfloat16 x) { return __bfloat162float(x); }, [](float x) { return __float2bfloat16_rn(x); }); }
static inline uint4 mc_ld_reduce_f16(const void *mc)
{ return emu_mc_reduce_acc_f32<__half>(mc, [](__half x) { return __half2float(x); }, [](float x) { return __float2half_rn(x); }); }
#define NVL_EMU_RED(_name, _E, _expr) static inline uint4 _name(const void *mc) { return emu_mc_reduce<_E>(mc, [](_E a, _E b) { return (_E)(_expr); }); }
NVL_EMU_RED(mc_red_add_s32, int32_t, a + b) NVL_EMU_RED(mc_red_add_u32, uint32_t, a + b) NVL_EMU_RED(mc_red_min_s32, int32_t, a < b ? a : b) NVL_EMU_RED(mc_red_max_s32, int32_t, a > b ? a : b)
NVL_EMU_RED(mc_red_min_u32, uint32_t, a < b ? a : b) NVL_EMU_RED(mc_red_max_u32, uint32_t, a > b ? a : b) NVL_EMU_RED(mc_red_and_b32, uint32_t, a & b) NVL_EMU_RED(mc_red_or_b32, uint32_t, a | b)
NVL_EMU_RED(mc_red_xor_b32, uint32_t, a ^ b)
NVL_EMU_RED(mc_red_add_u64, uint64_t, a + b) NVL_EMU_RED(mc_red_min_s64, int64_t, a < b ? a : b) NVL_EMU_RED(mc_red_max_s64, int64_t, a > b ? a : b) NVL_EMU_RED(mc_red_min_u64, uint64_t, a < b ? a : b)
NVL_EMU_RED(mc_red_max_u64, uint64_t, a > b ? a : b) NVL_EMU_RED(mc_red_and_b64, uint64_t, a & b) NVL_EMU_RED(mc_red_or_b64, uint64_t, a | b) NVL_EMU_RED(mc_red_xor_b64, uint64_t, a ^ b)
static inline void mc_st_v4(void *mc, uint4 v) { const size_t off = emu_mc_off(mc); for (int p = 0; p < g_emu.n; p++) memcpy(g_emu.heaps[p] + off, &v, 16); }
#endif
