// Numerics of every tl/nvl reduction kernel, compiled as host C++ (NVL_HOST_EMU) for ONE datatype (-DNUM_DT=<nvl_dt_t>):
// one-shot allreduce, one-shot reduce_scatter(v), staged P2P, staged NVLS, zero-copy direct, ring, rhd, nvls_pipe and symm, with
// every operator nvl_dt_supports_op() accepts (NVLS kernels: what nvl_nvls_supports() accepts), as allreduce, reduce (root != 0)
// and reduce_scatter(v), over counts around the vector width and the staging capacity, shifted by one element and in place.
//
// Inputs are chosen so that every result can be checked bit for bit whatever order a kernel reduces in (the in-switch reduction
// of the NVLS kernels has no defined order):
//   exact-sum   signed k * 2^e, |k| <= 127, e in [-4, 4], and +-0: every partial sum of <= 8 terms is a multiple of 2^-4 below
//               2^14, exact in float.  SUM = the exact sum rounded once; AVG = acc(sum) * acc(1/N) rounded once; MAX / MIN exact
//   exact-prod  {+-0.5, +-0.75, +-1, +-1.5, +-2}: a product of <= 8 terms has at most 13 significant bits, exact in float
//   special     exact-prod values, with NaN / +Inf / +Inf and -Inf (two ranks) on chosen elements: NaN resp. Inf on every rank
//   random      k * 2^-m, |k| < 2^m, m = significand bits: allreduce outputs bitwise equal on every rank, and
//               |got - sum| <= (N-1) u_acc sum|x| + ulp(got)/2 (recursive summation: N-1 roundings of partial sums bounded by
//               sum|x|, to first order; then one rounding to the storage type); AVG: see check_elem()
//   integers    random full-width bits (logical operators: zero and non-zero values whose low byte is zero); SUM / PROD wrap,
//               AVG = trunc(wrapped sum / N), all exact
// Exceptions that are properties of the algorithm, not defects:
//   - ring / rhd keep partial sums in the heap in the STORAGE type, so for f16 / bf16 they get inputs whose partial sums and
//     products are exact in the storage type (integers |v| <= 31, powers of two), and no error bound on random inputs
//   - in-switch AVG of f16 / bf16: the switch rounds the sum to the storage type, the kernel scales it and rounds again:
//     round(round(sum) * f32(1/N))
// Every destination has one guard element on each side that must stay untouched.
#define NVL_EMU_SUPPORT_TABLES 1
#include "nvl_emu_world.h"
#include <algorithm>
#include <set>

#ifndef NUM_DT
#error "build with -DNUM_DT=<nvl_dt_t value>"
#endif

template <int DT> struct DtOf;
#define NVL_DT_OF(_dt, _T, _name) template <> struct DtOf<_dt> { typedef _T type; static constexpr const char *name = _name; };
NVL_DT_OF(NVL_DT_I8, int8_t, "int8") NVL_DT_OF(NVL_DT_I16, int16_t, "int16") NVL_DT_OF(NVL_DT_I32, int32_t, "int32") NVL_DT_OF(NVL_DT_I64, int64_t, "int64")
NVL_DT_OF(NVL_DT_U8, uint8_t, "uint8") NVL_DT_OF(NVL_DT_U16, uint16_t, "uint16") NVL_DT_OF(NVL_DT_U32, uint32_t, "uint32") NVL_DT_OF(NVL_DT_U64, uint64_t, "uint64")
NVL_DT_OF(NVL_DT_F16, __half, "float16") NVL_DT_OF(NVL_DT_F32, float, "float32") NVL_DT_OF(NVL_DT_F64, double, "float64") NVL_DT_OF(NVL_DT_BF16, __nv_bfloat16, "bfloat16")
NVL_DT_OF(NVL_DT_C64, nvl_c64, "float32_complex") NVL_DT_OF(NVL_DT_C128, nvl_c128, "float64_complex")
typedef DtOf<NUM_DT>::type T;
constexpr int E = 16 / sizeof(T);
constexpr bool IS_FLOAT = IsFloatLike<T>::v, IS_CPLX = IsComplex<T>::v, IS_HALF = sizeof(T) == 2 && IS_FLOAT;
/* significand bits of the storage type and unit roundoff of the accumulator */
constexpr int MBITS = NUM_DT == NVL_DT_F16 ? 11 : NUM_DT == NVL_DT_BF16 ? 8 : (NUM_DT == NVL_DT_F32 || NUM_DT == NVL_DT_C64) ? 24 : 53;
constexpr long double U_ACC = (NUM_DT == NVL_DT_F64 || NUM_DT == NVL_DT_C128) ? 0x1p-53L : 0x1p-24L;

static const char *opn[NVL_OP_LAST] = {"sum", "prod", "max", "min", "land", "lor", "lxor", "band", "bor", "bxor", "avg"};
enum Set { S_SUM, S_PROD, S_SPECIAL, S_RANDOM, S_INT };
static const char *setn[] = {"exact-sum", "exact-prod", "special", "random", "int"};
static int g_fail = 0, g_cases = 0;

static uint64_t mix(uint64_t x)
{
    x += 0x9e3779b97f4a7c15ull; x = (x ^ (x >> 30)) * 0xbf58476d1ce4e5b9ull; x = (x ^ (x >> 27)) * 0x94d049bb133111ebull; return x ^ (x >> 31);
}
static uint64_t rnd(int seed, int r, size_t i) { return mix(mix(mix((uint64_t)seed) ^ (uint64_t)r) ^ (uint64_t)i); }

struct Case {
    int set, op, seed, N;
    bool storage_exact;   /* ring / rhd on f16 / bf16: partial results live in the storage type */
    bool nvls_avg_twice;  /* in-switch AVG of f16 / bf16 */
};

/* ---------------- floating-point inputs and oracle (as long double: every exact input and result fits) ---------------- */
static long double fin(const Case &c, int r, size_t i)
{
    const uint64_t h = rnd(c.seed, r, i);
    switch (c.set) {
    case S_SUM:
        if (i % 97 == 5) return -0.0L;                                  /* -0 on every rank: the sum is -0 */
        if ((h >> 40) % 16 == 0) return (h >> 45) & 1 ? -0.0L : 0.0L;
        if (c.storage_exact) return (long double)((int)(h % 63) - 31);
        return std::ldexp((long double)((int)(h % 255) - 127), (int)((h >> 8) % 9) - 4);
    case S_PROD: case S_SPECIAL: {
        static const long double pv[] = {0.5L, 0.75L, 1.0L, 1.5L, 2.0L}, pe[] = {0.5L, 1.0L, 2.0L};
        const long double v = c.storage_exact ? pe[h % 3] : pv[h % 5];
        if (c.set == S_SPECIAL) {
            const size_t cls = i % 13, who = i % c.N;
            if (cls == 1 && (size_t)r == who) return NAN;
            if ((cls == 4 || cls == 7) && (size_t)r == who) return INFINITY;
            if (cls == 7 && (size_t)r == (who + 1) % c.N) return -INFINITY;
        }
        return (h >> 20) & 1 ? -v : v;
    }
    default: {   /* random: k * 2^-m, |k| < 2^m */
        const int64_t k = (int64_t)(h >> (64 - MBITS - 1)) - ((int64_t)1 << MBITS);
        return std::ldexp((long double)k, -MBITS);
    }
    }
}
template <typename X> static X to_t(long double v) { return from_acc<X>((typename AccOf<X>::type)v); }
template <typename X> static long double of_t(X x) { return (long double)to_acc<X>(x); }
template <typename X> static uint64_t bits(X x) { uint64_t b = 0; memcpy(&b, &x, sizeof(X)); return b; }
template <typename X> static long double ulp_of(X x)   /* distance from |x| to the next representable magnitude */
{
    X a = x; unsigned char *p = (unsigned char *)&a; p[sizeof(X) - 1] &= 0x7f;
    uint64_t b = bits(a) + 1; X n; memcpy(&n, &b, sizeof(X));
    return of_t(n) - of_t(a);
}

/* ---------------- integer inputs and oracle ---------------- */
template <typename I> static I iin(const Case &c, int r, size_t i)
{
    const uint64_t h = rnd(c.seed, r, i);
    if (c.op == NVL_OP_LAND || c.op == NVL_OP_LOR || c.op == NVL_OP_LXOR) {
        static const uint64_t pool[] = {0, 0, 0, 1, 0x80, 0x100, 0x8000, 0x10000, 0x80000000ull, 1ull << 32, 1ull << 63, ~0ull};
        uint64_t v = pool[h % 12] & (sizeof(I) == 8 ? ~0ull : ((1ull << (8 * sizeof(I))) - 1));
        return (I)v;
    }
    return (I)h;
}

/* ---------------- buffers ---------------- */
static const unsigned char GUARD = 0xa5;
struct Buf {   /* 64-byte aligned storage: element E + mis (16-byte aligned for mis = 0) is the first one the kernel sees, the one in front a guard */
    std::vector<unsigned char> raw; T *base;
    void init(size_t n) { raw.assign((n + 2 * E + 8) * sizeof(T) + 128, GUARD); base = (T *)(((uintptr_t)raw.data() + 63) & ~(uintptr_t)63); }
};
static bool guard_ok(const T *p) { const unsigned char *b = (const unsigned char *)p; for (size_t i = 0; i < sizeof(T); i++) if (b[i] != GUARD) return false; return true; }

static void fail(const char *what, int r, size_t i, const char *msg)
{
    if (g_fail < 40) printf("EMU FAIL %s: rank %d elem %zu: %s\n", what, r, i, msg);
    g_fail++;
}

/* ---------------- expected value of one output element ---------------- */
template <typename X = T> static void check_elem(const char *what, const Case &c, int r, size_t i, X got)
{
    char msg[256];
    const int N = c.N;
    if constexpr (std::is_integral<X>::value) {
        typedef typename std::make_unsigned<X>::type UX;
        X acc = iin<X>(c, 0, i);
        uint64_t s = (uint64_t)(UX)acc, pr = s; bool all = acc != 0, any = acc != 0; int nz = acc != 0; X mx = acc, mn = acc, ba = acc, bo = acc, bx = acc;
        for (int p = 1; p < N; p++) {
            const X x = iin<X>(c, p, i);
            s += (uint64_t)(UX)x; pr *= (uint64_t)(UX)x; all = all && x; any = any || x; nz += x != 0;
            mx = std::max(mx, x); mn = std::min(mn, x); ba &= x; bo |= x; bx ^= x;
        }
        X e = 0;
        switch (c.op) {
        case NVL_OP_SUM: e = (X)(UX)s; break;
        case NVL_OP_PROD: e = (X)(UX)pr; break;
        case NVL_OP_MAX: e = mx; break;
        case NVL_OP_MIN: e = mn; break;
        case NVL_OP_LAND: e = all; break;
        case NVL_OP_LOR: e = any; break;
        case NVL_OP_LXOR: e = nz & 1; break;
        case NVL_OP_BAND: e = ba; break;
        case NVL_OP_BOR: e = bo; break;
        case NVL_OP_BXOR: e = bx; break;
        case NVL_OP_AVG: e = (X)((X)(UX)s / (X)N); break;   /* truncating, on the wrapped sum */
        }
        if (got != e) { snprintf(msg, sizeof(msg), "got %lld (0x%llx) expected %lld (0x%llx)", (long long)got, (unsigned long long)(UX)got, (long long)e, (unsigned long long)(UX)e); fail(what, r, i, msg); }
    } else {
        long double s = 0, sabs = 0, pr = 1, mx = -INFINITY, mn = INFINITY; bool allneg0 = true;
        for (int p = 0; p < N; p++) {
            const long double x = fin(c, p, i);
            s += x; sabs += std::fabs(x); pr *= x; mx = std::max(mx, x); mn = std::min(mn, x);
            allneg0 = allneg0 && x == 0 && std::signbit(x);
        }
        if (s == 0) s = allneg0 ? -0.0L : 0.0L;
        typedef typename AccOf<X>::type AX;
        const AX inv = (AX)1 / (AX)N;
        if (c.set == S_RANDOM) {
            if (c.storage_exact) return;   /* partial sums rounded to the storage type (ring / rhd, f16 / bf16): only the ranks' agreement is checked */
            const long double exact = c.op == NVL_OP_AVG ? s / N : s;
            long double bound = ulp_of(got) / 2;
            if (c.op == NVL_OP_SUM) bound += (N - 1) * U_ACC * sabs;
            else {
                /* AVG: fl(fl(S^ * fl(1/N))) with |S^ - S| <= (N-1) u sum|x| (SUM above); fl(1/N) and the product add a relative 2u
                 * each unless N is a power of two (both exact then): <= u sum|x| ((N-1) + 2 [N not a power of two]) / N (1 + 4u) */
                const bool pow2 = (N & (N - 1)) == 0;
                bound += U_ACC * sabs * ((N - 1) + (pow2 ? 0 : 2)) / N * (1 + 4 * U_ACC);
            }
            if (!(std::fabs(of_t(got) - exact) <= bound)) { snprintf(msg, sizeof(msg), "got %.21Lg exact %.21Lg error %.3Lg > bound %.3Lg", of_t(got), exact, std::fabs(of_t(got) - exact), bound); fail(what, r, i, msg); }
            return;
        }
        X e;
        switch (c.op) {
        case NVL_OP_PROD: e = to_t<X>(pr); break;
        case NVL_OP_MAX: e = to_t<X>(mx); break;
        case NVL_OP_MIN: e = to_t<X>(mn); break;
        case NVL_OP_AVG:
            if (c.nvls_avg_twice) e = from_acc<X>(to_acc<X>(to_t<X>(s)) * inv);
            else e = from_acc<X>((AX)s * inv);
            break;
        default: e = to_t<X>(s); break;
        }
        const long double g = of_t(got), x = of_t(e);
        bool ok;
        if (std::isnan(x)) ok = std::isnan(g);
        else if (c.op == NVL_OP_MAX || c.op == NVL_OP_MIN) ok = g == x;   /* compared by value: -0 == +0 */
        else ok = bits(got) == bits(e);
        if (!ok) { snprintf(msg, sizeof(msg), "got %.17Lg (0x%llx) expected %.17Lg (0x%llx)", g, (unsigned long long)bits(got), x, (unsigned long long)bits(e)); fail(what, r, i, msg); }
    }
}

template <typename X> static void fill_input(const Case &c, int r, X *p, size_t n)
{
    for (size_t i = 0; i < n; i++) {
        if constexpr (std::is_integral<X>::value) p[i] = iin<X>(c, r, i);
        else if constexpr (IsComplex<X>::v) { typedef decltype(X::re) R; const uint64_t h = rnd(c.seed, r, i), g = rnd(c.seed + 1, r, i);
            p[i] = X{(R)std::ldexp((long double)((int64_t)(h >> (64 - MBITS - 1)) - ((int64_t)1 << MBITS)), -MBITS), (R)std::ldexp((long double)((int64_t)(g >> (64 - MBITS - 1)) - ((int64_t)1 << MBITS)), -MBITS)}; }
        else p[i] = to_t<X>(fin(c, r, i));
    }
}
template <typename X> static void check_range(const char *what, const Case &c, int r, size_t first, const X *got, size_t n)
{
    if constexpr (!IsComplex<X>::v) for (size_t i = 0; i < n; i++) check_elem<X>(what, c, r, first + i, got[i]);
}

/* would tl_nvl_coll.c run kernel k on this collective? */
static bool kern_fits(const World &w, int k, int kind, size_t count, const std::vector<size_t> *rs)
{
    const int N = w.N;
    size_t slice = 0;
    if (kind == NVL_RED_REDUCE_SCATTER) { for (int p = 0; p < N; p++) slice = std::max(slice, rs ? (*rs)[p] : count / N); }
    else slice = (count + N - 1) / N;
    const size_t cap_e = (w.data_size / N / 16) * E;
    if (k == K_RING || k == K_RHD) return slice <= cap_e;                      /* single round: larger vectors take the two-shot kernels */
    if (k == K_ONESHOT) return count * sizeof(T) <= NVL_LL_MAX;
    if (k == K_ONESHOT_RS) return slice * sizeof(T) <= NVL_LL_MAX;
    if ((k == K_DIRECT || k == K_SYMM) && kind == NVL_RED_REDUCE_SCATTER) {   /* the host takes neither for blocks off a 16-byte boundary */
        size_t o = 0; for (int p = 0; p < N; p++) { if ((o * sizeof(T)) & 15) return false; o += rs ? (*rs)[p] : count / N; }
    }
    return true;
}

enum Place { P_ALIGNED, P_SHIFTED, P_INPLACE };
static const char *placen[] = {"", " shifted", " inplace"};

/* one collective; `rs` = block counts of a reduce_scatterv (nullptr: equal blocks) */
static void run_case(World &w, int k, int kind, const Case &c, size_t count, int place, const std::vector<size_t> *rs = nullptr)
{
    if (!kern_fits(w, k, kind, count, rs)) return;
    const int N = w.N, root = kind == NVL_RED_REDUCE ? N - 1 : 0;
    const bool symm = k == K_SYMM;
    const size_t mis = place == P_SHIFTED ? 1 : 0;
    std::vector<size_t> cnt(N), off(N);
    for (int p = 0, o = 0; p < N; p++) { cnt[p] = kind == NVL_RED_REDUCE_SCATTER ? (rs ? (*rs)[p] : count / N) : count; off[p] = o; o += (int)cnt[p]; }
    std::vector<Buf> sb(N), db(N);
    std::vector<T *> src(N), dst(N);
    const size_t ub = (count * sizeof(T) + 255) / 256 * 256 + 256;
    for (int r = 0; r < N; r++) {
        if (symm) {
            CHECK(2 * ub + 256 <= w.user_size);
            memset(w.user(r), GUARD, 2 * ub + 256);
            src[r] = (T *)(w.user(r) + 256);
        } else { sb[r].init(count); src[r] = sb[r].base + E + mis; }
        fill_input<T>(c, r, src[r], count);
        const size_t dn = kind == NVL_RED_REDUCE_SCATTER ? cnt[r] : count;
        if (place == P_INPLACE) dst[r] = kind == NVL_RED_REDUCE_SCATTER ? src[r] + off[r] : src[r];
        else if (symm && kind != NVL_RED_REDUCE_SCATTER) dst[r] = (T *)(w.user(r) + 256 + ub);
        else { db[r].init(dn); dst[r] = db[r].base + E + mis; }
        if (kind == NVL_RED_REDUCE && r != root) dst[r] = nullptr;
    }
    launch<T>(w, k, kind, c.op, count, src, dst, root, rs);
    g_cases++;
    char what[256];
    snprintf(what, sizeof(what), "%s %s %s %s N %d count %zu %s%s%s", kname[k], DtOf<NUM_DT>::name,
             kind == NVL_RED_ALLREDUCE ? "allreduce" : kind == NVL_RED_REDUCE ? "reduce" : rs ? "reduce_scatterv" : "reduce_scatter",
             opn[c.op], N, count, setn[c.set], placen[place], c.storage_exact ? " storage-exact" : "");
    for (int r = 0; r < N; r++) {
        if (!dst[r]) continue;
        const size_t n = kind == NVL_RED_REDUCE_SCATTER ? cnt[r] : count, first = kind == NVL_RED_REDUCE_SCATTER ? off[r] : 0;
        check_range<T>(what, c, r, first, dst[r], n);
        if (place != P_INPLACE && !guard_ok(dst[r] - 1)) fail(what, r, (size_t)-1, "guard element in front of the destination overwritten");
        if ((place != P_INPLACE || kind != NVL_RED_REDUCE_SCATTER) && !guard_ok(dst[r] + n)) fail(what, r, n, "guard element behind the destination overwritten");
        if (kind == NVL_RED_ALLREDUCE && r > 0 && memcmp(dst[r], dst[0], count * sizeof(T))) {
            size_t i = 0; while (!memcmp(&dst[r][i], &dst[0][i], sizeof(T))) i++;
            size_t nd = 0; for (size_t j = 0; j < count; j++) nd += memcmp(&dst[r][j], &dst[0][j], sizeof(T)) != 0;
            char msg[128]; snprintf(msg, sizeof(msg), "differs from rank 0 (first difference; %zu of %zu elements differ)", nd, count); fail(what, r, i, msg);
        }
    }
}

int main(int argc, char **argv)
{
    setvbuf(stdout, nullptr, _IOLBF, 0);   /* keep what was printed if an emulated access aborts */
    CHECK(argc > 1);
    const int N = atoi(argv[1]);
    const int dt = NUM_DT;
    // 16 KB data region: a few thousand elements already need several staging rounds
    World w(N, 16 * 1024, 1 << 20);
    const size_t cap_e = (w.data_size / N / 16) * E, multi = 2 * N * cap_e + N * (cap_e / 3) + 1;   /* two full staging rounds + a ragged third */
    const bool pow2 = (N & (N - 1)) == 0;

    if constexpr (IS_CPLX) {
        /* random complex values through the one-shot allreduce: every rank stores the same bits */
        for (int op : {NVL_OP_SUM, NVL_OP_AVG, NVL_OP_PROD})
            for (size_t count : {(size_t)N * E + 1, (size_t)4097}) run_case(w, K_ONESHOT, NVL_RED_ALLREDUCE, Case{S_RANDOM, op, 7 + (int)count, N, false, false}, count, P_ALIGNED);
    } else {
        const std::set<size_t> counts_all = {1, (size_t)std::max(E - 1, 1), (size_t)E, (size_t)E + 1, (size_t)N * E - 1, (size_t)N * E + 1, 4097, multi};
        const int allred_k[] = {K_ONESHOT, K_STAGED, K_STAGED_NVLS, K_DIRECT, K_RING, K_RHD, K_PIPE, K_SYMM};
        const int rs_k[] = {K_ONESHOT_RS, K_STAGED, K_STAGED_NVLS, K_DIRECT, K_RING, K_RHD, K_SYMM};
        auto kern_ok = [&](int k, int op) { return nvl_dt_supports_op(dt, op) && (!kern_nvls(k) || nvl_nvls_supports(dt, op)) && (k != K_RHD || pow2); };
        auto mk = [&](int k, int op, int set, int seed) {
            const bool se = IS_HALF && (k == K_RING || k == K_RHD);
            if (!IS_FLOAT) set = S_INT;
            return Case{set, op, seed, N, se, IS_HALF && kern_nvls(k) && op == NVL_OP_AVG};
        };
        auto exact_set = [](int op) { return op == NVL_OP_PROD ? S_PROD : S_SUM; };
        std::vector<size_t> rsv(N), rsv_al(N);   /* unequal blocks with an empty one; rsv_al: every block a whole number of vectors */
        for (int p = 0; p < N; p++) { rsv[p] = p == 1 ? 0 : 3 + 37 * (size_t)p; rsv_al[p] = p == 1 ? 0 : (size_t)E * (p + 2); }

        for (int k : allred_k) {
            for (int op = 0; op < NVL_OP_LAST; op++) {
                if (!kern_ok(k, op)) continue;
                /* every operator on the exact set at a ragged size, then the size sweep for SUM (and AVG: the scaling) */
                run_case(w, k, NVL_RED_ALLREDUCE, mk(k, op, exact_set(op), 1), (size_t)N * E + 1, P_ALIGNED);
                if (op == NVL_OP_SUM || (op == NVL_OP_AVG && IS_FLOAT))
                    for (size_t c : counts_all) if (kern_fits(w, k, NVL_RED_ALLREDUCE, c, nullptr)) run_case(w, k, NVL_RED_ALLREDUCE, mk(k, op, S_SUM, 2 + (int)c), c, P_ALIGNED);
                if (IS_FLOAT && (op == NVL_OP_SUM || op == NVL_OP_AVG || op == NVL_OP_PROD)) run_case(w, k, NVL_RED_ALLREDUCE, mk(k, op, S_SPECIAL, 3), (size_t)N * E + 3, P_ALIGNED);
                /* random full-mantissa values: same bits on every rank, error within the summation bound */
                if (IS_FLOAT && (op == NVL_OP_SUM || (op == NVL_OP_AVG && !(IS_HALF && kern_nvls(k)))) && !(IS_HALF && (k == K_RING || k == K_RHD)))
                    run_case(w, k, NVL_RED_ALLREDUCE, Case{S_RANDOM, op, 4, N, false, false}, kern_fits(w, k, NVL_RED_ALLREDUCE, 4097, nullptr) ? 4097 : (size_t)N * E + 1, P_ALIGNED);
            }
            if (IS_HALF && (k == K_RING || (k == K_RHD && pow2)))   /* ring / rhd on random f16 / bf16 inputs: the ranks agree (no bound, see above) */
                run_case(w, k, NVL_RED_ALLREDUCE, Case{S_RANDOM, NVL_OP_SUM, 5, N, true, false}, (size_t)N * E + 1, P_ALIGNED);
            /* placement: shifted by one element (the guarded element path) and in place */
            if (k == K_RHD && !pow2) continue;
            const size_t c = kern_fits(w, k, NVL_RED_ALLREDUCE, 4097, nullptr) ? 4097 : (size_t)N * E + 1;
            const int pop = IS_FLOAT && kern_ok(k, NVL_OP_AVG) ? NVL_OP_AVG : NVL_OP_SUM;
            if (kern_ok(k, NVL_OP_SUM) && k != K_SYMM && k != K_DIRECT) run_case(w, k, NVL_RED_ALLREDUCE, mk(k, NVL_OP_SUM, S_SUM, 6), c, P_SHIFTED);
            if (kern_ok(k, pop)) run_case(w, k, NVL_RED_ALLREDUCE, mk(k, pop, S_SUM, 7), c, P_INPLACE);
            printf("  ok allreduce %-12s N %d\n", kname[k], N);
        }
        for (int k : rs_k) {
            for (int op = 0; op < NVL_OP_LAST; op++) {
                if (!kern_ok(k, op)) continue;
                run_case(w, k, NVL_RED_REDUCE_SCATTER, mk(k, op, exact_set(op), 11), (size_t)N * (E + 1), P_ALIGNED);
                if (op != NVL_OP_SUM) continue;
                for (size_t blk : {(size_t)1, (size_t)E, (size_t)1000, multi / N})
                    if (kern_fits(w, k, NVL_RED_REDUCE_SCATTER, blk * N, nullptr)) run_case(w, k, NVL_RED_REDUCE_SCATTER, mk(k, op, S_SUM, 12), blk * N, P_ALIGNED);
                for (const std::vector<size_t> *v : {&rsv, &rsv_al}) {
                    size_t tot = 0; for (size_t x : *v) tot += x;
                    if (kern_fits(w, k, NVL_RED_REDUCE_SCATTER, tot, v)) run_case(w, k, NVL_RED_REDUCE_SCATTER, mk(k, op, S_SUM, 13), tot, P_ALIGNED, v);
                }
                const size_t bp = kern_fits(w, k, NVL_RED_REDUCE_SCATTER, (size_t)N * 999, nullptr) ? 999 : (size_t)E + 1;
                if (k != K_SYMM && k != K_DIRECT) run_case(w, k, NVL_RED_REDUCE_SCATTER, mk(k, op, S_SUM, 14), (size_t)N * bp, P_SHIFTED);
                if (k != K_SYMM) run_case(w, k, NVL_RED_REDUCE_SCATTER, mk(k, op, S_SUM, 15), (size_t)N * (bp + 1), P_INPLACE);
            }
            printf("  ok reduce_scatter %-12s N %d\n", kname[k], N);
        }
        for (int k : {K_STAGED, K_STAGED_NVLS, K_DIRECT}) {
            for (int op = 0; op < NVL_OP_LAST; op++) {
                if (!kern_ok(k, op)) continue;
                run_case(w, k, NVL_RED_REDUCE, mk(k, op, exact_set(op), 21), (size_t)N * E + 1, P_ALIGNED);
                if (op != NVL_OP_SUM) continue;
                run_case(w, k, NVL_RED_REDUCE, mk(k, op, S_SUM, 22), multi, P_ALIGNED);
                if (k != K_DIRECT) run_case(w, k, NVL_RED_REDUCE, mk(k, op, S_SUM, 23), 4097, P_SHIFTED);
            }
            printf("  ok reduce %-12s N %d\n", kname[k], N);
        }
    }
    printf("%d collectives checked, %d failures\n", g_cases, g_fail);
    if (g_fail) return 1;
    printf("NVL_EMU_OK\n");
    return 0;
}
