// Host emulation of the tl/nvl reduction kernels on complex elements (nvl_c64 / nvl_c128): every reduction kernel x {SUM, PROD,
// AVG} x N in {2, 3, 4, 8}, compiled as plain C++ (NVL_HOST_EMU) like tests/emu/nvl_emu.cpp.  Inputs are Gaussian integers with
// parts in [-2, 2]: sums and products of up to 8 of them are exact in f32, so results are compared exactly.  Random-valued inputs
// are compared with a tolerance, and c64 SUM is compared bitwise with f32 SUM of the same bytes.
#include <complex>
#include "nvl_emu_world.h"

static const char *opname(int op) { return op == NVL_OP_SUM ? "sum" : op == NVL_OP_PROD ? "prod" : "avg"; }

template <typename C> struct Cx { typedef decltype(C::re) R; };
static uint64_t lcg(uint64_t &s) { s = s * 6364136223846793005ull + 1442695040888963407ull; return s >> 33; }

/* input element i of rank r: a Gaussian integer (exact) or a random value in [-1, 1) */
template <typename C> static C input(int r, size_t i, int seed, bool exact)
{
    typedef typename Cx<C>::R R;
    if (exact) {
        int re = (int)((i * 7 + (size_t)r * 13 + (size_t)seed) % 5) - 2, im = (int)((i * 3 + (size_t)r * 11 + (size_t)seed * 5) % 5) - 2;
        if (!re && !im) re = 1;
        return C{(R)re, (R)im};
    }
    uint64_t s = (i * 2654435761ull) ^ ((uint64_t)r << 40) ^ ((uint64_t)seed << 52); lcg(s); lcg(s);
    return C{(R)((double)lcg(s) / 2147483648.0 * 2 - 1), (R)((double)lcg(s) / 2147483648.0 * 2 - 1)};
}

/* oracle in complex128; AVG scales the sum by 1/N computed in the component precision */
template <typename C> static std::complex<double> expect(int N, int op, size_t i, int seed, bool exact)
{
    typedef typename Cx<C>::R R;
    std::complex<double> e;
    for (int p = 0; p < N; p++) {
        const C x = input<C>(p, i, seed, exact);
        const std::complex<double> v((double)x.re, (double)x.im);
        if (p == 0) e = v;
        else if (op == NVL_OP_PROD) e = std::complex<double>(e.real() * v.real() - e.imag() * v.imag(), e.real() * v.imag() + e.imag() * v.real());
        else e += v;
    }
    if (op == NVL_OP_AVG) { const R s = (R)1 / (R)N; e = std::complex<double>((double)((R)e.real() * s), (double)((R)e.imag() * s)); }
    return e;
}

template <typename C> static void compare(const char *what, const C *got, size_t n, size_t first, int N, int op, int seed, bool exact, int r)
{
    const double tol = sizeof(C) == 8 ? 1e-5 : 1e-12;
    for (size_t i = 0; i < n; i++) {
        const std::complex<double> e = expect<C>(N, op, first + i, seed, exact);
        const double dr = std::fabs((double)got[i].re - e.real()), di = std::fabs((double)got[i].im - e.imag());
        const bool ok = exact ? (dr == 0 && di == 0) : (dr <= tol * (1 + std::fabs(e.real())) && di <= tol * (1 + std::fabs(e.imag())));
        if (!ok) { printf("EMU FAIL %s: rank %d elem %zu got (%.9g, %.9g) expected (%.9g, %.9g)\n", what, r, first + i, (double)got[i].re, (double)got[i].im, e.real(), e.imag()); exit(1); }
    }
}

/* run kernel k for one (kind, op, count) and check it; `mis` shifts the source by one element (8-byte aligned c64 buffers) */
template <typename C> static void check_one(World &w, int k, int kind, int op, size_t count, bool exact, size_t mis = 0)
{
    const int N = w.N, seed = (int)count % 17 + op, root = N - 1;
    const bool symm = k == K_SYMM;
    std::vector<std::vector<C>> sb(N, std::vector<C>(count + 8)), db(N, std::vector<C>(count + 8));
    std::vector<C *> src(N), dst(N);
    const C guard{(typename Cx<C>::R)77, (typename Cx<C>::R)-77};
    for (int r = 0; r < N; r++) {
        src[r] = symm ? (C *)w.user(r) : sb[r].data() + 2 + mis;
        dst[r] = symm ? src[r] : db[r].data() + 2;
        if (symm) CHECK(count * sizeof(C) + 64 <= w.user_size);
        for (size_t i = 0; i < count; i++) src[r][i] = input<C>(r, i, seed, exact);
        if (!symm) { db[r][1] = guard; db[r][2 + count] = guard; }
    }
    if (kind == NVL_RED_REDUCE_SCATTER) for (int r = 0; r < N; r++) dst[r] = db[r].data() + 2, db[r][2 + count / N] = guard;
    if (kind == NVL_RED_REDUCE) for (int r = 0; r < N; r++) if (r != root) dst[r] = nullptr;
    launch<C>(w, k, kind, op, count, src, dst, root);
    char what[128]; snprintf(what, sizeof(what), "%s %s %s N %d count %zu%s%s", kname[k], sizeof(C) == 8 ? "c64" : "c128", opname(op), N, count, exact ? "" : " random", mis ? " unaligned" : "");
    for (int r = 0; r < N; r++) {
        if (kind == NVL_RED_ALLREDUCE) compare<C>(what, dst[r], count, 0, N, op, seed, exact, r);
        else if (kind == NVL_RED_REDUCE_SCATTER) { const size_t b = count / N; compare<C>(what, dst[r], b, (size_t)r * b, N, op, seed, exact, r); CHECK(!memcmp(&db[r][2 + b], &guard, sizeof(C))); }
        else if (r == root) compare<C>(what, dst[r], count, 0, N, op, seed, exact, r);
        if (!symm && kind != NVL_RED_REDUCE_SCATTER && dst[r]) { CHECK(!memcmp(&db[r][1], &guard, sizeof(C))); CHECK(!memcmp(&db[r][2 + count], &guard, sizeof(C))); }
    }
}

/* c64 SUM through kernel k == f32 SUM of the same bytes, bit for bit (random values: any difference in order would show) */
static void check_c64_is_f32(World &w, int k, size_t count)
{
    const int N = w.N;
    std::vector<std::vector<nvl_c64>> s(N, std::vector<nvl_c64>(count + 4)), dc(N, std::vector<nvl_c64>(count + 4)), df(N, std::vector<nvl_c64>(count + 4));
    std::vector<nvl_c64 *> sc(N), oc(N); std::vector<float *> sf(N), of(N);
    for (int r = 0; r < N; r++) {
        for (size_t i = 0; i < count; i++) s[r][2 + i] = input<nvl_c64>(r, i, 3, false);
        if (k == K_SYMM) { sc[r] = (nvl_c64 *)w.user(r); memcpy(sc[r], s[r].data() + 2, count * 8); } else sc[r] = s[r].data() + 2;
        oc[r] = k == K_SYMM ? sc[r] : dc[r].data() + 2; sf[r] = (float *)sc[r]; of[r] = k == K_SYMM ? sf[r] : (float *)(df[r].data() + 2);
    }
    launch<nvl_c64>(w, k, NVL_RED_ALLREDUCE, NVL_OP_SUM, count, sc, oc);
    std::vector<std::vector<nvl_c64>> res(N);
    for (int r = 0; r < N; r++) res[r].assign(oc[r], oc[r] + count);
    if (k == K_SYMM) for (int r = 0; r < N; r++) memcpy(sc[r], s[r].data() + 2, count * 8);
    launch<float>(w, k, NVL_RED_ALLREDUCE, NVL_OP_SUM, 2 * count, sf, of);
    for (int r = 0; r < N; r++) if (memcmp(res[r].data(), of[r], count * 8)) { printf("EMU FAIL %s: c64 SUM differs from f32 SUM, N %d count %zu rank %d\n", kname[k], N, count, r); exit(1); }
}

int main(int argc, char **argv)
{
    const std::string what = argc > 1 ? argv[1] : "all";
    for (int N : {2, 3, 4, 8}) {
        if (what != "all" && what != "n" + std::to_string(N)) continue;
        // 48 KB data region: a few thousand elements already need several staging rounds
        World w(N, 48 * 1024, 1 << 20);
        for (int k = 0; k < K_LAST; k++) {
            if (k == K_RHD && (N & (N - 1))) continue;
            const bool c64_only = k == K_STAGED_NVLS || k == K_PIPE || k == K_SYMM;    // in-switch reduction: c64 SUM / AVG only
            const bool one_round = k == K_RING || k == K_RHD;                          // single round: the vector has to fit the heap
            const int kind = k == K_ONESHOT_RS ? NVL_RED_REDUCE_SCATTER : NVL_RED_ALLREDUCE;
            const std::vector<size_t> counts = kind == NVL_RED_REDUCE_SCATTER ? std::vector<size_t>{(size_t)N, 333 * (size_t)N}
                                             : one_round ? std::vector<size_t>{1, 3, 999} : std::vector<size_t>{1, 3, 999, 7001};
            for (int op : {NVL_OP_SUM, NVL_OP_PROD, NVL_OP_AVG}) {
                if (c64_only && op == NVL_OP_PROD) continue;
                for (size_t c : counts) check_one<nvl_c64>(w, k, kind, op, c, true);
                if (!c64_only) for (size_t c : counts) check_one<nvl_c128>(w, k, kind, op, c, true);
                check_one<nvl_c64>(w, k, kind, op, counts.back(), false);
                if (!c64_only) check_one<nvl_c128>(w, k, kind, op, counts.back(), false);
                if (k != K_SYMM && k != K_DIRECT) check_one<nvl_c64>(w, k, kind, op, counts.back() - (kind == NVL_RED_REDUCE_SCATTER ? 0 : 2), true, 1);
            }
            if (kind == NVL_RED_ALLREDUCE) check_c64_is_f32(w, k, one_round ? 999 : 7001);
            printf("  ok %-12s N %d\n", kname[k], N);
        }
        // the staged and step kernels also produce reduce_scatter and reduce
        for (int op : {NVL_OP_SUM, NVL_OP_PROD, NVL_OP_AVG}) {
            check_one<nvl_c64>(w, K_STAGED, NVL_RED_REDUCE_SCATTER, op, 1001 * (size_t)N, true, 1);
            check_one<nvl_c128>(w, K_STAGED, NVL_RED_REDUCE_SCATTER, op, 1001 * (size_t)N, true);
            check_one<nvl_c64>(w, K_RING, NVL_RED_REDUCE_SCATTER, op, 99 * (size_t)N, true);
            check_one<nvl_c128>(w, K_STAGED, NVL_RED_REDUCE, op, 3001, true);
            check_one<nvl_c64>(w, K_STAGED, NVL_RED_REDUCE, op, 3001, false, 1);
        }
        printf("  ok %-12s N %d\n", "rs / reduce", N);
    }
    printf("NVL_EMU_OK\n");
    return 0;
}
