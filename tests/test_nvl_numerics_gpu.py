"""Numerics of the tl/nvl reduction kernels on a real GPU, through the public API: every real datatype x every operator tl/nvl
accepts, under every forced algorithm and the default selection.  N emulated ranks share cuda:0 as in tests/test_nvl_gpu.py.

Inputs and oracles are those of the host emulation (tests/emu/nvl_emu_numerics.cpp), written here in numpy:
  exact-sum   signed k * 2^e, |k| <= 127, e in [-4, 4], and +-0: partial sums of <= 8 terms are exact in float, so SUM is the
              exact sum rounded once to the storage type and AVG is acc(sum) * acc(1/N) rounded once, bit for bit
  exact-prod  {+-0.5, +-0.75, +-1, +-1.5, +-2}: products of <= 8 terms are exact in float
  random      k * 2^-m (m = significand bits): every rank stores the same bits, |got - sum| <= (N-1) u_acc sum|x| + ulp(got)/2
  integers    random full-width bits; logical operators get zero and non-zero values whose low byte is zero
Ring and rhd keep partial sums in the storage type, so f16 / bf16 get inputs exact in the storage type there.  Unsigned types
travel through numpy byte buffers (torch supports uint16 / uint32 / uint64 only partly on CUDA).  Every destination has one
guard element on each side."""
import os
import re
import subprocess
import sys

import numpy as np
import pytest

os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from ucc_b200 import capi as U  # noqa: E402
from ucc_b200.harness import UccJob, coll_args  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CUDA = U.UCC_MEMORY_TYPE_CUDA
FLOATS = ["float32", "float64", "float16", "bfloat16"]
INTS = ["int8", "int16", "int32", "int64", "uint8", "uint16", "uint32", "uint64"]
NP = {"float32": np.float32, "float64": np.float64, "float16": np.float16, "bfloat16": np.uint16, "int8": np.int8, "int16": np.int16,
      "int32": np.int32, "int64": np.int64, "uint8": np.uint8, "uint16": np.uint16, "uint32": np.uint32, "uint64": np.uint64}
MBITS = {"float32": 24, "float64": 53, "float16": 11, "bfloat16": 8}
FOPS = ["sum", "prod", "max", "min", "avg"]
IOPS = ["sum", "prod", "max", "min", "land", "lor", "lxor", "band", "bor", "bxor", "avg"]
ENV = {"UCC_TL_NVL_MAX_BLOCKS": "4", "UCC_TL_NVL_TIMEOUT": "5s", "UCC_TL_NVL_SYMMETRIC_SIZE": "8Mb", "UCC_TL_NVL_P2P_TIMEOUT": "20s"}
ALGS = ["default", "oneshot", "twoshot", "twoshot-zcopy", "ring", "rhd"]
TEAM_SIZES = (2, 3, 5, 8)


def alg_env(alg):
    if alg == "default":
        return dict(ENV, UCC_TL_NVL_ZCOPY="n")
    name = alg.split("-")[0]
    colls = ["allreduce", "reduce_scatter", "reduce_scatterv"] + (["reduce"] if name == "twoshot" else [])
    env = dict(ENV, UCC_TL_NVL_TUNE="#".join(f"{c}:cuda:inf:@{name}" for c in colls),
               UCC_TL_NVL_ALLREDUCE_ONESHOT_THRESH="1M" if name == "oneshot" else "0")
    env.update({"UCC_TL_NVL_ZCOPY": "y", "UCC_TL_NVL_ZCOPY_THRESH": "0"} if alg.endswith("zcopy") else {"UCC_TL_NVL_ZCOPY": "n"})
    return env


# ---------------------------------------------------------------- storage conversions
def bf16_round(x32):
    """float32 -> bfloat16 bits, round to nearest even (NaN kept quiet)"""
    b = np.asarray(x32, np.float32).view(np.uint32).astype(np.uint64)
    r = ((b + 0x7FFF + ((b >> 16) & 1)) >> 16).astype(np.uint16)
    return np.where(np.isnan(x32), np.uint16(0x7FC0), r)


def to_store(dt, v):
    """exactly-representable-in-float32 (or float64) values -> storage, one rounding"""
    if dt == "float64":
        return np.asarray(v, np.float64)
    f = np.asarray(v, np.float32)
    return bf16_round(f) if dt == "bfloat16" else f.astype(NP[dt])


def to_f64(dt, a):
    if dt == "bfloat16":
        return (a.astype(np.uint32) << 16).view(np.float32).astype(np.float64)
    return a.astype(np.float64)


def ulp(dt, a):
    if dt == "bfloat16":
        m = a & np.uint16(0x7FFF)
        return to_f64(dt, m + np.uint16(1)) - to_f64(dt, m)
    return np.spacing(np.abs(a)).astype(np.float64)


# ---------------------------------------------------------------- inputs
def f_inputs(kind, dt, n, count, seed, storage_exact):
    g = np.random.default_rng(seed)
    if kind == "sum":
        if storage_exact:
            v = g.integers(-31, 32, (n, count)).astype(np.float64)
        else:
            v = np.ldexp(g.integers(-127, 128, (n, count)).astype(np.float64), g.integers(-4, 5, (n, count)))
        z = g.integers(0, 16, (n, count)) == 0
        v[z] = np.where(g.integers(0, 2, (n, count))[z] == 1, -0.0, 0.0)
        v[:, 5::97] = -0.0                                                  # -0 on every rank: the sum is -0
        return v
    if kind == "prod":
        pool = np.array([0.5, 1.0, 2.0] if storage_exact else [0.5, 0.75, 1.0, 1.5, 2.0])
        return pool[g.integers(0, len(pool), (n, count))] * np.where(g.integers(0, 2, (n, count)) == 1, -1.0, 1.0)
    m = MBITS[dt]                                                           # random: k * 2^-m, |k| < 2^m
    return g.integers(-(1 << m), 1 << m, (n, count), dtype=np.int64)


def i_inputs(dt, op, n, count, seed):
    g = np.random.default_rng(seed)
    if op in ("land", "lor", "lxor"):
        pool = np.array([0, 0, 0, 1, 0x80, 0x100, 0x8000, 0x10000, 0x80000000, 1 << 32, 1 << 63, (1 << 64) - 1], dtype=np.uint64)
        u = pool[g.integers(0, len(pool), (n, count))]
    else:
        u = g.integers(0, np.iinfo(np.uint64).max, (n, count), dtype=np.uint64, endpoint=True)
    return u.astype(np.dtype(NP[dt]).newbyteorder("=").str.replace("i", "u")).view(NP[dt])


# ---------------------------------------------------------------- oracles
def f_expect(dt, op, v, nvls_avg_twice=False):
    n = v.shape[0]
    if op in ("sum", "avg"):
        s = v[0].copy()
        for p in range(1, n):
            s = s + v[p]                                                    # exact in float64
        if op == "sum":
            return to_store(dt, s)
        if dt == "float64":
            return s * (1.0 / n)
        acc = np.float32(s) if not nvls_avg_twice else to_f64(dt, to_store(dt, s)).astype(np.float32)
        return to_store(dt, acc * (np.float32(1) / np.float32(n)))
    if op == "prod":
        return to_store(dt, np.prod(v, axis=0))
    return to_store(dt, v.max(0) if op == "max" else v.min(0))


def i_expect(dt, op, x):
    n, t = x.shape[0], NP[dt]
    u = x.view(np.dtype(t).str.replace("i", "u"))
    if op in ("sum", "avg", "prod"):
        acc = u[0].astype(np.uint64)
        for p in range(1, n):
            acc = acc + u[p].astype(np.uint64) if op != "prod" else acc * u[p].astype(np.uint64)
        w = acc.astype(u.dtype).view(t)                                     # wrapped in the storage type
        if op != "avg":
            return w
        if np.issubdtype(t, np.signedinteger):
            s = w.astype(np.int64)
            q = s // n
            q = q + ((s % n != 0) & (s < 0))                                # truncating division
            return q.astype(t)
        return (w // t(n)).astype(t)
    nz = x != 0
    return {"max": lambda: x.max(0), "min": lambda: x.min(0), "land": lambda: nz.all(0).astype(t), "lor": lambda: nz.any(0).astype(t),
            "lxor": lambda: (nz.sum(0) & 1).astype(t), "band": lambda: np.bitwise_and.reduce(x, 0), "bor": lambda: np.bitwise_or.reduce(x, 0),
            "bxor": lambda: np.bitwise_xor.reduce(x, 0)}[op]()


# ---------------------------------------------------------------- device buffers
GUARD = 0xA5


class DevBuf:
    """bytes on cuda:0; the kernel sees element 0 at byte 16 (+ one element when shifted), guards on both sides"""

    def __init__(self, dt, count, shifted=False):
        self.es = np.dtype(NP[dt]).itemsize
        self.off = 16 + (self.es if shifted else 0)
        self.count = count
        self.t = torch.full((self.off + (count + 1) * self.es + 16,), GUARD, dtype=torch.uint8, device="cuda")
        self.ptr = self.t.data_ptr() + self.off
        self.np_t = NP[dt]

    def put(self, a):
        self.t[self.off:self.off + a.nbytes].copy_(torch.from_numpy(np.ascontiguousarray(a).view(np.uint8)))

    def get(self):
        b = self.t.cpu().numpy()
        guards_ok = bool((b[self.off - self.es:self.off] == GUARD).all() and (b[self.off + self.count * self.es:self.off + (self.count + 1) * self.es] == GUARD).all())
        return b[self.off:self.off + self.count * self.es].view(self.np_t), guards_ok


def run(team, args):
    req = team.coll(args)
    st = req.run()
    req.finalize()
    torch.cuda.synchronize()
    assert st == U.UCC_OK, U.status_str(st)


def ca(coll, src, dst, dt, **kw):
    return coll_args(coll, dt=dt, mem_type=CUDA, src_ptr=src.ptr if src is not None else None, dst_ptr=dst.ptr if dst is not None else None,
                     count_src=src.count if src is not None else 0, count_dst=dst.count if dst is not None else 0, **kw)


def compare(fails, what, dt, got, exp, by_value=False):
    if dt in INTS:
        ok = np.array_equal(got, exp)
    elif by_value:
        ok = np.array_equal(to_f64(dt, got), to_f64(dt, exp))
    else:
        g, e = to_f64(dt, got), to_f64(dt, exp)
        ok = np.array_equal(np.asarray(got).view(np.uint8), np.asarray(exp).view(np.uint8)) or (np.isnan(e) == np.isnan(g)).all() and \
            np.array_equal(np.asarray(got)[~np.isnan(e)].view(np.uint8), np.asarray(exp)[~np.isnan(e)].view(np.uint8))
    if not ok:
        bad = np.nonzero(to_f64(dt, got) != to_f64(dt, exp) if dt not in INTS else got != exp)[0]
        i = int(bad[0]) if len(bad) else -1
        fails.append(f"{what}: elem {i} got {got[i] if i >= 0 else '?'} expected {exp[i] if i >= 0 else '?'} ({len(bad)} differ)")


# ---------------------------------------------------------------- fixtures
@pytest.fixture(scope="module", params=ALGS)
def alg_job(request):
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    torch.cuda.set_device(0)
    job = UccJob(8, env=alg_env(request.param))
    teams = {n: job.create_team(range(n)) for n in TEAM_SIZES}
    yield request.param, teams
    job.cleanup()


def ops_of(dt):
    return FOPS if dt in FLOATS else IOPS


def inputs(dt, op, n, count, seed, storage_exact):
    """(values in storage type per rank, oracle input) for the exact sets / integers"""
    if dt in INTS:
        x = i_inputs(dt, op, n, count, seed)
        return x, x
    v = f_inputs("prod" if op == "prod" else "sum", dt, n, count, seed, storage_exact)
    return np.stack([to_store(dt, v[r]) for r in range(n)]), v


def expect(dt, op, v):
    return i_expect(dt, op, v) if dt in INTS else f_expect(dt, op, v)


@pytest.mark.parametrize("n", TEAM_SIZES)
def test_allreduce_every_dtype_op(alg_job, n):
    """allreduce, every (datatype, operator), exact oracle, all ranks equal, guards intact; shifted by one element and in place"""
    alg, teams = alg_job
    team, fails = teams[n], []
    if alg == "rhd" and n & (n - 1):
        pytest.skip("recursive halving / doubling pairs ranks by xor: power-of-two teams")
    for dt in FLOATS + INTS:
        E = 16 // np.dtype(NP[dt]).itemsize
        se = dt in ("float16", "bfloat16") and alg in ("ring", "rhd")
        for op in ops_of(dt):
            counts = (1, E + 1, n * E - 1, 4097) if op in ("sum", "avg") else (n * E + 1,)
            for count in counts:
                for place in ("aligned", "shifted", "inplace") if (op == "sum" and count == 4097) else ("aligned",):
                    x, v = inputs(dt, op, n, count, 1000 * n + count, se)
                    src = [DevBuf(dt, count, place == "shifted") for _ in range(n)]
                    dst = src if place == "inplace" else [DevBuf(dt, count, place == "shifted") for _ in range(n)]
                    for r in range(n):
                        src[r].put(x[r])
                    torch.cuda.synchronize()
                    run(team, [ca("allreduce", None if place == "inplace" else src[r], dst[r], dt, op=op, inplace=place == "inplace") for r in range(n)])
                    exp = expect(dt, op, v)
                    outs = [dst[r].get() for r in range(n)]
                    what = f"{alg} allreduce {dt} {op} N {n} count {count} {place}"
                    compare(fails, what, dt, outs[0][0], exp, by_value=op in ("max", "min"))
                    for r in range(n):
                        if outs[r][0].tobytes() != outs[0][0].tobytes():
                            fails.append(f"{what}: rank {r} differs from rank 0")
                        if place != "inplace" and not outs[r][1]:
                            fails.append(f"{what}: rank {r} guard overwritten")
    assert not fails, f"{len(fails)} failures:\n" + "\n".join(fails[:30])


@pytest.mark.parametrize("n", TEAM_SIZES)
def test_allreduce_random_ranks_agree(alg_job, n):
    """full-mantissa inputs: every rank stores the same bits; SUM / AVG within the recursive-summation bound (see the module doc)"""
    alg, teams = alg_job
    team, fails = teams[n], []
    if alg == "rhd" and n & (n - 1):
        pytest.skip("power-of-two teams only")
    for dt in FLOATS:
        m, u = MBITS[dt], (2.0 ** -53 if dt == "float64" else 2.0 ** -24)
        for op in ("sum", "avg"):
            for count in (7, 4097, 100003):
                k = f_inputs("random", dt, n, count, 7 * n + count, False)
                x = np.stack([to_store(dt, np.ldexp(k[r].astype(np.float64), -m)) for r in range(n)])
                src = [DevBuf(dt, count) for _ in range(n)]
                dst = [DevBuf(dt, count) for _ in range(n)]
                for r in range(n):
                    src[r].put(x[r])
                torch.cuda.synchronize()
                run(team, [ca("allreduce", src[r], dst[r], dt, op=op) for r in range(n)])
                outs = [dst[r].get()[0] for r in range(n)]
                what = f"{alg} allreduce {dt} {op} N {n} count {count} random"
                for r in range(1, n):
                    if outs[r].tobytes() != outs[0].tobytes():
                        fails.append(f"{what}: rank {r} differs from rank 0 in {int((outs[r].view(np.uint8) != outs[0].view(np.uint8)).sum())} bytes")
                if dt in ("float16", "bfloat16") and alg in ("ring", "rhd"):
                    continue                                                # partial sums rounded to the storage type: agreement only
                S = np.ldexp(k.sum(0).astype(np.longdouble), -m)             # exact (integer sum of the k)
                sabs = np.ldexp(np.abs(k).sum(0).astype(np.longdouble), -m)
                exact = S / n if op == "avg" else S
                if op == "sum":
                    bound = (n - 1) * u * sabs
                else:   # fl(fl(S^ * fl(1/N))): (N-1)/N u sum|x| from the sum, 2u more unless 1/N and the product are exact
                    bound = u * sabs * ((n - 1) + (0 if (n & (n - 1)) == 0 else 2)) / n * (1 + 4 * u)
                bound = bound + ulp(dt, outs[0]) / 2
                err = np.abs(to_f64(dt, outs[0]).astype(np.longdouble) - exact)
                if (err > bound).any():
                    i = int(np.argmax(err > bound))
                    fails.append(f"{what}: elem {i} error {float(err[i]):.3g} > bound {float(bound[i]):.3g}")
    assert not fails, f"{len(fails)} failures:\n" + "\n".join(fails[:30])


@pytest.mark.parametrize("n", TEAM_SIZES)
def test_reduce_scatter_and_reduce_every_dtype_op(alg_job, n):
    """reduce_scatter (equal blocks), reduce_scatterv (unequal blocks, one empty) and reduce to root N-1 (two-shot algorithms)"""
    alg, teams = alg_job
    team, fails = teams[n], []
    if alg == "rhd" and n & (n - 1):
        pytest.skip("power-of-two teams only")
    for dt in FLOATS + INTS:
        E = 16 // np.dtype(NP[dt]).itemsize
        se = dt in ("float16", "bfloat16") and alg in ("ring", "rhd")
        for op in ops_of(dt):
            # reduce_scatter, equal blocks
            for blk in ((1, E + 1, 1000) if op == "sum" else (E + 1,)):
                x, v = inputs(dt, op, n, blk * n, 31 * n + blk, se)
                exp = expect(dt, op, v)
                src = [DevBuf(dt, blk * n) for _ in range(n)]
                dst = [DevBuf(dt, blk) for _ in range(n)]
                for r in range(n):
                    src[r].put(x[r])
                torch.cuda.synchronize()
                run(team, [ca("reduce_scatter", src[r], dst[r], dt, op=op) for r in range(n)])
                for r in range(n):
                    got, gok = dst[r].get()
                    what = f"{alg} reduce_scatter {dt} {op} N {n} blk {blk} rank {r}"
                    compare(fails, what, dt, got, exp[r * blk:(r + 1) * blk], by_value=op in ("max", "min"))
                    if not gok:
                        fails.append(f"{what}: guard overwritten")
            if op not in ("sum", "max"):
                continue
            # reduce_scatterv: unequal blocks, block 1 empty
            cnts = [0 if p == 1 else 3 + 37 * p for p in range(n)]
            offs = np.concatenate([[0], np.cumsum(cnts)[:-1]]).astype(int)
            x, v = inputs(dt, op, n, sum(cnts), 77 * n, se)
            exp = expect(dt, op, v)
            src = [DevBuf(dt, sum(cnts)) for _ in range(n)]
            dst = [DevBuf(dt, cnts[r]) for r in range(n)]
            for r in range(n):
                src[r].put(x[r])
            torch.cuda.synchronize()
            run(team, [ca("reduce_scatterv", src[r], dst[r], dt, op=op, dst_counts=cnts, dst_displs=offs) for r in range(n)])
            for r in range(n):
                got, gok = dst[r].get()
                what = f"{alg} reduce_scatterv {dt} {op} N {n} rank {r}"
                compare(fails, what, dt, got, exp[offs[r]:offs[r] + cnts[r]], by_value=op == "max")
                if not gok:
                    fails.append(f"{what}: guard overwritten")
            # reduce, root != 0
            if alg not in ("twoshot", "twoshot-zcopy", "default"):
                continue
            root, count = n - 1, 4097
            x, v = inputs(dt, op, n, count, 5 * n, se)
            src = [DevBuf(dt, count) for _ in range(n)]
            res = DevBuf(dt, count)
            for r in range(n):
                src[r].put(x[r])
            torch.cuda.synchronize()
            run(team, [coll_args("reduce", dt=dt, mem_type=CUDA, src_ptr=src[r].ptr, dst_ptr=res.ptr if r == root else None, count_src=count,
                                 count_dst=count if r == root else 0, op=op, root=root) for r in range(n)])
            got, gok = res.get()
            compare(fails, f"{alg} reduce {dt} {op} N {n}", dt, got, expect(dt, op, v), by_value=op == "max")
            if not gok:
                fails.append(f"{alg} reduce {dt} {op} N {n}: guard overwritten")
    assert not fails, f"{len(fails)} failures:\n" + "\n".join(fails[:30])


TRACE_SCRIPT = r"""
import sys, numpy as np, torch
sys.path.insert(0, sys.argv[1]); sys.path.insert(0, sys.argv[1] + "/tests")
import test_nvl_numerics_gpu as T
from ucc_b200.harness import UccJob
torch.cuda.set_device(0)
for alg in T.ALGS:
    with UccJob(4, env=dict(T.alg_env(alg), UCC_COLL_TRACE="info")) as job:
        team = job.create_team()
        for dt in ("float64", "bfloat16", "uint16", "uint64", "int8"):
            for op in ("sum", "avg", "max"):
                x, v = T.inputs(dt, op, 4, 4097, 1, False)
                src = [T.DevBuf(dt, 4097) for _ in range(4)]
                dst = [T.DevBuf(dt, 4097) for _ in range(4)]
                for r in range(4):
                    src[r].put(x[r])
                torch.cuda.synchronize()
                T.run(team, [T.ca("allreduce", src[r], dst[r], dt, op=op) for r in range(4)])
        team.destroy()
print("NUMERICS_TRACE_OK", flush=True)
"""


def test_trace_shows_tl_nvl():
    """the collectives above run on tl/nvl: a case that fell back to another transport would pass the oracle without testing a kernel"""
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    env = dict(os.environ, PYTHONPATH=ROOT)
    for k in ("UCC_TL_NVL_TUNE", "UCC_TLS"):
        env.pop(k, None)
    out = subprocess.run([sys.executable, "-c", TRACE_SCRIPT, ROOT], env=env, capture_output=True, text=True, timeout=600)
    log = out.stdout + out.stderr
    assert out.returncode == 0 and "NUMERICS_TRACE_OK" in out.stdout, log[-4000:]
    lines = [ln for ln in log.splitlines() if "coll_init:" in ln and re.search(r"allreduce", ln, re.I)]
    assert len(lines) >= len(ALGS) * 15, log[-3000:]
    bad = [ln for ln in lines if "{TL_NVL}" not in ln]
    assert not bad, bad[:5]
