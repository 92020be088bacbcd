"""Worker of tests/test_nvl_complex.py: complex reductions (float32_complex / float64_complex) through the public UCC API on the
tl/nvl plugin built against the emulated CUDA runtime (tests/emu/build_hostemu_complex.sh), N ranks in this process, "device"
buffers from the emulated cudaMalloc, UCC_COLL_TRACE=info (the test reads which TL served every collective).  Results are compared
exactly with numpy: the inputs are Gaussian integers."""
import ctypes as C
import faulthandler
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EMU = os.path.join(ROOT, "build-emu", "complex", "lib")
os.environ["UCC_MODULE_DIR"] = os.path.join(EMU, "ucc")
faulthandler.dump_traceback_later(600, exit=True)
rt = C.CDLL(os.path.join(EMU, "libcudart_emu.so"), mode=C.RTLD_GLOBAL)
sys.path.insert(0, ROOT)
from ucc_b200 import capi as U  # noqa: E402
from ucc_b200.harness import UccJob, coll_args  # noqa: E402

CUDA = U.UCC_MEMORY_TYPE_CUDA
BASE = {"UCC_TL_NVL_MAX_BLOCKS": "2", "UCC_TL_NVL_NTHREADS": "64", "UCC_TL_NVL_TIMEOUT": "30s", "UCC_TL_NVL_SYMMETRIC_SIZE": "1Mb", "UCC_TLS": "nvl,shm,self",
        "UCC_COLL_TRACE": "info"}
ZC = {"UCC_TL_NVL_ZCOPY": "y", "UCC_TL_NVL_ZCOPY_THRESH": "0"}
NOZC = {"UCC_TL_NVL_ZCOPY": "n"}


class Dev:
    """numpy view of a buffer allocated with the emulated cudaMalloc (never freed)"""

    def __init__(self, n, dtype, fill=None):
        p = C.c_void_p()
        nbytes = max(n, 1) * np.dtype(dtype).itemsize
        assert rt.cudaMalloc(C.byref(p), C.c_size_t(nbytes)) == 0
        self.ptr = p.value
        self.a = np.frombuffer((C.c_char * nbytes).from_address(p.value), dtype=dtype)[:n]
        if fill is not None:
            self.a[:] = fill


def ca(coll, src, dst, dt, **kw):
    kw.setdefault("count_src", src.a.size if src is not None else 0)
    kw.setdefault("count_dst", dst.a.size if dst is not None else 0)
    return coll_args(coll, dt=dt, mem_type=CUDA, src_ptr=src.ptr if src is not None else None, dst_ptr=dst.ptr if dst is not None else None, **kw)


def run(team, args):
    q = team.coll(args)
    st = q.run()
    q.finalize()
    assert st == U.UCC_OK, U.status_str(st)
    rt.cudaDeviceSynchronize()


def gauss(n, seed, dtype):
    """Gaussian integers with parts in [-2, 2], never 0: sums and products of a few of them are exact"""
    g = np.random.default_rng(seed)
    re, im = g.integers(-2, 3, n), g.integers(-2, 3, n)
    re[(re == 0) & (im == 0)] = 1
    return (re + 1j * im).astype(dtype)


def complex_reduce(op, xs):
    a = np.stack([x.astype(np.complex128) for x in xs])
    if op == "prod":
        return a.prod(0).astype(xs[0].dtype)
    s = a.sum(0).astype(xs[0].dtype)
    if op == "avg":   # the sum times 1/N computed in the component precision
        c = s.real.dtype.type
        s = (s.view(s.real.dtype) * (c(1) / c(len(xs)))).view(s.dtype)
    return s


def complex_colls():
    """float32_complex / float64_complex SUM, AVG, PROD: allreduce, reduce_scatter(v), reduce under the default selection and every
    forced algorithm, in place, persistent, zero-copy and staged; a complex MAX is declined on a team of tl/nvl alone"""
    variants = [("default", {})]
    for alg in ("oneshot", "twoshot", "ring", "rhd"):
        colls = ["allreduce", "reduce_scatter", "reduce_scatterv"] + (["reduce"] if alg == "twoshot" else [])
        variants.append((alg, dict(NOZC, UCC_TL_NVL_TUNE="#".join(f"{c}:cuda:inf:@{alg}" for c in colls),
                                   UCC_TL_NVL_ALLREDUCE_ONESHOT_THRESH="1M" if alg == "oneshot" else "0")))
    variants.append(("twoshot-zcopy", dict(ZC, UCC_TL_NVL_TUNE="allreduce:cuda:inf:@twoshot#reduce_scatter:cuda:inf:@twoshot#reduce:cuda:inf:@twoshot",
                                           UCC_TL_NVL_ALLREDUCE_ONESHOT_THRESH="0")))
    for name, extra in variants:
        with UccJob(4, env=dict(BASE, **extra)) as j:
            for n in (3, 4):
                if name == "rhd" and n == 3:
                    continue
                team = j.create_team(range(n))
                for dt, npdt in (("float32_complex", np.complex64), ("float64_complex", np.complex128)):
                    for op in ("sum", "avg", "prod"):
                        for count in (1, 7, 1003, 40001):   # 40001 x 4 ranks: more than one 1 MB heap round
                            src = [Dev(count * n, npdt, fill=gauss(count * n, 10 * r + count, npdt)) for r in range(n)]
                            exp = complex_reduce(op, [s.a for s in src])
                            dst = [Dev(count * n, npdt, fill=0) for _ in range(n)]
                            run(team, [ca("allreduce", src[r], dst[r], dt=dt, op=op) for r in range(n)])
                            for r in range(n):
                                assert np.array_equal(dst[r].a, exp), (name, "allreduce", n, dt, op, count, r)
                            blk = [Dev(count, npdt, fill=0) for _ in range(n)]
                            run(team, [ca("reduce_scatter", src[r], blk[r], dt=dt, op=op) for r in range(n)])
                            for r in range(n):
                                assert np.array_equal(blk[r].a, exp[r * count:(r + 1) * count]), (name, "reduce_scatter", n, dt, op, count, r)
                            if name != "twoshot-zcopy":
                                cnts = [count + 3 * r for r in range(n)]
                                offs = np.concatenate([[0], np.cumsum(cnts)[:-1]])
                                sv = [Dev(sum(cnts), npdt, fill=gauss(sum(cnts), r + 5, npdt)) for r in range(n)]
                                ev = complex_reduce(op, [s.a for s in sv])
                                dv = [Dev(cnts[r], npdt, fill=0) for r in range(n)]
                                run(team, [ca("reduce_scatterv", sv[r], dv[r], dt=dt, op=op, dst_counts=cnts, dst_displs=offs) for r in range(n)])
                                for r in range(n):
                                    assert np.array_equal(dv[r].a, ev[offs[r]:offs[r] + cnts[r]]), (name, "reduce_scatterv", n, dt, op, count, r)
                            if name in ("default", "twoshot", "twoshot-zcopy"):
                                out = Dev(count * n, npdt, fill=0)
                                run(team, [ca("reduce", src[r], out if r == n - 1 else None, dt=dt, op=op, root=n - 1, count_dst=count * n if r == n - 1 else 0) for r in range(n)])
                                assert np.array_equal(out.a, exp), (name, "reduce", n, dt, op, count)
                    # in place: allreduce and reduce_scatter; persistent in-place allreduce posted three times
                    src = [Dev(5003, npdt, fill=gauss(5003, r + 70, npdt)) for r in range(n)]
                    exp = complex_reduce("sum", [s.a.copy() for s in src])
                    run(team, [ca("allreduce", None, src[r], dt=dt, inplace=True) for r in range(n)])
                    for r in range(n):
                        assert np.array_equal(src[r].a, exp), (name, "allreduce inplace", n, dt, r)
                    blk = 1001
                    src = [Dev(blk * n, npdt, fill=gauss(blk * n, r + 80, npdt)) for r in range(n)]
                    exp = complex_reduce("prod", [s.a.copy() for s in src])
                    run(team, [ca("reduce_scatter", None, src[r], dt=dt, op="prod", inplace=True) for r in range(n)])
                    for r in range(n):
                        assert np.array_equal(src[r].a[r * blk:(r + 1) * blk], exp[r * blk:(r + 1) * blk]), (name, "reduce_scatter inplace", n, dt, r)
                    buf = [Dev(2049, npdt, fill=0) for _ in range(n)]
                    q = team.coll([ca("allreduce", None, buf[r], dt=dt, op="avg", inplace=True, persistent=True) for r in range(n)])
                    for it in range(3):
                        vals = [gauss(2049, 10 * it + r, npdt) for r in range(n)]
                        for r in range(n):
                            buf[r].a[:] = vals[r]
                        assert q.run() == U.UCC_OK
                        rt.cudaDeviceSynchronize()
                        for r in range(n):
                            assert np.array_equal(buf[r].a, complex_reduce("avg", vals)), (name, "persistent", n, dt, it, r)
                    q.finalize()
                team.destroy()
        print(f"  complex {name} ok", flush=True)
    with UccJob(3, env=dict(BASE, UCC_TL_SHM_TUNE="allreduce:0")) as j:   # allreduce: tl/nvl alone
        team = j.create_team(range(3))
        x = [Dev(16, np.complex64, fill=gauss(16, r, np.complex64)) for r in range(3)]
        try:
            team.coll([ca("allreduce", x[r], x[r], dt="float32_complex", op="max") for r in range(3)]).finalize()
            raise AssertionError("complex MAX was accepted")
        except U.UccError as e:
            assert e.status == U.UCC_ERR_NOT_SUPPORTED, e
        team.destroy()
    print("  complex MAX declined ok", flush=True)


if __name__ == "__main__":
    complex_colls()
    print("HOSTEMU_WORKER_OK", flush=True)
