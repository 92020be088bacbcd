"""Worker of tests/test_nvl_complex_gpu.py: complex reductions (float32_complex / float64_complex) on CUDA buffers.

    complex_worker.py trace   one process, 4 ranks emulated on cuda:0, UCC_COLL_TRACE=info: every complex allreduce,
                              reduce_scatter(v) and reduce under the default selection and under every forced algorithm
    complex_worker.py nvl     under torchrun, one process per GPU: forced @nvls / @nvls_pipe, cross-process zero-copy (IPC
                              mappings), in-place allreduce on symm_empty() tensors
    complex_worker.py nccl    under torchrun with UCC_TLS=nccl,self: SUM / AVG correct, PROD declined
    complex_worker.py torch   under torchrun: the ucc_b200 torch.distributed backend, reduce_scatter_tensor and reduce on complex64

Inputs are Gaussian integers with parts in [-2, 2], so sums and products of up to 8 of them are exact and results are compared
exactly; AVG is the sum times 1/N computed in the component precision, as the kernels compute it."""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from ucc_b200 import capi as U  # noqa: E402

DTS = {"float32_complex": torch.complex64, "float64_complex": torch.complex128}
FAIL = []


def gauss(n, seed, dtype):
    g = np.random.default_rng(seed)
    re, im = g.integers(-2, 3, n), g.integers(-2, 3, n)
    re[(re == 0) & (im == 0)] = 1
    return torch.complex(torch.from_numpy(re).double(), torch.from_numpy(im).double()).to(dtype)


def expected(op, xs):
    """the reduction of the CPU tensors xs, computed in complex128 and rounded the way the kernels round"""
    dtype, n = xs[0].dtype, len(xs)
    a = torch.stack([x.cpu().to(torch.complex128) for x in xs])
    if op == "prod":
        r = a[0]
        for x in a[1:]:
            r = r * x
        return r.to(dtype)
    s = a.sum(0).to(dtype)
    if op == "avg":
        inv = np.float32(1) / np.float32(n) if dtype == torch.complex64 else 1.0 / n
        s = torch.view_as_complex(torch.view_as_real(s) * torch.tensor(float(inv), dtype=torch.view_as_real(s).dtype))
    return s


def check(ok, what):
    if not ok:
        FAIL.append(what)
        print("FAIL", what, flush=True)


def trace():
    """default selection + every forced algorithm on one GPU; the test reads the trace"""
    from ucc_b200.harness import UccJob, coll_args
    torch.cuda.set_device(0)
    CUDA = U.UCC_MEMORY_TYPE_CUDA

    def ca(coll, src, dst, dt, **kw):
        kw.setdefault("count_src", src.numel() if src is not None else 0)
        kw.setdefault("count_dst", dst.numel() if dst is not None else 0)
        return coll_args(coll, dt=dt, mem_type=CUDA, src_ptr=src.data_ptr() if src is not None else None, dst_ptr=dst.data_ptr() if dst is not None else None, **kw)

    def run(team, args):
        q = team.coll(args)
        st = q.run()
        q.finalize()
        torch.cuda.synchronize()
        check(st == U.UCC_OK, f"status {U.status_str(st)}")

    base = {"UCC_TL_NVL_MAX_BLOCKS": "4", "UCC_TL_NVL_TIMEOUT": "5s", "UCC_TL_NVL_SYMMETRIC_SIZE": "8Mb", "UCC_COLL_TRACE": "info"}
    variants = [("default", {})]
    for alg in ("oneshot", "twoshot", "ring", "rhd"):
        colls = ["allreduce", "reduce_scatter", "reduce_scatterv"] + (["reduce"] if alg == "twoshot" else [])
        variants.append((alg, {"UCC_TL_NVL_TUNE": "#".join(f"{c}:cuda:inf:@{alg}" for c in colls), "UCC_TL_NVL_ZCOPY": "n",
                               "UCC_TL_NVL_ALLREDUCE_ONESHOT_THRESH": "1M" if alg == "oneshot" else "0"}))
    variants.append(("twoshot-zcopy", {"UCC_TL_NVL_TUNE": "allreduce:cuda:inf:@twoshot#reduce_scatter:cuda:inf:@twoshot#reduce:cuda:inf:@twoshot",
                                       "UCC_TL_NVL_ZCOPY": "y", "UCC_TL_NVL_ZCOPY_THRESH": "0", "UCC_TL_NVL_ALLREDUCE_ONESHOT_THRESH": "0"}))
    n = 4
    for name, extra in variants:
        with UccJob(n, env=dict(base, **extra)) as job:
            team = job.create_team()
            for dt, tdt in DTS.items():
                for op in ("sum", "avg", "prod"):
                    for count in (7, 40001):
                        xs = [gauss(count * n, 100 * r + count, tdt).cuda() for r in range(n)]
                        out = [torch.zeros(count * n, dtype=tdt, device="cuda") for _ in range(n)]
                        run(team, [ca("allreduce", xs[r], out[r], dt, op=op) for r in range(n)])
                        exp = expected(op, xs)
                        check(all(torch.equal(o.cpu(), exp) for o in out), f"trace {name} allreduce {dt} {op} {count}")
                        blk = [torch.zeros(count, dtype=tdt, device="cuda") for _ in range(n)]
                        run(team, [ca("reduce_scatter", xs[r], blk[r], dt, op=op) for r in range(n)])
                        check(all(torch.equal(blk[r].cpu(), exp[r * count:(r + 1) * count]) for r in range(n)), f"trace {name} reduce_scatter {dt} {op}")
                        if name not in ("twoshot-zcopy",):
                            cnts = [count + 3 * r for r in range(n)]
                            offs = np.concatenate([[0], np.cumsum(cnts)[:-1]])
                            xv = [gauss(sum(cnts), 5 * r + count, tdt).cuda() for r in range(n)]
                            ov = [torch.zeros(cnts[r], dtype=tdt, device="cuda") for r in range(n)]
                            run(team, [ca("reduce_scatterv", xv[r], ov[r], dt, op=op, dst_counts=cnts, dst_displs=offs) for r in range(n)])
                            ev = expected(op, xv)
                            check(all(torch.equal(ov[r].cpu(), ev[offs[r]:offs[r] + cnts[r]]) for r in range(n)), f"trace {name} reduce_scatterv {dt} {op}")
                        if name in ("default", "twoshot", "twoshot-zcopy"):
                            root = n - 1
                            res = torch.zeros(count * n, dtype=tdt, device="cuda")
                            run(team, [ca("reduce", xs[r], res if r == root else None, dt, op=op, root=root, count_dst=count * n if r == root else 0) for r in range(n)])
                            check(torch.equal(res.cpu(), exp), f"trace {name} reduce {dt} {op}")
            team.destroy()
    # MAX is not defined on complex numbers: on a team of tl/nvl alone it is declined at init
    with UccJob(n, env=dict(base, UCC_TL_SHM_TUNE="allreduce:0")) as job:   # allreduce: tl/nvl alone
        team = job.create_team()
        x = [gauss(16, r, torch.complex64).cuda() for r in range(n)]
        try:
            team.coll([ca("allreduce", x[r], x[r], "float32_complex", op="max") for r in range(n)]).finalize()
            check(False, "complex MAX was accepted")
        except U.UccError as e:
            check(e.status == U.UCC_ERR_NOT_SUPPORTED, f"complex MAX: {e}")
        team.destroy()


def nvl():
    from ucc_b200.dist import Communicator, init_distributed
    rank, world, _ = init_distributed("cpu:gloo,cuda:nccl")
    dev = torch.device("cuda", torch.cuda.current_device())

    def allreduce(comm, src, dst, op):
        req = comm.allreduce_init(src, dst, op=op)
        req.post_on_stream()
        req.wait()
        req.finalize()
        torch.cuda.synchronize()

    # forced in-switch kernels: c64 SUM / AVG (c128 and PROD are declined by @nvls and fall back to the two-shot kernels)
    for tune, want in (("allreduce:cuda:inf:@nvls#reduce_scatter:cuda:inf:@nvls", "nvls_staged"), ("allreduce:cuda:inf:@nvls_pipe", "nvls_pipe")):
        os.environ["UCC_TL_NVL_TUNE"] = tune
        os.environ["UCC_TL_NVL_ALLREDUCE_ONESHOT_THRESH"] = "0"
        comm = Communicator(symm_size="16M")
        has_nvls = bool(comm.symm_region() and comm.symm_region()[2])
        for dtype in (torch.complex64, torch.complex128):
            for op in ("sum", "avg", "prod"):
                for count in (1, 4097, 3000001):
                    alls = [gauss(count, 7 * r + count, dtype) for r in range(world)]
                    out = torch.zeros(count, dtype=dtype, device=dev)
                    allreduce(comm, alls[rank].to(dev), out, op)
                    check(torch.equal(out.cpu(), expected(op, alls)), f"{want} allreduce {dtype} {op} {count}")
                    if has_nvls and dtype == torch.complex64 and op != "prod":
                        check(want in comm.request_info_last(), f"{want} not taken for c64 {op}: {comm.request_info_last()}")
        comm.destroy()
    os.environ.pop("UCC_TL_NVL_TUNE")
    os.environ.pop("UCC_TL_NVL_ALLREDUCE_ONESHOT_THRESH")
    # zero-copy across processes: the members' user buffers are mapped with CUDA IPC and reduced in place
    os.environ.update(UCC_TL_NVL_ZCOPY="y", UCC_TL_NVL_ZCOPY_THRESH="0",
                      UCC_TL_NVL_TUNE="allreduce:cuda:inf:@twoshot#reduce_scatter:cuda:inf:@twoshot#reduce:cuda:inf:@twoshot",
                      UCC_TL_NVL_ALLREDUCE_ONESHOT_THRESH="0")
    comm = Communicator()
    for dtype in (torch.complex64, torch.complex128):
        for op in ("sum", "avg", "prod"):
            count = 1 << 20
            alls = [gauss(count, 11 * r + 1, dtype) for r in range(world)]
            out = torch.zeros(count, dtype=dtype, device=dev)
            allreduce(comm, alls[rank].to(dev), out, op)
            exp = expected(op, alls)
            check(torch.equal(out.cpu(), exp), f"zcopy allreduce {dtype} {op}")
            check("zcopy" in comm.request_info_last(), f"zero-copy kernel not taken: {comm.request_info_last()}")
            blk = count // world
            rs = torch.zeros(blk, dtype=dtype, device=dev)
            req = comm.coll_init("reduce_scatter", alls[rank].to(dev), rs, op=op)
            req.post_on_stream()
            req.wait()
            req.finalize()
            torch.cuda.synchronize()
            check(torch.equal(rs.cpu(), exp[rank * blk:(rank + 1) * blk]), f"zcopy reduce_scatter {dtype} {op}")
    comm.destroy()
    for k in ("UCC_TL_NVL_ZCOPY", "UCC_TL_NVL_ZCOPY_THRESH", "UCC_TL_NVL_TUNE", "UCC_TL_NVL_ALLREDUCE_ONESHOT_THRESH"):
        os.environ.pop(k)
    # symmetric user memory: in-place c64 SUM takes the in-switch kernel exactly as float32 does
    comm = Communicator(symm_size="256M")
    reg = comm.symm_region()
    for count in (4, 262147, 8 * 1024 * 1024):
        comm.symm_reset()
        alls = [gauss(count, 3 * r + count, torch.complex64) for r in range(world)]
        buf = comm.symm_empty(count, torch.complex64)
        guard = comm.symm_empty(64, torch.int32)
        guard.fill_(4242)
        buf.copy_(alls[rank].to(dev))
        torch.cuda.synchronize()
        comm.barrier()
        allreduce(comm, buf, buf, "sum")
        check(torch.equal(buf.cpu(), expected("sum", alls)), f"symm c64 sum {count}")
        check(bool((guard == 4242).all()), f"symm guard {count}")
        if reg and reg[2]:
            check("nvls_symm_inplace" in comm.request_info_last(), f"symm kernel not taken: {comm.request_info_last()}")
    comm.destroy()
    return rank, world


def nccl():
    from ucc_b200.dist import Communicator, init_distributed
    rank, world, _ = init_distributed("cpu:gloo,cuda:nccl")
    dev = torch.device("cuda", torch.cuda.current_device())
    comm = Communicator()
    for dtype in (torch.complex64, torch.complex128):
        for op in ("sum", "avg"):
            count = 100003 * world
            alls = [gauss(count, 5 * r + 2, dtype) for r in range(world)]
            exp = expected(op, alls)
            out = torch.zeros(count, dtype=dtype, device=dev)
            comm.run(comm.allreduce_init(alls[rank].to(dev), out, op=op), torch.cuda.current_stream())
            torch.cuda.synchronize()
            check(torch.equal(out.cpu(), exp), f"nccl allreduce {dtype} {op}")
            blk = count // world
            rs = torch.zeros(blk, dtype=dtype, device=dev)
            comm.run(comm.coll_init("reduce_scatter", alls[rank].to(dev), rs, op=op), torch.cuda.current_stream())
            torch.cuda.synchronize()
            check(torch.equal(rs.cpu(), exp[rank * blk:(rank + 1) * blk]), f"nccl reduce_scatter {dtype} {op}")
            res = torch.zeros(count, dtype=dtype, device=dev)
            src = alls[rank].to(dev)
            comm.run(comm.coll_init("reduce", src, res if rank == 0 else None, op=op, root=0), torch.cuda.current_stream())
            torch.cuda.synchronize()
            if rank == 0:
                check(torch.equal(res.cpu(), exp), f"nccl reduce {dtype} {op}")
        x = torch.ones(16, dtype=dtype, device=dev)
        try:
            comm.allreduce_init(x, x, op="prod").finalize()
            check(False, f"nccl accepted complex PROD {dtype}")
        except U.UccError:
            pass
    comm.destroy()
    return rank, world


def torch_backend():
    import torch.distributed as dist
    import ucc_b200.torch_backend  # noqa: F401
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", rank)) % torch.cuda.device_count())
    dev = torch.device("cuda", torch.cuda.current_device())
    dist.init_process_group("ucc_b200", rank=rank, world_size=world)
    blk = 4099
    g = torch.Generator().manual_seed(1)
    alls = [torch.randn(blk * world, generator=g, dtype=torch.complex64) for _ in range(world)]
    ref = sum(a.to(torch.complex128) for a in alls)
    out = torch.zeros(blk, dtype=torch.complex64, device=dev)
    dist.reduce_scatter_tensor(out, alls[rank].to(dev))
    torch.cuda.synchronize()
    check(out.dtype == torch.complex64 and torch.allclose(out.cpu().to(torch.complex128), ref[rank * blk:(rank + 1) * blk], rtol=1e-5, atol=1e-5), "torch reduce_scatter_tensor complex64")
    t = alls[rank][:blk].to(dev)
    dist.reduce(t, dst=0)
    torch.cuda.synchronize()
    if rank == 0:
        check(torch.allclose(t.cpu().to(torch.complex128), sum(a[:blk].to(torch.complex128) for a in alls), rtol=1e-5, atol=1e-5), "torch reduce complex64")
    outs = [torch.zeros(blk, dtype=torch.complex64, device=dev) for _ in range(1)]
    dist.reduce_scatter(outs[0], [c.to(dev) for c in alls[rank].chunk(world)])
    torch.cuda.synchronize()
    check(torch.allclose(outs[0].cpu().to(torch.complex128), ref[rank * blk:(rank + 1) * blk], rtol=1e-5, atol=1e-5), "torch reduce_scatter complex64")
    return rank, world


def main():
    mode = sys.argv[1]
    if mode == "trace":
        trace()
        print("COMPLEX_WORKER_OK" if not FAIL else f"COMPLEX_WORKER_FAIL {FAIL[:5]}", flush=True)
        return 0 if not FAIL else 1
    import torch.distributed as dist
    rank, world = {"nvl": nvl, "nccl": nccl, "torch": torch_backend}[mode]()
    flag = torch.tensor([0 if FAIL else 1], device="cuda" if mode == "torch" else "cpu")
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    if rank == 0:
        print(f"COMPLEX_WORKER_OK n_gpus={world}" if flag.item() == 1 else "COMPLEX_WORKER_FAIL", flush=True)
    dist.destroy_process_group()
    return 0 if flag.item() == 1 else 1


if __name__ == "__main__":
    sys.exit(main())
