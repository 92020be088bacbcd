#!/usr/bin/env python
"""Multi-process functional test driver with an oracle - the role of the reference's `ucc_test_mpi` (test/mpi/main.cc:87-120,
test/mpi/test_mpi.cc), launched with torchrun instead of mpirun:

    python -m torch.distributed.run --nproc-per-node 4 --master-addr 127.0.0.1 tools/ucc_test_dist.py \
        -c allreduce,alltoallv -t world,half,odd_even,reverse -M host -d int32,float32 -o sum,max -I 2 -P 2 -m 8:65536:8

Every rank generates every rank's input from (seed, case, rank), so the expected result is computed locally - no second
communication library is needed as the oracle.  A case whose init returns NOT_SUPPORTED counts as skipped.
The report at the end has the reference's shape (total / passed / skipped / failed).
"""
from __future__ import annotations

import argparse
import faulthandler
import ctypes as C
import itertools
import os
import sys
import time

import numpy as np
import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from ucc_b200 import capi as U  # noqa: E402
from ucc_b200.dist import Communicator, init_distributed  # noqa: E402
from ucc_b200.harness import coll_args  # noqa: E402

ALL_COLLS = ["barrier", "allreduce", "allgather", "allgatherv", "bcast", "alltoall", "alltoallv", "reduce", "reduce_scatter",
             "reduce_scatterv", "gather", "gatherv", "scatter", "scatterv"]
REDUCTIONS = {"allreduce", "reduce", "reduce_scatter", "reduce_scatterv"}
ROOTED = {"bcast", "reduce", "gather", "gatherv", "scatter", "scatterv"}
NO_DATA = {"barrier"}
NP_DT = {"int8": np.int8, "uint8": np.uint8, "int16": np.int16, "uint16": np.uint16, "int32": np.int32, "uint32": np.uint32,
         "int64": np.int64, "uint64": np.uint64, "float16": np.float16, "float32": np.float32, "float64": np.float64,
         "bfloat16": None, "float32_complex": np.complex64, "float64_complex": np.complex128}
INT_OPS = {"sum", "prod", "max", "min", "land", "lor", "lxor", "band", "bor", "bxor"}
FLOAT_OPS = {"sum", "prod", "max", "min", "avg"}
COMPLEX_OPS = {"sum", "prod", "avg"}   # what the reference's ec/cuda defines for complex types
MEM = {"host": U.UCC_MEMORY_TYPE_HOST, "cuda": U.UCC_MEMORY_TYPE_CUDA, "cudaManaged": U.UCC_MEMORY_TYPE_CUDA_MANAGED}


def dt_size(dt):
    return 2 if dt == "bfloat16" else np.dtype(NP_DT[dt]).itemsize


def is_float(dt):
    return dt in ("float16", "float32", "float64", "bfloat16", "float32_complex", "float64_complex")


def is_complex(dt):
    return dt in ("float32_complex", "float64_complex")


def logical_dt(dt):
    """numpy type the logical contents of a `dt` buffer travel in"""
    return np.complex128 if is_complex(dt) else np.float64 if is_float(dt) else np.int64


class Buf:
    """`count` elements of `dt` in host or CUDA memory; contents move as logical float64/int64 numpy arrays"""

    def __init__(self, dt, count, mtype):
        self.dt, self.count, self.mtype = dt, count, mtype
        self.t = torch.zeros(max(count, 1) * dt_size(dt), dtype=torch.uint8, device="cuda" if mtype == "cuda" else "cpu")

    def reset(self):
        """back to the initial contents (persistent collectives are posted several times, in-place ones consume their input)"""
        if getattr(self, "init", None) is not None:
            self.set(self.init)
        else:
            self.t.zero_()

    @property
    def ptr(self):
        return self.t.data_ptr()

    def set(self, vals):
        vals = np.asarray(vals)
        assert vals.size == self.count
        self.init = vals
        if self.count == 0:
            return
        if self.dt == "bfloat16":
            raw = torch.from_numpy(vals.astype(np.float32)).to(torch.bfloat16).view(torch.uint8)
        else:
            raw = torch.from_numpy(vals.astype(NP_DT[self.dt]).view(np.uint8).copy())
        self.t[:raw.numel()].copy_(raw)

    def get(self):
        raw = self.t[:self.count * dt_size(self.dt)].cpu()
        if self.dt == "bfloat16":
            return raw.view(torch.bfloat16).float().numpy().astype(np.float64)
        v = raw.numpy().view(NP_DT[self.dt])
        return v.astype(np.uint64 if self.dt == "uint64" else logical_dt(self.dt))


def gen(seed, case, rank, count, dt, op="sum"):
    """logical input of `rank`: small non-negative values, exactly representable in every datatype"""
    g = np.random.default_rng([seed, case, rank])
    if is_complex(dt):   # Gaussian integers: sums exact; PROD parts in [-1, 1] (never 0) keep products of many ranks small
        lo, hi = (-1, 2) if op == "prod" else (-4, 5)
        re, im = g.integers(lo, hi, count), g.integers(lo, hi, count)
        if op == "prod":
            re[(re == 0) & (im == 0)] = 1
        return (re + 1j * im).astype(np.complex128)
    if op == "prod":
        return g.integers(1, 3, count).astype(np.float64 if is_float(dt) else np.int64)
    hi = 4 if dt in ("int8", "uint8", "float16", "bfloat16") else 100
    return g.integers(0, hi, count).astype(np.float64 if is_float(dt) else np.int64)


def reduce_oracle(op, arrs, dt):
    a = np.stack(arrs)
    if op == "sum":
        r = a.sum(0)
    elif op == "avg" and is_complex(dt):   # the sum times 1/N computed in the component precision
        c = NP_DT[dt](0).real.dtype.type
        r = (a.sum(0).astype(NP_DT[dt]) * (c(1) / c(len(arrs)))).astype(np.complex128)
    elif op == "avg":
        r = a.sum(0) / len(arrs)
    elif op == "prod":
        r = a.prod(0)
    elif op == "max":
        r = a.max(0)
    elif op == "min":
        r = a.min(0)
    elif op in ("land", "lor", "lxor"):
        b = a != 0
        r = {"land": b.all(0), "lor": b.any(0), "lxor": (b.sum(0) % 2) == 1}[op].astype(a.dtype)
    else:
        ai = a.astype(np.int64)
        f = {"band": np.bitwise_and, "bor": np.bitwise_or, "bxor": np.bitwise_xor}[op]
        r = ai[0]
        for x in ai[1:]:
            r = f(r, x)
    if not is_float(dt):   # wrap like the fixed-width type does
        r = r.astype(np.int64).astype(NP_DT[dt]).astype(np.uint64 if dt == "uint64" else np.int64)
    return r


def close(got, exp, dt, n):
    if not is_float(dt):
        return np.array_equal(got.astype(np.int64), np.asarray(exp).astype(np.int64))
    tol = {"float64": 1e-12, "float32": 1e-5, "float16": 2e-2, "bfloat16": 6e-2, "float64_complex": 1e-12, "float32_complex": 1e-5}[dt] * max(1, n)
    if is_complex(dt):   # per part, with the tolerance of the component type
        exp = np.asarray(exp)
        return np.allclose(got.real, exp.real, rtol=tol, atol=tol) and np.allclose(got.imag, exp.imag, rtol=tol, atol=tol)
    return np.allclose(got, exp, rtol=tol, atol=tol)


class Team:
    def __init__(self, kind, rank, world):
        self.kind = kind
        self.comm = None
        self.members = None
        self.group = None          # gloo group of the members (None = everybody) for the pass/fail agreement
        if kind == "world":
            self.members = list(range(world))
            self.comm = Communicator()
        elif kind == "reverse":
            self.members = [world - 1 - u for u in range(world)]     # UCC rank u is torch rank world-1-u
            self.comm = Communicator(perm=[world - 1 - g for g in range(world)])
        elif kind == "half":
            m = list(range((world + 1) // 2))
            g = dist.new_group(m, backend="gloo")                     # collective over the world: everybody calls it
            if rank in m and len(m) > 1:
                self.members, self.comm, self.group = m, Communicator(g), g
        elif kind == "odd_even":
            ev, od = [r for r in range(world) if r % 2 == 0], [r for r in range(world) if r % 2 == 1]
            ge, go = dist.new_group(ev, backend="gloo"), dist.new_group(od, backend="gloo")
            m, g = (ev, ge) if rank % 2 == 0 else (od, go)
            if len(m) > 1:
                self.members, self.comm, self.group = m, Communicator(g), g
        else:
            raise ValueError(f"incorrect team type: {kind}")

    def destroy(self):
        if self.comm:
            self.comm.destroy()


def v_counts(seed, case, n, count):
    g = np.random.default_rng([seed, case, 7777])
    return [int(x) for x in g.integers(0, max(count, 1) + 1, n)]


def build_case(coll, team, urank, n, seed, case, dt, op, mtype, count, root, inplace):
    """returns (args, check) where check() -> bool compares the destination with the oracle; or None when the combination
    does not exist (e.g. in-place alltoall)"""
    mt = MEM[mtype]
    inp = lambda r, c, salt=0: gen(seed, case * 131 + salt, r, c, dt, op)  # noqa: E731
    keep = []

    def buf(c, vals=None):
        b = Buf(dt, c, mtype)
        if vals is not None:
            b.set(vals)
        keep.append(b)
        return b

    def done(args, check):
        args._bufs = keep
        return args, check
    if coll == "barrier":
        return done(coll_args("barrier"), lambda: True)
    if coll == "allreduce":
        data = [inp(r, count) for r in range(n)]
        exp = reduce_oracle(op, data, dt)
        dst = buf(count, data[urank] if inplace else None)
        src = None if inplace else buf(count, data[urank])
        a = coll_args(coll, dt=dt, op=op, inplace=inplace, mem_type=mt, src_ptr=src.ptr if src else None, dst_ptr=dst.ptr,
                      count_src=0 if inplace else count, count_dst=count)
        return done(a, lambda: close(dst.get(), exp, dt, n))
    if coll == "reduce":
        data = [inp(r, count) for r in range(n)]
        exp = reduce_oracle(op, data, dt)
        is_root = urank == root
        if inplace and is_root:
            dst = buf(count, data[urank])
            a = coll_args(coll, dt=dt, op=op, root=root, inplace=True, mem_type=mt, dst_ptr=dst.ptr, count_dst=count, count_src=0)
        else:
            src = buf(count, data[urank])
            dst = buf(count) if is_root else None
            a = coll_args(coll, dt=dt, op=op, root=root, inplace=inplace, mem_type=mt, src_ptr=src.ptr, dst_ptr=dst.ptr if dst else None,
                          count_src=count, count_dst=count if is_root else 0)
        return done(a, lambda: (not is_root) or close(dst.get(), exp, dt, n))
    if coll == "bcast":
        if inplace:
            return None
        data = inp(root, count)
        b = buf(count, data if urank == root else None)
        a = coll_args(coll, dt=dt, root=root, mem_type=mt, src_ptr=b.ptr, count_src=count, count_dst=0)
        return done(a, lambda: close(b.get(), data, dt, 1))
    if coll == "allgather":
        data = [inp(r, count) for r in range(n)]
        exp = np.concatenate(data)
        dst = buf(count * n)
        if inplace:
            full = np.zeros(count * n, exp.dtype)
            full[urank * count:(urank + 1) * count] = data[urank]
            dst.set(full)
            a = coll_args(coll, dt=dt, inplace=True, mem_type=mt, dst_ptr=dst.ptr, count_dst=count * n, count_src=0)
        else:
            src = buf(count, data[urank])
            a = coll_args(coll, dt=dt, mem_type=mt, src_ptr=src.ptr, dst_ptr=dst.ptr, count_src=count, count_dst=count * n)
        return done(a, lambda: close(dst.get(), exp, dt, 1))
    if coll == "allgatherv":
        counts = v_counts(seed, case, n, count)
        displs = [int(x) for x in np.concatenate([[0], np.cumsum(counts)[:-1]])]
        data = [inp(r, counts[r]) for r in range(n)]
        exp = np.concatenate(data) if sum(counts) else np.zeros(0)
        dst = buf(sum(counts))
        if inplace:
            full = np.zeros(sum(counts), logical_dt(dt))
            full[displs[urank]:displs[urank] + counts[urank]] = data[urank]
            dst.set(full)
            a = coll_args(coll, dt=dt, inplace=True, mem_type=mt, dst_ptr=dst.ptr, dst_counts=counts, dst_displs=displs, count_src=0)
        else:
            src = buf(counts[urank], data[urank])
            a = coll_args(coll, dt=dt, mem_type=mt, src_ptr=src.ptr, count_src=counts[urank], dst_ptr=dst.ptr, dst_counts=counts, dst_displs=displs)
        return done(a, lambda: close(dst.get(), exp, dt, 1))
    if coll == "alltoall":
        data = [inp(r, count * n) for r in range(n)]
        exp = np.concatenate([data[p][urank * count:(urank + 1) * count] for p in range(n)])
        if inplace:
            dst = buf(count * n, data[urank])
            a = coll_args(coll, dt=dt, inplace=True, mem_type=mt, dst_ptr=dst.ptr, count_dst=count * n, count_src=0)
            return done(a, lambda: close(dst.get(), exp, dt, 1))
        src, dst = buf(count * n, data[urank]), buf(count * n)
        a = coll_args(coll, dt=dt, mem_type=mt, src_ptr=src.ptr, dst_ptr=dst.ptr, count_src=count * n, count_dst=count * n)
        return done(a, lambda: close(dst.get(), exp, dt, 1))
    if coll == "alltoallv":
        if inplace:
            return None
        g = np.random.default_rng([seed, case, 4242])
        m = g.integers(0, max(count, 1) + 1, (n, n))                  # m[s][d]: elements s sends to d
        sc, rc = [int(x) for x in m[urank]], [int(x) for x in m[:, urank]]
        sd = [int(x) for x in np.concatenate([[0], np.cumsum(sc)[:-1]])]
        rd = [int(x) for x in np.concatenate([[0], np.cumsum(rc)[:-1]])]
        data = [inp(r, int(m[r].sum())) for r in range(n)]
        parts = []
        for p in range(n):
            off = int(m[p][:urank].sum())
            parts.append(data[p][off:off + int(m[p][urank])])
        exp = np.concatenate(parts) if sum(rc) else np.zeros(0)
        src, dst = buf(sum(sc), data[urank]), buf(sum(rc))
        a = coll_args(coll, dt=dt, mem_type=mt, src_ptr=src.ptr, dst_ptr=dst.ptr, src_counts=sc, src_displs=sd, dst_counts=rc, dst_displs=rd)
        return done(a, lambda: close(dst.get(), exp, dt, 1))
    if coll == "reduce_scatter":
        data = [inp(r, count * n) for r in range(n)]
        exp = reduce_oracle(op, data, dt)[urank * count:(urank + 1) * count]
        if inplace:
            dst = buf(count * n, data[urank])
            a = coll_args(coll, dt=dt, op=op, inplace=True, mem_type=mt, dst_ptr=dst.ptr, count_dst=count * n, count_src=0)
            return done(a, lambda: close(dst.get()[urank * count:(urank + 1) * count], exp, dt, n))
        src, dst = buf(count * n, data[urank]), buf(count)
        a = coll_args(coll, dt=dt, op=op, mem_type=mt, src_ptr=src.ptr, dst_ptr=dst.ptr, count_src=count * n, count_dst=count)
        return done(a, lambda: close(dst.get(), exp, dt, n))
    if coll == "reduce_scatterv":
        if inplace:
            return None
        counts = v_counts(seed, case, n, count)
        displs = [int(x) for x in np.concatenate([[0], np.cumsum(counts)[:-1]])]
        data = [inp(r, sum(counts)) for r in range(n)]
        exp = reduce_oracle(op, data, dt)[displs[urank]:displs[urank] + counts[urank]] if sum(counts) else np.zeros(0)
        src, dst = buf(sum(counts), data[urank]), buf(counts[urank])
        a = coll_args(coll, dt=dt, op=op, mem_type=mt, src_ptr=src.ptr, count_src=sum(counts), dst_ptr=dst.ptr, dst_counts=counts, dst_displs=displs)
        return done(a, lambda: close(dst.get(), exp, dt, n))
    if coll in ("gather", "gatherv"):
        counts = [count] * n if coll == "gather" else v_counts(seed, case, n, count)
        displs = [int(x) for x in np.concatenate([[0], np.cumsum(counts)[:-1]])]
        data = [inp(r, counts[r]) for r in range(n)]
        exp = np.concatenate(data) if sum(counts) else np.zeros(0)
        is_root = urank == root
        src = buf(counts[urank], data[urank])
        dst = buf(sum(counts)) if is_root else None
        if inplace and is_root:
            full = np.zeros(sum(counts), logical_dt(dt))
            full[displs[urank]:displs[urank] + counts[urank]] = data[urank]
            dst.set(full)
            if coll == "gather":
                a = coll_args(coll, dt=dt, root=root, inplace=True, mem_type=mt, dst_ptr=dst.ptr, count_dst=count * n, count_src=0)
            else:
                a = coll_args(coll, dt=dt, root=root, inplace=True, mem_type=mt, dst_ptr=dst.ptr, dst_counts=counts, dst_displs=displs, count_src=0)
        elif coll == "gather":
            a = coll_args(coll, dt=dt, root=root, mem_type=mt, src_ptr=src.ptr, count_src=count, dst_ptr=dst.ptr if dst else None,
                          count_dst=count * n if is_root else 0)
        elif is_root:
            a = coll_args(coll, dt=dt, root=root, mem_type=mt, src_ptr=src.ptr, count_src=counts[urank], dst_ptr=dst.ptr, dst_counts=counts, dst_displs=displs)
        else:
            a = coll_args(coll, dt=dt, root=root, mem_type=mt, src_ptr=src.ptr, count_src=counts[urank], count_dst=0)
        return done(a, lambda: (not is_root) or close(dst.get(), exp, dt, 1))
    if coll in ("scatter", "scatterv"):
        counts = [count] * n if coll == "scatter" else v_counts(seed, case, n, count)
        displs = [int(x) for x in np.concatenate([[0], np.cumsum(counts)[:-1]])]
        data = inp(root, sum(counts))
        exp = data[displs[urank]:displs[urank] + counts[urank]]
        is_root = urank == root
        src = buf(sum(counts), data) if is_root else None
        dst = buf(counts[urank])
        if inplace and is_root:      # the root keeps its block where it is: nothing to check on that rank
            if coll == "scatter":
                a = coll_args(coll, dt=dt, root=root, inplace=True, mem_type=mt, src_ptr=src.ptr, count_src=count * n, count_dst=0)
            else:
                a = coll_args(coll, dt=dt, root=root, inplace=True, mem_type=mt, src_ptr=src.ptr, src_counts=counts, src_displs=displs, count_dst=0)
            return done(a, lambda: close(src.get(), data, dt, 1))
        if coll == "scatter":
            a = coll_args(coll, dt=dt, root=root, mem_type=mt, src_ptr=src.ptr if src else None, count_src=count * n if is_root else 0,
                          dst_ptr=dst.ptr, count_dst=count)
        elif is_root:
            a = coll_args(coll, dt=dt, root=root, mem_type=mt, src_ptr=src.ptr, src_counts=counts, src_displs=displs, dst_ptr=dst.ptr, count_dst=counts[urank])
        else:
            a = coll_args(coll, dt=dt, root=root, mem_type=mt, dst_ptr=dst.ptr, count_dst=counts[urank], count_src=0)
        return done(a, lambda: close(dst.get(), exp, dt, 1))
    raise ValueError(coll)


def run_batch(comm, batch, iters, use_cuda, timeout=120.0):
    """Run the cases of `batch` (dicts with args/persistent/triggered) CONCURRENTLY on one team: init all, post all in the same
    order on every rank, progress until all are done.  Fills case["res"] with 'ok' | 'skip' | 'fail:<why>'."""
    from ucc_b200.dist import Request
    live = []
    for c in batch:
        args = c["args"]
        if c["persistent"]:
            args.mask |= U.UCC_COLL_ARGS_FIELD_FLAGS
            args.flags |= U.UCC_COLL_ARGS_FLAG_PERSISTENT
        r = C.POINTER(U.ucc_coll_req_t)()
        st = U.ucc_collective_init(C.byref(args), C.byref(r), comm.team)
        if st in (U.UCC_ERR_NOT_SUPPORTED, U.UCC_ERR_NOT_IMPLEMENTED):
            c["res"] = "skip"
        elif st != U.UCC_OK:
            c["res"] = f"fail:init {st}"
        else:
            c["res"], c["req"] = "ok", Request(comm, r, (args,))
            live.append(c)
    max_it = max([iters if c["persistent"] else 1 for c in live], default=0)
    for it in range(max_it):
        cur = [c for c in live if c["res"] == "ok" and it < (iters if c["persistent"] else 1)]
        for c in cur:
            if it:
                for b in c["args"]._bufs:
                    b.reset()
            if c["triggered"] and use_cuda:
                c["req"].post_on_stream()
            else:
                c["req"].post()
        t0 = time.time()
        while any(c["req"].test() == U.UCC_INPROGRESS for c in cur):
            comm.progress()
            if time.time() - t0 > timeout:
                break
        for c in cur:
            st = c["req"].test()
            if st == U.UCC_INPROGRESS:
                c["res"] = "fail:timeout"
            elif st != U.UCC_OK:
                c["res"] = f"fail:status {st}"
        if use_cuda:
            torch.cuda.synchronize()
    for c in live:
        if c["req"].test() != U.UCC_INPROGRESS:
            c["req"].finalize()


def parse_args(argv):
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("-c", "--colls", default="all")
    ap.add_argument("-t", "--teams", default="world")
    ap.add_argument("-M", "--mtypes", default="host")
    ap.add_argument("-d", "--dtypes", default="int32,float32")
    ap.add_argument("-o", "--ops", default="sum,max")
    ap.add_argument("-I", "--inplace", type=int, default=0, help="0 - no inplace, 1 - inplace, 2 - both")
    ap.add_argument("-P", "--persistent", type=int, default=0, help="0 - no persistent, 1 - persistent, 2 - both")
    ap.add_argument("-m", "--msgsize", default="8:65536:8", help="min:max[:power] in bytes")
    ap.add_argument("-r", "--root", default="single:0", help="single:<value>, random:<n>, all")
    ap.add_argument("-s", "--seed", type=int, default=None)
    ap.add_argument("-Z", "--max_size", type=int, default=1 << 30, help="cases whose largest buffer exceeds this are skipped")
    ap.add_argument("-N", "--num_tests", type=int, default=1, help="number of tests to run in parallel (outstanding on the same team)")
    ap.add_argument("-i", "--iter", type=int, default=1)
    ap.add_argument("--triggered", type=int, default=0, help="0 - post, 1 - triggered post (CUDA memory), 2 - both")
    ap.add_argument("-v", "--verbose", action="store_true")
    return ap.parse_args(argv)


def main(argv=None):
    faulthandler.enable()
    a = parse_args(argv)
    colls = ALL_COLLS if a.colls == "all" else a.colls.split(",")
    for c in colls:
        if c not in ALL_COLLS:
            raise SystemExit(f"incorrect coll type: {c}")
    mtypes = a.mtypes.split(",")
    use_cuda = "cuda" in mtypes
    rank, world, _ = init_distributed("cpu:gloo,cuda:nccl" if use_cuda else "gloo")
    if a.seed is None:
        s = torch.tensor([int(time.time()) & 0x7fffffff])
        dist.broadcast(s, 0)
        a.seed = int(s.item())
    p = a.msgsize.split(":")
    lo, hi, power = int(p[0]), int(p[1]), int(p[2]) if len(p) > 2 else 2
    sizes, sz = [], max(lo, 1)
    while sz <= hi:
        sizes.append(sz)
        sz *= max(power, 2)
    inplaces = {0: [False], 1: [True], 2: [False, True]}[a.inplace]
    persists = {0: [False], 1: [True], 2: [False, True]}[a.persistent]
    trigs = {0: [False], 1: [True], 2: [False, True]}[a.triggered]
    if rank == 0:
        print("===== UCC DIST TEST INFO =======")
        print(f"seed:         {a.seed}\ncollectives:  {', '.join(colls)}\ndata types:   {a.dtypes}\nmemory types: {a.mtypes}\nteams:        {a.teams}", flush=True)
    totals = np.zeros(4, np.int64)   # total, passed, skipped, failed
    failures = []
    case = 0
    for ki, kind in enumerate(a.teams.split(",")):
        case = ki * 10_000_000      # not every process takes part in every team kind: keep the case ids aligned
        team = Team(kind, rank, world)
        if team.comm is None:
            team.destroy()
            continue
        comm, n, urank = team.comm, team.comm.size, team.comm.rank
        rk, rv = (a.root.split(":") + ["0"])[:2]
        roots = list(range(n)) if rk == "all" else ([int(rv) % n] if rk == "single" else
                                                    [int(x) for x in np.random.default_rng([a.seed, 99]).integers(0, n, int(rv))])
        batch = []

        def flush(batch):
            """run the pending cases concurrently, agree on the verdicts across the team, tally"""
            if not batch:
                return
            run_batch(comm, batch, a.iter, any(c["cuda"] for c in batch))
            codes = []
            for c in batch:
                if c["res"] == "ok" and not c["check"]():
                    c["res"] = "fail:data mismatch"
                codes.append(0 if c["res"] == "ok" else (1 if c["res"] == "skip" else 2))
            # a case passes only if it passed everywhere; NOT_SUPPORTED must be unanimous too
            code = torch.tensor(codes)
            dist.all_reduce(code, op=dist.ReduceOp.MAX, group=team.group)
            for c, worst in zip(batch, code.tolist()):
                if worst == 0:
                    totals[1] += 1
                elif worst == 1:
                    totals[2] += 1
                else:
                    totals[3] += 1
                    failures.append(f"{c['name']}: rank {rank} {c['res']}")
                if a.verbose and rank == 0:
                    print(f"[{'OK' if worst == 0 else 'SKIP' if worst == 1 else 'FAIL'}] {c['name']}", flush=True)
            batch.clear()
        for coll in colls:
            dts = ["int32"] if coll in NO_DATA else a.dtypes.split(",")
            ops = a.ops.split(",") if coll in REDUCTIONS else ["sum"]
            szs = [0] if coll in NO_DATA else sizes
            for mtype, dt, op, size, root, inplace, persistent, trig in itertools.product(
                    mtypes, dts, ops, szs, roots if coll in ROOTED else [0], inplaces, persists, trigs):
                case += 1
                if dt not in NP_DT or mtype not in MEM:
                    raise SystemExit(f"incorrect dtype/mtype: {dt}/{mtype}")
                if coll in REDUCTIONS and op not in (COMPLEX_OPS if is_complex(dt) else FLOAT_OPS if is_float(dt) else INT_OPS):
                    continue
                if trig and mtype != "cuda":
                    continue
                count = max(size // dt_size(dt), 1) if coll not in NO_DATA else 0
                name = f"{kind}/{coll}/{mtype}/{dt}/{op}/count={count}/root={root}/inplace={int(inplace)}/persistent={int(persistent)}/triggered={int(trig)}"
                totals[0] += 1
                if count * dt_size(dt) * (n if coll not in ("allreduce", "reduce", "bcast") else 1) > a.max_size or mtype == "cudaManaged":
                    totals[2] += 1
                    continue
                built = build_case(coll, team, urank, n, a.seed, case, dt, op, mtype, count, root, inplace)
                if built is None:
                    totals[2] += 1
                    continue
                batch.append({"name": name, "args": built[0], "check": built[1], "persistent": persistent, "triggered": trig,
                              "cuda": mtype == "cuda"})
                if len(batch) >= max(a.num_tests, 1):
                    flush(batch)
        flush(batch)
        comm.barrier()
        team.destroy()
    # sub-teams run on a subset of the processes: merge the per-process tallies
    fails = [None] * world
    dist.all_gather_object(fails, failures)
    allt = [None] * world
    dist.all_gather_object(allt, totals.tolist())
    if rank == 0:
        tot = np.max(np.array(allt), axis=0)      # same case list on every process that ran a team kind
        nfail = sum(1 for f in fails for _ in f)
        print("\n===== UCC DIST TEST REPORT =====")
        print(f"   total tests : {int(tot[0])}\n   passed      : {int(tot[1])}\n   skipped     : {int(tot[2])}\n   failed      : {int(tot[3])}")
        for f in fails:
            for ln in f[:20]:
                print("   FAILED " + ln)
        if tot[0] and tot[0] == tot[2]:
            print("\n All tests have been skipped, indicating most likely a problem with the requested memory type / transport")
        print("UCC_TEST_DIST_" + ("OK" if nfail == 0 and tot[3] == 0 else "FAIL"), flush=True)
    bad = torch.tensor([sum(len(f) for f in fails)])
    dist.destroy_process_group()
    return 1 if bad.item() else 0


if __name__ == "__main__":
    sys.exit(main())
