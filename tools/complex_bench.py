#!/usr/bin/env python3
"""Complex allreduce / reduce_scatter on CUDA buffers: tl/nvl vs the float32 control on the same bytes, NCCL and the host transport.

    torchrun --nproc-per-node N tools/complex_bench.py [--out FILE] [--reps R]

Rows (bytes per rank: 4 KB, 64 KB, 1 MB, 16 MB, 256 MB, 1 GiB):
  allreduce c64 SUM, c64 PROD, c128 SUM   default selection of this library
  allreduce f32 SUM control               the same bytes as float32 (view_as_real): the c64 SUM row runs the same kernels
  allreduce nccl f32 SUM                  torch.distributed (NCCL) on view_as_real
  allreduce c64 SUM shm                   UCC_TLS=shm,self, the only path complex data had before tl/nvl took it (up to 1 MB)
  reduce_scatter c64 SUM                  16 MB and 256 MB
Time = device time from CUDA events around ITERS back-to-back collectives on one stream after a warm-up, max over ranks.  The
rows of one size alternate R times; the median is reported with the min / max as the run-to-run spread.  Every result is checked
(Gaussian-integer inputs, exact).  busbw = 2 (N-1)/N * bytes / time (allreduce), (N-1)/N * bytes / time (reduce_scatter).  The card
name and its power limit are read in the same run."""
import argparse
import json
import os
import subprocess
import sys

import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from ucc_b200.dist import Communicator, init_distributed  # noqa: E402

SIZES = [4 << 10, 64 << 10, 1 << 20, 16 << 20, 256 << 20, 1 << 30]
RS_SIZES = [16 << 20, 256 << 20]
SHM_MAX = 1 << 20
WARM = 3


def gpu_info():
    name = torch.cuda.get_device_name()
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", str(torch.cuda.current_device())],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        q = f"unavailable ({e})"
    return {"gpu": name, "power_limit_and_max_sm_clock": q}


def pattern(count, rank, dtype, dev):
    """Gaussian integers with parts in [-2, 2] (never 0): exact sums and products up to 8 ranks"""
    i = torch.arange(count, device=dev, dtype=torch.int64)
    re = (i * 7 + rank * 13) % 5 - 2
    im = (i * 3 + rank * 11 + 1) % 5 - 2
    re = torch.where((re == 0) & (im == 0), torch.ones_like(re), re)
    return torch.complex(re.double(), im.double()).to(dtype)


def expected(count, world, dtype, op, dev):
    r = pattern(count, 0, torch.complex128, dev)
    for p in range(1, world):
        x = pattern(count, p, torch.complex128, dev)
        r = r * x if op == "prod" else r + x
    return r.to(dtype)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="", help="JSON file (rank 0); stdout when empty")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--max-bytes", type=int, default=SIZES[-1])
    args = ap.parse_args()
    rank, world, _ = init_distributed("cpu:gloo,cuda:nccl")
    dev = torch.device("cuda", torch.cuda.current_device())
    stream = torch.cuda.Stream()
    comm = Communicator()
    os.environ["UCC_TLS"] = "shm,self"
    comm_shm = Communicator()
    os.environ.pop("UCC_TLS")

    def maxr(x):
        t = torch.tensor([x], dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.item()

    def timed(post, iters, finish=None):
        with torch.cuda.stream(stream):
            for _ in range(WARM):
                post()
            if finish:
                finish()
            torch.cuda.synchronize()
            dist.barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            for _ in range(iters):
                post()
            e1.record(stream)
            if finish:
                finish()
            torch.cuda.synchronize()
        return maxr(e0.elapsed_time(e1) * 1e3 / iters)

    def ours(c, coll, src, dst, op, iters):
        reqs = []

        def post():
            r = c.coll_init(coll, src, dst, op=op)
            r.post_on_stream(stream)
            reqs.append(r)

        def finish():
            for r in reqs:
                r.wait()
                r.finalize()
            reqs.clear()
        t = timed(post, iters, finish)
        return t, c.request_info_last()

    def nccl(x, buf, iters):
        """NCCL reduces in place: time it on zeros (the values stay put), then one more call on the input for the check"""
        buf.zero_()
        t = timed(lambda: dist.all_reduce(buf), iters)
        buf.copy_(x)
        dist.all_reduce(buf)
        torch.cuda.synchronize()
        return t, "nccl"

    rows = []
    ok = True
    for nbytes in [s for s in SIZES if s <= args.max_bytes]:
        iters = 20 if nbytes <= (16 << 20) else 5
        n64, n128 = nbytes // 8, nbytes // 16
        x64, x128 = pattern(n64, rank, torch.complex64, dev), pattern(n128, rank, torch.complex128, dev)
        o64, o128 = torch.empty_like(x64), torch.empty_like(x128)
        xf, of = torch.view_as_real(x64).reshape(-1), torch.empty(2 * n64, device=dev)
        nz = torch.zeros_like(of)
        cases = {
            "allreduce_c64_sum": lambda: ours(comm, "allreduce", x64, o64, "sum", iters),
            "allreduce_f32_sum_control": lambda: ours(comm, "allreduce", xf, of, "sum", iters),
            "allreduce_c64_prod": lambda: ours(comm, "allreduce", x64, o64, "prod", iters),
            "allreduce_c128_sum": lambda: ours(comm, "allreduce", x128, o128, "sum", iters),
            "allreduce_nccl_f32_sum": lambda: nccl(xf, nz, iters),
        }
        if nbytes <= SHM_MAX:
            cases["allreduce_c64_sum_shm"] = lambda: ours(comm_shm, "allreduce", x64, o64, "sum", iters)
        if nbytes in RS_SIZES:
            rs_out = torch.empty(n64 // world, dtype=torch.complex64, device=dev)
            cases["reduce_scatter_c64_sum"] = lambda: ours(comm, "reduce_scatter", x64[:rs_out.numel() * world], rs_out, "sum", iters)
        times = {k: [] for k in cases}
        kern = {}
        for _ in range(args.reps):
            for k, fn in cases.items():
                t, kern[k] = fn()
                times[k].append(t)
                # verify what the last timed step computed
                if k.startswith("allreduce_c64") or k == "allreduce_c128_sum":
                    o, dt, op = (o128, torch.complex128, "sum") if "c128" in k else (o64, torch.complex64, "prod" if "prod" in k else "sum")
                    good = torch.equal(o, expected(o.numel(), world, dt, op, dev))
                elif k == "allreduce_f32_sum_control":
                    good = torch.equal(of, torch.view_as_real(expected(n64, world, torch.complex64, "sum", dev)).reshape(-1))
                elif k == "reduce_scatter_c64_sum":
                    e = expected(rs_out.numel() * world, world, torch.complex64, "sum", dev)
                    good = torch.equal(rs_out, e[rank * rs_out.numel():(rank + 1) * rs_out.numel()])
                else:
                    good = torch.equal(nz, torch.view_as_real(expected(n64, world, torch.complex64, "sum", dev)).reshape(-1))
                flag = torch.tensor([1 if good else 0])
                dist.all_reduce(flag, op=dist.ReduceOp.MIN)
                if flag.item() != 1:
                    ok = False
                    if rank == 0:
                        print(f"MISMATCH {k} {nbytes}", flush=True)
        for k, ts in times.items():
            ts = sorted(ts)
            med = ts[len(ts) // 2]
            f = (world - 1) / world * (1 if k.startswith("reduce_scatter") else 2)
            rb = rs_out.numel() * world * 8 if k.startswith("reduce_scatter") else nbytes
            rows.append({"row": k, "bytes": rb, "us": round(med, 2), "us_min": round(ts[0], 2), "us_max": round(ts[-1], 2),
                         "busbw_GBs": round(f * rb / (med * 1e-6) / 1e9, 1), "kernel": kern[k]})
        del x64, x128, o64, o128, xf, of, nz
        torch.cuda.empty_cache()
    res = {"n_gpus": world, **gpu_info(), "iters": "20 (<= 16 MB) / 5", "reps": args.reps, "verified": ok, "rows": rows}
    # c64 SUM over the f32 control, and PROD over SUM, per size (median times)
    by = {(r["row"], r["bytes"]): r["us"] for r in rows}
    res["c64_sum_over_f32_control"] = {b: round(by[("allreduce_c64_sum", b)] / by[("allreduce_f32_sum_control", b)], 3) for b in SIZES if ("allreduce_c64_sum", b) in by}
    res["c64_prod_over_c64_sum"] = {b: round(by[("allreduce_c64_prod", b)] / by[("allreduce_c64_sum", b)], 3) for b in SIZES if ("allreduce_c64_prod", b) in by}
    if rank == 0:
        txt = json.dumps(res, indent=1)
        if args.out:
            with open(args.out, "w") as fh:
                fh.write(txt + "\n")
        print(txt, flush=True)
        print("COMPLEX_BENCH_OK" if ok else "COMPLEX_BENCH_FAIL", flush=True)
    comm_shm.destroy()
    comm.destroy()
    dist.destroy_process_group()
    return 0 if ok else 1


if __name__ == "__main__":
    sys.exit(main())
