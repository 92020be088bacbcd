#!/usr/bin/env python3
"""Headline benchmark: ucc_perftest-style allreduce bus bandwidth / latency on CUDA buffers.

    python bench.py --gpus N --steps K --warmup W [--impl reference]

Metric (BASELINE.json): allreduce bus bandwidth at 1 GiB float32 on CUDA buffers plus a 1 KB..1 GiB sweep with latency.
Per-GPU bus bandwidth = S/t * 2(N-1)/N (reference formula, tools/perf/ucc_pt_coll_allreduce.cc:84-93); `value` is the
whole-job aggregate, i.e. the sum over the N GPUs (N * busbw; `busbw_per_gpu_GBps` carries the familiar per-GPU figure, the one
to hold against 900 GB/s per direction).  One rank per GPU (torchrun for N > 1).  A "step" is one allreduce of the headline
size on ordinary cudaMalloc buffers:

  --impl ours       through the library's public C API (ucc_collective_init / triggered_post / test / finalize), executed by
                    one fused tl/nvl NVLink kernel
  --impl reference  the reference's own tl/cuda NVLS kernels compiled unmodified from an openucx/ucc checkout and driven through
                    its stock host sequence (oracle/ref_arm), next to tl/nccl's ncclAllReduce - what its score map falls back to
                    for messages above NVLS_SYMMETRIC_SIZE; the better of the two is the reference's value

Device time = CUDA events on the launching stream, max over ranks.  The result vector is verified in full against a
seeded, rank-dependent, non-constant input (exact integer-valued floats, so the comparison is bitwise)."""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--size", type=int, default=1 << 30, help="headline message size in bytes")
    ap.add_argument("--dtype", default="float32")
    ap.add_argument("--e2e-chunks", type=int, default=0,
                    help="end-to-end step of --impl ours: number of chunks whose H2D copy overlaps the previous chunk's allreduce "
                         "(ops.all_reduce_from_host); 0 = library default, 1 = no overlap")
    ap.add_argument("--symm", default="", help="put the device buffers into a symmetric user region of this size, e.g. 3G "
                    "(Communicator(symm_size=...).symm_empty, the ncclMemAlloc analogue): in-place in-switch allreduce")
    ap.add_argument("--no-sweep", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-nccl", action="store_true")
    ap.add_argument("--out", default="")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="after the timed steps write what the last timed step of --impl ours computed to DIR/<name>_rank<r>.npy "
                         "(float32, float64 for --dtype float64; a fixed seeded sample of each vector, at most 32 MB in all): the inputs are "
                         "the same from run to run, so two builds can be compared output for output")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "ours":
        ap.error("--dump-outputs records the timed path of --impl ours")
    return a


class ClockSampler:
    """nvidia-smi sampling of SM clocks / throttle reasons during the timed region."""
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu):
        self.gpu, self.rows, self.proc = gpu, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm = sorted(int(r[0]) for r in self.rows if r and r[0].isdigit())
        mx = [int(r[1]) for r in self.rows if len(r) > 1 and r[1].isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 6 for i in range(4) if r[2 + i].lower().startswith("active")})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons, "samples": len(self.rows)}


# ---------------------------------------------------------------------------------------------------------------------
# data: rank-dependent, non-constant, integer valued (<= 19 per rank, <= 152 summed over 8 ranks: exact even in bf16)
# ---------------------------------------------------------------------------------------------------------------------
def pattern(torch, cnt, r, dt, dev, out=None):
    CH = 1 << 26
    out = torch.empty(cnt, dtype=dt, device=dev) if out is None else out
    for o in range(0, cnt, CH):
        n = min(CH, cnt - o)
        i = torch.arange(o, o + n, device=dev, dtype=torch.int64)
        out[o:o + n] = (((i + 17 * r) % 13) + r).to(dt)
    return out


DUMP_BYTES = 16 << 20           # per dumped vector, summed over the ranks


def dump_output(torch, d, name, x, rank, N):
    """DIR/<name>_rank<rank>.npy: the whole of `x` when it fits DUMP_BYTES / N, else its first and last 64 Ki elements plus
    positions in between drawn from a fixed seed (the same for every run of the same size), in ascending order"""
    import numpy as np
    out_dt = torch.float64 if x.dtype == torch.float64 else torch.float32
    x = x.reshape(-1)
    k = DUMP_BYTES // (out_dt.itemsize * N)
    if x.numel() > k:
        n, edge = x.numel(), min(1 << 16, k // 4)
        mid = torch.randint(edge, n - edge, (k - 2 * edge,), generator=torch.Generator().manual_seed(20240917))
        idx = torch.cat([torch.arange(edge), mid, torch.arange(n - edge, n)]).unique()
        x = x[idx.to(x.device)]
    os.makedirs(d, exist_ok=True)
    np.save(os.path.join(d, f"{name}_rank{rank}.npy"), x.to(out_dt).cpu().numpy())


def expected_sum(torch, cnt, N, dt, dev):
    CH = 1 << 26
    exp = torch.empty(cnt, dtype=dt, device=dev)
    for o in range(0, cnt, CH):
        n = min(CH, cnt - o)
        i = torch.arange(o, o + n, device=dev, dtype=torch.int64)
        acc = torch.zeros(n, dtype=torch.int64, device=dev)
        for r in range(N):
            acc += ((i + 17 * r) % 13) + r
        exp[o:o + n] = acc.to(dt)
    return exp


class Bench:
    """what both arms share: sizes, timing, verification, JSON.  An arm provides
         ar(src, dst, stream) -> handle      enqueue one allreduce on `stream` (stream ordered)
         settle(handles)                     host-side completion / cleanup of those allreduces (after the timed region)"""

    def __init__(self, a):
        import torch
        import torch.distributed as dist
        self.a, self.torch, self.dist = a, torch, dist
        self.rank = int(os.environ.get("RANK", "0"))
        self.N = int(os.environ.get("WORLD_SIZE", "1"))
        lrank = int(os.environ.get("LOCAL_RANK", str(self.rank)))
        torch.cuda.set_device(lrank % torch.cuda.device_count())
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("MASTER_PORT", "29555")
        if not dist.is_initialized():
            dist.init_process_group(backend="cpu:gloo,cuda:nccl", rank=self.rank, world_size=self.N)
        if self.N != a.gpus and self.rank == 0:
            print(f"warning: --gpus {a.gpus} but WORLD_SIZE {self.N}", file=sys.stderr)
        self.dev = torch.device("cuda", torch.cuda.current_device())
        self.dt = getattr(torch, a.dtype)
        self.esz = torch.empty(0, dtype=self.dt).element_size()
        self.stream = torch.cuda.Stream()

    def maxr(self, x):
        if self.N == 1:
            return x
        t = self.torch.tensor([x], dtype=self.torch.float64)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return t.item()

    def all_ok(self, ok):
        if self.N == 1:
            return bool(ok)
        t = self.torch.tensor([1.0 if ok else 0.0], dtype=self.torch.float64)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MIN)
        return bool(t.item() > 0.5)

    def barrier(self):
        if self.N > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def busbw(self, nbytes, us):
        """per-GPU bus bandwidth, GB/s.  N = 1 has no bus: plain S/t of the local copy is reported and flagged."""
        f = 2.0 * (self.N - 1) / self.N if self.N > 1 else 1.0
        return nbytes / us / 1e3 * f

    def time_arm(self, ar, settle, nbytes, iters, warm, alloc=None, dump=None):
        """device time per allreduce (us, max over ranks) of `iters` allreduces posted back to back on one stream, and whether
        the WHOLE result vector of the last one equals the exact expected sum on every rank; `dump` names the file that result
        goes to under --dump-outputs"""
        torch = self.torch
        cnt = nbytes // self.esz
        mk = alloc or (lambda c: torch.empty(c, dtype=self.dt, device=self.dev))
        src = pattern(torch, cnt, self.rank, self.dt, self.dev, out=mk(cnt))
        dst = mk(cnt).zero_()
        # the buffers were produced on the default stream and are used on a side stream: without this the first collectives run
        # while the producer kernels are still queued (and the caching allocator hands the producer's temporaries out as `dst`)
        torch.cuda.synchronize()
        with torch.cuda.stream(self.stream):
            hs = [ar(src, dst, self.stream) for _ in range(warm)]
            settle(hs)
            self.barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            dst.zero_()
            e0.record(self.stream)
            hs = [ar(src, dst, self.stream) for _ in range(iters)]
            hs = self.flush(hs)
            e1.record(self.stream)
            settle(hs)
            torch.cuda.synchronize()
        us = e0.elapsed_time(e1) * 1e3 / iters
        exp = expected_sum(torch, cnt, self.N, self.dt, self.dev)
        ok = bool(torch.equal(dst, exp))
        if dump and self.a.dump_outputs:
            dump_output(torch, self.a.dump_outputs, dump, dst, self.rank, self.N)
        del src, dst, exp
        return self.maxr(us), self.all_ok(ok)

    def flush(self, hs):
        return hs

    def time_e2e(self, step_fn, nbytes):
        """end to end: every step copies its input host (pinned) -> device, all-reduces, and reads a result word back"""
        for _ in range(max(3, min(self.a.warmup, 5))):
            step_fn()
        self.barrier()
        t0 = time.perf_counter()
        for _ in range(self.a.steps):
            last = step_fn()
        self.torch.cuda.synchronize()
        us = self.maxr((time.perf_counter() - t0) * 1e6 / self.a.steps)
        return us, last


# ---------------------------------------------------------------------------------------------------------------------
def run_ours(a):
    B = Bench(a)
    torch, dist, N = B.torch, B.dist, B.N
    from ucc_b200.dist import Communicator
    from ucc_b200 import ops
    comm = Communicator(symm_size=a.symm) if a.symm else Communicator()
    use_symm = bool(a.symm) and comm.symm_region() is not None

    def alloc(cnt):
        return comm.symm_empty(cnt, B.dt)

    def ar(src, dst, stream):
        r = comm.allreduce_init(src, dst)                    # ucc_collective_init
        r.post_on_stream(stream, wait_posted=False)          # ucc_collective_triggered_post
        return r

    def flush(hs):
        for r in hs:
            r.wait_posted()                                  # zero-copy kernels enter the stream once the peers' buffers are mapped
        return hs
    B.flush = flush

    def settle(hs):
        for r in hs:
            r.wait_posted()
        for r in hs:
            r.wait()                                         # ucc_collective_test + ucc_context_progress
            r.finalize()                                     # ucc_collective_finalize

    def time_ours(nbytes, iters, warm, dump=None):
        if use_symm:
            comm.symm_reset()
        return B.time_arm(ar, settle, nbytes, iters, warm, alloc if use_symm else None, dump)

    def time_nccl(nbytes, iters, warm):
        if N == 1 or a.no_nccl:
            return None
        x = torch.ones(nbytes // B.esz, dtype=B.dt, device=B.dev)
        with torch.cuda.stream(B.stream):
            for _ in range(warm):
                dist.all_reduce(x)
            B.barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(B.stream)
            for _ in range(iters):
                dist.all_reduce(x)
            e1.record(B.stream)
            torch.cuda.synchronize()
        del x
        return B.maxr(e0.elapsed_time(e1) * 1e3 / iters)

    S = a.size
    sampler = ClockSampler(torch.cuda.current_device())
    sampler.start()
    us, ok = time_ours(S, a.steps, a.warmup, dump="allreduce")
    headline_alg = comm.request_info_last()
    value = B.busbw(S, us)
    nccl_us = time_nccl(S, a.steps, a.warmup)

    e2e = None
    if not a.no_e2e:
        cnt = S // B.esz
        host = pattern(torch, cnt, B.rank, B.dt, "cpu").pin_memory()
        if use_symm:
            comm.symm_reset()
        mk = alloc if use_symm else (lambda c: torch.empty(c, dtype=B.dt, device=B.dev))
        src, dst = mk(cnt), mk(cnt)
        out = torch.empty(16, dtype=B.dt).pin_memory()
        torch.cuda.synchronize()
        chunks = a.e2e_chunks or None

        def step():
            with torch.cuda.stream(B.stream):
                # public API: H2D of this step's input from pinned memory (copy engine) overlapped chunk by chunk with the
                # NVLink allreduce kernels of the chunks that already arrived; the whole input crosses PCIe, the whole vector is reduced
                ops.all_reduce_from_host(host, dst, staging=src, comm=comm, chunks=chunks, stream=B.stream)
                out.copy_(dst[:16], non_blocking=True)             # D2H read of the result
                B.stream.synchronize()
            return out[0].item()

        e2e_us, last = B.time_e2e(step, S)
        exp = expected_sum(torch, cnt, N, B.dt, B.dev)
        e2e_ok = B.all_ok(bool(torch.equal(dst, exp)))
        if a.dump_outputs:
            dump_output(torch, a.dump_outputs, "all_reduce_from_host", dst, B.rank, N)
        e2e = {"value": round(N * B.busbw(S, e2e_us), 3), "busbw_per_gpu_GBps": round(B.busbw(S, e2e_us), 3), "unit": "GB/s", "h2d_bytes_per_step": S,
               "d2h_bytes_per_step": 16 * B.esz, "us_per_step": round(e2e_us, 1), "chunks": ops.last_from_host_chunks(), "correct": e2e_ok,
               "api": "ucc_b200.ops.all_reduce_from_host (pinned host -> device copy pipelined with the tl/nvl allreduce kernels)"}
        del host, src, dst, exp
    clocks = sampler.stop()

    sweep = []
    if not a.no_sweep:
        nb = 1 << 10
        while nb <= (1 << 30):
            iters = 50 if nb <= (1 << 22) else (20 if nb <= (1 << 26) else 8)
            u, okk = time_ours(nb, iters, 5)
            nu = time_nccl(nb, iters, 5)
            sweep.append({"bytes": nb, "us": round(u, 2), "busbw": round(B.busbw(nb, u), 2), "ok": okk, "alg": comm.request_info_last(),
                          "nccl_us": round(nu, 2) if nu else None, "nccl_busbw": round(B.busbw(nb, nu), 2) if nu else None})
            nb <<= 2

    res = result_json(B, a, "ours", value, us, ok, clocks, a.steps, e2e, sweep)
    res["config"]["algorithm"] = f"tl/nvl fused kernel chosen by coll_score: {headline_alg}"
    res["config"]["symmetric_memory"] = use_symm
    res["nccl_same_box"] = {"us": round(nccl_us, 2), "busbw_per_gpu_GBps": round(B.busbw(S, nccl_us), 2)} if nccl_us else None
    comm.destroy()
    finish(B, a, res)
    return 0


# ---------------------------------------------------------------------------------------------------------------------
def run_reference(a):
    lib = os.path.join(ROOT, "oracle", "_ref", "libref_tlcuda.so")
    if not os.path.exists(lib):
        print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref/libref_tlcuda.so is not built (run oracle/ref_arm/build.sh with REFERENCE_DIR set to an openucx/ucc checkout)"}))
        return 0
    sys.path.insert(0, os.path.join(ROOT, "oracle", "ref_arm"))
    B = Bench(a)
    torch, dist, N = B.torch, B.dist, B.N
    S = a.size
    STOCK_SYMM = 512 << 20                      # reference default UCC_TL_CUDA_NVLS_SYMMETRIC_SIZE (tl_cuda.c:55)
    tlcuda = None

    def make_tlcuda():
        # created AFTER tl/nccl was measured: its 8 x (symmetric size) multicast-bound region must not compete with NCCL's own
        # NVLS resources while NCCL is being timed (each transport gets the box for itself, as in separate ucc_perftest runs)
        from ref_arm import RefTlCuda
        # the headline message is larger than the stock symmetric size: the stock build hands it to tl/nccl.  The region is
        # sized to fit the headline too so that tl/cuda's NVLS path is ALSO measured there (UCC_TL_CUDA_NVLS_SYMMETRIC_SIZE raised).
        symm = max(STOCK_SYMM, (S + 16 * N - 1) // (16 * N) * (16 * N))
        t = RefTlCuda(B.rank, N, torch.cuda.current_device(), symm_size=symm, slots=8, sm_count=4, threads=1024)
        return t if t.ok else None

    def settle(hs):
        pass

    def ar_self(src, dst, stream):              # tl/self: team of one
        dst.copy_(src, non_blocking=True)

    def ar_tlcuda(src, dst, stream):
        st = tlcuda.allreduce(src, dst, stream)
        if st != 0:
            raise RuntimeError(f"ref_allreduce failed: {st}")

    def time_nccl(nbytes, iters, warm):
        cnt = nbytes // B.esz
        src = pattern(torch, cnt, B.rank, B.dt, B.dev)
        x = src.clone()
        torch.cuda.synchronize()
        with torch.cuda.stream(B.stream):
            for _ in range(warm):
                dist.all_reduce(x)
            x.copy_(src)
            dist.all_reduce(x)
            torch.cuda.synchronize()
            ok = bool(torch.equal(x, expected_sum(torch, cnt, N, B.dt, B.dev)))
            B.barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(B.stream)
            for _ in range(iters):
                dist.all_reduce(x)
            e1.record(B.stream)
            torch.cuda.synchronize()
        del x, src
        return B.maxr(e0.elapsed_time(e1) * 1e3 / iters), B.all_ok(ok)

    sampler = ClockSampler(torch.cuda.current_device())
    sampler.start()
    arms = {}
    nccl_sweep = {}
    if N == 1:
        u, okk = B.time_arm(ar_self, settle, S, a.steps, a.warmup)
        arms["tl_self(cudaMemcpyAsync)"] = (u, okk)
    else:
        if not a.no_nccl:
            arms["tl_nccl(ncclAllReduce)"] = time_nccl(S, a.steps, a.warmup)
            if not a.no_sweep:
                nb = 1 << 10
                while nb <= (1 << 30):
                    nccl_sweep[nb] = time_nccl(nb, 50 if nb <= (1 << 22) else (20 if nb <= (1 << 26) else 8), 5)
                    nb <<= 2
        tlcuda = make_tlcuda()
        if tlcuda is not None:
            arms["tl_cuda_nvls(stock kernels, 4x1024, NVLS_SYMMETRIC_SIZE raised to fit)" if S > STOCK_SYMM else "tl_cuda_nvls(stock kernels, 4x1024)"] = \
                B.time_arm(ar_tlcuda, settle, S, a.steps, a.warmup)
    best = min(arms, key=lambda k: arms[k][0])
    us, ok = arms[best]
    value = B.busbw(S, us)
    stock = "tl_self" if N == 1 else ("tl_nccl" if (S > STOCK_SYMM or tlcuda is None) else "tl_cuda_nvls")

    sweep = []
    if not a.no_sweep and N > 1:
        nb = 1 << 10
        while nb <= (1 << 30):
            iters = 50 if nb <= (1 << 22) else (20 if nb <= (1 << 26) else 8)
            row = {"bytes": nb}
            if tlcuda is not None and nb >= 16 * N:
                u, okk = B.time_arm(ar_tlcuda, settle, nb, iters, 5)
                row.update({"tl_cuda_us": round(u, 2), "tl_cuda_busbw": round(B.busbw(nb, u), 2), "tl_cuda_ok": okk, "tl_cuda_stock_selectable": nb <= STOCK_SYMM})
            if nb in nccl_sweep:
                u, okk = nccl_sweep[nb]
                row.update({"nccl_us": round(u, 2), "nccl_busbw": round(B.busbw(nb, u), 2)})
            sweep.append(row)
            nb <<= 2

    if tlcuda is not None and not best.startswith("tl_cuda"):
        tlcuda.destroy()          # the end-to-end steps below run tl/nccl: give NCCL the box back
        tlcuda = None


    e2e = None
    if not a.no_e2e:
        cnt = S // B.esz
        host = pattern(torch, cnt, B.rank, B.dt, "cpu").pin_memory()
        src = torch.empty(cnt, dtype=B.dt, device=B.dev)
        dst = torch.empty(cnt, dtype=B.dt, device=B.dev)
        out = torch.empty(16, dtype=B.dt).pin_memory()
        torch.cuda.synchronize()
        use = best

        def step():
            with torch.cuda.stream(B.stream):
                if use.startswith("tl_nccl"):
                    dst.copy_(host, non_blocking=True)             # H2D of this step's input from pinned memory
                    dist.all_reduce(dst)
                else:
                    src.copy_(host, non_blocking=True)
                    (ar_self if N == 1 else ar_tlcuda)(src, dst, B.stream)
                out.copy_(dst[:16], non_blocking=True)             # D2H read of the result
                B.stream.synchronize()
            return out[0].item()
        e2e_us, _ = B.time_e2e(step, S)
        exp = expected_sum(torch, cnt, N, B.dt, B.dev)
        e2e = {"value": round(N * B.busbw(S, e2e_us), 3), "busbw_per_gpu_GBps": round(B.busbw(S, e2e_us), 3), "unit": "GB/s", "h2d_bytes_per_step": S,
               "d2h_bytes_per_step": 16 * B.esz, "us_per_step": round(e2e_us, 1), "correct": B.all_ok(bool(torch.equal(dst, exp))), "transport": use}
        del host, src, dst, exp
    clocks = sampler.stop()
    res = result_json(B, a, "reference", value, us, ok, clocks, a.steps * (3 if best.startswith("tl_cuda") else 1), e2e, sweep)
    res["reference_class"] = best
    res["reference_stock_selection"] = stock
    res["reference_arms"] = {k: {"us": round(v[0], 2), "busbw_per_gpu_GBps": round(B.busbw(S, v[0]), 2), "correct": v[1]} for k, v in arms.items()}
    res["config"]["algorithm"] = "reference openucx/ucc: tl/cuda NVLS kernels (unmodified, oracle/_ref) through the stock memcpy-kernel-memcpy sequence; " \
                                 "tl/nccl = ncclAllReduce; value = the faster of the two at the headline size"
    res["gpu_launches_note"] = "launches of the reference's kernels / copies in the timed region (none of the repo's own code is loaded)"
    if tlcuda is not None:
        tlcuda.destroy()
    finish(B, a, res)
    return 0


def result_json(B, a, impl, busbw, us, ok, clocks, launches, e2e, sweep):
    N, S = B.N, a.size
    res = {
        "metric": "allreduce_busbw_GBps", "value": round(N * busbw, 3), "unit": "GB/s", "n_gpus": N, "steps": a.steps, "warmup": a.warmup,
        "ms_per_step": round(us / 1e3, 5), "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": a.dtype,
        "data": "synthetic (seeded rank-dependent integer-valued pattern), CUDA device buffers (cudaMalloc)", "impl": impl,
        "busbw_per_gpu_GBps": round(busbw, 3),
        "metric_note": "value = N x per-GPU bus bandwidth (whole-job aggregate of S/t*2(N-1)/N); per-GPU figure in busbw_per_gpu_GBps. "
                       "N=1 has no bus: S/t of the local device copy is reported, it is not comparable with N>1",
        "config": {"model": "ucc_perftest allreduce", "collective": "allreduce", "op": "sum", "message_bytes": S, "global_batch": S * N,
                   "seq_len": S // B.esz, "parallelism": f"dp{N}", "timing": "cuda events on the posting stream, max over ranks",
                   "l2": "message (1 GiB) is larger than the 126 MB L2", "memtype": "cuda", "inplace": False},
        "correct": bool(ok), "verified": "whole vector, bitwise, every rank", "clocks": clocks, "gpu_launches": launches,
        "latency_us": round(us, 2), "roofline_frac_of_900": round(busbw / 900.0, 4) if N > 1 else None,
        "roofline_frac_of_hbm_copy": round(2.0 * busbw / peak_copy_gbps(), 4) if N == 1 else None,
    }
    if e2e:
        res["e2e"] = e2e
    if sweep:
        res["sweep"] = sweep
    return res


def peak_copy_gbps():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        for k in ("hbm_gbs", "copy_GBps", "hbm_copy_GBps", "copy_bandwidth_GBps"):
            if k in p:
                return float(p[k])
        for v in p.values():
            if isinstance(v, dict):
                for k2, v2 in v.items():
                    if "copy" in k2.lower() and isinstance(v2, (int, float)):
                        return float(v2)
    except Exception:
        pass
    return 6478.3


def finish(B, a, res):
    if B.rank == 0:
        print(json.dumps(res), flush=True)
        if a.out:
            with open(a.out, "w") as f:
                json.dump(res, f, indent=1)
    if B.dist.is_initialized():
        B.dist.destroy_process_group()


def main():
    a = parse()
    return run_reference(a) if a.impl == "reference" else run_ours(a)


if __name__ == "__main__":
    sys.exit(main())
