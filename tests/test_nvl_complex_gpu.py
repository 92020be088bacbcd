"""Complex reductions (float32_complex / float64_complex) on the tl/nvl kernels on a real GPU.

N emulated ranks share cuda:0 as in tests/test_nvl_gpu.py; the multi-process runs (in-switch kernels, zero-copy over CUDA IPC,
symmetric memory, tl/nccl, the torch backend) go through tests/complex_worker.py under torchrun.  Inputs are Gaussian integers
with parts in [-2, 2]: sums and products of up to 8 of them are exact in float32, so every result is compared exactly."""
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
sys.path.insert(0, os.path.join(ROOT, "tests"))
from complex_worker import expected, gauss  # noqa: E402

CUDA = U.UCC_MEMORY_TYPE_CUDA
TDT = {"float32_complex": torch.complex64, "float64_complex": torch.complex128}
ZC = {"UCC_TL_NVL_ZCOPY": "y", "UCC_TL_NVL_ZCOPY_THRESH": "0"}
NOZC = {"UCC_TL_NVL_ZCOPY": "n"}
ENV = {"UCC_TL_NVL_MAX_BLOCKS": "4", "UCC_TL_NVL_TIMEOUT": "5s", "UCC_TL_NVL_SYMMETRIC_SIZE": "8Mb",
       "UCC_TL_NVL_P2P_TIMEOUT": "20s"}
ALGS = ["oneshot", "twoshot", "twoshot-zcopy", "ring", "rhd"]


def need_cuda():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    torch.cuda.set_device(0)


def cargs(coll, src, dst, dt, **kw):
    kw.setdefault("count_src", src.numel() if src is not None else 0)
    kw.setdefault("count_dst", dst.numel() if dst is not None else 0)
    return coll_args(coll, dt=dt, mem_type=CUDA, src_ptr=src.data_ptr() if src is not None else None,
                     dst_ptr=dst.data_ptr() if dst is not None else None, **kw)


def run(team, args):
    req = team.coll(args)
    st = req.run()
    req.finalize()
    assert st == U.UCC_OK, U.status_str(st)
    torch.cuda.synchronize()


def alg_env(alg):
    name = alg.split("-")[0]
    colls = ["allreduce", "reduce_scatter", "reduce_scatterv"] + (["reduce"] if name == "twoshot" else [])
    env = dict(ENV, UCC_TL_NVL_TUNE="#".join(f"{c}:cuda:inf:@{name}" for c in colls),
               UCC_TL_NVL_ALLREDUCE_ONESHOT_THRESH="1M" if name == "oneshot" else "0")
    env.update(ZC if alg.endswith("zcopy") else NOZC)
    return env


@pytest.fixture(scope="module", params=ALGS)
def alg_job(request):
    need_cuda()
    job = UccJob(8, env=alg_env(request.param))
    teams = {n: job.create_team(range(n)) for n in (2, 3, 4, 8)}
    yield request.param, teams
    job.cleanup()


@pytest.mark.parametrize("n", [2, 3, 4, 8])
@pytest.mark.parametrize("dt", ["float32_complex", "float64_complex"])
@pytest.mark.parametrize("op", ["sum", "avg", "prod"])
def test_complex_reductions(alg_job, n, dt, op):
    alg, teams = alg_job
    if alg == "rhd" and n == 3:
        pytest.skip("recursive halving / doubling pairs ranks by xor: power-of-two teams")
    team, tdt = teams[n], TDT[dt]
    counts = (1, 7, 4097, 40001) + ((700001,) if alg.startswith("twoshot") else ())   # 700001 x c128: several heap rounds
    for count in counts:
        xs = [gauss(count, 31 * r + count, tdt).cuda() for r in range(n)]
        dst = [torch.zeros(count, dtype=tdt, device="cuda") for _ in range(n)]
        run(team, [cargs("allreduce", xs[r], dst[r], dt, op=op) for r in range(n)])
        exp = expected(op, xs)
        for r in range(n):
            assert torch.equal(dst[r].cpu(), exp), (alg, "allreduce", n, dt, op, count, r)
    for blk in (1, 7, 4097):
        xs = [gauss(blk * n, 17 * r + blk, tdt).cuda() for r in range(n)]
        exp = expected(op, xs)
        dst = [torch.zeros(blk, dtype=tdt, device="cuda") for _ in range(n)]
        run(team, [cargs("reduce_scatter", xs[r], dst[r], dt, op=op) for r in range(n)])
        for r in range(n):
            assert torch.equal(dst[r].cpu(), exp[r * blk:(r + 1) * blk]), (alg, "reduce_scatter", n, dt, op, blk, r)
        cnts = [blk + 3 * r for r in range(n)]
        offs = np.concatenate([[0], np.cumsum(cnts)[:-1]])
        xv = [gauss(sum(cnts), 5 * r + blk, tdt).cuda() for r in range(n)]
        ev = expected(op, xv)
        dv = [torch.zeros(cnts[r], dtype=tdt, device="cuda") for r in range(n)]
        run(team, [cargs("reduce_scatterv", xv[r], dv[r], dt, op=op, dst_counts=cnts, dst_displs=offs) for r in range(n)])
        for r in range(n):
            assert torch.equal(dv[r].cpu(), ev[offs[r]:offs[r] + cnts[r]]), (alg, "reduce_scatterv", n, dt, op, blk, r)
    # reduce has no one-shot / ring / rhd kernel: those teams run it on the default (two-shot) selection of the same TL
    root = n - 1
    xs = [gauss(9001, 3 * r, tdt).cuda() for r in range(n)]
    res = torch.zeros(9001, dtype=tdt, device="cuda")
    run(team, [cargs("reduce", xs[r], res if r == root else None, dt, op=op, root=root, count_dst=9001 if r == root else 0) for r in range(n)])
    assert torch.equal(res.cpu(), expected(op, xs)), (alg, "reduce", n, dt, op)


@pytest.mark.parametrize("n", [2, 3, 4, 8])
def test_c64_sum_is_f32_sum(alg_job, n):
    """float32_complex SUM runs the float32 kernels on the same bytes: results are bitwise equal on random values"""
    alg, teams = alg_job
    if alg == "rhd" and n == 3:
        pytest.skip("power-of-two teams only")
    team = teams[n]
    for count in (5, 4097, 100003):
        g = torch.Generator().manual_seed(count + n)
        xs = [torch.randn(count, generator=g, dtype=torch.complex64).cuda() for _ in range(n)]
        dc = [torch.zeros(count, dtype=torch.complex64, device="cuda") for _ in range(n)]
        df = [torch.zeros(2 * count, dtype=torch.float32, device="cuda") for _ in range(n)]
        run(team, [cargs("allreduce", xs[r], dc[r], "float32_complex") for r in range(n)])
        run(team, [cargs("allreduce", torch.view_as_real(xs[r]).reshape(-1), df[r], "float32") for r in range(n)])
        for r in range(n):
            assert torch.equal(torch.view_as_real(dc[r]).reshape(-1), df[r]), (alg, n, count, r)


def test_unaligned_and_persistent_inplace(alg_job):
    alg, teams = alg_job
    n, count = 4, 3001
    team = teams[n]
    # float32_complex one element into an allocation: 8-byte aligned source and destination (the guarded element path)
    for op in ("sum", "prod"):
        xb = [torch.zeros(count + 1, dtype=torch.complex64, device="cuda") for _ in range(n)]
        db = [torch.zeros(count + 1, dtype=torch.complex64, device="cuda") for _ in range(n)]
        xs = [gauss(count, r + 40, torch.complex64) for r in range(n)]
        for r in range(n):
            xb[r][1:].copy_(xs[r])
        run(team, [cargs("allreduce", xb[r][1:], db[r][1:], "float32_complex", op=op) for r in range(n)])
        for r in range(n):
            assert torch.equal(db[r][1:].cpu(), expected(op, xs)), (alg, "unaligned", op, r)
            assert db[r][0].item() == 0
    req = team.coll([cargs("allreduce", None, xb[r][1:], "float32_complex", op="avg", inplace=True, persistent=True) for r in range(n)])
    for it in range(3):
        xs = [gauss(count, 10 * it + r, torch.complex64) for r in range(n)]
        for r in range(n):
            xb[r][1:].copy_(xs[r])
        torch.cuda.synchronize()
        assert req.run() == U.UCC_OK
        torch.cuda.synchronize()
        for r in range(n):
            assert torch.equal(xb[r][1:].cpu(), expected("avg", xs)), (alg, "persistent", it, r)
    req.finalize()


def test_trace_shows_tl_nvl():
    """every complex allreduce / reduce_scatter(v) / reduce, default selection and forced algorithms, is initialised on tl/nvl;
    a complex MAX is declined at init on a tl/nvl-only team"""
    need_cuda()
    env = dict(os.environ, PYTHONPATH=ROOT)
    for k in ("UCC_TL_NVL_TUNE", "UCC_TLS"):
        env.pop(k, None)
    out = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "complex_worker.py"), "trace"], env=env, capture_output=True, text=True, timeout=600)
    log = out.stdout + out.stderr
    assert out.returncode == 0 and "COMPLEX_WORKER_OK" in out.stdout, log[-4000:]
    lines = [ln for ln in log.splitlines() if "coll_init:" in ln and re.search(r"float(32|64)_complex", ln, re.I)]
    assert len(lines) > 100, log[-3000:]
    bad = [ln for ln in lines if "{TL_NVL}" not in ln]
    assert not bad, bad[:5]


def _torchrun(n, mode, port, extra_env=None):
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={n}", "--master-addr", "127.0.0.1",
           "--master-port", str(port), os.path.join(ROOT, "tests", "complex_worker.py"), mode]
    env = dict(os.environ, PYTHONPATH=ROOT)
    for k in ("UCC_TL_NVL_TUNE", "UCC_TLS"):
        env.pop(k, None)
    env.update(extra_env or {})
    out = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=600)
    assert "COMPLEX_WORKER_OK" in out.stdout, out.stdout[-3000:] + out.stderr[-4000:]


def _gpu_counts():
    n = torch.cuda.device_count() if torch.cuda.is_available() else 0
    return sorted({2, n}) if n >= 2 else []


@pytest.mark.parametrize("which", ["2", "all"])
def test_multiproc_nvl(which):
    """forced @nvls / @nvls_pipe (c64 SUM / AVG in the switch), zero-copy over CUDA IPC, symm_empty() in place"""
    counts = _gpu_counts()
    if not counts or (which == "all" and counts[-1] == 2):
        pytest.skip("needs >= 2 GPUs" if not counts else "only 2 GPUs")
    _torchrun(2 if which == "2" else counts[-1], "nvl", 29810 if which == "2" else 29811)


def test_multiproc_nccl_complex():
    """UCC_TLS=nccl,self: complex SUM / AVG as real vectors twice as long, PROD declined"""
    if not _gpu_counts():
        pytest.skip("needs >= 2 GPUs")
    _torchrun(2, "nccl", 29812, {"UCC_TLS": "nccl,self"})


def test_multiproc_torch_backend_complex():
    """reduce_scatter_tensor / reduce_scatter / reduce on complex64 through the ucc_b200 torch.distributed backend"""
    if not _gpu_counts():
        pytest.skip("needs >= 2 GPUs")
    _torchrun(2, "torch", 29813)
