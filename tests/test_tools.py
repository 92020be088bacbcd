"""ucc_info and ucc_perftest (reference tools/info/ucc_info.c, tools/perf/*): CLI behaviour on host memory."""
import os
import re
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "ucc_b200", "bin")


def _need(tool):
    p = os.path.join(BIN, tool)
    if not os.path.exists(p):
        subprocess.run(["make", "-C", ROOT, "-j8", "core", "tools"], capture_output=True)
    if not os.path.exists(p):
        pytest.skip(f"{tool} not built")
    return p


def test_ucc_info_flags():
    exe = _need("ucc_info")
    out = subprocess.run([exe, "-v"], capture_output=True, text=True, timeout=60).stdout
    assert re.search(r"1\.\d+", out)
    out = subprocess.run([exe, "-c", "-a"], capture_output=True, text=True, timeout=60).stdout
    assert "UCC_CLS" in out and "UCC_TL_SHM_TUNE" in out
    out = subprocess.run([exe, "-A"], capture_output=True, text=True, timeout=60).stdout
    assert "sra_knomial" in out and "allreduce" in out.lower()
    out = subprocess.run([exe, "-s"], capture_output=True, text=True, timeout=60).stdout
    assert "shm" in out.lower()


def _perftest(args, n=2, port=29500):
    exe = _need("ucc_perftest")
    procs = []
    for r in range(n):
        env = dict(os.environ, RANK=str(r), WORLD_SIZE=str(n), MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), CUDA_VISIBLE_DEVICES="")
        procs.append(subprocess.Popen([exe] + args, env=env, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True))
    outs = [p.communicate(timeout=180) for p in procs]
    for p, (o, e) in zip(procs, outs):
        assert p.returncode == 0, e[-2000:] + o[-1000:]
    return outs[0][0]


def test_perftest_allreduce_host_sweep():
    out = _perftest(["-c", "allreduce", "-m", "host", "-b", "8", "-e", "4096", "-n", "20", "-w", "5", "-d", "float32", "-o", "sum"], port=29510)
    rows = [ln.split() for ln in out.splitlines() if re.match(r"^\s*\d+\s+\d+", ln)]
    assert len(rows) >= 8, out
    counts = [int(r[0]) for r in rows]
    assert counts[0] == 8 and counts[-1] >= 2048 and all(b == 2 * a for a, b in zip(counts, counts[1:]))
    full = _perftest(["-c", "allreduce", "-m", "host", "-b", "1024", "-e", "1024", "-n", "10", "-w", "2", "-F"], port=29511)
    assert "bandwidth" in full.lower() or "GB/s" in full, full


@pytest.mark.parametrize("coll", ["alltoall", "allgather", "bcast", "barrier", "reduce_scatter"])
def test_perftest_other_colls(coll):
    port = 29520 + hash(coll) % 50
    out = _perftest(["-c", coll, "-m", "host", "-b", "16", "-e", "256", "-n", "10", "-w", "2"], n=3, port=port)
    assert coll in out.lower()


def test_perftest_persistent_inplace_and_executor_ops():
    out = _perftest(["-c", "allreduce", "-m", "host", "-b", "64", "-e", "64", "-n", "10", "-w", "2", "-F", "-i", "-p"], port=29590)
    assert re.search(r"^\s*64\s", out, re.M)
    out = _perftest(["-c", "memcpy", "-m", "host", "-b", "1024", "-e", "1024", "-n", "10", "-w", "2"], n=1, port=29591)
    assert re.search(r"^\s*1024\s", out, re.M)


def test_profile_log_and_reader(tmp_path):
    """UCC_PROFILE_MODE=log,accum writes the .prof file at exit; tools/read_profile.py turns it into tables / a chrome trace
    (reference: UCS profile + ucx_read_profile, utils/profile/ucc_profile_on.h:34-96)."""
    import json
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    prof = tmp_path / "run.prof"
    code = (
        "import numpy as np\n"
        "from ucc_b200.harness import UccJob, coll_args\n"
        "j = UccJob(3); t = j.create_team()\n"
        "for k in range(5):\n"
        "    s = [np.full(256, r + 1.0, np.float32) for r in range(3)]; d = [np.zeros(256, np.float32) for _ in range(3)]\n"
        "    q = t.coll([coll_args('allreduce', s[r], d[r]) for r in range(3)]); assert q.run() == 0; q.finalize()\n"
        "    q = t.coll([coll_args('barrier') for r in range(3)]); assert q.run() == 0; q.finalize()\n"
        "j.cleanup()\n")
    env = dict(os.environ, PYTHONPATH=root, UCC_PROFILE_MODE="log,accum", UCC_PROFILE_FILE=str(prof))
    out = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=120)
    assert out.returncode == 0, out.stderr[-2000:]
    assert prof.exists()
    chrome = tmp_path / "t.json"
    r = subprocess.run([sys.executable, os.path.join(root, "tools", "read_profile.py"), str(prof), "--json", "--chrome", str(chrome)],
                       capture_output=True, text=True, timeout=60)
    assert r.returncode == 0, r.stderr
    rep = json.loads(r.stdout)
    names = {a["name"]: a for a in rep["accum"]}
    assert names["ucc_collective_init"]["count"] >= 30 and names["ucc_collective_post"]["count"] >= 30
    # 15 user allreduces + the service allreduces of team creation
    assert names["shm_allreduce_start"]["count"] == names["shm_allreduce_done"]["count"] >= 15
    assert rep["latency_us"]["shm_allreduce"]["n"] >= 15 and rep["latency_us"]["shm_barrier"]["n"] == 15
    assert rep["latency_us"]["shm_allreduce"]["min"] >= 0
    tr = json.loads(chrome.read_text())
    assert len(tr["traceEvents"]) == rep["n_log"] > 0
    txt = subprocess.run([sys.executable, os.path.join(root, "tools", "read_profile.py"), str(prof)], capture_output=True, text=True, timeout=60)
    assert "shm_allreduce" in txt.stdout and "ucc_collective_post" in txt.stdout


def test_install_and_consumer_exports(tmp_path):
    """`make install` + the pkg-config file and the CMake package a consumer of openucx/ucc expects (reference ucc.pc.in, cmake/*.in)"""
    prefix = str(tmp_path / "inst")
    r = subprocess.run(["make", "-C", ROOT, "install", f"PREFIX={prefix}"], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    pc = open(os.path.join(prefix, "lib", "pkgconfig", "ucc.pc")).read()
    assert "-lucc" in pc and prefix in pc
    assert os.path.exists(os.path.join(prefix, "lib", "cmake", "ucc", "ucc-config.cmake"))
    r = subprocess.run(["bash", os.path.join(ROOT, "tools", "test_consumer_export.sh"), prefix], capture_output=True, text=True, timeout=600)
    assert "CONSUMER_EXPORT_OK" in r.stdout, r.stdout[-2000:] + r.stderr[-2000:]


def test_reference_arm_builds_from_unmodified_reference_sources():
    """oracle/ref_arm/build.sh: the reference's NVLS kernels are copied byte for byte and compile with the two shim headers;
    bench.py --impl reference then reports through them.  tests/golden/ref_arm_sources.sha256 holds the sha256 of the reference
    sources the arm was written and measured against: with an openucx/ucc checkout in REFERENCE_DIR the arm is rebuilt from it,
    and an arm found in oracle/_ref must have been built from exactly those files."""
    golden = sorted(l for l in open(os.path.join(ROOT, "tests", "golden", "ref_arm_sources.sha256")).read().splitlines() if l)
    assert len(golden) == 9
    recipe = open(os.path.join(ROOT, "oracle", "ref_arm", "build.sh")).read()
    for line in golden:
        assert os.path.basename(line.split()[1]) in recipe, line
    # the arm never imports the repository's own package or libraries
    src = open(os.path.join(ROOT, "oracle", "ref_arm", "ref_arm.py")).read() + open(os.path.join(ROOT, "oracle", "ref_arm", "ref_harness.cpp")).read()
    assert "ucc_b200" not in src and "libucc" not in src
    out = os.path.join(ROOT, "oracle", "_ref")
    ref = os.environ.get("REFERENCE_DIR")
    if ref and os.path.isdir(os.path.join(ref, "src", "components", "tl", "cuda", "kernels")) and os.path.exists("/usr/local/cuda/bin/nvcc"):
        env = {k: v for k, v in os.environ.items() if k != "LD_PRELOAD"}   # (tools/run_asan.sh preloads libasan; nvcc does not survive that)
        r = subprocess.run(["bash", os.path.join(ROOT, "oracle", "ref_arm", "build.sh")], capture_output=True, text=True, timeout=900, env=env)
        assert r.returncode == 0, r.stdout[-1500:] + r.stderr[-1500:]
        assert sorted(l for l in open(os.path.join(out, "MANIFEST.ref.txt")).read().splitlines() if l) == golden, \
            "REFERENCE_DIR is not the reference version the arm was written against"
    if not os.path.exists(os.path.join(out, "libref_tlcuda.so")):
        return
    built = sorted(l for l in open(os.path.join(out, "MANIFEST.txt")).read().splitlines() if l)
    assert built == golden, "a reference source file was altered on its way into oracle/_ref"
    syms = subprocess.run(["nm", "-D", os.path.join(out, "libref_tlcuda.so")], capture_output=True, text=True).stdout
    for s in ("post_allreduce_kernel", "post_reduce_scatter_kernel", "post_allgatherv_kernel", "ref_allreduce"):
        assert s in syms


def test_bench_pattern_is_exact_in_every_dtype():
    """bench.py verifies bitwise: the per-rank pattern and its sum over 8 ranks must be exactly representable, also in bfloat16"""
    torch = pytest.importorskip("torch")
    import importlib.util
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    for dt in (torch.float32, torch.bfloat16, torch.float16, torch.int32):
        parts = [bench.pattern(torch, 1000, r, dt, "cpu") for r in range(8)]
        exact = sum(p.to(torch.float64) for p in parts)
        assert torch.equal(bench.expected_sum(torch, 1000, 8, dt, "cpu").to(torch.float64), exact)
        assert len({float(v) for v in parts[3].to(torch.float64)}) > 5          # not a constant vector
        assert not torch.equal(parts[0], parts[1])


def test_bench_dump_output_is_a_fixed_sample(tmp_path):
    """bench.py --dump-outputs: a large result is sampled at the same positions every run (both ends kept whole) within its byte
    budget; a small one is written whole; float64 stays float64, every other dtype is written as float32"""
    torch = pytest.importorskip("torch")
    import importlib.util
    import numpy as np
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    x = bench.expected_sum(torch, 2_000_003, 3, torch.bfloat16, "cpu")
    for d in ("a", "b"):
        bench.dump_output(torch, str(tmp_path / d), "ar", x, 1, 8)
    a, b = np.load(tmp_path / "a" / "ar_rank1.npy"), np.load(tmp_path / "b" / "ar_rank1.npy")
    assert a.dtype == np.float32 and np.array_equal(a, b)
    assert 0 < a.nbytes <= bench.DUMP_BYTES // 8 and a.size < x.numel()
    ref = x.float().numpy()
    assert np.array_equal(a[:1 << 16], ref[:1 << 16]) and np.array_equal(a[-(1 << 16):], ref[-(1 << 16):])
    y = bench.pattern(torch, 1000, 2, torch.float64, "cpu")
    bench.dump_output(torch, str(tmp_path / "c"), "small", y, 0, 1)
    c = np.load(tmp_path / "c" / "small_rank0.npy")
    assert c.dtype == np.float64 and np.array_equal(c, y.numpy())
