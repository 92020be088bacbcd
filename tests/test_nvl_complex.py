"""Complex datatypes (float32_complex / float64_complex) on the tl/nvl reduction kernels, without a GPU.

  - the kernels compiled as host C++ (tests/emu/nvl_emu_complex.cpp): every reduction kernel x {SUM, PROD, AVG} x N in
    {2, 3, 4, 8}, exact on Gaussian integers, c64 SUM bitwise equal to f32 SUM of the same bytes
  - the whole plugin on the emulated CUDA runtime (tests/emu/build_hostemu_complex.sh, tests/hostemu_complex_worker.py): the
    public API, default selection and every forced algorithm, and the trace shows tl/nvl for every complex collective
  - the built sm_100a objects: the PROD instantiations keep the register budget without a stack frame"""
import os
import re
import shutil
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CUDA_INC = "/usr/local/cuda/include"


@pytest.fixture(scope="module")
def emu(tmp_path_factory):
    if not os.path.exists(os.path.join(CUDA_INC, "cuda_fp16.h")):
        pytest.skip("CUDA headers not installed")
    exe = tmp_path_factory.mktemp("emu") / "nvl_emu_complex"
    k = os.path.join(ROOT, "src", "components", "tl", "nvl", "kernels")
    cc = subprocess.run(["g++", "-O1", "-g", "-std=c++17", "-pthread", f"-I{CUDA_INC}", f"-I{k}", f"-I{ROOT}/include", f"-I{ROOT}/src",
                         os.path.join(ROOT, "tests", "emu", "nvl_emu_complex.cpp"), "-o", str(exe)], capture_output=True, text=True)
    assert cc.returncode == 0, cc.stderr[-4000:]
    return str(exe)


@pytest.mark.parametrize("n", [2, 3, 4, 8])
def test_complex_kernels_host_emulation(emu, n):
    out = subprocess.run([emu, f"n{n}"], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0 and "NVL_EMU_OK" in out.stdout, out.stdout[-3000:] + out.stderr[-2000:]
    assert out.stdout.count("  ok ") == (10 if n in (2, 4, 8) else 9)   # every kernel ran (rhd: power-of-two teams)


@pytest.fixture(scope="module")
def emu_build():
    if not os.path.exists(os.path.join(CUDA_INC, "cuda_fp16.h")):
        pytest.skip("CUDA headers not installed")
    out = subprocess.run(["bash", os.path.join(ROOT, "tests", "emu", "build_hostemu_complex.sh")], capture_output=True, text=True, timeout=900)
    assert "HOSTEMU_BUILD_OK" in out.stdout, out.stdout[-2000:] + out.stderr[-3000:]


def test_complex_host_emulation(emu_build):
    env = dict(os.environ, PYTHONPATH=ROOT)
    for k in ("UCC_TL_NVL_TUNE", "UCC_MODULE_DIR", "UCC_TLS"):
        env.pop(k, None)
    out = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "hostemu_complex_worker.py")], env=env, capture_output=True, text=True, timeout=900)
    assert out.returncode == 0 and "HOSTEMU_WORKER_OK" in out.stdout, out.stdout[-2500:] + out.stderr[-2500:]
    lines = [ln for ln in (out.stdout + out.stderr).splitlines() if "coll_init:" in ln and re.search(r"float(32|64)_complex", ln, re.I)]
    assert len(lines) > 500, (out.stdout + out.stderr)[-2000:]
    bad = [ln for ln in lines if "{TL_NVL}" not in ln]
    assert not bad, bad[:5]


def _res_usage(obj):
    txt = subprocess.run(["cuobjdump", "-res-usage", obj], capture_output=True, text=True).stdout
    names = subprocess.run(["c++filt"], input=txt, capture_output=True, text=True).stdout
    res, fn = {}, None
    for ln in names.splitlines():
        m = re.match(r"\s*Function (.+):$", ln)
        if m:
            fn = m.group(1)
            continue
        m = re.search(r"REG:(\d+) STACK:(\d+)", ln)
        if m and fn:
            res[fn] = (int(m.group(1)), int(m.group(2)))
            fn = None
    return res


@pytest.mark.parametrize("t", ["c64", "c128"])
def test_complex_prod_kernels_have_no_stack(t):
    """complex PROD is the one new reduction body: its zero-copy (team-size classes 2, 4 and generic) and one-shot instantiations
    keep 2 CTAs x 512 threads (64 registers) with no local-memory stack"""
    obj = os.path.join(ROOT, "build", "src", "components", "tl", "nvl", "kernels", f"nvl_red_{t}.cu.o")
    if not os.path.exists(obj) or not shutil.which("cuobjdump") or not shutil.which("c++filt"):
        pytest.skip("sm_100a build or cuobjdump not present")
    res = _res_usage(obj)
    T = {"c64": "nvl_c64", "c128": "nvl_c128"}[t]
    want = [f"void nvl_reduce_direct_kernel_t<{T}, 1, {cn}>(nvl_red_args)" for cn in (2, 4, 0)] + [f"void nvl_allreduce_oneshot_kernel_t<{T}, 1>(nvl_red_args)"]
    for k in want:
        assert k in res, (k, sorted(res)[:8])
        assert res[k][1] == 0, (k, res[k])
    for k in want[:3]:
        assert res[k][0] <= 64, (k, res[k])
