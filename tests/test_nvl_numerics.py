"""Numerics of every tl/nvl reduction kernel, without a GPU (tests/emu/nvl_emu_numerics.cpp compiled as host C++).

One executable per datatype (the 12 real types and the two complex ones) runs one-shot allreduce, one-shot reduce_scatter(v),
staged P2P / NVLS, zero-copy, ring, rhd, nvls_pipe and symm with every operator the type supports, as allreduce, reduce and
reduce_scatter(v), at counts around the vector width and the staging capacity, shifted by one element and in place.  Inputs are
chosen so that every result is checked bit for bit against an exact oracle; random full-mantissa inputs check that every rank of
an allreduce stores the same bits and that the error stays within the recursive-summation bound."""
import os
import subprocess
from concurrent.futures import ThreadPoolExecutor

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CUDA_INC = "/usr/local/cuda/include"
# nvl_dt_t values (src/components/tl/nvl/kernels/nvl_kernels.h)
DTS = {"int8": 0, "int16": 1, "int32": 2, "int64": 3, "uint8": 4, "uint16": 5, "uint32": 6, "uint64": 7,
       "float16": 8, "float32": 9, "float64": 10, "bfloat16": 11, "float32_complex": 12, "float64_complex": 13}


@pytest.fixture(scope="module")
def emu(tmp_path_factory):
    if not os.path.exists(os.path.join(CUDA_INC, "cuda_fp16.h")):
        pytest.skip("CUDA headers not installed")
    out = tmp_path_factory.mktemp("emu_numerics")
    k = os.path.join(ROOT, "src", "components", "tl", "nvl", "kernels")

    def build(name):
        exe = str(out / f"nvl_emu_numerics_{name}")
        # -fwrapv: integer SUM / PROD wrap as they do on the GPU
        cc = subprocess.run(["g++", "-O1", "-fwrapv", "-std=c++17", "-pthread", f"-DNUM_DT={DTS[name]}", f"-I{CUDA_INC}", f"-I{k}",
                             f"-I{ROOT}/include", f"-I{ROOT}/src", os.path.join(ROOT, "tests", "emu", "nvl_emu_numerics.cpp"), "-o", exe],
                            capture_output=True, text=True)
        assert cc.returncode == 0, cc.stderr[-4000:]
        return name, exe

    with ThreadPoolExecutor(max_workers=max(2, os.cpu_count() or 2)) as ex:
        return dict(ex.map(build, DTS))


@pytest.mark.parametrize("n", [2, 3, 4, 5, 8])
def test_reduction_kernels_numerics(emu, n):
    """every datatype at team size n (2 / 4 / 8: the unrolled size classes; 3 / 5: the generic one, 5 with a source group of one)"""
    def run(name):
        return name, subprocess.run([emu[name], str(n)], capture_output=True, text=True, timeout=170)

    with ThreadPoolExecutor(max_workers=4) as ex:
        res = dict(ex.map(run, emu))
    bad = {name: (r.stdout[-2500:] + r.stderr[-1000:]) for name, r in res.items() if r.returncode != 0 or "NVL_EMU_OK" not in r.stdout}
    assert not bad, "\n".join(f"--- {k}\n{v}" for k, v in bad.items())
