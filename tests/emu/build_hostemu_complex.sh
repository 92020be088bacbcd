#!/bin/bash
# Host-emulated build of the CUDA plugins whose kernels also serve float32_complex / float64_complex (tests/test_nvl_complex.py):
# build-emu/complex/lib/ucc/{libucc_tl_nvl.so,libucc_mc_cuda.so} + build-emu/complex/lib/libcudart_emu.so.  The same recipe as
# build_hostemu.sh with tests/emu/nvl_emu_launch_complex.cpp as the launcher; EMU_CC / EMU_CXX / EMU_EXTRA work the same way.
set -e
cd "$(dirname "$0")/../.."
OUT=build-emu/complex/lib; MOD=$OUT/ucc; OBJ=build-emu/complex/obj
mkdir -p $MOD $OBJ
CUDA_INC=/usr/local/cuda/include
CF="-O0 $EMU_EXTRA -fPIC -D_GNU_SOURCE -Iinclude -Isrc -I$CUDA_INC -Wall -Wno-unused-parameter -Wno-unused-function"
${EMU_CXX:-g++} $CF -std=c++17 -pthread -shared tests/emu/cudart_emu.cpp -o $OUT/libcudart_emu.so
for f in src/components/tl/nvl/tl_nvl.c src/components/tl/nvl/tl_nvl_coll.c src/components/tl/nvl/tl_nvl_team.c src/components/tl/nvl/tl_nvl_direct.c src/components/tl/nvl/tl_nvl_memh.c src/utils/cuda/ucc_cuda_util.c src/components/mc/cuda/mc_cuda.c; do
  ${EMU_CC:-gcc} $CF -std=gnu11 -c $f -o $OBJ/$(basename $f).o &
done
${EMU_CXX:-g++} $CF -std=c++17 -pthread -Isrc/components/tl/nvl/kernels -c tests/emu/nvl_emu_launch_complex.cpp -o $OBJ/nvl_emu_launch_complex.o &
wait
${EMU_CXX:-g++} $EMU_EXTRA -shared -o $MOD/libucc_tl_nvl.so $OBJ/tl_nvl.c.o $OBJ/tl_nvl_coll.c.o $OBJ/tl_nvl_team.c.o $OBJ/tl_nvl_direct.c.o $OBJ/tl_nvl_memh.c.o $OBJ/ucc_cuda_util.c.o $OBJ/nvl_emu_launch_complex.o \
    -Lucc_b200/lib -lucc -L$OUT -lcudart_emu -Wl,-rpath,'$ORIGIN/..' -Wl,-rpath,$PWD/ucc_b200/lib -lpthread -ldl
${EMU_CC:-gcc} $EMU_EXTRA -shared -o $MOD/libucc_mc_cuda.so $OBJ/mc_cuda.c.o $OBJ/ucc_cuda_util.c.o -Lucc_b200/lib -lucc -L$OUT -lcudart_emu -Wl,-rpath,'$ORIGIN/..' -Wl,-rpath,$PWD/ucc_b200/lib -lpthread -ldl
echo "HOSTEMU_BUILD_OK $MOD"
