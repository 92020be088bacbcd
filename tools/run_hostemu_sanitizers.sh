#!/bin/bash
# The full tl/nvl stack in the host emulation (tests/test_nvl_hostemu.py) under ThreadSanitizer and AddressSanitizer: the plugin's
# host code (team creation, launch queue, exchange board, ...) cannot be sanitised on a GPU box without the CUDA runtime getting in
# the way; against the emulated runtime it can.  HOSTEMU_BUILD / HOSTEMU_WORKER select another build script / worker, e.g. the
# complex datatypes: HOSTEMU_BUILD=tests/emu/build_hostemu_complex.sh HOSTEMU_WORKER=tests/hostemu_complex_worker.py HOSTEMU_SCENARIOS=all
cd "$(dirname "$0")/.."
export EMU_CC=/usr/bin/gcc EMU_CXX=/usr/bin/g++
rc=0
for san in thread address; do
  EMU_EXTRA="-fsanitize=$san -g" bash ${HOSTEMU_BUILD:-tests/emu/build_hostemu.sh} > /dev/null 2>&1 || { echo "build failed ($san)"; exit 1; }
  rm -f /tmp/ucc_b200_he_$san.*
  lib=$(/usr/bin/gcc -print-file-name=$([ $san = thread ] && echo libtsan.so || echo libasan.so))
  for s in ${HOSTEMU_SCENARIOS:-allreduce colls_staged colls_zcopy colls_push colls_ce misc triggered p2p memh lanes}; do
    LD_PRELOAD=$lib TSAN_OPTIONS="log_path=/tmp/ucc_b200_he_$san:halt_on_error=0:report_signal_unsafe=0" \
      ASAN_OPTIONS="detect_leaks=0:detect_odr_violation=0:log_path=/tmp/ucc_b200_he_$san" timeout 1500 python ${HOSTEMU_WORKER:-tests/hostemu_worker.py} $s > /tmp/ucc_b200_he_${san}_$s.log 2>&1
    ok=$(grep -c HOSTEMU_WORKER_OK /tmp/ucc_b200_he_${san}_$s.log)
    echo "$san $s: $([ "$ok" = 1 ] && echo ok || echo FAILED)"; [ "$ok" = 1 ] || rc=1
  done
  n=$(ls /tmp/ucc_b200_he_$san.* 2>/dev/null | wc -l)
  echo "$san: sanitizer report files: $n"; [ "$n" = 0 ] || rc=1
done
bash ${HOSTEMU_BUILD:-tests/emu/build_hostemu.sh} > /dev/null 2>&1   # back to the plain build
exit $rc
