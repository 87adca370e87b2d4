#!/bin/bash
# compute-sanitizer is closed on this GPU pool.  Substitute: the CUDA kernel sources of the block-push family, compiled
# unchanged by g++ on the SIMT emulator (tests/simt_emu: one std::thread per CUDA thread, shared memory = a host buffer),
# under AddressSanitizer + UndefinedBehaviorSanitizer (memcheck: every shared / global access of the kernels is a host
# access ASan checks, including the per-warp slices and the block-shared tables) and under ThreadSanitizer (racecheck:
# lanes are threads, __syncwarp / __syncthreads / shuffles are barriers, so two lanes touching one shared-memory word
# without a barrier between them is a data race TSan reports).   usage: tools/emu_sanitize.sh  -> profiles/r02_emu_*.log
# tools/emu_sanitize.sh cap4: ASan + UBSan only, every kernel at a contact capacity of 4 on states that overflow it
# -> profiles/r03_emu_asan_cap4.log
set -u
cd "$(dirname "$0")/.."
OUT=profiles
if [ "${1:-}" == cap4 ]; then
  SAN="-fsanitize=address,undefined -fno-omit-frame-pointer"; PRE=$(gcc -print-file-name=libasan.so)
  EMU="-O1 -g -std=c++17 -fPIC -shared -ffp-contract=off $SAN -D__CUDACC__ -DHSRB_SIMT_EMU -include tests/simt_emu/simt_emu.h -I tests/simt_emu"
  g++ $EMU -DHSR_COMPACT -DPUSH_MAXCON=4 -DWPE_MAXCON=4 -o /tmp/libpush_emu_cap4_asan.so tests/simt_emu/emu_push.cpp -lpthread || exit 1
  g++ $EMU -o /tmp/libstep_emu_asan.so tests/simt_emu/emu_step.cpp -lpthread || exit 1
  LOG=$OUT/r03_emu_asan_cap4.log
  ASAN_OPTIONS=detect_leaks=0:halt_on_error=0 LD_PRELOAD=$PRE EMU_CAP=4 EMU_LIB=/tmp/libpush_emu_cap4_asan.so \
  EMU_LIB_G=/tmp/libstep_emu_asan.so timeout 3000 python tools/emu_sanitize_case.py > $LOG 2>&1
  echo "exit $?" >> $LOG
  echo "== asan cap4"; grep -cE "ERROR: AddressSanitizer|runtime error" $LOG; tail -n 6 $LOG
  exit 0
fi
# tools/emu_sanitize.sh episode: ASan + UBSan, the episode kernel (hsrb_episode.cuh: TimeLimit + auto-reset) through
# tests/test_episode_emu.py -> profiles/r04_emu_asan_episode.log
if [ "${1:-}" == episode ]; then
  SAN="-fsanitize=address,undefined -fno-omit-frame-pointer"; PRE=$(gcc -print-file-name=libasan.so)
  g++ -O1 -g -std=c++17 -fPIC -shared -ffp-contract=off $SAN -D__CUDACC__ -DHSRB_SIMT_EMU -include tests/simt_emu/simt_emu.h \
      -I tests/simt_emu -o /tmp/libepisode_emu_asan.so tests/simt_emu/emu_episode.cpp -lpthread || exit 1
  LOG=$OUT/r04_emu_asan_episode.log
  ASAN_OPTIONS=detect_leaks=0:halt_on_error=0 LD_PRELOAD=$PRE EMU_EPISODE_LIB=/tmp/libepisode_emu_asan.so \
  timeout 3000 python -m pytest tests/test_episode_emu.py -q -p no:cacheprovider > $LOG 2>&1
  echo "exit $?" >> $LOG
  echo "== asan episode"; grep -cE "ERROR: AddressSanitizer|runtime error" $LOG; tail -n 6 $LOG
  exit 0
fi
for MODE in asan tsan; do
  if [ $MODE == asan ]; then SAN="-fsanitize=address,undefined -fno-omit-frame-pointer"; PRE=$(gcc -print-file-name=libasan.so); else SAN="-fsanitize=thread"; PRE=$(gcc -print-file-name=libtsan.so); fi
  LIB=/tmp/libpush_emu_$MODE.so
  g++ -O1 -g -std=c++17 -fPIC -shared -ffp-contract=off $SAN -D__CUDACC__ -DHSRB_SIMT_EMU -DHSR_COMPACT \
      -include tests/simt_emu/simt_emu.h -I tests/simt_emu -o $LIB tests/simt_emu/emu_push.cpp -lpthread || exit 1
  ASAN_OPTIONS=detect_leaks=0:halt_on_error=0 TSAN_OPTIONS="halt_on_error=0 report_signal_unsafe=0 history_size=4" \
  LD_PRELOAD=$PRE EMU_LIB=$LIB timeout 3000 python tools/emu_sanitize_case.py > $OUT/r02_emu_$MODE.log 2>&1
  echo "exit $?" >> $OUT/r02_emu_$MODE.log
  echo "== $MODE"; grep -cE "ERROR: AddressSanitizer|runtime error|WARNING: ThreadSanitizer" $OUT/r02_emu_$MODE.log; tail -n 6 $OUT/r02_emu_$MODE.log
done
