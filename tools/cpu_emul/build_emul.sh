#!/bin/sh
# Developer aid: compile the CUDA sources for the CPU fiber emulator (see cuda_emul.h).
# Output: tools/cpu_emul/libsoftgnss_emul.so (git-ignored, never loaded by the package).
# Objects are cached under tools/cpu_emul/obj and rebuilt when a source or header is newer.
set -e
HERE=$(cd "$(dirname "$0")" && pwd)
ROOT=$(cd "$HERE/../.." && pwd)
SRC=$ROOT/softgnss_python_b200/csrc
mkdir -p "$HERE/obj"
NEWEST_HDR=$(ls -t "$SRC"/*.cuh "$SRC"/*.h "$HERE/cuda_emul.h" "$ROOT/include/softgnss_b200.h" | head -1)
OBJS=""
for f in sgx_api.cu sgx_track.cu sgx_synth.cu sgx_acq.cu sgx_pfa.cu sgx_fine.cu sgx_bitsync.cu sgx_nav.cu sgx_quality.cu; do
  [ -f "$SRC/$f" ] || continue
  o="$HERE/obj/${f%.cu}.o"
  OBJS="$OBJS $o"
  if [ ! -f "$o" ] || [ "$SRC/$f" -nt "$o" ] || [ "$NEWEST_HDR" -nt "$o" ]; then
    g++ -x c++ -std=c++17 -O2 -g -DSGX_EMUL -ffp-contract=off -fPIC -pthread \
        -Wno-unknown-pragmas -Wno-attributes -I"$HERE" -I"$SRC" -c "$SRC/$f" -o "$o" &
  fi
done
wait
g++ -shared -pthread $OBJS -o "$HERE/libsoftgnss_emul.so"
echo "$HERE/libsoftgnss_emul.so"
