#!/bin/bash
# Build an experimental copy of libnsf.so: scripts/build_variant.sh <name> [csrc_dir] [extra nvcc flags...]
# Output: neurosync_trainer_lite_b200/_lib/variants/<name>.so (select it with NSF_LIB_PATH). Experiments only.
set -e
ROOT=$(cd "$(dirname "$0")/.." && pwd)
NAME=$1; shift
SRC=${1:-$ROOT/neurosync_trainer_lite_b200/csrc}; shift || true
OUT=$ROOT/neurosync_trainer_lite_b200/_lib/variants
TMP=$(mktemp -d)
mkdir -p "$OUT"
# the library's own source list (neurosync_trainer_lite_b200/build.py SOURCES)
SOURCES=$(python3 -c 'import runpy, sys; print(" ".join(runpy.run_path(sys.argv[1])["SOURCES"]))' \
          "$ROOT/neurosync_trainer_lite_b200/build.py")
pids=()
for f in $SOURCES; do
  [ -f "$SRC/$f" ] || continue      # older source trees (A/B against an earlier commit) lack the newer files
  nvcc -gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -std=c++17 -Xcompiler -fPIC,-O3,-fvisibility=hidden \
       -x cu -cudart static -I "$ROOT/include" -I "$SRC" -DNSF_BUILDING=1 "$@" -c "$SRC/$f" -o "$TMP/${f%.*}.o" &
  pids+=($!)
done
for p in "${pids[@]}"; do wait "$p"; done
nvcc -shared -cudart static -gencode arch=compute_100a,code=sm_100a -o "$OUT/$NAME.so" "$TMP"/*.o
rm -rf "$TMP"
echo "$OUT/$NAME.so"
