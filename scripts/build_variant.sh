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
pids=()
for f in nsf_plan.cpp nsf_kernels.cu nsf_autocorr_mma.cu nsf_stft_tc.cu nsf_convert.cu nsf_api.cu; do
  [ -f "$SRC/$f" ] || continue      # older source trees (A/B against an earlier commit) lack the newer files
  nvcc -gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -std=c++17 -Xcompiler -fPIC,-O3,-fvisibility=hidden \
       -x cu -cudart static -I "$ROOT/include" -I "$SRC" -DNSF_BUILDING=1 "$@" -c "$SRC/$f" -o "$TMP/${f%.*}.o" &
  pids+=($!)
done
for p in "${pids[@]}"; do wait "$p"; done
nvcc -shared -cudart static -gencode arch=compute_100a,code=sm_100a -o "$OUT/$NAME.so" "$TMP"/*.o
rm -rf "$TMP"
echo "$OUT/$NAME.so"
