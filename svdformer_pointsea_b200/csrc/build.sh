#!/usr/bin/env bash
# Builds libpointsea_b200.so (sm_100a only) next to the Python package.
set -euo pipefail
HERE="$(cd "$(dirname "${BASH_SOURCE[0]}")" && pwd)"
OUT="$HERE/../lib"
mkdir -p "$OUT"
NVCC="${NVCC:-/usr/local/cuda/bin/nvcc}"
FLAGS=(-gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -std=c++17 -Xcompiler -fPIC -Xptxas -v)
SRCS=(runtime.cu comm.cu step.cu chamfer.cu chamfer_sym.cu fps.cu gather_group.cu neighbors.cu knn_select.cu host_pipeline.cu feature_knn.cu metrics.cu scatter.cu chamfer_loss.cu crop.cu)
OBJS=()
pids=()
for s in "${SRCS[@]}"; do
  o="$OUT/${s%.cu}.o"
  OBJS+=("$o")
  "$NVCC" "${FLAGS[@]}" -c "$HERE/$s" -o "$o" > "$OUT/${s%.cu}.ptxas.log" 2>&1 &
  pids+=($!)
done
rc=0
for p in "${pids[@]}"; do wait "$p" || rc=1; done
if [ $rc -ne 0 ]; then cat "$OUT"/*.ptxas.log; exit 1; fi
"$NVCC" -shared -o "$OUT/libpointsea_b200.so" "${OBJS[@]}" -gencode arch=compute_100a,code=sm_100a
echo "built $OUT/libpointsea_b200.so"
