#!/usr/bin/env bash
# Builds lib/libroi3d_b200.so for sm_100a (B200) in-tree.  nvcc cross-compiles without a GPU.
# No torch, no CUTLASS: plain CUDA runtime, C ABI (include/roi3d_b200.h).
set -euo pipefail
HERE=$(cd "$(dirname "$0")" && pwd)
NVCC=${NVCC:-/usr/local/cuda/bin/nvcc}
OUT=$HERE/lib
mkdir -p "$OUT" "$HERE/build"
FLAGS=(-gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -lineinfo -Xcompiler -fPIC --expt-relaxed-constexpr -DROI3D_BUILD)
[ "${VERBOSE_PTXAS:-0}" = "1" ] && FLAGS+=(-Xptxas -v)
[ -n "${ROI3D_EXTRA_NVCC_FLAGS:-}" ] && FLAGS+=(${ROI3D_EXTRA_NVCC_FLAGS})
pids=()
for f in roi_align3d roi_align3d_stream roi_align3d_planar roi_align3d_det nms3d soft_nms3d multiclass_nms proposal assign mask_paste host_api; do
  src=$HERE/csrc/$f.cu
  obj=$HERE/build/$f.o
  if [ ! -f "$obj" ] || [ "$src" -nt "$obj" ] || [ "$HERE/csrc/common.cuh" -nt "$obj" ] || [ "$HERE/csrc/roi_align3d_shared.cuh" -nt "$obj" ] \
     || [ "$HERE/../include/roi3d_b200.h" -nt "$obj" ]; then
    "$NVCC" "${FLAGS[@]}" -c "$src" -o "$obj" &
    pids+=($!)
  fi
done
for p in "${pids[@]:-}"; do [ -n "$p" ] && wait "$p"; done
"$NVCC" -gencode arch=compute_100a,code=sm_100a -shared -o "$OUT/libroi3d_b200.so" "$HERE"/build/{roi_align3d,roi_align3d_stream,roi_align3d_planar,roi_align3d_det,nms3d,soft_nms3d,multiclass_nms,proposal,assign,mask_paste,host_api}.o -cudart static
echo "built $OUT/libroi3d_b200.so"
