#!/bin/bash
# Builds libgnnx.so (sm_100a only) in-tree: gnn-model-explainer_b200/gnnx/lib/libgnnx.so
set -e
HERE="$(cd "$(dirname "$0")" && pwd)"
ROOT="$(cd "$HERE/../.." && pwd)"
OUT="${GNNX_BUILD_OUT:-$HERE/../gnnx/lib}"   # GNNX_BUILD_OUT + GNNX_NVCC_EXTRA: A-B builds for tools/ (e.g. -DGXG_UNROLL=4)
mkdir -p "$OUT"
NVCC=${NVCC:-/usr/local/cuda/bin/nvcc}
FLAGS="-gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -std=c++17 -Xcompiler -fPIC -I$ROOT/include -I$HERE ${GNNX_NVCC_EXTRA}"
PIDS=()
for f in api khop explain_node explain_graph explain_graph_var explain_stream explain_gang explain_var forward trace denoise comm; do
  if [ ! -f "$OUT/$f.o" ] || [ "$HERE/$f.cu" -nt "$OUT/$f.o" ] || [ "$HERE/gnnx_internal.cuh" -nt "$OUT/$f.o" ] || [ "$ROOT/include/gnnx.h" -nt "$OUT/$f.o" ] || [ "$HERE/explain_common.cuh" -nt "$OUT/$f.o" ]; then
    rm -f "$OUT/$f.o"   # a failed compile must not leave an older object for the link below
    $NVCC $FLAGS -c "$HERE/$f.cu" -o "$OUT/$f.o" &
    PIDS+=($!)
  fi
done
for p in "${PIDS[@]}"; do wait "$p"; done   # set -e: the first failed compile stops the build
$NVCC -gencode arch=compute_100a,code=sm_100a -shared -o "$OUT/libgnnx.so.tmp" "$OUT/api.o" "$OUT/khop.o" "$OUT/explain_node.o" "$OUT/explain_graph.o" "$OUT/explain_graph_var.o" "$OUT/explain_stream.o" "$OUT/explain_gang.o" "$OUT/explain_var.o" "$OUT/forward.o" "$OUT/trace.o" "$OUT/denoise.o" "$OUT/comm.o" -ldl
mv -f "$OUT/libgnnx.so.tmp" "$OUT/libgnnx.so"   # atomic: a snapshot never sees a half-written library
echo "built $OUT/libgnnx.so"
