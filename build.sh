#!/bin/sh
# Builds libpsg_b200.so (sm_100a only) in-tree.  The .so travels to the GPU box with the snapshot.
set -e
HERE="$(cd "$(dirname "$0")" && pwd)"
SRC="$HERE/pointsecguard_b200/csrc"
OUT="$HERE/pointsecguard_b200/libpsg_b200.so"
OBJ="$SRC/_obj"
mkdir -p "$OBJ"
NVCC="${NVCC:-nvcc}"
FLAGS="-gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -std=c++17 -Xcompiler -fPIC"
pids=""
set --      # the objects to link: exactly the sources listed here, whatever else _obj/ holds
for f in fps neighbors ballgrid gather gemm_simt gemm_tc sa_fused compact chain_fused geomgrad elementwise nu slicer train streambench knn net api; do
  set -- "$@" "$OBJ/$f.o"
  if [ ! -f "$OBJ/$f.o" ] || [ "$SRC/$f.cu" -nt "$OBJ/$f.o" ] || [ "$SRC/psg_common.cuh" -nt "$OBJ/$f.o" ] || \
     [ "$SRC/psg_internal.h" -nt "$OBJ/$f.o" ] || [ "$SRC/psg_loss.cuh" -nt "$OBJ/$f.o" ] || [ "$SRC/psg_epi.cuh" -nt "$OBJ/$f.o" ] || [ "$SRC/psg_tc.cuh" -nt "$OBJ/$f.o" ] || [ "$HERE/include/psg_b200.h" -nt "$OBJ/$f.o" ]; then
    $NVCC $FLAGS -c "$SRC/$f.cu" -o "$OBJ/$f.o" &
    pids="$pids $!"
  fi
done
for p in $pids; do wait $p; done
$NVCC -shared -gencode arch=compute_100a,code=sm_100a -o "$OUT" "$@" -lcudart
echo "built $OUT"
