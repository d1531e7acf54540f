#!/bin/bash
# Build libsemk.so in-tree for sm_100a (nvcc cross-compiles without a GPU).
set -euo pipefail
cd "$(dirname "$0")"
NVCC=${NVCC:-/usr/local/cuda/bin/nvcc}
FLAGS="-gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -std=c++17 -Xcompiler -fPIC -Xcompiler -O3"
OBJS=""
PIDS=""
for f in semk_api.cu semk_geom.cu semk_apply.cu semk_box.cu semk_vec.cu semk_peer.cu semk_sc.cu semk_field.cu semk_ml.cu semk_ho.cu semk_locate.cu semk_stokes.cu semk_block.cu; do
  [ -f "$f" ] || continue
  o="${f%.cu}.o"
  if [ ! -f "$o" ] || [ "$f" -nt "$o" ] || [ semk_common.cuh -nt "$o" ] || [ semk_elem.cuh -nt "$o" ] || [ semk_patch.cuh -nt "$o" ] || [ ../../include/semk.h -nt "$o" ]; then
    rm -f "$o"      # a failed compile must not leave a stale, linkable object behind
    $NVCC $FLAGS ${SEMK_EXTRA_FLAGS:-} ${SEMK_PTXAS_V:+-Xptxas -v} -c "$f" -o "$o" &
    PIDS="$PIDS $!"
  fi
  OBJS="$OBJS $o"
done
o=semk_hostplan.o
if [ ! -f "$o" ] || [ semk_hostplan.cpp -nt "$o" ] || [ ../../include/semk.h -nt "$o" ]; then
  rm -f "$o"
  g++ -O3 -std=c++17 -fPIC -fopenmp -c semk_hostplan.cpp -o "$o" &
  PIDS="$PIDS $!"
fi
o=semk_hostnum.o
if [ ! -f "$o" ] || [ semk_hostnum.cpp -nt "$o" ] || [ ../../include/semk.h -nt "$o" ]; then
  rm -f "$o"
  g++ -O3 -std=c++17 -fPIC -fopenmp -c semk_hostnum.cpp -o "$o" &
  PIDS="$PIDS $!"
fi
for pid in $PIDS; do
  wait "$pid" || { echo "build.sh: a compile job failed" >&2; exit 1; }
done
$NVCC -gencode arch=compute_100a,code=sm_100a -shared -Xcompiler -fopenmp -o libsemk.so $OBJS semk_hostplan.o semk_hostnum.o
echo "built $(pwd)/libsemk.so"
