#!/bin/bash
# Builds affnet_b200/lib/libaffnet_b200.so for sm_100a (nvcc cross-compiles without a GPU).
set -e
HERE="$(cd "$(dirname "$0")" && pwd)"
OUT="$HERE/../lib"
mkdir -p "$OUT" "$HERE/obj"
NVCC="${NVCC:-/usr/local/cuda/bin/nvcc}"
FLAGS="${AG_EXTRA_FLAGS:-} -gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -std=c++17 -Xcompiler -fPIC -Xptxas -v"
pids=()
objs=()   # objects of the current sources only: one left behind by a deleted source must not be linked
for f in "$HERE"/*.cu; do
  o="$HERE/obj/$(basename "${f%.cu}").o"
  objs+=("$o")
  stale=0
  for d in "$f" "$HERE"/*.cuh "$HERE/../../include/affnet_b200.h"; do [ "$d" -nt "$o" ] && stale=1; done
  if [ ! -f "$o" ] || [ $stale = 1 ]; then
    ( $NVCC $FLAGS -c "$f" -o "$o" > "$o.log" 2>&1 || { cat "$o.log"; exit 1; } ) &
    pids+=($!)
  fi
done
fail=0
for p in "${pids[@]}"; do wait $p || fail=1; done
if [ $fail = 1 ]; then echo "build failed" >&2; rm -f "$HERE"/obj/*.o.failed; for l in "$HERE"/obj/*.o.log; do grep -l "error" "$l" >/dev/null 2>&1 && rm -f "${l%.log}"; done; exit 1; fi
$NVCC -gencode arch=compute_100a,code=sm_100a -shared -o "$OUT/libaffnet_b200.so" "${objs[@]}" -lcudart
echo "built $OUT/libaffnet_b200.so"
if [ "${AG_XPROF:-0}" = "1" ]; then mkdir -p "$HERE/obj_prof";   # developer build with the warp-role cycle counters of the second-generation engine (scripts/role_prof_x.py)
  $NVCC $FLAGS -DAG_ROLE_PROF -c "$HERE/nets_tcx.cu" -o "$HERE/obj_prof/nets_tcx.o" > "$HERE/obj_prof/nets_tcx.log" 2>&1 || { cat "$HERE/obj_prof/nets_tcx.log"; exit 1; }
  xobjs=("${objs[@]/*nets_tcx.o/$HERE/obj_prof/nets_tcx.o}")
  $NVCC -gencode arch=compute_100a,code=sm_100a -shared -o "$OUT/libaffnet_b200_xprof.so" "${xobjs[@]}" -lcudart
  echo "built $OUT/libaffnet_b200_xprof.so"
fi
