#!/bin/bash
# Builds libmrl_b200.so in-tree for sm_100a.  Usage: build.sh [extra nvcc flags]
set -e
HERE="$(cd "$(dirname "$0")" && pwd)"
OUT="$HERE/../libmrl_b200.so"
NVCC="${NVCC:-/usr/local/cuda/bin/nvcc}"
FLAGS="-gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -std=c++17 -Xcompiler -fPIC -Xcompiler -O2 --expt-relaxed-constexpr -Xptxas -v"
mkdir -p "$HERE/obj"
pids=()
for f in geom batch_params mlp_l1_tc mlp_mid mlp_layers mlp_chain mlp_fvp_tc peak_tc population vec_kernels scan_kernels rollout cem_search api comm; do
  ( $NVCC $FLAGS "$@" -c "$HERE/$f.cu" -o "$HERE/obj/$f.o" > "$HERE/obj/$f.log" 2>&1 || { cat "$HERE/obj/$f.log"; exit 1; } ) &
  pids+=($!)
done
rc=0
for p in "${pids[@]}"; do wait $p || rc=1; done
[ $rc -eq 0 ] || exit 1
$NVCC -shared -o "$OUT" "$HERE"/obj/{geom,batch_params,mlp_l1_tc,mlp_mid,mlp_layers,mlp_chain,mlp_fvp_tc,peak_tc,population,vec_kernels,scan_kernels,rollout,cem_search,api,comm}.o -lcudart -ldl
echo "built $OUT"
