#!/bin/bash
# Build libdmip_sm100.so in-tree (sm_100a only; nvcc cross-compiles without a GPU).
# DMIP_DEBUG=1 bash build.sh  compiles the DMIP_DBG ablation bits and the kernel timeline in (slower issue loops).
set -euo pipefail
cd "$(dirname "$0")"
OUT=${DMIP_OUT:-../libdmip_sm100.so}
NVCC=${NVCC:-/usr/local/cuda/bin/nvcc}
FLAGS="-gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -std=c++17 -Xcompiler -fPIC -Xptxas -v ${DMIP_DEBUG:+-DDMIP_DEBUG} ${DMIP_EXP:+-DDMIP_EXP=$DMIP_EXP} ${DMIP_JOBMARKS:+-DDMIP_JOBMARKS} ${DMIP_TILE:+-DDMIP_TILE_$DMIP_TILE} ${DMIP_DEFS:-}"
mkdir -p build
pids=()
SRCS="dmip_api dmip_pack dmip_tc dmip_f32 dmip_loss dmip_tcl dmip_surrogate dmip_surrogate_tc dmip_metrics dmip_mmd dmip_mmd_test dmip_ksd dmip_tsample"
for f in $SRCS; do
  ( $NVCC $FLAGS -c $f.cu -o build/$f.o > build/$f.log 2>&1 || { cat build/$f.log; exit 1; } ) &
  pids+=($!)
done
for p in "${pids[@]}"; do wait $p; done
OBJS=""; for f in $SRCS; do OBJS="$OBJS build/$f.o"; done
$NVCC -gencode arch=compute_100a,code=sm_100a -shared -o $OUT $OBJS
echo "built $(realpath $OUT)"
