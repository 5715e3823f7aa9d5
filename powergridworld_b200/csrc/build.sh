#!/usr/bin/env bash
# Build libpgw_b200.so in-tree for sm_100a (B200).  nvcc cross-compiles without a GPU.
set -euo pipefail
HERE="$(cd "$(dirname "${BASH_SOURCE[0]}")" && pwd)"
OUT="${PGW_OUT:-$HERE/../libpgw_b200.so}"          # PGW_OUT / PGW_EXTRA_FLAGS: instrumented builds (tools/)
BUILD="${PGW_BUILD_DIR:-$HERE/build}"
NVCC="${NVCC:-/usr/local/cuda/bin/nvcc}"
ARCH="-gencode arch=compute_100a,code=sm_100a"
COMMON="-O3 -std=c++17 -lineinfo -Xcompiler -fPIC $ARCH ${PGW_EXTRA_FLAGS:-}"
mkdir -p "$BUILD"
# component kernels: no FMA contraction, so float64 rounds exactly like the reference
"$NVCC" $COMMON -fmad=false ${PTXAS_V:+-Xptxas -v} -c "$HERE/components.cu" -o "$BUILD/components.o"
"$NVCC" $COMMON ${PTXAS_V:+-Xptxas -v} -c "$HERE/powerflow.cu" -o "$BUILD/powerflow.o"
"$NVCC" $COMMON ${PTXAS_V:+-Xptxas -v} -c "$HERE/powerflow_tc.cu" -o "$BUILD/powerflow_tc.o"
"$NVCC" $COMMON ${PTXAS_V:+-Xptxas -v} -c "$HERE/powerflow_tc2.cu" -o "$BUILD/powerflow_tc2.o"
"$NVCC" $COMMON -fmad=false ${PTXAS_V:+-Xptxas -v} -c "$HERE/step_fused.cu" -o "$BUILD/step_fused.o"
"$NVCC" $COMMON -c "$HERE/api.cu" -o "$BUILD/api.o"
"$NVCC" $COMMON -c "$HERE/tables.cpp" -o "$BUILD/tables.o"   # host only: same host flags as api.cu
"$NVCC" -shared $ARCH -o "$OUT" "$BUILD/components.o" "$BUILD/powerflow.o" "$BUILD/powerflow_tc.o" "$BUILD/powerflow_tc2.o" "$BUILD/step_fused.o" "$BUILD/api.o" "$BUILD/tables.o" -lcudart
echo "built $OUT"
