#!/usr/bin/env bash
# Builds libcsic.so in-tree for sm_100a (B200).  nvcc cross-compiles without a GPU.
# The row kernel is compiled once per spatial factor, in parallel.
set -euo pipefail
cd "$(dirname "$0")"
NVCC=${NVCC:-/usr/local/cuda/bin/nvcc}
OUT=../libcsic.so
OBJ=../build/obj
mkdir -p "$OBJ"
FLAGS=(-gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -std=c++17 -Xcompiler -fPIC,-Wall,-fvisibility=hidden -Xptxas -v)
pids=()
for f in 1 2 4 8; do
  "$NVCC" "${FLAGS[@]}" -DCSIC_ROWS_F=$f -c csic_rows_kernel.cu -o "$OBJ/rows_f$f.o" 2> "$OBJ/rows_f$f.log" & pids+=($!)
done
for f in 2 4 8; do
  "$NVCC" "${FLAGS[@]}" -DCSIC_POOL_F=$f -c csic_pool_kernel.cu -o "$OBJ/pool_f$f.o" 2> "$OBJ/pool_f$f.log" & pids+=($!)
done
"$NVCC" "${FLAGS[@]}" -c csic_flex_kernel.cu -o "$OBJ/flex.o" 2> "$OBJ/flex.log" & pids+=($!)
"$NVCC" "${FLAGS[@]}" -c csic_decode_kernel.cu -o "$OBJ/decode.o" 2> "$OBJ/decode.log" & pids+=($!)
"$NVCC" "${FLAGS[@]}" -c csic_kernels.cu -o "$OBJ/kernels.o" 2> "$OBJ/kernels.log" & pids+=($!)
"$NVCC" "${FLAGS[@]}" -c csic_api.cu -o "$OBJ/api.o" 2> "$OBJ/api.log" & pids+=($!)
"$NVCC" "${FLAGS[@]}" -x cu -c csic_params.cpp -o "$OBJ/params.o" 2> "$OBJ/params.log" & pids+=($!)
g++ -O3 -std=c++17 -fPIC -Wall -fvisibility=hidden -c csic_plan.cpp -o "$OBJ/plan.o" 2> "$OBJ/plan.log" & pids+=($!)
rc=0
for p in "${pids[@]}"; do wait "$p" || rc=1; done
cat "$OBJ"/*.log > build.log
if [ $rc -ne 0 ]; then grep -v "ptxas info" build.log; exit 1; fi
"$NVCC" -gencode arch=compute_100a,code=sm_100a --shared -cudart static -Xlinker --version-script=csic.map -o "$OUT" "$OBJ"/rows_f1.o "$OBJ"/rows_f2.o "$OBJ"/rows_f4.o "$OBJ"/rows_f8.o "$OBJ"/pool_f2.o "$OBJ"/pool_f4.o "$OBJ"/pool_f8.o "$OBJ"/flex.o "$OBJ"/decode.o "$OBJ"/kernels.o "$OBJ"/api.o "$OBJ"/params.o "$OBJ"/plan.o
# native host program mirroring the reference CLI (uses only the C ABI + zlib)
g++ -O2 -std=c++17 -Wall -o ../csic_app host/csic_app.cpp host/png_io.cpp -L.. -lcsic -lz -Wl,-rpath,'$ORIGIN'
grep -E "error|warning" build.log | grep -v "ptxas info" || true
echo "built $(realpath $OUT)"
