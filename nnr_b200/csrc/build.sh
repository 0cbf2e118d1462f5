#!/bin/bash
# Build libnnr_b200.so for sm_100a (in-tree; the .so travels to the GPU box with the snapshot).
set -e
HERE="$(cd "$(dirname "$0")" && pwd)"
OUT="$HERE/../_lib"
mkdir -p "$OUT" "$HERE/.obj"
NVCC=${NVCC:-/usr/local/cuda/bin/nvcc}
FLAGS="-gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -std=c++17 -Xcompiler -fPIC -Xcompiler -O2 --expt-relaxed-constexpr ${NVCC_EXTRA}"
pids=()
for f in api_common seq_embed misc_kernels gemm_simt gemm_api gemm_tc lstm lstm_mma attn_pool sue sue_tail topk; do
  src="$HERE/$f.cu"; obj="$HERE/.obj/$f.o"
  if [ ! -f "$obj" ] || [ "$src" -nt "$obj" ] || [ "$HERE/common.cuh" -nt "$obj" ] || [ "$HERE/gemm_epilogue.cuh" -nt "$obj" ] || [ "$HERE/lstm_common.cuh" -nt "$obj" ] || [ "$HERE/../../include/nnr_b200.h" -nt "$obj" ]; then
    ( $NVCC $FLAGS ${PTXAS_V:+-Xptxas -v} -c "$src" -o "$obj" 2>&1 | sed "s/^/[$f] /" ; exit ${PIPESTATUS[0]} ) &
    pids+=($!)
  fi
done
rc=0
for p in "${pids[@]}"; do wait $p || rc=1; done
[ $rc -eq 0 ] || { echo "compile failed"; exit 1; }
$NVCC -gencode arch=compute_100a,code=sm_100a -shared -o "$OUT/libnnr_b200.so" "$HERE"/.obj/*.o -lcudart_static -lcuda -ldl -lrt -lpthread
echo "built $OUT/libnnr_b200.so"
