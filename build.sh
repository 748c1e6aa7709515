#!/bin/bash
# Builds libb200compact.so (sm_100a only) in-tree, the CPU oracle (test infrastructure) and the input generator bench.py loads.
set -e
cd "$(dirname "$0")"
NVCC=${NVCC:-/usr/local/cuda/bin/nvcc}
OUT=cassandra_b200/libb200compact.so
SRCS=$(ls cassandra_b200/csrc/*.cu)
$NVCC -gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -std=c++17 -Xcompiler -fPIC,-Wall,-Wno-unused-function \
      -Xptxas -v -shared -o $OUT.tmp $SRCS 2> build_ptxas.log || { cat build_ptxas.log; rm -f $OUT.tmp; exit 1; }
mv -f $OUT.tmp $OUT          # atomically: a gpurun snapshot taken meanwhile sees the old or the new library, never half of one
grep -E "error|warning" build_ptxas.log | grep -v "ptxas info" | head -20 || true
make -C oracle -s
make -C synth -s
echo "built $OUT"
