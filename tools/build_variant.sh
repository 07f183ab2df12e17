#!/bin/bash
# Developer tool: builds build/variants/libmlb200_<name>.so with extra nvcc flags (e.g. -maxrregcount=96) so that
# tools/quick_bench.py can time experimental kernels side by side (MLB200_LIB=<path> python tools/quick_bench.py ...).
set -e
name=$1; shift
cd "$(dirname "$0")/.."
mkdir -p build/variants/$name
for f in context seeding em kmeans selftest; do
  /usr/local/cuda/bin/nvcc -O3 -std=c++17 -gencode arch=compute_100a,code=sm_100a -lineinfo -Xcompiler -fPIC "$@" \
      -c ml_b200/csrc/$f.cu -o build/variants/$name/$f.o &
done
wait
/usr/local/cuda/bin/nvcc -gencode arch=compute_100a,code=sm_100a -shared -o build/variants/libmlb200_$name.so build/variants/$name/*.o -ldl
echo build/variants/libmlb200_$name.so
