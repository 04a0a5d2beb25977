#!/bin/bash
# dev tool: build an experimental variant of the library into build/var_<name>/:
#   tools/build_variant.sh <name> [--only file.cu] <extra nvcc flags...>     (objects of untouched files are reused from build/)
set -e
cd "$(dirname "$0")/.."
name=$1; shift
only=""
if [ "$1" = "--only" ]; then only=$2; shift 2; fi
mkdir -p build/var_$name
# the kernel headers as text for the run-time compiled Gram kernels (gram_jit.cpp), generated from csrc/ as rosdyn_b200/build.py does
python -c "from rosdyn_b200 import build; build._write_jit_headers()"
for src in kernels.cu gram.cu gram_fused.cu gram_jit.cpp components.cu aux.cu ik.cu group.cu capi.cu urdf.cpp solve.cpp fold.cpp ../../build/gram_jit_headers.cpp; do
  f=$(basename ${src%.*})
  if [ -n "$only" ] && [ "$src" != "$only" ] && [ -f build/$f.o ]; then cp build/$f.o build/var_$name/$f.o; continue; fi
  /usr/local/cuda/bin/nvcc -O3 -std=c++17 -gencode arch=compute_100a,code=sm_100a -lineinfo -Xcompiler -fPIC -ccbin /usr/bin/g++ "$@" -c rosdyn_b200/csrc/$src -o build/var_$name/$f.o &
done
wait
/usr/local/cuda/bin/nvcc -shared -cudart static -ccbin /usr/bin/g++ -gencode arch=compute_100a,code=sm_100a -o build/var_$name/librosdyn_b200.so build/var_$name/*.o -ldl
rm -f build/var_$name/*.o
echo build/var_$name/librosdyn_b200.so
