#!/bin/bash
# dev tool: A/B builds of the Gram kernels on top of a -DRDB_DEV_SWITCHES build (RDB_GRAM_IMPL=ring|slots selects the kernel at run time)
set -e
cd "$(dirname "$0")/.."
NV="/usr/local/cuda/bin/nvcc -O3 -std=c++17 -gencode arch=compute_100a,code=sm_100a -lineinfo -Xcompiler -fPIC -ccbin /usr/bin/g++ -DRDB_DEV_SWITCHES"
mkdir -p build/obj_dev
for src in kernels.cu gram.cu gram_fused.cu gram_ring.cu gram_jit.cpp gram_jit_headers.cpp components.cu aux.cu ik.cu group.cu capi.cu urdf.cpp solve.cpp fold.cpp; do
  f=${src%.*}
  if [ "$src" = gram.cu ] || [ "$src" = gram_fused.cu ] || [ "$src" = gram_ring.cu ]; then
    $NV -c rosdyn_b200/csrc/$src -o build/obj_dev/$f.o &
  else
    cp build/$f.o build/obj_dev/$f.o
  fi
done
wait
link() { # name, extra objects override
  mkdir -p build/var_$1
  /usr/local/cuda/bin/nvcc -shared -cudart static -ccbin /usr/bin/g++ -gencode arch=compute_100a,code=sm_100a -o build/var_$1/librosdyn_b200.so "${@:2}" -ldl
}
objs() { for f in kernels gram gram_fused gram_ring gram_jit gram_jit_headers components aux ik group capi urdf solve fold; do echo build/obj_dev/$f.o; done; }
link dev $(objs)
for v in "$@"; do
  case $v in
    unpaired) $NV -DRING_UNPAIRED -c rosdyn_b200/csrc/gram_ring.cu -o build/obj_dev/gram_ring_$v.o ;;
    nofence) $NV -DRING_NO_THREADFENCE -c rosdyn_b200/csrc/gram_ring.cu -o build/obj_dev/gram_ring_$v.o ;;
    eager)   $NV -DRING_EAGER_LOADS -c rosdyn_b200/csrc/gram_ring.cu -o build/obj_dev/gram_ring_$v.o ;;
    nofence_eager) $NV -DRING_NO_THREADFENCE -DRING_EAGER_LOADS -c rosdyn_b200/csrc/gram_ring.cu -o build/obj_dev/gram_ring_$v.o ;;
    *) $NV $RING_FLAGS -c rosdyn_b200/csrc/gram_ring.cu -o build/obj_dev/gram_ring_$v.o ;;
  esac
  link $v $(objs | sed "s#gram_ring.o#gram_ring_$v.o#")
done
ls build/var_*/librosdyn_b200.so
