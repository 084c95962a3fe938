#!/bin/bash
# Build a differently-compiled libchaos_b200 under build/variants/ for A/B runs on the GPU box:
#   tools/build_variant.sh NAME [-DMACRO=VALUE ...]   ->  build/variants/lib_NAME.so
# Select it at run time with CHAOS_B200_LIB=build/variants/lib_NAME.so
set -e
cd "$(dirname "$0")/.."
name=$1; shift
out=build/variants; mkdir -p $out/obj_$name
A="-gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -std=c++17 -Xcompiler -fPIC -Xcompiler -fno-fast-math"
S=gym_lorenz_b200/csrc
nvcc $A -fmad=false "$@" -c $S/tu_parity.cu -o $out/obj_$name/tu_parity.o &
nvcc $A "$@" -c $S/tu_northstar.cu -o $out/obj_$name/tu_northstar.o &
nvcc $A -fmad=false "$@" -c $S/tu_rl_ops.cu -o $out/obj_$name/tu_rl_ops.o &
nvcc $A -fmad=false "$@" -c $S/tu_policy.cu -o $out/obj_$name/tu_policy.o &
nvcc $A "$@" -c $S/chaos_b200.cu -o $out/obj_$name/chaos_b200.o &
wait
nvcc -gencode arch=compute_100a,code=sm_100a -shared -cudart static -o $out/lib_$name.so $out/obj_$name/*.o
echo $out/lib_$name.so
