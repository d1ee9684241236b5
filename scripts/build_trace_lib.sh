#!/bin/bash
# Trace build of the 128-wide gradient kernel: qb_grad_tc128.cu with -DQB_TG8_TRACE, the other objects from build/obj.
set -e
cd "$(dirname "$0")/.."
nvcc -gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -std=c++17 -c -Xcompiler -fPIC -DQB_TG8_TRACE -I include -I quinn_b200/csrc \
     -o build/obj/qb_grad_tc128_trace.o quinn_b200/csrc/qb_grad_tc128.cu
nvcc -gencode arch=compute_100a,code=sm_100a --shared -o quinn_b200/lib/libquinn_b200_trace.so build/obj/qb_kernels.o build/obj/qb_launch.o build/obj/qb_grad_tc.o \
     build/obj/qb_grad_tc128_trace.o build/obj/qb_value_tc3.o build/obj/qb_post.o
