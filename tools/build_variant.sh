#!/bin/bash
# Build a kernel variant of libhgi_b200.so for tools/ab_bench.py:  tools/build_variant.sh NAME [-DFLAG ...]
# Recompiles the fast tile kernel with the extra flags into build/NAME/ and links it with the stock objects.
# Compile-time hooks of the kernel:
#   -DHGI_FAST_MIN_BLOCKS=n / -DHGI_FAST_MIN_BLOCKS_LIGHT=n   CTAs per SM (quantizing encode / light kernels)
#   -DHGI_VAR_POISON_SMEM=0xXX   the shared-memory planes start as this byte pattern (see hgi_tile_fast.cu)
# Run-time knobs for tools/ab_bench.py (name=lib.so,ENV=VALUE): HGI_B200_PREFETCH, HGI_B200_SPLIT_MIN
set -e
cd "$(dirname "$0")/../rustyhgi_b200/csrc"
name=$1; shift
out=../../build/$name; mkdir -p $out
NV="/usr/local/cuda/bin/nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -lineinfo -Xcompiler -fPIC -fmad=false"
$NV "$@" -c -o $out/hgi_tile_fast.o hgi_tile_fast.cu
$NV -shared -cudart static -o ../../build/libhgi_$name.so $out/hgi_tile_fast.o hgi_capi.o hgi_reduce_kernels.o hgi_region.o hgi_archive.o -lz
echo built build/libhgi_$name.so
