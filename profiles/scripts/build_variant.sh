#!/bin/bash
# build_variant.sh <name> <file.cu> [-DMACRO=val ...]: rebuild ONE translation unit with extra defines and
# link it with the other (already built) objects into build_variants/<name>.so (select with DCB_LIB_PATH).
set -e
name=$1; src=$2; shift 2
R=$(cd "$(dirname "$0")/../.." && pwd)
C=$R/diffcodec-controlling-latent-diffusion-for-perceptual-video-compression_b200/csrc
B=$R/build_variants
mkdir -p $B
nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -lineinfo -Xcompiler -fPIC --expt-relaxed-constexpr -Xptxas -v \
  -I$R/include -I$C "$@" -c $C/$src -o $B/variant_$name.o 2> $B/variant_$name.log
others=$(ls $C/*.o | grep -v "/${src%.cu}.o")
nvcc -gencode arch=compute_100a,code=sm_100a -shared -o $B/$name.so $B/variant_$name.o $others -cudart static
grep -A1 "k_backwarp_fwd4\|$name" $B/variant_$name.log | grep -i "registers" | head -3
