#!/bin/bash
# Library variants for same-box A/B runs of compile-time switches: tools/build_variants.sh "name:-DFLAG=.. -DFLAG2=.." ...
# (only the L=8 objects k1 / k2 are rebuilt per variant); results in gpu_variants/libpolar_b200_<name>.so
set -e
ROOT=$(cd "$(dirname "$0")/.." && pwd)
OUT=$ROOT/gpu_variants
cd "$ROOT/quantized_decoder_polar_codes_b200"
F="-gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -std=c++17 -fmad=false -Xcompiler -fPIC"
mkdir -p "$OUT"
OBJS=$(ls build/*.o | grep -v "_v_\|/k1.o\|/k2.o")
for spec in "$@"; do
  name=${spec%%:*}; flags=${spec#*:}
  nvcc $F -DPB_TU=1 $flags -c csrc/pb_kernels.cu -o build/k1_v_$name.o &
  nvcc $F -DPB_TU=2 $flags -c csrc/pb_kernels.cu -o build/k2_v_$name.o &
done
wait
for spec in "$@"; do
  name=${spec%%:*}
  nvcc -shared -gencode arch=compute_100a,code=sm_100a -o "$OUT/libpolar_b200_$name.so" $OBJS build/k1_v_$name.o build/k2_v_$name.o
done
ls -la "$OUT"
