#!/bin/bash
# A/B helper: builds flowcompare_b200/variants/lib_<name>.so with extra -D flags for ONE source file.
#   scripts/build_variant.sh spl2 attention_tc "-DA_SPL=2"
# and run with FLOWCOMPARE_B200_LIB=flowcompare_b200/variants/lib_spl2.so python bench.py ...
set -e
name=$1; src=$2; flags=$3
mkdir -p build/var_$name flowcompare_b200/variants
nvcc -gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -std=c++17 -Xcompiler -fPIC -Xcompiler -fvisibility=hidden -diag-suppress 177 -Wno-deprecated-gpu-targets $flags \
  -c flowcompare_b200/csrc/$src.cu -o build/var_$name/$src.o
objs=$(ls build/*.o | grep -v "/$src.o")
nvcc -shared -o flowcompare_b200/variants/lib_$name.so $objs build/var_$name/$src.o -lcuda
echo built flowcompare_b200/variants/lib_$name.so
