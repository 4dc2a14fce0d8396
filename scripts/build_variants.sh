#!/bin/bash
# Build A/B variants of libgsx.so that differ only in the compile-time switches of one translation unit.
#   scripts/build_variants.sh gsx_sor.cu  base:""  tma:"-DGSX_KNN_TMA=1"  i64:"-DGSX_KNN_I32=0"
# -> 3dgsconverter_b200/lib/variants/libgsx_<name>.so (not tracked; they travel to the GPU box with gpurun)
# GSX_VARIANT_DIR=<dir> puts the objects and libraries under <dir> instead (the tests build theirs in a temporary
# directory, so the tree is only read).
set -e
cd "$(dirname "$0")/../3dgsconverter_b200/csrc"
make -j8 >/dev/null
TU=$1; shift
LIBDIR=${GSX_VARIANT_DIR:-../lib/variants}
OBJDIR=${GSX_VARIANT_DIR:-../build_var}
mkdir -p "$LIBDIR" "$OBJDIR"
NV="/usr/local/cuda/bin/nvcc -gencode arch=compute_100a,code=sm_100a -O3 -lineinfo --fmad=false -prec-div=true -prec-sqrt=true -std=c++17 -Xcompiler -fPIC,-O2 -ccbin /usr/bin/g++"
OBJS=$(ls ../build/*.o | grep -v "/${TU%.cu}.o")
for spec in "$@"; do
  name=${spec%%:*}; flags=${spec#*:}
  $NV $flags -c -o "$OBJDIR/${TU%.cu}_$name.o" $TU
  /usr/local/cuda/bin/nvcc -gencode arch=compute_100a,code=sm_100a -shared -o "$LIBDIR/libgsx_$name.so" $OBJS "$OBJDIR/${TU%.cu}_$name.o" -ccbin /usr/bin/g++ -Xcompiler -pthread
  echo "built libgsx_$name.so ($flags)"
done
