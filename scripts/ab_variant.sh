#!/bin/bash
# A/B helper: build a variant of libfdcm_b200.so with extra -D flags into build/ab/<name>/libfdcm_b200.so
#   scripts/ab_variant.sh <name> "<-D flags>" file1.cu [file2.cu ...]     (only the listed sources are recompiled)
# run it with: python scripts/ab_run.py build/ab/<name>/libfdcm_b200.so scripts/bench_build.py L2 10
set -e
name=$1; flags=$2; shift 2
src=openfdcm_b200/csrc
out=build/ab/$name
mkdir -p $out
NVCCFLAGS="-gencode arch=compute_100a,code=sm_100a -std=c++17 -O3 -lineinfo -fmad=false -prec-div=true -prec-sqrt=true -Xcompiler -fPIC,-O3,-fno-math-errno,-ffp-contract=off"
objs=""
for cu in $(sed -n 's/^SRCS *= *//p' $src/Makefile); do   # every source the library links, as the Makefile lists them
  f=${cu%.cu}
  if [[ " $* " == *" $f.cu "* ]]; then
    /usr/local/cuda/bin/nvcc $NVCCFLAGS $flags -c $src/$f.cu -o $out/$f.o
    objs="$objs $out/$f.o"
  else
    objs="$objs $src/$f.o"
  fi
done
/usr/local/cuda/bin/nvcc -gencode arch=compute_100a,code=sm_100a -shared -o $out/libfdcm_b200.so $objs -lcudart_static -lpthread -ldl -lrt
echo built $out/libfdcm_b200.so
