#!/bin/bash
# Experiment helper: rebuild ONE translation unit with extra -D flags and link it with the production objects into
# speech_separation_b200/variants/libvatss_<name>.so (git-ignored; select it with VATSS_LIB_OVERRIDE=<path>).
#   tools/build_variant.sh poly2 tc_attn3 -DA3_POLY=2
# VARIANT_SRC=<file.cu> compiles that file in place of <unit>.cu (an edited copy kept outside the tree, e.g. a mutant
# for checking that the tests catch a bug); its #includes resolve against csrc/.
set -e
name=$1; unit=$2; shift 2
src=$(realpath "${VARIANT_SRC:-$(dirname "$0")/../speech_separation_b200/csrc/$unit.cu}")
cd "$(dirname "$0")/../speech_separation_b200/csrc"
mkdir -p build/var ../variants
ARCH="-gencode arch=compute_100a,code=sm_100a"
/usr/local/cuda/bin/nvcc -O3 -std=c++17 -lineinfo $ARCH -Xcompiler -fPIC,-Wall,-Wno-unused-function -I. "$@" -c "$src" -o build/var/${unit}_$name.o
# every translation unit of the production library, in the Makefile's order (SRCS)
units=$(make -s --no-print-directory -f Makefile -f - print-srcs <<<'print-srcs: ; @echo $(SRCS:.cu=)')
[ -n "$units" ] || { echo "no SRCS in Makefile" >&2; exit 1; }
make -s -j "$(nproc)" $(for o in $units; do echo build/$o.o; done)
objs=""
for o in $units; do
  if [ $o == $unit ]; then objs="$objs build/var/${unit}_$name.o"; else objs="$objs build/$o.o"; fi
done
/usr/local/cuda/bin/nvcc $ARCH -shared -o ../variants/libvatss_$name.so $objs -lcudart_static -lpthread -ldl -lrt
echo built ../variants/libvatss_$name.so
