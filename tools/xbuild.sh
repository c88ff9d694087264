#!/bin/bash
# Build the working tree's decode library under another name for kernel experiments (A/B runs against base):
#   bash tools/xbuild.sh <name> [extra nvcc flags, e.g. -Xptxas -v]   ->  structuredetector_b200/csrc/exp/lib_<name>.so
# and run with SDNET_DECODE_LIB=structuredetector_b200/csrc/exp/lib_<name>.so, or time it with tools/sweep.py base <name>
name=$1; shift
mkdir -p structuredetector_b200/csrc/exp
nvcc -gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -std=c++17 -prec-div=true -prec-sqrt=true -ftz=false \
  -Xcompiler -fPIC -shared -Iinclude "$@" -o structuredetector_b200/csrc/exp/lib_$name.so structuredetector_b200/csrc/sdnet_decode.cu
