#!/bin/bash
# Builds an A/B variant of libising_b200.so with extra nvcc flags into scratch_ab/lib_<tag>.so (git-ignored, ships to
# the GPU box); select it at run time with ISING_B200_LIB=$PWD/scratch_ab/lib_<tag>.so.
#   scripts/build_variant.sh timing -DISB_TC_TIMING
set -eu
tag=$1; shift
root=$(cd "$(dirname "$0")/.." && pwd)
w=$(mktemp -d)
mkdir -p "$w/pkg/csrc" "$w/include" "$root/scratch_ab"
cp "$root"/isingmodel.jl_b200/csrc/*.cu "$root"/isingmodel.jl_b200/csrc/*.cuh "$root"/isingmodel.jl_b200/csrc/*.hpp \
   "$root"/isingmodel.jl_b200/csrc/Makefile "$w/pkg/csrc/"
cp "$root"/include/*.h "$w/include/"
make -C "$w/pkg/csrc" -j8 EXTRA="$*" > /dev/null
cp "$w/pkg/libising_b200.so" "$root/scratch_ab/lib_$tag.so"
rm -rf "$w"
echo "scratch_ab/lib_$tag.so"
