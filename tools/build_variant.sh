#!/bin/bash
# Builds an experimental variant of the library into build_variants/lib_<name>.so:
#   tools/build_variant.sh <name> <copy.cu> [nvcc flags...]
# <copy.cu> is an edited copy of one csrc/ source under the same file name (e.g. /tmp/v1/attn_tcgen05.cu): it replaces
# that source's object, the other objects come from the normal build (make first).  The sources have no tuning knobs, so a
# variant is an edit of the copy; the only defines are -DCMT_ATTN_TRACE (attention event trace) and -DCMT_TRAP_REPORT
# (wait-timeout records).
set -e
name=$1; src=$(realpath "$2"); shift 2
cd "$(dirname "$0")/../cmt-cooperative-perception_b200/csrc"
mkdir -p ../../build_variants
obj=../../build_variants/${name}_$(basename $src .cu).o
nvcc -O3 -std=c++17 -lineinfo -gencode arch=compute_100a,code=sm_100a -Xcompiler -fPIC -Xptxas -v --expt-relaxed-constexpr -I. "$@" -c $src -o $obj 2> ../../build_variants/${name}.ptxas.log
others=$(ls *.o | grep -v "^$(basename $src .cu).o$")
nvcc -gencode arch=compute_100a,code=sm_100a -shared -o ../../build_variants/lib_${name}.so $obj $others -cudart static
grep -A1 "tc_attn_db_kernel\|Compiling.*$(basename $src .cu)" ../../build_variants/${name}.ptxas.log | grep -E "registers|spill" | head -4
