#!/bin/bash
# A/B timing of library variants built by tools/build_variant.sh: tools/ab.sh <mode> <reps> <variant>...
# Runs `tools/prof_kernels.py <mode> <reps>` once per variant with build_variants/lib_<variant>.so in place of the
# shipped library, then restores it.  Output -> stdout and gpurun_out/ab.log.
mode=$1; reps=$2; shift 2
lib=cmt-cooperative-perception_b200/libcmtcoop_b200.so
mkdir -p gpurun_out
shipped=$(mktemp)
cp $lib $shipped || exit 1
# put the shipped library back however the script ends, so that no variant is left in the tree
trap 'cp $shipped $lib; rm -f $shipped' EXIT
for v in "$@"; do
  cp build_variants/lib_$v.so $lib
  echo "== $v: $(timeout 300 python tools/prof_kernels.py $mode $reps 2>&1 | tr '\n' ' ')" | tee -a gpurun_out/ab.log
done
