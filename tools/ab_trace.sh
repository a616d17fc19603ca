#!/bin/bash
# tools/ab_trace.sh <lo> <hi> <variant>...: tools/attn_trace.py under each trace-built variant (see tools/ab.sh)
lo=$1; hi=$2; shift 2
lib=cmt-cooperative-perception_b200/libcmtcoop_b200.so
mkdir -p gpurun_out
shipped=$(mktemp)
cp $lib $shipped || exit 1
# put the shipped library back however the script ends, so that no variant is left in the tree
trap 'cp $shipped $lib; rm -f $shipped' EXIT
for v in "$@"; do
  cp build_variants/lib_$v.so $lib
  echo "== $v" | tee -a gpurun_out/trace.log
  timeout 300 python tools/attn_trace.py $lo $hi 2>&1 | tee -a gpurun_out/trace.log
done
