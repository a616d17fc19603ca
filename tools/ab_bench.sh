#!/bin/bash
# In-step A/B of library variants (tools/build_variant.sh): runs bench.py with each build_variants/lib_<v>.so in place of the
# shipped library and prints value / attention per-launch time (static + online) -- the attention kernel's clock depends on
# what runs around it, so back-to-back launches of the kernel alone (tools/ab.sh) rank variants differently.
lib=cmt-cooperative-perception_b200/libcmtcoop_b200.so
mkdir -p gpurun_out
shipped=$(mktemp)
cp $lib $shipped || exit 1
# put the shipped library back however the script ends, so that no variant is left in the tree
trap 'cp $shipped $lib; rm -f $shipped' EXIT
for v in "$@"; do
  cp build_variants/lib_$v.so $lib
  timeout 300 python bench.py --steps 20 --warmup 4 --no-cpu-baseline --no-parity --no-shared-conv-leg > /tmp/ab_$v.json 2> /tmp/ab_$v.err
  python - "$v" <<'PY' | tee -a gpurun_out/ab_bench.log
import json, sys
v = sys.argv[1]
try:
    d = json.loads(open(f"/tmp/ab_{v}.json").read().strip().splitlines()[-1])
    r = d["roofline"]
    print(f"== {v}: value {d['value']:.1f} ms/step {d['ms_per_step']:.3f} attn {r['avg_launch_ms']*1e3:.1f} us online {r['online_kernel']['avg_launch_ms']*1e3:.1f} us clk {r['sm_clock_ghz_under_kernel']:.3f} e2e {d['e2e']['value']:.1f}")
except Exception as e:
    print(f"== {v}: FAILED {e}", open(f"/tmp/ab_{v}.err").read()[-500:])
PY
done
