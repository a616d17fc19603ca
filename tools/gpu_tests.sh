#!/bin/bash
# Runs the GPU parity suites one file/group at a time under a timeout so that a fault in one
# kernel family cannot take the others (or the box) down with it.  Logs -> gpurun_out/.
mkdir -p gpurun_out
nvidia-smi --query-gpu=name,clocks.sm,clocks.max.sm,power.draw --format=csv > gpurun_out/smi.txt 2>&1
run() {
  name=$1; shift
  echo "=== $name"
  timeout 900 python -m pytest -m gpu -q --no-header -p no:cacheprovider "$@" > gpurun_out/test_$name.log 2>&1
  echo "exit=$? $(tail -n 3 gpurun_out/test_$name.log | tr '\n' ' ')"
}
run simple tests/test_gpu_kernels.py -k "not gemm and not attention"
run gemm tests/test_gpu_kernels.py -k "gemm"
run gemm_geometry tests/test_gpu_gemm_geometry.py
run forward_replay tests/test_gpu_forward_replay.py
run attn tests/test_gpu_kernels.py -k "attention"
run attn_edges tests/test_gpu_attention_edges.py
run heads tests/test_gpu_heads.py
run decoder tests/test_gpu_decoder.py
run multi tests/test_gpu_multi.py
run decode tests/test_gpu_bbox_decode.py
run fp16 tests/test_gpu_fp16.py
run node_mask tests/test_gpu_coop_node_mask.py
run sensor_mask tests/test_gpu_sensor_mask.py
