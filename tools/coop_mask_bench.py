"""Cost of the per-frame node mask (`node_valid`) of the cooperative heads on the B200.

    python tools/coop_mask_bench.py [--steps 20] [--rounds 4] [--out results/coop_mask_bench.json]

Prints the GPU name and power limit of the same run, then for coop_lidar and coop_fusion at B = 8 (bench.py's workloads
and scope, bf16 features, graph replay including the batched box decode):
  1. ms per step of three captured graphs: no mask, an all-true mask, a mixed mask (every frame state present),
     alternated `--rounds` times;
  2. CUDA-event time per launch of cmt_split3_bf16 (the decoder's real output shape, both nodes stacked) and of
     cmt_bbox_topk_decode (900 queries x 7 classes, K = 300), with and without the mixed mask, alternated.
Medians over the rounds; the spread (min-max) is printed next to every number.  An absent node's frames still run
through the decoder, so the step times are expected to differ by noise only."""
import argparse
import json
import os
import statistics
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from bench import build_case  # noqa: E402
from cmtcoop_b200 import ops, synth  # noqa: E402
from cmtcoop_b200.plugin import MultiTaskBBoxCoder, build_head  # noqa: E402
from cmtcoop_b200.runtime import GraphedForward  # noqa: E402

DEV = torch.device("cuda", 0)
B = 8
MIXED = [[True, True, False, False, True, True, True, False], [True, False, True, False, True, False, True, True]]


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.TimeoutExpired):
        q = ""
    return q or torch.cuda.get_device_name(0)


def spread(xs):
    return dict(median=statistics.median(xs), min=min(xs), max=max(xs))


def fmt(d, unit):
    return f"{d['median']:.4f} {unit} ({d['min']:.4f}-{d['max']:.4f})"


def timed(fn, n):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n


def alternate(fns, n, rounds):
    out = {k: [] for k in fns}
    for _ in range(rounds):
        for k, fn in fns.items():
            out[k].append(timed(fn, n))
    return {k: spread(v) for k, v in out.items()}


def bench_workload(workload, steps, rounds):
    kind, cfg, inputs = build_case(workload, B)
    head = build_head({k: v for k, v in cfg.items() if not k.startswith("_")})
    synth.load_synth_weights(head, 0)
    head = head.to(DEV).eval().set_precision("bf16")
    head.apply_shared_conv = False
    metas = inputs["img_metas"]
    feats = {k: torch.from_numpy(v).to(torch.bfloat16).to(DEV) for k, v in inputs.items() if isinstance(v, np.ndarray)}
    modes = {"no_mask": None, "all_true": torch.ones(2, B, dtype=torch.bool, device=DEV),
             "mixed": torch.tensor(MIXED, dtype=torch.bool, device=DEV)}
    with torch.no_grad():
        graphs = {k: GraphedForward(head, metas, feats if m is None else dict(feats, node_valid=m), adopt_inputs=True,
                                    decode_boxes=True) for k, m in modes.items()}
        for g in graphs.values():
            for _ in range(3):
                g()
        step = alternate(graphs, steps, rounds)
    del graphs
    return step


def bench_kernels(reps, rounds):
    L, Nq = 6, 900
    g = torch.Generator().manual_seed(0)
    outs = torch.randn(L, 2 * B, Nq, 256, generator=g).to(DEV)
    mask = torch.tensor(MIXED, dtype=torch.bool, device=DEV)
    coder = MultiTaskBBoxCoder(pc_range=synth.TUMTRAF_RANGE, post_center_range=[-80, -80, -10.0, 80, 80, 10.0],
                               max_num=300, num_classes=7)
    preds = [[{n: torch.randn(1, B, Nq, w, generator=g).to(DEV)
               for n, w in dict(center=2, height=1, dim=3, rot=2, vel=2, cls_logits=7).items()}]]
    fns = {"split3": lambda: ops.split3(outs, stacked_nodes=True),
           "split3_masked": lambda: ops.split3(outs, stacked_nodes=True, node_valid=mask),
           "decode": lambda: coder.decode_batched(preds, bottom_center=True),
           "decode_masked": lambda: coder.decode_batched(preds, bottom_center=True, node_valid=mask)}
    for fn in fns.values():
        for _ in range(5):
            fn()
    return {k: {s: 1e3 * v for s, v in d.items()} for k, d in alternate(fns, reps, rounds).items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20, help="graph replays per timed window")
    ap.add_argument("--rounds", type=int, default=4, help="alternations of the modes")
    ap.add_argument("--reps", type=int, default=200, help="kernel launches per timed window")
    ap.add_argument("--out", default=None, help="also write the results as JSON here")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("coop_mask_bench needs a CUDA device")
    res = dict(gpu=gpu_info(), B=B, mixed_mask=MIXED)
    print(f"GPU (name, power limit, max SM clock): {res['gpu']}")
    for w in ("coop_lidar", "coop_fusion"):
        res[w] = bench_workload(w, args.steps, args.rounds)
        print(f"{w} B={B} graph step (heads + decode): " +
              " | ".join(f"{k} {fmt(v, 'ms')}" for k, v in res[w].items()))
    res["kernels_us"] = bench_kernels(args.reps, args.rounds)
    print("per launch (CUDA events): " + " | ".join(f"{k} {fmt(v, 'us')}" for k, v in res["kernels_us"].items()))
    print(json.dumps(res))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
