"""Cost of the single-node heads' per-frame sensor mask (`sensor_valid`) on the B200.

    python tools/sensor_mask_bench.py [--steps 20] [--rounds 4] [--out results/sensor_mask_bench.json]

Prints the GPU name and power limit of the same run, then for bench.py's default workload (nusc: CmtHead, 6 cameras x
40x100 + 180x180 BEV = 56 400 tokens, B = 8, bf16 features, bench.py's scope) the ms per step of three captured graphs
(heads + batched box decode): no mask, an all-true mask and a mixed mask (a missing camera, a missing LiDAR sweep, a
frame with no sensor), alternated `--rounds` times.  Medians over the rounds with the spread (min-max).  An absent
sensor's work is not skipped, so a masked step differs from the unmasked one by the masked attention instantiation,
the key-keep build and one key-mask pack per decoder layer."""
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
from cmtcoop_b200 import synth  # noqa: E402
from cmtcoop_b200.plugin import build_head  # noqa: E402
from cmtcoop_b200.runtime import GraphedForward  # noqa: E402

DEV = torch.device("cuda", 0)
B = 8
V = 6
# per frame (LiDAR, camera 0..5): all present, camera 3 missing, LiDAR missing, cameras 0 and 5 missing, nothing,
# cameras only, LiDAR only, all present
MIXED_FRAMES = [(1, 1, 1, 1, 1, 1, 1), (1, 1, 1, 1, 0, 1, 1), (0, 1, 1, 1, 1, 1, 1), (1, 0, 1, 1, 1, 1, 0),
                (0, 0, 0, 0, 0, 0, 0), (0, 1, 1, 1, 1, 1, 1), (1, 0, 0, 0, 0, 0, 0), (1, 1, 1, 1, 1, 1, 1)]


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


def bench_workload(steps, rounds):
    kind, cfg, inputs = build_case("nusc", B)
    head = build_head({k: v for k, v in cfg.items() if not k.startswith("_")})
    synth.load_synth_weights(head, 0)
    head = head.to(DEV).eval().set_precision("bf16")
    head.apply_shared_conv = False
    metas = inputs["img_metas"]
    feats = {k: torch.from_numpy(v).to(torch.bfloat16).to(DEV) for k, v in inputs.items() if isinstance(v, np.ndarray)}
    mixed = torch.tensor(MIXED_FRAMES, dtype=torch.bool).t().contiguous().to(DEV)   # [1 + V, B]
    modes = {"no_mask": None, "all_true": torch.ones(1 + V, B, dtype=torch.bool, device=DEV), "mixed": mixed}
    with torch.no_grad():
        graphs = {k: GraphedForward(head, metas, feats if m is None else dict(feats, sensor_valid=m), adopt_inputs=True,
                                    decode_boxes=True) for k, m in modes.items()}
        for g in graphs.values():
            for _ in range(3):
                g()
        step = alternate(graphs, steps, rounds)
    return step


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20, help="graph replays per timed window")
    ap.add_argument("--rounds", type=int, default=4, help="alternations of the modes")
    ap.add_argument("--out", default=None, help="also write the results as JSON here")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("sensor_mask_bench needs a CUDA device")
    res = dict(gpu=gpu_info(), workload="nusc", B=B, mixed_frames=MIXED_FRAMES)
    print(f"GPU (name, power limit, max SM clock): {res['gpu']}")
    res["step_ms"] = bench_workload(args.steps, args.rounds)
    print(f"nusc B={B} graph step (heads + decode): " + " | ".join(f"{k} {fmt(v, 'ms')}" for k, v in res["step_ms"].items()))
    print(json.dumps(res))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
