"""Box decode on the B200: the eager torch coder (CmtHead.get_bboxes) against the batched kernel (get_bboxes_batched,
cmt_bbox_topk_decode), and what moving the decode into the graph does to a serving step.

    python tools/decode_bench.py [--steps 20] [--out results/decode_bench.json]

Prints the GPU name and power limit of the same run, then
  1. at the nuScenes decode shape (900 queries x 10 classes, K = 300) for B = 8 and B = 64: host wall time of
     get_bboxes ending in a synchronise, host wall time of get_bboxes_batched ending in a synchronise, and the kernel's
     CUDA-event time per launch (200 back-to-back launches);
  2. the graph step time of the default bench workload (CmtHead nuScenes, B = 8) with and without decode_boxes,
     alternating the two graphs three times;
  3. PipelinedRunner end to end (graph replay) with outputs="heads" against outputs="boxes": frames/s and D2H bytes
     per step, alternating twice.
Medians over repeats; the spread (min-max) is printed next to every number."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from bench import build_case  # noqa: E402
from cmtcoop_b200 import synth  # noqa: E402
from cmtcoop_b200.plugin import MultiTaskBBoxCoder, build_head  # noqa: E402
from cmtcoop_b200.plugin.cmt_head import CmtHead  # noqa: E402
from cmtcoop_b200.runtime import GraphedForward, PipelinedRunner  # noqa: E402

DEV = torch.device("cuda", 0)


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
    return f"{d['median']:.3f} {unit} ({d['min']:.3f}-{d['max']:.3f})"


def decode_preds(B, Nq=900, C=10, seed=0):
    g = torch.Generator().manual_seed(seed)
    widths = dict(center=2, height=1, dim=3, rot=2, vel=2, cls_logits=C)
    d = {n: torch.randn(1, B, Nq, w, generator=g).to(DEV) for n, w in widths.items()}
    d["center"] *= 40.0
    return [[d]]


def bench_decode(B, reps):
    preds = decode_preds(B)
    coder = MultiTaskBBoxCoder(pc_range=synth.NUSC_RANGE, post_center_range=[-61.2, -61.2, -10.0, 61.2, 61.2, 10.0],
                               max_num=300, num_classes=10)
    head = type("H", (), {"bbox_coder": coder})()
    metas = [dict(box_type_3d=None) for _ in range(B)]

    def wall(fn):
        out = []
        for _ in range(reps):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            fn()
            torch.cuda.synchronize()
            out.append(1e3 * (time.perf_counter() - t0))
        return spread(out)

    eager = lambda: CmtHead.get_bboxes(head, preds, metas)                 # noqa: E731
    batched = lambda: CmtHead.get_bboxes_batched(head, preds, metas)       # noqa: E731
    for _ in range(5):
        eager()
        batched()
    r = dict(B=B, get_bboxes_wall_ms=wall(eager), get_bboxes_batched_wall_ms=wall(batched))
    ev = []
    for _ in range(5):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(200):
            batched()
        e1.record()
        torch.cuda.synchronize()
        ev.append(1e3 * e0.elapsed_time(e1) / 200)
    r["kernel_event_us"] = spread(ev)
    return r


def timed(fn, steps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--reps", type=int, default=30, help="repeats of each host-timed decode")
    ap.add_argument("--out", default=None, help="also write the results as JSON here")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("decode_bench needs a CUDA device")
    res = dict(gpu=gpu_info())
    print(f"GPU (name, power limit, max SM clock): {res['gpu']}")

    res["decode"] = [bench_decode(B, args.reps) for B in (8, 64)]
    for r in res["decode"]:
        print(f"decode B={r['B']:3d} 900x10 K=300: get_bboxes {fmt(r['get_bboxes_wall_ms'], 'ms')} host wall | "
              f"get_bboxes_batched {fmt(r['get_bboxes_batched_wall_ms'], 'ms')} host wall | "
              f"kernel {fmt(r['kernel_event_us'], 'us')} per launch (CUDA events)")

    B = 8
    kind, cfg, inputs = build_case("nusc", B)
    head = build_head({k: v for k, v in cfg.items() if not k.startswith("_")})
    synth.load_synth_weights(head, 0)
    head = head.to(DEV).eval().set_precision("bf16")
    head.apply_shared_conv = False
    metas = inputs["img_metas"]
    keys = [k for k, v in inputs.items() if isinstance(v, np.ndarray)]
    host = {k: torch.from_numpy(inputs[k]).to(torch.bfloat16).pin_memory() for k in keys}
    resident = {k: v.to(DEV) for k, v in host.items()}
    with torch.no_grad():
        graphs = {False: GraphedForward(head, metas, resident, adopt_inputs=True),
                  True: GraphedForward(head, metas, resident, adopt_inputs=True, decode_boxes=True)}
        for g in graphs.values():
            for _ in range(3):
                g()
        step = {False: [], True: []}
        for _ in range(3):
            for dec, g in graphs.items():
                step[dec].append(timed(g, args.steps) / args.steps)
    res["graph_step_ms"] = {"heads": spread(step[False]), "heads+decode_boxes": spread(step[True])}
    print(f"graph step, default workload (B={B}): without decode {fmt(res['graph_step_ms']['heads'], 'ms')} | "
          f"with decode_boxes {fmt(res['graph_step_ms']['heads+decode_boxes'], 'ms')}")
    del graphs

    runners = {o: PipelinedRunner(head, metas, host, DEV, use_cuda_graph=True, outputs=o) for o in ("heads", "boxes")}
    for r in runners.values():
        r.run([host] * 3)
    fps = {o: [] for o in runners}
    for _ in range(2):
        for o, r in runners.items():
            ms = timed(lambda: r.run([host] * args.steps), 1)
            fps[o].append(1e3 * B * args.steps / ms)
    res["runner"] = {o: dict(frames_per_s=spread(fps[o]), d2h_bytes_per_step=runners[o].d2h_bytes) for o in runners}
    for o, r in res["runner"].items():
        print(f"PipelinedRunner outputs={o!r}: {fmt(r['frames_per_s'], 'frames/s')}, D2H {r['d2h_bytes_per_step']} bytes/step")
    print(json.dumps(res))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
