"""bf16 against fp16 compute precision on the default bench workload (CmtHead nuScenes, configs[2], B = 8, bf16 features),
in one process: step time from CUDA-graph replays, which attention instantiation the items take, and frame-0 parity.

    python tools/precision_bench.py [--steps 20] [--warmup 5] [--rounds 3] [--out results/precision_bench.json]

One head per precision (same synthetic weights), each captured in its own graph.  The timed windows alternate
bf16, fp16, bf16, fp16, ... (`--rounds` windows of `--steps` replays each per precision, every window between two
device synchronisations, CUDA events), so both see the same clocks and neighbours.  Prints one JSON line with
  gpu                    name, power limit and max SM clock of the card (read-only nvidia-smi query);
  ms_per_step            per precision: median over the windows, and min / max;
  static_item_fraction   per precision: share of the cross-attention items (layer, frame, head) whose operand-norm score
                         bound is within the dtype's static-shift limit (60 bf16, 14 fp16), from fused_decoder.last_norms;
  rel_l2                 per precision and output: frame 0 of the batch, all six decoder layers, against the fp32 CPU
                         oracle on the same inputs."""
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

from bench import build_case, frame0_inputs  # noqa: E402
from cmtcoop_b200 import ops, synth  # noqa: E402
from cmtcoop_b200.plugin import build_head, fused_decoder  # noqa: E402
from cmtcoop_b200.runtime import GraphedForward  # noqa: E402

PRECISIONS = ("bf16", "fp16")


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.TimeoutExpired):
        q = ""
    return q or torch.cuda.get_device_name(0)


def static_fraction(precision):
    """Share of the last forward's attention items on the static-shift kernel (the kernels' own predicate)."""
    if fused_decoder.last_norms is None:
        return 0.0
    qn2, kn2 = fused_decoder.last_norms
    kn = torch.cat([c.permute(1, 0, 2) for c in kn2], 1)            # [L, frames, H]
    bound = torch.sqrt(qn2 * kn) * 1.0079 + 1e-3
    return float((bound <= fused_decoder.STATIC_LIMIT[ops.compute_dtype(precision)]).float().mean())


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--steps", type=int, default=20, help="graph replays per timed window (>= 20)")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=3, help="timed windows per precision, alternating")
    ap.add_argument("--out", help="also write the JSON line to this file")
    args = ap.parse_args()
    if args.steps < 20 or args.warmup < 3 or args.rounds < 1:
        ap.error("--steps >= 20, --warmup >= 3, --rounds >= 1")
    if not torch.cuda.is_available():
        sys.exit("precision_bench.py measures on the GPU: no CUDA device")
    dev = torch.device("cuda", 0)
    B = 8
    kind, cfg, inputs = build_case("nusc", B)   # cfg["_apply_shared_conv"] = False also tells the oracle the bench scope
    feats = {k: torch.from_numpy(v).to(torch.bfloat16).to(dev) for k, v in inputs.items() if isinstance(v, np.ndarray)}
    metas = inputs["img_metas"]

    heads, graphs, static, rets = {}, {}, {}, {}
    with torch.no_grad():
        for p in PRECISIONS:
            head = build_head({k: v for k, v in cfg.items() if not k.startswith("_")})
            synth.load_synth_weights(head, 0)
            head = head.to(dev).eval().set_precision(p)
            head.apply_shared_conv = False   # bench scope: the BEV input is the post-shared_conv map
            for _ in range(args.warmup):
                rets[p] = head.forward_single(feats["pts_feats"], feats["img_feats"], metas)
            torch.cuda.synchronize()
            static[p] = static_fraction(p)
            rets[p] = [{n: t.float().cpu() for n, t in r.items()} for r in rets[p]]
            graphs[p] = GraphedForward(head, metas, feats, adopt_inputs=True)
            for _ in range(args.warmup):
                graphs[p]()
            heads[p] = head
        times = {p: [] for p in PRECISIONS}
        for _ in range(args.rounds):
            for p in PRECISIONS:
                torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(args.steps):
                    graphs[p]()
                e1.record()
                torch.cuda.synchronize()
                times[p].append(e0.elapsed_time(e1) / args.steps)

    from oracle import cmt_oracle as O
    torch.set_num_threads(os.cpu_count() or 1)
    sd = {k: v.detach().float().cpu() for k, v in heads["bf16"].state_dict().items()}
    with torch.no_grad():
        want = O.head_forward(sd, cfg, frame0_inputs(inputs, B, False, torch.bfloat16))[0][0]
    rel = {p: {n: O.rel_l2(rets[p][0][n][:, :1], want[n]) for n in want} for p in PRECISIONS}

    line = dict(
        tool="precision_bench", workload="nusc (CmtHead, configs[2]): 6 cams x 40x100 + 180x180 BEV, 900 queries, 6 layers",
        batch=B, feat_dtype="bf16", gpu=gpu_info(), steps_per_window=args.steps, windows=args.rounds,
        ms_per_step={p: dict(median=statistics.median(times[p]), min=min(times[p]), max=max(times[p]), windows=times[p])
                     for p in PRECISIONS},
        static_item_fraction=static, static_limit={p: fused_decoder.STATIC_LIMIT[ops.compute_dtype(p)] for p in PRECISIONS},
        rel_l2=rel, rel_l2_worst={p: max(rel[p].values()) for p in PRECISIONS},
        rel_l2_note="frame 0 of the batch, all 6 decoder layers, against the fp32 CPU oracle on the same bf16 features")
    text = json.dumps(line)
    print(text, flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
