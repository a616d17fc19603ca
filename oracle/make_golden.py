"""TEST INFRASTRUCTURE ONLY.  Generates tests/golden/*.npz by running the UNMODIFIED reference
code (imported through oracle/ref_stub.py from the checkout CMT_REFERENCE_ROOT names) on CPU in fp32, with
the deterministic synthetic weights / inputs of cmtcoop_b200.synth:

    CMT_REFERENCE_ROOT=<checkout of the original project> python oracle/make_golden.py

Each file holds the reference outputs for one head class on the "mini" case
(synth.mini_case): outs_dec, every task-head tensor, top-k indices/scores, and for the
multimodal head the intermediate stages (ray coords, rv/bev position embeddings, query embeds).
"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from cmtcoop_b200 import synth  # noqa: E402
from oracle import ref_stub  # noqa: E402

GOLDEN_DIR = os.path.join(ROOT, "tests", "golden")


def run_reference(kind, cfg, inputs, seed=0, capture=None):
    head = ref_stub.build_reference_head(kind, cfg)
    synth.load_synth_weights(head, seed)
    head.eval()
    t = lambda a: None if a is None else torch.from_numpy(a)
    metas = inputs["img_metas"]
    hooks = []
    if capture is not None:
        def grab(name):
            def hook(_m, _i, out):
                capture[name] = (out[0] if isinstance(out, tuple) else out).detach().clone()
            return hook
        hooks.append(head.transformer.register_forward_hook(grab("outs_dec")))
        if getattr(head, "rv_embedding", None) is not None:
            calls = []
            hooks.append(head.rv_embedding.register_forward_hook(
                lambda _m, i, o: calls.append((i[0].detach().clone(), o.detach().clone()))))
            capture["_rv_calls"] = calls
        if getattr(head, "shared_conv", None) is not None:
            bcalls = []
            hooks.append(head.bev_embedding.register_forward_hook(
                lambda _m, i, o: bcalls.append((i[0].detach().clone(), o.detach().clone()))))
            capture["_bev_calls"] = bcalls
    with torch.no_grad():
        if kind.endswith("Coop"):
            rets = head.forward_single(t(inputs["vehicle_pts_feats"]), t(inputs["infrastructure_pts_feats"]),
                                       t(inputs["vehicle_img_feats"]), t(inputs["infrastructure_img_feats"]), metas)
        else:
            rets = head.forward_single(t(inputs["pts_feats"]), t(inputs["img_feats"]), metas)
        for m in metas:
            m["box_type_3d"] = lambda b, box_dim=9: b
        boxes = head.get_bboxes([[r] for r in rets], metas)
    for h in hooks:
        h.remove()
    return head, rets, boxes


def main():
    os.makedirs(GOLDEN_DIR, exist_ok=True)
    torch.manual_seed(0)
    torch.set_num_threads(8)
    for kind in synth.HEAD_KINDS:
        cfg, inputs = synth.mini_case(kind)
        cap = {}
        head, rets, boxes = run_reference(kind, cfg, inputs, capture=cap)
        out = {}
        for t, d in enumerate(rets):
            for k, v in d.items():
                out[f"task{t}.{k}"] = v.numpy()
        for i, (bb, sc, lb) in enumerate(boxes):
            out[f"boxes{i}.bboxes"] = bb.numpy()
            out[f"boxes{i}.scores"] = sc.numpy()
            out[f"boxes{i}.labels"] = lb.numpy()
        if not kind.endswith("Coop"):
            out["outs_dec"] = cap["outs_dec"].numpy()  # [L,B,Nq,C] (already transposed by the transformer)
        if kind == "CmtHead":
            rv = cap["_rv_calls"]      # call 0: _rv_pe (coords -> rv_pos); call 1: _rv_query_embed
            out["ray_coords"] = rv[0][0].numpy()
            out["rv_pos"] = rv[0][1].numpy()
            out["rv_query_feats"] = rv[1][0].numpy()
            bv = cap["_bev_calls"]     # call 0: bev_pos (pos2embed(coords_bev)); call 1: query bev embed
            out["bev_sincos"] = bv[0][0].numpy()
            out["bev_pos"] = bv[0][1].numpy()
        path = os.path.join(GOLDEN_DIR, f"{kind}_mini.npz")
        np.savez_compressed(path, **{k: np.ascontiguousarray(v) for k, v in out.items()})
        print(kind, "->", path, f"{os.path.getsize(path) / 1e6:.2f} MB", {k: v.shape for k, v in list(out.items())[:3]})


if __name__ == "__main__":
    main()
