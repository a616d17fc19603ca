"""Per-frame node availability in the cooperative heads (`node_valid`, a torch.bool [2, B] device mask, row 0 the vehicle,
row 1 the infrastructure): the V2I merge (cmt_split3_bf16) and the batched box decode (cmt_bbox_topk_decode) apply it
per frame, and an absent node's features change no output bit.

The head inputs are the mini_case shapes with B = 4, so that one batch holds the four frame states of MASK: both nodes,
vehicle only, infrastructure only, neither."""
import numpy as np
import pytest
import torch

from cmtcoop_b200 import ops, synth
from cmtcoop_b200.plugin import build_head
from cmtcoop_b200.plugin.detector_glue import batched_to_results, coop_simple_test
from cmtcoop_b200.runtime import GraphedForward, PipelinedRunner
from oracle import cmt_oracle as O

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
B = 4
COOP_KINDS = ["CmtHeadCoop", "CmtLidarHeadCoop", "CmtImageHeadCoop"]
FEATS = ("vehicle_pts_feats", "infrastructure_pts_feats", "vehicle_img_feats", "infrastructure_img_feats")
MASK = [[True, True, False, False], [True, False, True, False]]
MASKS = [MASK, [[True] * B, [True] * B], [[False, True, True, False], [True, True, False, False]], [[False] * B, [False] * B]]
FLT_MAX = torch.finfo(torch.float32).max


def _mask(m, device=DEV):
    return torch.tensor(m, dtype=torch.bool, device=device)


def _case(kind, precision):
    cfg = synth.head_cfg(kind, num_query=96, num_layers=2, grid=8 * 24, max_num=50)
    inputs = synth.make_inputs(kind, B=B, bev_hw=24, n_views=2, img_hw=(6, 10), vehicle_views=1, infra_views=2, seed=0)
    head = build_head(cfg)
    synth.load_synth_weights(head, 0)
    head = head.to(DEV).eval().set_precision(precision)
    feats = {k: torch.from_numpy(inputs[k]).to(DEV) for k in FEATS if inputs.get(k) is not None}
    return head, feats, inputs["img_metas"]


def _fwd(head, f, metas, node_valid=None):
    with torch.no_grad():
        return head.forward_single(*[f.get(k) for k in FEATS], metas, node_valid=node_valid)


def _refill(f, mask, value):
    """The features with every absent (node, frame) overwritten by `value`."""
    out = {k: v.clone() for k, v in f.items()}
    for k, t in out.items():
        node = 0 if k.startswith("vehicle") else 1
        per = t.shape[0] // B
        for b in range(B):
            if not mask[node][b]:
                t[b * per:(b + 1) * per] = value
    return out


def _drop(f, node):
    return {k: v for k, v in f.items() if not k.startswith(node)}


def _equal(a, b, frames=slice(None)):
    for ta, tb in zip(a, b):
        assert set(ta) == set(tb)
        for n in ta:
            assert torch.equal(ta[n][:, frames], tb[n][:, frames]), n


# ---- cmt_split3_bf16 ------------------------------------------------------------------------------------------------
def _stacks(L=3, Nq=40, seed=0):
    g = torch.Generator().manual_seed(seed)
    v, i = (torch.randn(L, B, Nq, 256, generator=g) * 100 for _ in range(2))
    for t in (v, i):   # NaN and +-inf sprinkled in
        flat = t.view(-1)
        idx = torch.randperm(flat.numel(), generator=g)[:3000]
        flat[idx[:1000]] = float("nan")
        flat[idx[1000:2000]] = float("inf")
        flat[idx[2000:]] = -float("inf")
    return v.to(DEV), i.to(DEV)


def _expected_merged(v, i, m):
    out = torch.zeros_like(v)
    for b in range(B):
        if m[0][b] and m[1][b]:
            out[:, b] = torch.maximum(torch.nan_to_num(v[:, b]), torch.nan_to_num(i[:, b]))
        elif m[0][b]:
            out[:, b] = torch.nan_to_num(v[:, b])
        elif m[1][b]:
            out[:, b] = torch.nan_to_num(i[:, b])
    return out


@pytest.mark.parametrize("layout", ["stacked", "dense"])
def test_split3_follows_the_mask_exactly(layout):
    v, i = _stacks()

    def split(vv, ii, m):
        nv = None if m is None else _mask(m)
        if layout == "stacked":
            return ops.split3(torch.cat([vv, ii], 1).contiguous(), want_merged=True, stacked_nodes=True, node_valid=nv)
        return ops.split3(vv, ii, want_merged=True, node_valid=nv)

    for m in MASKS:
        xs, merged = split(v, i, m)
        want = _expected_merged(v, i, m)
        assert torch.equal(merged, want)
        assert torch.equal(xs, ops.split3(want))
        # an absent node's rows are not read: NaN there changes nothing
        vn, i_n = v.clone(), i.clone()
        for b in range(B):
            if not m[0][b]:
                vn[:, b] = float("nan")
            if not m[1][b]:
                i_n[:, b] = float("nan")
        xs2, merged2 = split(vn, i_n, m)
        assert torch.equal(xs2, xs) and torch.equal(merged2, merged)
    xs0, merged0 = split(v, i, None)
    xs1, merged1 = split(v, i, [[True] * B, [True] * B])
    assert torch.equal(xs1, xs0) and torch.equal(merged1, merged0)
    assert torch.equal(merged0, _expected_merged(v, i, [[True] * B, [True] * B]))
    assert bool((merged0.abs() <= FLT_MAX).all())


# ---- cmt_bbox_topk_decode -------------------------------------------------------------------------------------------
def _preds(counts=(4, 3), Nq=60, L=2, seed=1):
    g = torch.Generator().manual_seed(seed)
    preds = []
    for c in counts:
        d = {n: torch.randn(L, B, Nq, w, generator=g).to(DEV)
             for n, w in dict(center=2, height=1, dim=3, rot=2, vel=2, cls_logits=c).items()}
        d["center"] *= 40.0
        preds.append([d])
    return preds


def test_decode_frames_without_a_node_keep_nothing():
    from cmtcoop_b200.plugin import MultiTaskBBoxCoder
    coder = MultiTaskBBoxCoder(pc_range=synth.TUMTRAF_RANGE, post_center_range=[-80, -80, -10.0, 80, 80, 10.0],
                               max_num=40, num_classes=7)
    preds = _preds()
    want = coder.decode_batched(preds)
    assert bool((want["count"] > 0).all())
    for m in MASKS + [[[True, False, True, False]], [[False] * B, [True, False, False, True], [False] * B]]:
        got = coder.decode_batched(preds, node_valid=_mask(m))
        for b in range(B):
            if any(row[b] for row in m):
                for n in want:
                    assert torch.equal(got[n][b], want[n][b]), (m, b, n)
            else:
                assert int(got["count"][b]) == 0
                assert not bool(got["boxes"][b].any()) and not bool(got["scores"][b].any())
                assert bool((got["labels"][b] == -1).all()) and bool((got["topk_index"][b] == -1).all())


# ---- heads ----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("precision", ["bf16", "fp16", "fp32"])
@pytest.mark.parametrize("kind", COOP_KINDS)
def test_heads_follow_the_mask(kind, precision):
    head, f, metas = _case(kind, precision)
    m = _mask(MASK)
    for batch_nodes in (True, False):   # node-batched decoder pass, and the sequential one
        head.batch_nodes = batch_nodes
        none = _fwd(head, f, metas)
        _equal(_fwd(head, f, metas, _mask([[True] * B, [True] * B])), none)
        masked = _fwd(head, f, metas, m)
        for value in (1.0e4, float("nan")):   # the absent node's rows hold anything
            _equal(_fwd(head, _refill(f, MASK, value), metas, m), masked)
        _equal(masked, none, frames=slice(0, 1))   # both nodes present
        for b, absent in ((1, "infrastructure"), (2, "vehicle")):   # one node present: the single-node result
            single = _fwd(head, _drop(f, absent), metas)
            for ta, tb in zip(masked, single):
                for n in ta:
                    assert O.rel_l2(ta[n][:, b].float().cpu(), tb[n][:, b].float().cpu()) < 1e-5, (batch_nodes, b, n)
        for ta in masked:   # no node: defined, finite outputs
            for n, t in ta.items():
                assert bool(torch.isfinite(t[:, 3]).all()), n


def test_torch_task_head_path_takes_the_masked_merge():
    """Task heads the library does not fuse run torch's convolutions on split3's `merged` output."""
    head, f, metas = _case("CmtLidarHeadCoop", "fp32")
    m = _mask(MASK)
    fused = _fwd(head, f, metas, m)
    for t in head.task_heads:
        t.fusable = lambda x: False
    plain = _fwd(head, f, metas, m)
    _equal(_fwd(head, _refill(f, MASK, float("nan")), metas, m), plain)
    for ta, tb in zip(plain, fused):
        for n in ta:
            assert O.rel_l2(ta[n].cpu(), tb[n].cpu()) < 1e-5, n


# ---- graph and runner -----------------------------------------------------------------------------------------------
def test_graph_replays_every_mask_without_recapture():
    head, f, metas = _case("CmtLidarHeadCoop", "bf16")
    g = GraphedForward(head, metas, dict(f, node_valid=_mask(MASK)), decode_boxes=True)
    graph = g.graph
    for mk in MASKS:
        m = _mask(mk)
        want_rets = _fwd(head, f, metas, m)
        with torch.no_grad():
            want_boxes = head.get_bboxes_batched([[r] for r in want_rets], metas, node_valid=m)
        got_rets, got_boxes = g(dict(f, node_valid=m))
        torch.cuda.synchronize()
        assert g.graph is graph
        _equal(got_rets, want_rets)
        for n in want_boxes:
            assert torch.equal(got_boxes[n], want_boxes[n]), (mk, n)
        for b in range(B):
            if not (mk[0][b] or mk[1][b]):
                assert int(got_boxes["count"][b]) == 0


@pytest.mark.parametrize("outputs", ["heads", "boxes"])
@pytest.mark.parametrize("use_cuda_graph", [False, True])
def test_runner_takes_a_mask_per_batch(use_cuda_graph, outputs):
    head, f, metas = _case("CmtLidarHeadCoop", "bf16")
    host = {k: v.cpu() for k, v in f.items()}
    batches = [dict({k: (v * (1.0 - 0.1 * j)).pin_memory() for k, v in host.items()},
                    node_valid=torch.tensor(MASKS[j % len(MASKS)], dtype=torch.bool).pin_memory()) for j in range(5)]
    runner = PipelinedRunner(head, metas, batches[0], DEV, use_cuda_graph=use_cuda_graph, outputs=outputs)
    results = runner.run(batches)
    for j, res in enumerate(results):
        fj = {k: v.to(DEV) for k, v in batches[j].items()}
        m = fj.pop("node_valid")
        rets = _fwd(head, fj, metas, m)
        if outputs == "boxes":
            with torch.no_grad():
                want = head.get_bboxes_batched([[r] for r in rets], metas, node_valid=m)
            for n in want:
                assert torch.equal(res[n], want[n].cpu()), (j, n)
        else:
            _equal(res, [{n: t.cpu() for n, t in task.items()} for task in rets])


# ---- detector glue and argument checks ------------------------------------------------------------------------------
def test_coop_simple_test_with_a_mask():
    head, f, metas = _case("CmtLidarHeadCoop", "fp32")
    m = _mask(MASK)
    with torch.no_grad():
        res = coop_simple_test(head, [f["vehicle_pts_feats"]], [f["infrastructure_pts_feats"]], None, None, metas,
                               node_valid=m)
        outs = head([f["vehicle_pts_feats"]], [f["infrastructure_pts_feats"]], [None], [None], metas, node_valid=m)
        want = batched_to_results(head.get_bboxes_batched(outs, metas, node_valid=m), metas)
    def rows(d):   # order-free inside groups of bit-equal scores
        t = torch.cat([d["scores_3d"][:, None].view(torch.int32), d["labels_3d"][:, None].int(),
                       d["boxes_3d"].view(torch.int32)], 1)
        return sorted(map(tuple, t.tolist()))

    assert len(res) == B
    for r, w in zip(res, want):
        assert set(r["pts_bbox"]) == set(w) and rows(r["pts_bbox"]) == rows(w)
    assert res[3]["pts_bbox"]["scores_3d"].numel() == 0 and res[0]["pts_bbox"]["scores_3d"].numel() > 0


def test_bad_masks_raise():
    head, f, metas = _case("CmtLidarHeadCoop", "bf16")
    args = [f.get(k) for k in FEATS]
    bad = [torch.ones(2, B + 1, dtype=torch.bool, device=DEV), torch.ones(B, dtype=torch.bool, device=DEV),
           torch.ones(3, B, dtype=torch.bool, device=DEV), torch.ones(2, B, dtype=torch.uint8, device=DEV),
           torch.ones(2, B, dtype=torch.bool), [[True] * B, [True] * B]]
    with torch.no_grad():
        for nv in bad:
            with pytest.raises((ValueError, TypeError)):
                head.forward_single(*args, metas, node_valid=nv)
        with pytest.raises(ValueError):   # a node missing from the whole batch is None, without a mask
            head.forward_single(args[0], None, None, None, metas, node_valid=_mask(MASK))
        v, i = _stacks(L=1, Nq=8)
        with pytest.raises(ValueError):   # no second node to merge with
            ops.split3(v, node_valid=_mask(MASK))
        with pytest.raises(ValueError):
            ops.split3(v, i, node_valid=torch.ones(2, B, dtype=torch.bool))
        preds = _preds()
        from cmtcoop_b200.plugin import MultiTaskBBoxCoder
        coder = MultiTaskBBoxCoder(pc_range=synth.TUMTRAF_RANGE, post_center_range=[-80, -80, -10.0, 80, 80, 10.0],
                                   max_num=40, num_classes=7)
        for nv in (torch.ones(2, B + 1, dtype=torch.bool, device=DEV), torch.ones(0, B, dtype=torch.bool, device=DEV),
                   torch.ones(2, B, dtype=torch.int32, device=DEV), torch.ones(2, B, dtype=torch.bool)):
            with pytest.raises((ValueError, TypeError)):
                coder.decode_batched(preds, node_valid=nv)
