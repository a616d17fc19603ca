"""cmt_bbox_topk_decode (ops.bbox_topk_decode, MultiTaskBBoxCoder.decode_batched, CmtHead.get_bboxes_batched) against the
torch coder (MultiTaskBBoxCoder.decode / CmtHead.get_bboxes) on the same CUDA tensors.  The kernel is meant to give
the very bits torch computes, so every comparison is exact: top-k indices, labels, counts, and boxes / scores with
torch.equal.  Where bit-equal scores make torch.topk's order unspecified, the order rule is checked against
torch.sort(descending=True, stable=True) instead."""
import types

import numpy as np
import pytest
import torch

from cmtcoop_b200 import _lib, synth
from cmtcoop_b200.plugin import MultiTaskBBoxCoder, build_head
from cmtcoop_b200.plugin.cmt_head import CmtHead
from cmtcoop_b200.plugin.detector_glue import batched_to_results, simple_test
from cmtcoop_b200.runtime import GraphedForward, PipelinedRunner

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
WIDTH = {"center": 2, "height": 1, "dim": 3, "rot": 2, "vel": 2}
POST = [-61.2, -61.2, -10.0, 61.2, 61.2, 10.0]
# class setups: nuScenes (one task), TUMTraf (one task), nuScenes split into the six task groups of the multi-task head
SETUPS = {"nusc": [10], "tumtraf": [7], "split6": [1, 2, 2, 1, 2, 2]}


def _coder(n_cls, max_num, score_threshold=None, post=POST):
    return MultiTaskBBoxCoder(pc_range=synth.NUSC_RANGE, post_center_range=post, max_num=max_num,
                              score_threshold=score_threshold, num_classes=n_cls)


def _distinct_logits(x, gen):
    """Redraw last-layer logits until every frame's sigmoid scores are pairwise distinct (the CUDA sigmoid, as the coder
    computes them): then the top-k order is unique and torch.topk's order is the only one."""
    B = x.shape[1]
    last = x[-1].view(B, -1)
    for _ in range(100):
        s, order = last.sigmoid().sort(dim=1)
        dup = s[:, 1:] == s[:, :-1]
        if not bool(dup.any()):
            return x
        rows, cols = dup.nonzero(as_tuple=True)
        idx = order[rows, cols + 1]
        last[rows, idx] = torch.randn(len(rows), generator=gen).to(DEV)
    raise AssertionError("could not draw distinct scores")


def _preds(B, Nq, counts, seed, L=2, centre_sigma=40.0, distinct=True):
    """i.i.d. normal task-head outputs [L,B,Nq,c] (centres / heights spread so that some boxes leave the range)."""
    gen = torch.Generator().manual_seed(seed)
    logits = torch.randn(L, B, Nq, sum(counts), generator=gen).to(DEV)
    if distinct:
        logits = _distinct_logits(logits, gen)
    preds, c0 = [], 0
    for c in counts:
        d = {n: torch.randn(L, B, Nq, w, generator=gen).to(DEV) for n, w in WIDTH.items()}
        d["center"] *= centre_sigma
        d["height"] *= centre_sigma / 5.0
        d["cls_logits"] = logits[..., c0:c0 + c].contiguous()
        c0 += c
        preds.append([d])
    return preds


def _scores(preds, i):
    return torch.cat([p[0]["cls_logits"][-1][i] for p in preds], -1).sigmoid().flatten()


def _check_frame(got, i, boxes, scores, labels, topk_index):
    """Frame i of the batched decode equals one frame of the torch coder, padding included."""
    n = int(got["count"][i])
    K = got["scores"].shape[1]
    assert torch.equal(got["topk_index"][i], topk_index)
    assert n == scores.shape[0]
    assert torch.equal(got["labels"][i, :n], labels)
    assert torch.equal(got["scores"][i, :n], scores)
    assert torch.equal(got["boxes"][i, :n], boxes)
    assert bool((got["boxes"][i, n:] == 0).all()) and bool((got["scores"][i, n:] == 0).all())
    assert bool((got["labels"][i, n:] == -1).all()) and got["labels"][i, n:].numel() == K - n


@pytest.mark.parametrize("K", [1, 100, 300])
@pytest.mark.parametrize("B", [1, 3, 8])
@pytest.mark.parametrize("setup", list(SETUPS))
def test_decode_equals_torch_coder(setup, B, K):
    counts = SETUPS[setup]
    thr = {"nusc": None, "tumtraf": 0.7, "split6": 0.55}[setup]
    preds = _preds(B, 900, counts, seed=B * 1000 + K)
    coder = _coder(sum(counts), K, thr)
    want = coder.decode(preds)
    got = coder.decode_batched(preds)
    for i in range(B):
        w = want[i]
        _check_frame(got, i, w["bboxes"], w["scores"], w["labels"], w["topk_index"])
    # get_bboxes: the z shift applied in the kernel
    head = types.SimpleNamespace(bbox_coder=coder)
    metas = [dict(box_type_3d=None) for _ in range(B)]
    want_b = CmtHead.get_bboxes(head, preds, metas)
    got_b = CmtHead.get_bboxes_batched(head, preds, metas)
    for i in range(B):
        bb, sc, lb = want_b[i]
        _check_frame(got_b, i, bb, sc, lb, want[i]["topk_index"])


def _edge_preds(pcr32):
    """One class, 16 queries: for each of the six range bounds a centre exactly on it and one a float32 ulp outside,
    plus four interior centres."""
    B, Nq = 2, 16
    preds = _preds(B, Nq, [1], seed=5, centre_sigma=1.0)
    d = preds[0][0]
    xyz = torch.zeros(B, Nq, 3)
    expect_keep = torch.ones(Nq, dtype=torch.bool)
    for j in range(6):
        axis, lo = j % 3, j < 3
        bound = torch.tensor(pcr32[j], dtype=torch.float32)
        outside = torch.nextafter(bound, torch.tensor(-np.inf if lo else np.inf, dtype=torch.float32))
        xyz[:, 2 * j, axis] = bound
        xyz[:, 2 * j + 1, axis] = outside
        expect_keep[2 * j + 1] = False
    d["center"][-1].copy_(xyz[..., :2])
    d["height"][-1].copy_(xyz[..., 2:])
    return preds, expect_keep


def test_mask_edges():
    pcr32 = torch.tensor(POST, dtype=torch.float32).tolist()
    preds, expect_keep = _edge_preds(pcr32)
    B, Nq = 2, 16
    # frame 1: every centre outside the range -> count 0, all padding
    preds[0][0]["center"][-1][1] += 1000.0
    coder = _coder(1, Nq)
    want = coder.decode(preds)
    got = coder.decode_batched(preds)
    for i in range(B):
        _check_frame(got, i, want[i]["bboxes"], want[i]["scores"], want[i]["labels"], want[i]["topk_index"])
    assert int(got["count"][0]) == int(expect_keep.sum())
    assert int(got["count"][1]) == 0

    # a score exactly at the threshold is dropped (strict >); query 4 sits on a bound and is otherwise kept
    s0 = _scores(preds, 0)
    thr = float(s0[4])
    coder = _coder(1, Nq, score_threshold=thr)
    want = coder.decode(preds)
    got = coder.decode_batched(preds)
    for i in range(B):
        _check_frame(got, i, want[i]["bboxes"], want[i]["scores"], want[i]["labels"], want[i]["topk_index"])
    assert int(got["count"][0]) == int((s0[expect_keep.to(DEV)] > thr).sum())
    assert not bool((got["scores"][0, :int(got["count"][0])] == thr).any())

    # score_threshold = 0 is falsy: not applied, so a score of exactly 0 survives (query 12 is interior)
    preds[0][0]["cls_logits"][-1][0, 12] = -200.0       # sigmoid = 0.0
    coder = _coder(1, Nq, score_threshold=0)
    want = coder.decode(preds)
    got = coder.decode_batched(preds)
    for i in range(B):
        _check_frame(got, i, want[i]["bboxes"], want[i]["scores"], want[i]["labels"], want[i]["topk_index"])
    assert bool((got["scores"][0, :int(got["count"][0])] == 0).any())


@pytest.mark.parametrize("kind", ["quantised", "saturated", "nan"])
@pytest.mark.parametrize("K", [1, 100, 300, 1024])
def test_ties_follow_stable_sort(kind, K):
    B, Nq, C = 3, 900, 10
    preds = _preds(B, Nq, [C], seed=11, centre_sigma=1.0, distinct=False)
    x = preds[0][0]["cls_logits"][-1]
    gen = torch.Generator().manual_seed(K)
    if kind == "quantised":
        x.copy_((torch.randn(x.shape, generator=gen) * 2).round().div(2))
    else:
        sat = torch.rand(x.shape, generator=gen) < 0.4
        x.copy_(torch.where(sat, 17.0 + torch.rand(x.shape, generator=gen) * 10, torch.randn(x.shape, generator=gen)))
        if kind == "nan":
            x.view(-1)[torch.randperm(x.numel(), generator=gen)[:50]] = float("nan")
            x.view(-1)[:7] = -float("nan")
    coder = _coder(C, K)
    got = coder.decode_batched(preds)
    for i in range(B):
        s = _scores(preds, i)
        order = torch.sort(s, descending=True, stable=True).indices[:K]
        assert torch.equal(got["topk_index"][i], order)
        torch.testing.assert_close(s[got["topk_index"][i]], torch.topk(s, K).values, rtol=0, atol=0, equal_nan=True)
        n = int(got["count"][i])
        assert n == K     # every centre is inside the range
        torch.testing.assert_close(got["scores"][i], s[order], rtol=0, atol=0, equal_nan=True)
        assert torch.equal(got["labels"][i], order % C)


def _rows(boxes, scores, labels):
    """Detections as a sorted list of bit patterns (order-free comparison inside groups of bit-equal scores)."""
    t = torch.cat([scores[:, None].view(torch.int32), labels[:, None].int(), boxes.view(torch.int32)], 1)
    return sorted(map(tuple, t.cpu().tolist()))


def _build(kind, cfg, precision):
    head = build_head(cfg)
    synth.load_synth_weights(head, 0)
    return head.to(DEV).eval().set_precision(precision)


def _feats(inputs):
    return {k: torch.from_numpy(v).to(DEV) for k, v in inputs.items() if isinstance(v, np.ndarray)}


def _forward(head, kind, f, metas):
    with torch.no_grad():
        if kind.endswith("Coop"):
            return head.forward_single(f.get("vehicle_pts_feats"), f.get("infrastructure_pts_feats"),
                                       f.get("vehicle_img_feats"), f.get("infrastructure_img_feats"), metas)
        return head.forward_single(f.get("pts_feats"), f.get("img_feats"), metas)


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("kind", synth.HEAD_KINDS)
def test_heads_get_bboxes_batched(kind, precision):
    """Real head outputs (untrained decoder: bit-equal scores happen).  Top-k indices follow the stable-sort rule; the
    selected score values equal torch.topk's; index sets agree above the K-th score; detections agree exactly, compared
    order-free inside tie groups."""
    cfg, inputs = synth.mini_case(kind)
    head = _build(kind, cfg, precision)
    metas = inputs["img_metas"]
    preds = [[r] for r in _forward(head, kind, _feats(inputs), metas)]
    want = head.get_bboxes(preds, metas)
    want_idx = [d["topk_index"] for d in head.bbox_coder.decode(preds)]
    got = head.get_bboxes_batched(preds, metas)
    K = cfg["bbox_coder"]["max_num"]
    for i in range(len(metas)):
        s = _scores(preds, i)
        gi = got["topk_index"][i]
        assert torch.equal(gi, torch.sort(s, descending=True, stable=True).indices[:K])
        assert torch.equal(s[gi], s[want_idx[i]])
        kth = s[gi[-1]]
        assert set(gi[s[gi] > kth].tolist()) == set(want_idx[i][s[want_idx[i]] > kth].tolist())
        n = int(got["count"][i])
        bb, sc, lb = want[i]
        mine = (got["boxes"][i, :n], got["scores"][i, :n], got["labels"][i, :n])
        straddle = int((s == kth).sum()) > int((s[gi] == kth).sum())
        if straddle:   # the tie group at the K-th place: torch.topk may have picked other members
            m_mine, m_want = mine[1] > kth, sc > kth
            mine = (mine[0][m_mine], mine[1][m_mine], mine[2][m_mine])
            bb, sc, lb = bb[m_want], sc[m_want], lb[m_want]
        else:
            assert n == sc.shape[0]
        if torch.unique(s[gi]).numel() == K:
            assert torch.equal(mine[0], bb) and torch.equal(mine[1], sc) and torch.equal(mine[2], lb)
        else:
            assert _rows(*mine) == _rows(bb, sc, lb)
        assert bool((got["labels"][i, n:] == -1).all())


def test_graph_decode_boxes_replays_eager():
    kind = "CmtHead"
    cfg, inputs = synth.mini_case(kind)
    head = _build(kind, cfg, "bf16")
    metas = inputs["img_metas"]
    feats = _feats(inputs)

    def eager(f):
        rets = _forward(head, kind, f, metas)
        return rets, head.get_bboxes_batched([[r] for r in rets], metas)

    g = GraphedForward(head, metas, feats, decode_boxes=True)
    for f in (feats, {k: v * 0.5 + 0.1 for k, v in feats.items()}):
        want_rets, want_boxes = eager(f)
        got_rets, got_boxes = g(f)
        torch.cuda.synchronize()
        for n in want_rets[0]:
            assert torch.equal(got_rets[0][n], want_rets[0][n])
        for n in want_boxes:
            assert torch.equal(got_boxes[n], want_boxes[n]), n
        if f is feats:
            first = {n: t.clone() for n, t in got_boxes.items()}
    assert not torch.equal(first["topk_index"], got_boxes["topk_index"])


@pytest.mark.parametrize("use_cuda_graph", [False, True])
def test_runner_outputs_boxes(use_cuda_graph):
    kind = "CmtHead"
    cfg, inputs = synth.mini_case(kind)
    head = _build(kind, cfg, "bf16")
    metas = inputs["img_metas"]
    base = {k: torch.from_numpy(v) for k, v in inputs.items() if isinstance(v, np.ndarray)}
    batches = [{k: (v * (1.0 - 0.1 * j) + 0.05 * j).pin_memory() for k, v in base.items()} for j in range(5)]
    runner = PipelinedRunner(head, metas, batches[0], DEV, use_cuda_graph=use_cuda_graph, outputs="boxes")
    results = runner.run(batches)
    B, K = len(metas), cfg["bbox_coder"]["max_num"]
    assert runner.d2h_bytes == B * K * (9 * 4 + 4 + 8 + 8) + B * 4
    for j, res in enumerate(results):
        f = {k: v.to(DEV) for k, v in batches[j].items()}
        rets = _forward(head, kind, f, metas)
        want = head.get_bboxes_batched([[r] for r in rets], metas)
        assert set(res) == set(want)
        for n in want:
            assert not res[n].is_cuda
            assert torch.equal(res[n], want[n].cpu()), (j, n)


class _Boxes:
    """Stand-in for an mmdet3d box type: box_type_3d(tensor, box_dim)."""

    def __init__(self, tensor, box_dim):
        self.tensor, self.box_dim = tensor, box_dim

    def to(self, device):
        return _Boxes(self.tensor.to(device), self.box_dim)


def test_batched_to_results_equals_simple_test():
    kind = "CmtHead"
    cfg, inputs = synth.mini_case(kind)
    head = _build(kind, cfg, "fp32")
    metas = inputs["img_metas"]
    f = _feats(inputs)
    with torch.no_grad():
        want = [r["pts_bbox"] for r in simple_test(head, [f["pts_feats"]], [f["img_feats"]], metas)]
        outs = head([f["pts_feats"]], [f["img_feats"]], metas)
        got = batched_to_results(head.get_bboxes_batched(outs, metas), metas)
    assert len(got) == len(want)
    for g, w in zip(got, want):
        assert set(g) == set(w)
        if torch.unique(w["scores_3d"]).numel() == w["scores_3d"].numel():
            for n in w:
                assert not g[n].is_cuda and torch.equal(g[n], w[n]), n
        else:
            assert _rows(g["boxes_3d"], g["scores_3d"], g["labels_3d"]) == _rows(w["boxes_3d"], w["scores_3d"], w["labels_3d"])
    typed = [dict(m, box_type_3d=_Boxes) for m in metas]
    with torch.no_grad():
        got_t = batched_to_results(head.get_bboxes_batched(outs, typed), typed)
    for g, t in zip(got, got_t):
        assert isinstance(t["boxes_3d"], _Boxes) and t["boxes_3d"].box_dim == 9
        assert torch.equal(t["boxes_3d"].tensor, g["boxes_3d"])


def test_arguments_rejected():
    preds = _preds(2, 30, [3, 2], seed=3, distinct=False)
    with pytest.raises(_lib.CmtLibraryError):                        # CPU tensors: no fallback
        _coder(5, 10).decode_batched([[{n: t.cpu() for n, t in p[0].items()}] for p in preds])
    with pytest.raises(_lib.CmtLibraryError):                        # K > Nq * sum C (torch.topk raises too)
        _coder(5, 151).decode_batched(preds)
    with pytest.raises(RuntimeError):
        _coder(5, 151).decode(preds)
    with pytest.raises(ValueError):                                  # num_classes != sum C_t
        _coder(6, 10).decode_batched(preds)
    with pytest.raises(NotImplementedError):                         # like decode
        _coder(5, 10, post=None).decode_batched(preds)
    big = _preds(1, 1100, [10], seed=4, distinct=False)
    with pytest.raises(_lib.CmtLibraryError):                        # K > 1024
        _coder(10, 1025).decode_batched(big)
    huge = _preds(1, 5000, [10], seed=4, distinct=False)
    with pytest.raises(_lib.CmtLibraryError):                        # Nq * sum C above the shared-memory bound
        _coder(10, 300).decode_batched(huge)
    nine = _preds(1, 30, [1] * 9, seed=4, distinct=False)
    with pytest.raises(ValueError):                                  # more than 8 tasks
        _coder(9, 10).decode_batched(nine)
    # the largest candidate count the kernel holds (CMT_BOX_DECODE_MAX_CANDIDATES = 49152) still runs
    edge = _preds(2, 49152 // 10, [10], seed=6, distinct=False)
    got = _coder(10, 1024).decode_batched(edge)
    for i in range(2):
        assert torch.equal(got["topk_index"][i], torch.sort(_scores(edge, i), descending=True, stable=True).indices[:1024])

