"""Per-frame sensor availability in the single-node heads (`sensor_valid`, a torch.bool [S, B] device mask, one row per
sensor in token order: the LiDAR first for heads with BEV tokens, then the cameras in img_feats / lidar2img order).

A frame with at least one sensor must equal the CPU oracle run on that frame alone with only its present sensors; a
frame with none decodes to nothing; an absent sensor's features (and calibration) change no output bit.  The head inputs
are the mini_case shapes with B = 6, one frame per state of STATES."""
import numpy as np
import pytest
import torch

from cmtcoop_b200 import ops, synth
from cmtcoop_b200.plugin import build_head
from cmtcoop_b200.plugin.detector_glue import batched_to_results, simple_test
from cmtcoop_b200.runtime import GraphedForward, PipelinedRunner
from oracle import cmt_oracle as O

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
KINDS = ["CmtHead", "CmtImageHead", "CmtLidarHead"]
NAMES = ("center", "height", "dim", "rot", "vel", "cls_logits")
TOL = {"fp32": 1e-4, "bf16": 1e-2, "fp16": 1e-2}
V = 2
# (LiDAR, camera 0, camera 1) per frame: all present, one camera absent, all cameras absent, LiDAR absent,
# a single camera only, nothing present
STATES = [(1, 1, 1), (1, 1, 0), (1, 0, 0), (0, 1, 1), (0, 0, 1), (0, 0, 0)]
B = len(STATES)
FLT_MAX = torch.finfo(torch.float32).max


def _rows(kind, states=STATES):
    """The [S, B] mask of a head kind from per-frame (LiDAR, cam0, cam1) states."""
    cols = {"CmtHead": (0, 1, 2), "CmtImageHead": (1, 2), "CmtLidarHead": (0,)}[kind]
    return [[bool(st[c]) for st in states] for c in cols]


def _mask(rows):
    return torch.tensor(rows, dtype=torch.bool, device=DEV)


def _present(kind, b, states=STATES):
    """(LiDAR present, [present camera indices]) of frame b as the head kind sees it."""
    lidar, cams = bool(states[b][0]) and kind != "CmtImageHead", [v for v in range(V) if states[b][1 + v]]
    return lidar, (cams if kind != "CmtLidarHead" else [])


def _case(kind, precision):
    cfg = synth.head_cfg(kind, num_query=96, num_layers=2, grid=8 * 24, max_num=50)
    inputs = synth.make_inputs(kind, B=B, bev_hw=24, n_views=V, img_hw=(6, 10), seed=0)
    head = build_head(cfg)
    synth.load_synth_weights(head, 0)
    head = head.to(DEV).eval().set_precision(precision)
    return head, cfg, inputs


def _feats(inputs):
    return {k: torch.from_numpy(inputs[k]).to(DEV) for k in ("pts_feats", "img_feats") if inputs.get(k) is not None}


def _fwd(head, f, metas, sensor_valid=None):
    with torch.no_grad():
        return head.forward_single(f.get("pts_feats"), f.get("img_feats"), metas, sensor_valid=sensor_valid)


def _refill(kind, f, value, states=STATES):
    """The features with every absent (sensor, frame) overwritten by `value` ("random": fresh noise)."""
    out = {k: v.clone() for k, v in f.items()}
    g = torch.Generator(device=DEV).manual_seed(7)

    def fill(t):
        if value == "random":
            t.copy_(torch.randn(t.shape, generator=g, device=DEV) * 1e3)
        else:
            t.fill_(value)
    for b in range(B):
        lidar, cams = _present(kind, b, states)
        if "pts_feats" in out and not lidar:
            fill(out["pts_feats"][b])
        if "img_feats" in out:
            for v in range(V):
                if v not in cams:
                    fill(out["img_feats"][b * V + v])
    return out


def _garbage_calibration(kind, metas, states=STATES):
    """Metas whose absent cameras carry another (invertible) lidar2img."""
    out = [dict(m) for m in metas]
    for b, m in enumerate(out):
        if "lidar2img" not in m:
            continue
        _, cams = _present(kind, b, states)
        m["lidar2img"] = [M if v in cams else np.diag([3.0, -2.0, 0.5, 1.0]) @ np.asarray(M) + np.eye(4) * 7.0
                          for v, M in enumerate(m["lidar2img"])]
    return out


def _equal(a, b):
    for ta, tb in zip(a, b):
        assert set(ta) == set(tb)
        for n in ta:
            assert torch.equal(ta[n], tb[n]), n


_oracle_cache = {}


def _oracle_frame(kind, head, cfg, inputs, b, states=STATES, key=None):
    """O.head_forward on frame b alone with only its present sensors."""
    k = (kind, b, key)
    if k not in _oracle_cache:
        lidar, cams = _present(kind, b, states)
        meta = dict(inputs["img_metas"][b])
        one = dict(img_metas=[meta], pts_feats=None, img_feats=None)
        if lidar:
            one["pts_feats"] = inputs["pts_feats"][b:b + 1]
        if cams:
            n = inputs["img_feats"].shape[0] // len(inputs["img_metas"])
            one["img_feats"] = inputs["img_feats"][[b * n + v for v in cams]]
            meta["lidar2img"] = [meta["lidar2img"][v] for v in cams]
            meta["pad_shape"] = [meta["pad_shape"][v] for v in cams]
        sd = {n: t.detach().cpu() for n, t in head.state_dict().items()}
        _oracle_cache[k] = O.head_forward(sd, cfg, one)[0]
    return _oracle_cache[k]


def _check_against_oracle(kind, head, cfg, inputs, rets, precision, states=STATES, key=None):
    mask = _mask(_rows(kind, states))
    with torch.no_grad():
        dec = head.get_bboxes_batched([[r] for r in rets], inputs["img_metas"], node_valid=mask)
    worst = 0.0
    for b in range(len(states)):
        lidar, cams = _present(kind, b, states)
        if not lidar and not cams:   # nothing present: finite outputs, nothing decoded
            for n in NAMES:
                assert bool(torch.isfinite(rets[0][n][:, b]).all()), (b, n)
            assert int(dec["count"][b]) == 0 and bool((dec["topk_index"][b] == -1).all())
            continue
        want = _oracle_frame(kind, head, cfg, inputs, b, states, key)
        for n in NAMES:
            rel = O.rel_l2(rets[0][n][:, b].float().cpu(), want[0][n][:, 0])
            worst = max(worst, rel)
            assert rel <= TOL[precision], (b, n, rel)
        k = cfg["bbox_coder"]["max_num"]
        ours = rets[0]["cls_logits"][-1][b].float().cpu().sigmoid().flatten()
        ref = want[0]["cls_logits"][-1][0].sigmoid().flatten()
        tau = 2 * float((ours - ref).abs().max()) + 1e-7
        assert O.topk_tie_tolerant_equal(ours.topk(k).indices, ours, ref.topk(k).indices, ref, tau), b
    return worst


# ---- kernels --------------------------------------------------------------------------------------------------------
def _gather_case(fdt, n_bev_hw=(5, 7), img_hw=(6, 10), C=256, seed=0):
    g = torch.Generator().manual_seed(seed)
    xb = torch.randn(B, C, *n_bev_hw, generator=g).to(fdt).to(DEV)
    xi = torch.randn(B * V, C, *img_hw, generator=g).to(fdt).to(DEV)
    bev_pos = torch.randn(n_bev_hw[0] * n_bev_hw[1], C, generator=g).to(DEV)
    rv_pos = torch.randn(B * V, img_hw[0], img_hw[1], C, generator=g).to(DEV)
    return xb, xi, bev_pos, rv_pos


@pytest.mark.parametrize("out_dtype", [torch.float32, torch.bfloat16, torch.float16])
@pytest.mark.parametrize("fdt", [torch.float32, torch.bfloat16, torch.float16])
def test_gather_writes_zero_rows_for_absent_sensors(fdt, out_dtype):
    xb, xi, bev_pos, rv_pos = _gather_case(fdt)
    n_bev, n_img = xb.shape[2] * xb.shape[3], xi.shape[2] * xi.shape[3]
    for with_bev in (True, False):
        rows = _rows("CmtHead" if with_bev else "CmtImageHead")
        m = _mask(rows)
        nb = n_bev if with_bev else 0
        want_k, want_v = ops.gather_tokens(xb if with_bev else None, xi, bev_pos if with_bev else None, rv_pos, B, V,
                                           out_dtype=out_dtype)
        # absent sensors' features and position encodings hold NaN
        xb2, xi2, rv2 = xb.clone(), xi.clone(), rv_pos.clone()
        keep = torch.ones(B, nb + V * n_img, dtype=torch.bool)
        for b in range(B):
            if with_bev and not rows[0][b]:
                xb2[b] = float("nan")
                keep[b, :nb] = False
            for v in range(V):
                if not rows[(1 if with_bev else 0) + v][b]:
                    xi2[b * V + v] = float("nan")
                    rv2[b * V + v] = float("nan")
                    keep[b, nb + v * n_img: nb + (v + 1) * n_img] = False
        got_k, got_v = ops.gather_tokens(xb2 if with_bev else None, xi2, bev_pos if with_bev else None, rv2, B, V,
                                         out_dtype=out_dtype, sensor_valid=m)
        keep = keep.to(DEV)
        for got, want in ((got_k, want_k), (got_v, want_v)):
            assert torch.equal(got[keep], want[keep])
            assert not bool(got[~keep].float().abs().sum())
            assert not bool(torch.signbit(got[~keep].float()).any())
    # the image half only, behind BEV rows produced elsewhere (the fused shared_conv path): the mask keeps its LiDAR row
    m = _mask(_rows("CmtHead"))
    out = [torch.full((B, n_bev + V * n_img, 256), 5.0, dtype=out_dtype, device=DEV) for _ in range(2)]
    ops.gather_tokens(None, xi, None, rv_pos, B, V, out_dtype=out_dtype, n_bev_reserved=n_bev, out=out, sensor_valid=m)
    full_k, _ = ops.gather_tokens(xb, xi, bev_pos, rv_pos, B, V, out_dtype=out_dtype, sensor_valid=m)
    assert bool((out[0][:, :n_bev] == 5.0).all())
    assert torch.equal(out[0][:, n_bev:], full_k[:, n_bev:])


@pytest.mark.parametrize("fdt", [torch.float32, torch.bfloat16, torch.float16])
@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16])
def test_layout_kernel_zero_fills_absent_frames(fdt, dtype):
    g = torch.Generator().manual_seed(1)
    x = torch.randn(B, 128, 9, 12, generator=g).to(fdt).to(DEV)
    lidar = _mask(_rows("CmtLidarHead"))[0]
    want = ops.nchw_to_padded_nhwc(x, dtype=dtype)
    x2 = x.clone()
    x2[~lidar] = float("nan")
    got = ops.nchw_to_padded_nhwc(x2, dtype=dtype, frame_valid=lidar)
    out = torch.full_like(want, 3.0)   # a reused buffer: the interior of an absent frame is rewritten with zeros
    ops.nchw_to_padded_nhwc(x2, out, dtype=dtype, frame_valid=lidar)
    for b in range(B):
        if bool(lidar[b]):
            assert torch.equal(got[b], want[b])
        else:
            assert not bool(got[b].float().abs().sum())
    interior = want.new_zeros(want.shape[1], dtype=torch.bool)
    guard = ops.conv_guard_rows(12)
    for y in range(9):
        s = guard + (y + 1) * 14 + 1
        interior[s:s + 12] = True
    assert torch.equal(out[:, interior], got[:, interior])


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16, torch.float16])
def test_masked_view_sum_skips_absent_views(dtype):
    g = torch.Generator().manual_seed(2)
    Vs, Nq, C = 3, 70, 256
    states = [(1, 1, 1), (1, 0, 1), (0, 0, 0), (0, 1, 0), (1, 1, 0), (0, 0, 1)]
    vv = _mask([[bool(s[v]) for s in states] for v in range(Vs)])
    emb = torch.randn(B, Vs, Nq, C, generator=g).to(dtype).to(DEV)
    mask = (torch.rand(B, Vs, Nq, generator=g) > 0.3).float().to(DEV)   # the 0 / 1 visibility of ray_query_pe
    base = torch.randn(Nq, C, generator=g).to(DEV)
    emb2 = emb.clone()
    for b in range(B):
        for v in range(Vs):
            if not states[b][v]:
                emb2[b, v] = float("nan")
    got = ops.masked_view_sum(emb2, mask, base=base, view_valid=vv)
    acc = torch.zeros(B, Nq, C, device=DEV)
    for b in range(B):
        for v in range(Vs):
            if states[b][v]:
                acc[b] = acc[b] + emb[b, v].float() * mask[b, v][:, None]   # mask entries 0 / 1: exact products
    assert torch.equal(got, base + acc)
    # and equal to the unmasked kernel with the absent views' visibility zeroed
    m0 = mask.clone()
    m0[~vv.t()] = 0.0
    assert torch.equal(got, ops.masked_view_sum(emb, m0, base=base))


def test_key_keep_bytes():
    m = _mask(_rows("CmtHead"))
    for n_bev, Vk, n_img, rows in ((1000, 0, 0, m[:1]), (0, V, 33, m[1:]), (77, V, 33, m)):
        got = ops.sensor_key_keep(rows, B, n_bev, Vk, n_img)
        parts = ([rows[0][:, None].expand(B, n_bev)] if n_bev else []) + \
                [rows[(1 if n_bev else 0) + v][:, None].expand(B, n_img) for v in range(Vk)]
        want = torch.cat(parts, 1)
        assert got.dtype == torch.bool and torch.equal(got, want)


# ---- heads against the oracle -----------------------------------------------------------------------------------------
@pytest.mark.parametrize("precision", ["bf16", "fp16", "fp32"])
@pytest.mark.parametrize("kind", KINDS)
def test_heads_match_the_oracle_on_the_present_sensors(kind, precision):
    head, cfg, inputs = _case(kind, precision)
    f = _feats(inputs)
    m = _mask(_rows(kind))
    masked = _fwd(head, _refill(kind, f, float("nan")), inputs["img_metas"], m)
    worst = _check_against_oracle(kind, head, cfg, inputs, masked, precision)
    print(f"sensor mask {kind} {precision}: worst per-frame rel-L2 vs the oracle on present sensors {worst:.2e}")
    # independence: other garbage in the absent sensors (and another calibration for absent cameras): same bits
    metas2 = _garbage_calibration(kind, inputs["img_metas"])
    for value in (FLT_MAX, -FLT_MAX, "random", 0.0):
        _equal(_fwd(head, _refill(kind, f, value), metas2 if value == "random" else inputs["img_metas"], m), masked)
    # an all-true mask: the unmasked result up to the attention instantiation
    none = _fwd(head, f, inputs["img_metas"])
    full = _fwd(head, f, inputs["img_metas"], torch.ones_like(m))
    bitwise = all(torch.equal(ta[n], tb[n]) for ta, tb in zip(full, none) for n in ta)
    worst_full = max(O.rel_l2(ta[n].float().cpu(), tb[n].float().cpu()) for ta, tb in zip(full, none) for n in ta)
    print(f"sensor mask {kind} {precision}: all-true mask vs no mask bit-identical={bitwise} worst rel-L2 {worst_full:.1e}")
    assert worst_full <= 1e-6


def test_module_decoder_path_takes_the_mask():
    """The module-by-module decoder (PETRMultiheadFlashAttention -> FlashMHA key_padding_mask) with the sensor mask."""
    head, cfg, inputs = _case("CmtHead", "fp32")
    head.transformer.use_fused_decoder = False
    m = _mask(_rows("CmtHead"))
    rets = _fwd(head, _refill("CmtHead", _feats(inputs), float("nan")), inputs["img_metas"], m)
    _check_against_oracle("CmtHead", head, cfg, inputs, rets, "fp32")


def test_baseline_shape_with_missing_sensors():
    """configs[2] of test_gpu_configs (CmtHead, 6 cameras x 40x100 + 180x180 BEV = 56 400 tokens, B = 2, bf16) with
    camera 3 absent in frame 0 and the LiDAR absent in frame 1."""
    kind = "CmtHead"
    cfg = synth.head_cfg(kind, num_query=900, num_layers=6, grid=1440)
    inputs = synth.make_inputs(kind, seed=11, B=2, bev_hw=180, n_views=6, img_hw=(40, 100))
    head = build_head(cfg)
    synth.load_synth_weights(head, 0)
    head = head.to(DEV).eval().set_precision("bf16")
    rows = [[True, False]] + [[v != 3, True] for v in range(6)]
    f = _feats(inputs)
    f["pts_feats"][1] = float("nan")
    f["img_feats"][3] = float("nan")
    rets = _fwd(head, f, inputs["img_metas"], _mask(rows))
    torch.cuda.synchronize()
    sd = {n: t.detach().cpu() for n, t in head.state_dict().items()}
    torch.set_num_threads(max(torch.get_num_threads(), 8))
    for b, (lidar, cams) in enumerate(((True, [0, 1, 2, 4, 5]), (False, list(range(6))))):
        meta = dict(inputs["img_metas"][b])
        meta["lidar2img"] = [meta["lidar2img"][v] for v in cams]
        meta["pad_shape"] = [meta["pad_shape"][v] for v in cams]
        one = dict(img_metas=[meta], pts_feats=inputs["pts_feats"][b:b + 1] if lidar else None,
                   img_feats=inputs["img_feats"][[b * 6 + v for v in cams]])
        want = O.head_forward(sd, cfg, one)[0]
        worst = {n: O.rel_l2(rets[0][n][:, b].float().cpu(), want[0][n][:, 0]) for n in NAMES}
        print(f"configs[2] frame {b} with a missing sensor: " + " ".join(f"{k}={v:.2e}" for k, v in worst.items()))
        assert max(worst.values()) < 1e-2, worst


# ---- graph, runner, detector glue -------------------------------------------------------------------------------------
MASK_STATES = [STATES, [(1, 1, 1)] * B, [(0, 1, 0), (1, 0, 1), (0, 0, 0), (1, 1, 1), (1, 0, 0), (0, 1, 1)],
               [(0, 0, 0)] * B]


def test_graph_replays_every_mask_without_recapture():
    kind = "CmtHead"
    head, cfg, inputs = _case(kind, "bf16")
    f, metas = _feats(inputs), inputs["img_metas"]
    g = GraphedForward(head, metas, dict(f, sensor_valid=_mask(_rows(kind))), decode_boxes=True)
    graph = g.graph
    for states in MASK_STATES:
        m = _mask(_rows(kind, states))
        want_rets = _fwd(head, f, metas, m)
        with torch.no_grad():
            want_boxes = head.get_bboxes_batched([[r] for r in want_rets], metas, node_valid=m)
        got_rets, got_boxes = g(dict(f, sensor_valid=m))
        torch.cuda.synchronize()
        assert g.graph is graph
        _equal(got_rets, want_rets)
        for n in want_boxes:
            assert torch.equal(got_boxes[n], want_boxes[n]), (states, n)
        for b in range(B):
            if not any(states[b]):
                assert int(got_boxes["count"][b]) == 0


@pytest.mark.parametrize("outputs", ["heads", "boxes"])
@pytest.mark.parametrize("use_cuda_graph", [False, True])
def test_runner_takes_a_mask_per_batch(use_cuda_graph, outputs):
    kind = "CmtHead"
    head, cfg, inputs = _case(kind, "bf16")
    metas = inputs["img_metas"]
    host = {k: v.cpu() for k, v in _feats(inputs).items()}
    batches = [dict({k: (v * (1.0 - 0.1 * j)).pin_memory() for k, v in host.items()},
                    sensor_valid=torch.tensor(_rows(kind, MASK_STATES[j % len(MASK_STATES)]), dtype=torch.bool).pin_memory())
               for j in range(5)]
    runner = PipelinedRunner(head, metas, batches[0], DEV, use_cuda_graph=use_cuda_graph, outputs=outputs)
    results = runner.run(batches)
    for j, res in enumerate(results):
        fj = {k: v.to(DEV) for k, v in batches[j].items()}
        m = fj.pop("sensor_valid")
        rets = _fwd(head, fj, metas, m)
        if outputs == "boxes":
            with torch.no_grad():
                want = head.get_bboxes_batched([[r] for r in rets], metas, node_valid=m)
            for n in want:
                assert torch.equal(res[n], want[n].cpu()), (j, n)
        else:
            _equal(res, [{n: t.cpu() for n, t in task.items()} for task in rets])


def test_simple_test_with_a_mask():
    kind = "CmtHead"
    head, cfg, inputs = _case(kind, "fp32")
    f, metas = _feats(inputs), inputs["img_metas"]
    m = _mask(_rows(kind))
    with torch.no_grad():
        res = simple_test(head, [f["pts_feats"]], [f["img_feats"]], metas, sensor_valid=m)
        outs = head([f["pts_feats"]], [f["img_feats"]], metas, sensor_valid=m)
        want = batched_to_results(head.get_bboxes_batched(outs, metas, node_valid=m), metas)

    def rows(d):   # order-free inside groups of bit-equal scores
        t = torch.cat([d["scores_3d"][:, None].view(torch.int32), d["labels_3d"][:, None].int(),
                       d["boxes_3d"].view(torch.int32)], 1)
        return sorted(map(tuple, t.tolist()))

    assert len(res) == B
    for r, w in zip(res, want):
        assert set(r["pts_bbox"]) == set(w) and rows(r["pts_bbox"]) == rows(w)
    assert res[5]["pts_bbox"]["scores_3d"].numel() == 0 and res[0]["pts_bbox"]["scores_3d"].numel() > 0


def test_bad_masks_raise_on_the_device():
    head, cfg, inputs = _case("CmtHead", "bf16")
    f, metas = _feats(inputs), inputs["img_metas"]
    bad = [torch.ones(V, B, dtype=torch.bool, device=DEV), torch.ones(1 + V, B + 1, dtype=torch.bool, device=DEV),
           torch.ones(1 + V, B, dtype=torch.uint8, device=DEV), torch.ones(1 + V, B, dtype=torch.bool)]
    for m in bad:
        with pytest.raises((ValueError, TypeError)):
            _fwd(head, f, metas, m)
