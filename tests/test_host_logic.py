"""Host-side mirror of the reference interface: registry / config building, state-dict keys, the
torch-only stages (task heads, bbox coder) against the oracle on CPU, error behaviour, and the
multi-GPU partition helpers.  No GPU needed."""
import json
import os

import numpy as np
import pytest
import torch
from hypothesis import given, settings, strategies as st

from cmtcoop_b200 import _lib, ops, parallel, synth
from cmtcoop_b200 import plugin
from oracle import cmt_oracle as O
from oracle import ref_stub


@pytest.mark.parametrize("kind", synth.HEAD_KINDS)
def test_reference_config_builds_and_keys_match_reference(kind, golden_dir):
    cfg, _ = synth.mini_case(kind)
    head = plugin.build_head(cfg)
    assert type(head).__name__ == kind and not head.training
    want = json.load(open(os.path.join(golden_dir, "state_dict_keys_mini.json")))[kind]
    got = {k: list(v.shape) for k, v in head.state_dict().items()}
    assert got == want  # names and shapes of the reference class, checkpoint-compatible


def test_full_size_config_builds():
    head = plugin.build_head(synth.head_cfg("CmtHead"))
    assert head.num_query == 900 and len(head.transformer.decoder.layers) == 6
    assert tuple(head.coords_bev.shape) == (180 * 180, 2)
    ca = head.transformer.decoder.layers[0].attentions[1]
    assert isinstance(ca, plugin.PETRMultiheadFlashAttention) and ca.attn.in_proj_bias is not None  # bias quirk


def test_registry_names():
    for reg, names in dict(HEADS=synth.HEAD_KINDS + ("SeparateTaskHead",),
                           TRANSFORMER=("CmtTransformer", "CmtLidarTransformer", "CmtImageTransformer"),
                           ATTENTION=("MultiheadAttention", "PETRMultiheadAttention", "PETRMultiheadFlashAttention"),
                           TRANSFORMER_LAYER=("PETRTransformerDecoderLayer",),
                           TRANSFORMER_LAYER_SEQUENCE=("PETRTransformerDecoder",),
                           BBOX_CODERS=("MultiTaskBBoxCoder",)).items():
        for n in names:
            assert n in plugin.ALL[reg], (reg, n)
    with pytest.raises(KeyError):
        plugin.HEADS.get("NoSuchHead")


def test_no_cpu_fallback_and_inference_only():
    cfg, inputs = synth.mini_case("CmtLidarHead")
    head = plugin.build_head(cfg)
    x = torch.from_numpy(inputs["pts_feats"])
    with pytest.raises((RuntimeError, _lib.CmtLibraryError)):
        head.forward_single(x, None, inputs["img_metas"])          # CPU tensors are refused
    with pytest.raises(_lib.CmtLibraryError):
        ops.pos2embed(torch.rand(4, 2), 128)
    head.train()
    with pytest.raises(NotImplementedError):
        head.prepare_for_dn(1, head.reference_points.weight, None)
    mha = plugin.FlashMHA(256, 8, 0.1)
    assert mha.bias == 0.1 and mha.in_proj_bias is not None            # attn_drop lands in `bias` (petr_transformer.py:226)
    with pytest.raises(AssertionError):
        plugin.FlashMHA(256, 4)                                         # head_dim 64: not on the reference path


def test_task_heads_and_coder_match_oracle_cpu():
    """The torch-only tail (SeparateTaskHead, reference-point decode, MultiTaskBBoxCoder) on CPU."""
    for kind in ("CmtHead", "CmtLidarHead"):  # final_kernel 1 and 3
        cfg, _ = synth.mini_case(kind)
        head = plugin.build_head(cfg)
        synth.load_synth_weights(head, 1)
        g = torch.Generator().manual_seed(3)
        outs_dec = torch.randn(2, 2, 96, 256, generator=g)
        ref = head.reference_points.weight.detach().unsqueeze(0).repeat(2, 1, 1)
        sd = {k: v.detach() for k, v in head.state_dict().items()}
        want = O.decode_outputs(outs_dec, ref, sd, cfg)
        with torch.no_grad():
            got = head._finish(outs_dec, ref)
        for name in want[0]:
            # fp32 both sides; the k=1 heads run as batched GEMMs (different summation order than conv1d)
            assert torch.allclose(got[0][name], want[0][name], atol=2e-4, rtol=1e-4), (kind, name)
        wb = O.bbox_decode(want, cfg)
        gb = head.bbox_coder.decode([[got[0]]])
        for i in range(2):
            assert torch.equal(gb[i]["topk_index"], wb[i]["topk_index"])     # identical top-k query indices
            assert torch.equal(gb[i]["labels"], wb[i]["labels"])


def test_filter_img_metas():
    meta = dict(vehicle_lidar2img=1, infrastructure_lidar2img=2, box_type_3d=3, vehicle_pad_shape=4)
    v = plugin.get_vehicle_image_metas([meta])[0]
    assert v == dict(lidar2img=1, pad_shape=4, box_type_3d=3, node="vehicle_")
    i = plugin.get_infrastructure_image_metas([meta])[0]
    assert i == dict(lidar2img=2, box_type_3d=3, node="infrastructure_")


@settings(max_examples=200, deadline=None)
@given(n=st.integers(0, 100000), world=st.integers(1, 16))
def test_kv_split_ranges_partition_the_tokens(n, world):
    ranges = [parallel.kv_split_range(n, r, world) for r in range(world)]
    assert ranges[0][0] == 0 and ranges[-1][1] == n
    for (lo, hi), (lo2, _) in zip(ranges, ranges[1:]):
        assert lo <= hi == lo2
    assert all(lo % parallel.KV_TILE == 0 or lo == n for lo, _ in ranges)


@settings(max_examples=150, deadline=None)
@given(B=st.integers(1, 3), H=st.integers(1, 9), W=st.integers(1, 9), V=st.integers(0, 3), h=st.integers(1, 5),
       w=st.integers(1, 6), world=st.integers(1, 5), halo=st.integers(0, 1), data=st.data())
def test_token_rows_copy_plan_covers_the_ranks_tokens(B, H, W, V, h, w, world, halo, data):
    """The partial host->device hand-over of the KV-token split: applying the rank's rectangles to NaN-filled copies
    reproduces every feature value of the rank's tokens (and the halo rows), whatever the split point."""
    C = 2
    n_bev, n_img = H * W, V * h * w
    n_kv = n_bev + n_img
    cut = sorted(data.draw(st.lists(st.integers(0, n_kv), min_size=world - 1, max_size=world - 1)))
    bounds = [0] + cut + [n_kv]
    rng = np.random.RandomState(H * 131 + W * 17 + V)
    bev = rng.rand(B, C, H, W).astype(np.float32)
    img = rng.rand(B * V, C, h, w).astype(np.float32) if V else None
    for r in range(world):
        lo, hi = bounds[r], bounds[r + 1]
        plan = parallel.token_rows_copy_plan(bev.shape, None if img is None else img.shape, B, lo, hi, halo)
        for name, src in (("pts", bev), ("img", img)):
            if src is None:
                assert not plan[name]
                continue
            dst = np.full(src.size, np.nan, np.float32)
            flat = src.reshape(-1)
            for off, pitch, width, height in plan[name]:
                assert 0 < width <= pitch and off >= 0 and off + (height - 1) * pitch + width <= src.size
                for i in range(height):
                    dst[off + i * pitch: off + i * pitch + width] = flat[off + i * pitch: off + i * pitch + width]
            dst = dst.reshape(src.shape)
            if name == "pts":
                tok = dst.reshape(B, C, n_bev)
                a, b = min(lo, n_bev), min(hi, n_bev)
                assert np.array_equal(tok[:, :, a:b], bev.reshape(B, C, n_bev)[:, :, a:b])
                if b > a and halo:
                    y0, y1 = max(0, a // W - 1), min(H, (b + W - 1) // W + 1)
                    assert np.array_equal(dst[:, :, y0:y1], bev[:, :, y0:y1])
            else:
                tok = dst.reshape(B, V, C, h * w).transpose(0, 2, 1, 3).reshape(B, C, n_img)
                want = img.reshape(B, V, C, h * w).transpose(0, 2, 1, 3).reshape(B, C, n_img)
                a, b = max(lo, n_bev) - n_bev, max(hi, n_bev) - n_bev
                assert np.array_equal(tok[:, :, a:b], want[:, :, a:b])


@settings(max_examples=200, deadline=None)
@given(B=st.integers(1, 16), Nq=st.integers(1, 1200), H=st.integers(1, 8), slots=st.integers(2, 8))
def test_peer_exchange_layout(B, Nq, H, slots):
    """Buffers of the peer-memory exchange (parallel.PeerExchange): records, contexts and control words tile the
    allocation without overlap, and everything the kernel moves in 128-bit words is 16-byte aligned."""
    if (B * Nq * H) % 4:
        with pytest.raises(ValueError):
            parallel.peer_layout(B, Nq, H, slots)
        return
    lay = parallel.peer_layout(B, Nq, H, slots)
    assert lay["n_rec"] == B * Nq * H * 32 + B * H * Nq
    rec = [(i * lay["n_rec"], (i + 1) * lay["n_rec"]) for i in range(slots)]
    ctx = [(lay["ctx_off"] + i * lay["n_o"], lay["ctx_off"] + (i + 1) * lay["n_o"]) for i in range(slots)]
    spans = rec + ctx + [(lay["ctrl_off"], lay["total"])]
    assert spans[0][0] == 0 and all(a[1] == b[0] for a, b in zip(spans, spans[1:]))
    assert all(lo % 4 == 0 for lo, _ in spans)                       # 4-byte words -> 16-byte alignment
    assert lay["ctrl_off"] + 16 == lay["state_word"] < lay["total"]


@settings(max_examples=200, deadline=None)
@given(n=st.integers(0, 1000), world=st.integers(1, 16))
def test_frame_shards_partition_the_batch(n, world):
    ranges = [parallel.shard_frames(n, r, world) for r in range(world)]
    assert ranges[0][0] == 0 and ranges[-1][1] == n
    sizes = [hi - lo for lo, hi in ranges]
    assert max(sizes) - min(sizes) <= 1 and all(a[1] == b[0] for a, b in zip(ranges, ranges[1:]))


def test_synth_is_deterministic():
    a = synth.synth_tensor("transformer.decoder.layers.0.attentions.1.attn.in_proj_weight", (768, 256), 0)
    b = synth.synth_tensor("transformer.decoder.layers.0.attentions.1.attn.in_proj_weight", (768, 256), 0)
    assert np.array_equal(a, b) and a.dtype == np.float32
    assert abs(float(a[0, 0]) - float(a[0, 0])) == 0 and float(np.abs(a).max()) <= np.sqrt(6.0 / (256 + 768)) + 1e-7


def test_graph_runner_calibration_key():
    """runtime._metas_key: a CUDA graph bakes the calibration in, so the key must change exactly when lidar2img (of any
    node prefix) or the pad shape changes, and ignore everything else in img_metas."""
    import numpy as np
    from cmtcoop_b200.runtime import _metas_key
    rng = np.random.RandomState(0)
    m = [dict(lidar2img=[rng.randn(4, 4) for _ in range(3)], pad_shape=[(640, 1600, 3)] * 3, sample_idx="a"),
         dict(lidar2img=[rng.randn(4, 4) for _ in range(3)], pad_shape=[(640, 1600, 3)] * 3, sample_idx="b")]
    k0 = _metas_key(m)
    same = [dict(d, sample_idx="other", box_type_3d=object) for d in m]
    assert _metas_key(same) == k0
    moved = [dict(d) for d in m]
    moved[1] = dict(moved[1], lidar2img=[x + (1e-9 if i == 2 else 0.0) for i, x in enumerate(m[1]["lidar2img"])])
    assert _metas_key(moved) != k0
    padded = [dict(d, pad_shape=[(672, 1600, 3)] * 3) for d in m]
    assert _metas_key(padded) != k0
    coop = [dict(vehicle_lidar2img=[np.eye(4)], infrastructure_lidar2img=[np.eye(4)] * 3)]
    coop2 = [dict(vehicle_lidar2img=[np.eye(4)], infrastructure_lidar2img=[np.eye(4)] * 2 + [2 * np.eye(4)])]
    assert _metas_key(coop) != _metas_key(coop2)


# ---------------------------------------------------------------------------------------------
# the reference's own configs (when CMT_REFERENCE_ROOT names a checkout of the original project)
REF_CONFIGS = os.path.join(ref_stub.REFERENCE_ROOT, "projects", "configs")


def _reference_config_files():
    import glob
    return sorted(glob.glob(os.path.join(REF_CONFIGS, "**", "*.py"), recursive=True))


@pytest.mark.skipif(not ref_stub.reference_available(),
                    reason="CMT_REFERENCE_ROOT does not name a checkout of the original project")
def test_every_reference_config_builds_its_head_unchanged():
    """All 13 config files of the reference: exec the file (plain python dicts, no _base_ inheritance), take
    model['pts_bbox_head'] with the detector's train/test cfg folded in exactly as MVXTwoStageDetector.__init__ does
    (pts_bbox_head.update(train_cfg=train_cfg.pts, test_cfg=test_cfg.pts)), and build it through the plugin registry."""
    files = _reference_config_files()
    assert len(files) == 13, files
    seen = set()
    for f in files:
        ns = {}
        exec(compile(open(f).read(), f, "exec"), ns)
        model = ns["model"]
        head_cfg = dict(model["pts_bbox_head"])
        test_cfg = model.get("test_cfg") or {}
        head_cfg.update(train_cfg=None, test_cfg=test_cfg.get("pts"))
        head = plugin.build_head(head_cfg)
        assert type(head).__name__ == head_cfg["type"] and not head.training
        seen.add(head_cfg["type"])
        assert head.num_query == 900 and len(head.transformer.decoder.layers) == 6
        n_bev = head.coords_bev.shape[0] if head._has_bev else 0
        assert n_bev in (0, 128 * 128, 180 * 180), (f, n_bev)
        # every cross-attention is the FlashMHA drop-in, state-dict keys are the reference's
        for layer in head.transformer.decoder.layers:
            assert isinstance(layer.attentions[1], plugin.PETRMultiheadFlashAttention)
        sd = head.state_dict()
        assert "reference_points.weight" in sd and "transformer.decoder.post_norm.weight" in sd
        assert "transformer.decoder.layers.5.attentions.1.attn.in_proj_weight" in sd
        assert ("shared_conv.conv.weight" in sd) == head._has_bev and ("rv_embedding.0.weight" in sd) == head._has_img
    assert seen == set(synth.HEAD_KINDS)
