"""Decoder small ops on the GPU: the fused residual+LayerNorm kernel against torch, and the fused decoder
path (every op in libcmtcoop_b200) against the module-by-module path (torch self-attention / LN / FFN)."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from cmtcoop_b200 import ops, synth
from cmtcoop_b200.plugin import build_head
from oracle import cmt_oracle as O

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


@pytest.mark.parametrize("lp", [torch.bfloat16, torch.float32])
def test_add_layernorm(lp):
    g = torch.Generator().manual_seed(0)
    M, C = 1803, 256   # not a multiple of the rows per block
    x, r, add = (torch.randn(M, C, generator=g) for _ in range(3))
    w1, b1, w2, b2 = (torch.randn(C, generator=g) for _ in range(4))
    want_y = F.layer_norm(x + r, (C,), w1, b1, 1e-5)
    want_y2 = F.layer_norm(want_y, (C,), w2, b2, 1e-5)
    d = lambda t: t.to(DEV)
    y, y2, ylp, yadd = ops.add_layernorm(d(x), d(r), d(w1), d(b1), 1e-5, gamma2=d(w2), beta2=d(b2), add=d(add),
                                         lp_dtype=lp, want_ylp=True, want_yadd=True)
    assert torch.allclose(y.cpu(), want_y, atol=2e-5, rtol=1e-5)
    assert torch.allclose(y2.cpu(), want_y2, atol=5e-5, rtol=1e-5)
    assert torch.equal(ylp.cpu(), y.cpu().to(lp))                      # one rounding of the fp32 result
    assert torch.equal(yadd.cpu(), (y.cpu() + add).to(lp))
    y0, none2, none3, none4 = ops.add_layernorm(d(x), None, d(w1), d(b1), 1e-5)
    assert none2 is None and none3 is None and none4 is None
    assert torch.allclose(y0.cpu(), F.layer_norm(x, (C,), w1, b1, 1e-5), atol=2e-5, rtol=1e-5)


@pytest.mark.parametrize("precision,tol", [("fp32", 2e-5), ("bf16", 1e-2)])
@pytest.mark.parametrize("kind", ["CmtHead", "CmtLidarHeadCoop"])
def test_fused_decoder_equals_module_path(kind, precision, tol):
    cfg, inputs = synth.mini_case(kind)
    head = build_head(cfg)
    synth.load_synth_weights(head, 0)
    head = head.to(DEV).eval().set_precision(precision)
    d = {k: (torch.from_numpy(v).to(DEV) if isinstance(v, np.ndarray) else v) for k, v in inputs.items()}

    def run():
        with torch.no_grad():
            if kind.endswith("Coop"):
                return head.forward_single(d["vehicle_pts_feats"], d["infrastructure_pts_feats"],
                                           d["vehicle_img_feats"], d["infrastructure_img_feats"], d["img_metas"])
            return head.forward_single(d["pts_feats"], d["img_feats"], d["img_metas"])

    head.transformer.use_fused_decoder = True
    n0 = ops.launch_count()
    fused = run()
    n_fused = ops.launch_count() - n0
    head.transformer.use_fused_decoder = False
    n0 = ops.launch_count()
    modular = run()
    n_mod = ops.launch_count() - n0
    assert n_fused > n_mod                                  # the small ops moved into the library
    for name in fused[0]:
        assert O.rel_l2(fused[0][name].float().cpu(), modular[0][name].float().cpu()) < tol, name


@pytest.mark.parametrize("kind", ["CmtHead", "CmtImageHead", "CmtLidarHead"])
def test_reference_signature_transformer_forward(kind):
    """`head.transformer(...)` with the reference's arguments (cmt_transformer.py:84-127, :166-204, :243-282), called on
    the query embedding and position encodings the head computes, returns the head's own decoder output bit for bit
    and the token memory as [N_kv, B, C]."""
    cfg, inputs = synth.mini_case(kind)
    head = build_head(cfg)
    synth.load_synth_weights(head, 0)
    head = head.to(DEV).eval()
    head.apply_shared_conv = False   # the transformer's x is the map after shared_conv
    d = {k: (torch.from_numpy(v).to(DEV) if isinstance(v, np.ndarray) else v) for k, v in inputs.items()}
    x, x_img, metas = d.get("pts_feats"), d.get("img_feats"), d["img_metas"]
    B = len(metas)
    tr = head.transformer
    with torch.no_grad():
        if x is not None:
            x = head.shared_conv(x).contiguous()
        ref, attn_mask, _ = head.prepare_for_dn(B, head.reference_points.weight, metas)
        want = head.get_outs_dec(x, x_img, metas, ref, attn_mask)
        mats = head._matrices(metas, x_img.device) if x_img is not None else None
        query = head._query_embeds(ref, metas, mats)
        if kind == "CmtHead":
            out_dec, memory = tr(x, x_img, query, head._bev_pos_embed(x.device), head._rv_pe(x_img, metas, mats)[0],
                                 attn_masks=attn_mask)
        elif kind == "CmtLidarHead":
            out_dec, memory = tr(x, None, query, head._bev_pos_embed(x.device), attn_masks=attn_mask)
        else:
            out_dec, memory = tr(x_img, query, head._rv_pe(x_img, metas, mats)[0], attn_masks=attn_mask, bs=B)
    assert torch.isfinite(out_dec).all()   # so the head's nan_to_num leaves its output as the decoder wrote it
    assert torch.equal(out_dec, want)
    n_kv = (x.shape[2] * x.shape[3] if x is not None else 0) + (x_img[0, 0].numel() * (x_img.shape[0] // B) if x_img is not None else 0)
    assert memory.shape == (n_kv, B, out_dec.shape[-1])


@pytest.mark.parametrize("precision,tol", [("fp32", 1e-4), ("bf16", 1e-2)])
def test_flash_mha_key_padding_mask(precision, tol):
    """FlashMHA.forward(q, k, v, key_padding_mask) (attention.py:126-138 -> :76-90) against the oracle's
    nn.MultiheadAttention math with the padded keys dropped."""
    from cmtcoop_b200.plugin.attention import FlashMHA
    g = torch.Generator().manual_seed(3)
    B, Nq, S, E, H = 2, 50, 333, 256, 8
    mha = FlashMHA(E, H).eval()
    with torch.no_grad():
        for p in mha.parameters():
            p.copy_(torch.randn(p.shape, generator=g) * 0.05)
    sd = {"a." + k: v.detach().clone() for k, v in mha.state_dict().items()}
    mha = mha.to(DEV)
    mha.precision = precision
    q, k, v = (torch.randn(B, n, E, generator=g) for n in (Nq, S, S))
    keep = torch.rand(B, S, generator=g) > 0.35
    keep[0, :130] = False
    with torch.no_grad():
        out, _ = mha(q.to(DEV), k.to(DEV), v.to(DEV), key_padding_mask=keep.to(DEV))
    want = O.mha(q.transpose(0, 1), k.transpose(0, 1), v.transpose(0, 1), sd, "a", num_heads=H, key_keep=keep).transpose(0, 1)
    assert O.rel_l2(out.cpu(), want) < tol


@pytest.mark.parametrize("precision,tol", [("fp32", 1e-5), ("bf16", 2e-3)])
def test_zero_target_self_attention_shortcut(precision, tol):
    """Decoder layer 0 attends over the all-zero target (cmt_transformer.py:114): its self-attention block returns
    out_proj(b_v) for every query.  The one-row shortcut equals running the five launches."""
    from cmtcoop_b200.plugin import fused_decoder
    kind = "CmtHead"
    cfg, inputs = synth.mini_case(kind)
    head = build_head(cfg)
    synth.load_synth_weights(head, 0)
    head = head.to(DEV).eval().set_precision(precision)
    d = {k: (torch.from_numpy(v).to(DEV) if isinstance(v, np.ndarray) else v) for k, v in inputs.items()}
    outs = {}
    with torch.no_grad():
        head.forward_single(d["pts_feats"], d["img_feats"], d["img_metas"])   # fills the weight-only caches
    for skip in (True, False):
        fused_decoder.SKIP_ZERO_TARGET_SELF_ATTENTION = skip
        n0 = ops.launch_count()
        with torch.no_grad():
            outs[skip] = head.forward_single(d["pts_feats"], d["img_feats"], d["img_metas"])
        outs[skip] = (outs[skip], ops.launch_count() - n0)
    fused_decoder.SKIP_ZERO_TARGET_SELF_ATTENTION = True
    assert outs[True][1] < outs[False][1]
    for name in outs[True][0][0]:
        assert O.rel_l2(outs[True][0][0][name].float().cpu(), outs[False][0][0][name].float().cpu()) < tol, name
