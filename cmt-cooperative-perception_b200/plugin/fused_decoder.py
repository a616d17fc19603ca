"""Fused inference path of PETRTransformerDecoder for the standard layer
(`operation_order = self_attn, norm, cross_attn, norm, ffn, norm`, post-norm, eval, no attention mask;
projects/mmdet3d_plugin/models/utils/petr_transformer.py:347-487 + mmcv BaseTransformerLayer).

Same arithmetic as the module-by-module path in petr_transformer.py, but every op runs in
libcmtcoop_b200 and the activations stay batch-first [B,Nq,C] (the reference transposes to
sequence-first and back around every attention, petr_transformer.py:307-319):

  per layer (15 launches instead of ~60 eager ones):
    self-attention   Q/K/V^T projections (3 GEMMs) -> flash attention kernel -> out-proj GEMM
    norm0            fused (x + sa) LayerNorm, also emits lp(x1 + query_pos) for the next projection (lp: bf16 / fp16)
    cross-attention  Q GEMM -> flash attention over the hoisted K/V cache -> out-proj GEMM
    norm1            fused (x1 + ca) LayerNorm, also emits lp(x2) for the FFN
    ffn              GEMM+bias+ReLU, GEMM+bias
    norm2 (+post)    fused (x2 + ffn) LayerNorm + the shared post_norm written straight into the stacked
                     [L,B,Nq,C] output, also emits lp(x3), lp(x3 + query_pos) for the next layer
"""
from __future__ import annotations

import torch
import torch.nn as nn

from .. import ops
from .attention import KVCache, _Q_SCALE

_STD_ORDER = ("self_attn", "norm", "cross_attn", "norm", "ffn", "norm")

# Decoder layer 0 attends over an all-zero target: its self-attention is the constant row out_proj(b_v) (see _run).  False
# runs the five launches anyway (tests compare the two).
SKIP_ZERO_TARGET_SELF_ATTENTION = True

# diagnostics for bench.py: the operand-norm maxima of the last forward, (q_norm2 [L,B,H], [k_norm2 [B_i,L,H] per cache]) or None.
# An attention item (layer, frame, head) takes the static-shift kernel iff sqrt(qn * kn) * 1.0079 + 1e-3 <= limit, with
# limit STATIC_LIMIT[dtype] (the largest |score| whose weight 2^score is a normal number of the dtype).
STATIC_LIMIT = {torch.bfloat16: 60.0, torch.float16: 14.0}
last_norms = None


def _cached(module, tag, key, build):
    store = module.__dict__.setdefault("_cmt_cache", {})
    hit = store.get(tag)
    if hit is None or hit[0] != key:
        hit = (key, build())
        store[tag] = hit
    return hit[1]


def _pkey(*params):
    return tuple((p._version, p.data_ptr()) for p in params if p is not None)


def _mha_weights(attn: nn.MultiheadAttention, dt):
    """nn.MultiheadAttention parameters split per projection, in the compute dtype."""
    def build():
        E = attn.embed_dim
        w, b = attn.in_proj_weight.detach(), attn.in_proj_bias.detach().float()
        return dict(wq=w[:E].to(dt).contiguous(), wk=w[E:2 * E].to(dt).contiguous(), wv=w[2 * E:].to(dt).contiguous(),
                    bq=b[:E].contiguous(), bk=b[E:2 * E].contiguous(), bv=b[2 * E:].contiguous(),
                    wo=attn.out_proj.weight.detach().to(dt).contiguous(), bo=attn.out_proj.bias.detach().float().contiguous())
    return _cached(attn, "w", (dt,) + _pkey(attn.in_proj_weight, attn.in_proj_bias, attn.out_proj.weight,
                                             attn.out_proj.bias), build)


def _ffn_weights(ffn, dt):
    l0, l1 = ffn.layers[0][0], ffn.layers[1]

    def build():
        return (l0.weight.detach().to(dt).contiguous(), l0.bias.detach().float().contiguous(),
                l1.weight.detach().to(dt).contiguous(), l1.bias.detach().float().contiguous())
    return _cached(ffn, "w", (dt,) + _pkey(l0.weight, l0.bias, l1.weight, l1.bias), build)


def _ln(norm: nn.LayerNorm):
    return norm.weight.detach(), norm.bias.detach(), norm.eps


def supports(decoder, attn_masks, caches) -> bool:
    """True when the fused path computes exactly what the generic module path would.  caches: the list of KVCaches
    `run` would decode; several caches in one pass need every one unsplit and holding keys."""
    if len(caches) > 1 and any(c.group is not None or c.k is None for c in caches):
        return False
    if decoder.training or not decoder.return_intermediate or decoder.post_norm is None:
        return False
    if attn_masks is not None and any(m is not None for m in (attn_masks if isinstance(attn_masks, (list, tuple))
                                                               else [attn_masks])):
        return False
    eps = decoder.post_norm.eps
    for layer in decoder.layers:
        if any(n.eps != eps for n in layer.norms):
            return False
        if tuple(layer.operation_order) != _STD_ORDER or layer.pre_norm or layer.embed_dims != 256:
            return False
        sa = layer.attentions[0]
        if not isinstance(getattr(sa, "attn", None), nn.MultiheadAttention) or sa.attn.num_heads * ops.HEAD_DIM != 256:
            return False
        ffn = layer.ffns[0]
        if len(ffn.layers) != 3 or not ffn.add_identity:  # (Linear,ReLU,Dropout), Linear, Dropout
            return False
    return True


def run(decoder, query_pos: torch.Tensor, caches, precision: str) -> torch.Tensor:
    """query_pos [B,Nq,C] fp32 (batch-first).  Returns the stacked post-normed outputs [L,B,Nq,C] fp32.
    caches: a list of KVCaches covering consecutive frame ranges of the B frames -- one for all of them, or one per node
    for the cooperative heads: both nodes' frames in ONE decoder pass (shared weights and the same queries,
    cmt_head_coop.py:368-389) with one cross-attention launch per node because the nodes' token counts differ; every
    small op runs once over 2B frames."""
    cache = caches[0]
    dt = ops.compute_dtype(precision)
    B, Nq, C = query_pos.shape
    L = len(decoder.layers)
    H = decoder.layers[0].attentions[0].attn.num_heads
    dev = query_pos.device
    query_pos = query_pos.contiguous().float()
    out = torch.empty((L, B, Nq, C), dtype=torch.float32, device=dev)
    pw, pb, peps = _ln(decoder.post_norm)

    x = x_lp = xq_lp = None
    if not SKIP_ZERO_TARGET_SELF_ATTENTION:
        x = torch.zeros((B, Nq, C), dtype=torch.float32, device=dev)   # target = zeros (cmt_transformer.py:114)
        x_lp = torch.zeros((B, Nq, C), dtype=dt, device=dev)           # cast(x)
        xq_lp = query_pos.to(dt)                                       # cast(x + query_pos)

    # max |q|^2 per (layer, frame, head) of the cross-attention queries: with cache.k_norm2 the attention kernel gets a
    # bound on every score and drops the running row maximum (ops.cross_attn)
    static_shift = all(c.k_norm2 is not None for c in caches) and dt in STATIC_LIMIT
    qn2 = torch.zeros((L, B, H), dtype=torch.float32, device=dev) if static_shift else None

    global last_norms
    last_norms = (qn2, [c.k_norm2 for c in caches]) if static_shift else None   # k_norm2 per cache, frames in order
    for li, layer in enumerate(decoder.layers):
        # ---- self-attention over the queries: q = k = x + query_pos, v = x (key_pos = query_pos) ----
        sw = _mha_weights(layer.attentions[0].attn, dt)
        g, b, eps = _ln(layer.norms[0])
        if li == 0 and SKIP_ZERO_TARGET_SELF_ATTENTION:
            # The first layer's target is zero (cmt_transformer.py:114): every value row is the value bias b_v, so the
            # softmax-weighted mean is b_v for every query whatever the attention weights, and the block's output is the
            # single row out_proj(b_v) (operands rounded like the kernels round them).  x + attn_out is that row.
            sa_row = _cached(layer.attentions[0].attn, "zero_target_row", (dt,) + _pkey(*layer.attentions[0].attn.parameters()),
                             lambda: (sw["bv"].to(dt).float() @ sw["wo"].float().t() + sw["bo"]).contiguous())
            x1, _, _, x1q_lp = ops.add_layernorm(sa_row, None, g, b, eps, add=query_pos, lp_dtype=dt, want_yadd=True,
                                                 rows=(B, Nq))
        else:
            q = ops.linear(xq_lp, sw["wq"], sw["bq"], alpha=_Q_SCALE, out_dtype=dt)
            k = ops.project_keys(xq_lp, sw["wk"], sw["bk"], 1, H)
            vt = ops.project_values_t(x_lp, sw["wv"], sw["bv"], 1, H)
            ctx = ops.cross_attn(q, k, vt, 0, tag="self_attn")
            sa = ops.linear(ctx, sw["wo"], sw["bo"], out_dtype=torch.float32)
            x1, _, _, x1q_lp = ops.add_layernorm(x, sa, g, b, eps, add=query_pos, lp_dtype=dt, want_yadd=True)
        # ---- cross-attention over the hoisted K/V cache ----
        mha = layer.attentions[1].attn
        cw = mha.compute_weights()
        if static_shift:
            qc = ops.project_queries(x1q_lp, cw["wq"], cw["bq"], H, _Q_SCALE, norm2_max=qn2[li])
        else:
            qc = ops.linear(x1q_lp, cw["wq"], cw["bq"], alpha=_Q_SCALE, out_dtype=dt)
        if len(caches) > 1:
            ctx = torch.empty((B, Nq, C), dtype=dt, device=dev)
            f0 = 0
            for c in caches:
                nb = c.k.shape[0]
                ops.cross_attn(qc[f0:f0 + nb], c.k, c.vt, li, out=ctx[f0:f0 + nb], key_keep=c.key_keep,
                               q_norm2=qn2[li][f0:f0 + nb] if static_shift else None, k_norm2=c.k_norm2 if static_shift else None)
                f0 += nb
            assert f0 == B
        elif cache.group is None:
            # key_keep (sensor mask): the masked rows are finite (zero or ReLU(bias) features), so the operand-norm
            # bounds that include them still bound every attended score
            ctx = ops.cross_attn(qc, cache.k, cache.vt, li, key_keep=cache.key_keep,
                                 q_norm2=qn2[li] if static_shift else None, k_norm2=cache.k_norm2 if static_shift else None)
        else:
            ctx = mha._merge_kv_split(qc, cache, li, q_norm2=qn2[li] if static_shift else None)
        ca = ops.linear(ctx, cw["wo"], cw["bo"], out_dtype=torch.float32)
        g, b, eps = _ln(layer.norms[1])
        x2, _, x2_lp, _ = ops.add_layernorm(x1, ca, g, b, eps, lp_dtype=dt, want_ylp=True)
        # ---- FFN ----
        w0, b0, w1, b1 = _ffn_weights(layer.ffns[0], dt)
        h = ops.linear(x2_lp, w0, b0, relu=True, out_dtype=dt)
        f = ops.linear(h, w1, b1, out_dtype=torch.float32)
        g, b, eps = _ln(layer.norms[2])
        x, _, x_lp, xq_lp = ops.add_layernorm(x2, f, g, b, eps, gamma2=pw, beta2=pb, y2=out[li], add=query_pos,
                                              lp_dtype=dt, want_ylp=True, want_yadd=True)
    return out
