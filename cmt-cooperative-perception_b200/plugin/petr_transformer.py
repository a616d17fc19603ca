"""Decoder stack with the reference's class names, constructor arguments, forward signatures and
state-dict keys (projects/mmdet3d_plugin/models/utils/petr_transformer.py:37-487, which builds on
mmcv-full 1.6.2 BaseTransformerLayer / TransformerLayerSequence / FFN -- not installed here, so the
few behaviours the configs rely on are implemented directly: operation order loop, post-norm,
`key_pos=query_pos` for self-attention, FFN residual).

Two execution paths share these modules (and their state-dict keys):
  * the default inference path is plugin/fused_decoder.py: when the decoder has the standard layer
    (self_attn, norm, cross_attn, norm, ffn, norm; post-norm; no attention mask) every op -- the 900x900
    self-attention, the Q/K/V/out projections, LayerNorms and the FFN -- runs in libcmtcoop_b200, in bf16 on
    the tensor cores with fp32 accumulation, residuals and LayerNorm statistics (the reference runs these in
    fp32 nn.MultiheadAttention / nn.Linear; the bf16 budget of 1e-2 rel-L2 on the head outputs covers it, and
    `set_precision('fp32')` switches every kernel to the fp32 CUDA-core verification path);
  * the module-by-module path below (`transformer.use_fused_decoder = False`, or a DN attention mask /
    non-standard layer): cross-attention on libcmtcoop_b200, self-attention through torch's
    nn.MultiheadAttention, LayerNorm / FFN as torch CUDA ops.
"""
from __future__ import annotations

import copy
import warnings

import torch
import torch.nn as nn

from .attention import FlashMHA, KVCache
from .registry import (ATTENTION, FEEDFORWARD_NETWORK, TRANSFORMER_LAYER, TRANSFORMER_LAYER_SEQUENCE)


def _dropout_cfg(dropout_layer, kwargs, attn_drop):
    """Shared `dropout` -> (attn_drop, dropout_layer) deprecation handling (petr_transformer.py:68-76)."""
    dropout_layer = dict(dropout_layer) if dropout_layer else None
    if "dropout" in kwargs:
        attn_drop = kwargs["dropout"]
        if dropout_layer is not None:
            dropout_layer["drop_prob"] = kwargs.pop("dropout")
        else:
            kwargs.pop("dropout")
    return attn_drop, dropout_layer


def _resolve_pos(query, key, value, identity, query_pos, key_pos, cls_name):
    if key is None:
        key = query
    if value is None:
        value = key
    if identity is None:
        identity = query
    if key_pos is None and query_pos is not None:
        if query_pos.shape == key.shape:
            key_pos = query_pos
        else:
            warnings.warn(f"position encoding of key is missing in {cls_name}.")
    return key, value, identity, key_pos


@ATTENTION.register_module()
@ATTENTION.register_module(name="MultiheadAttention")
class PETRMultiheadAttention(nn.Module):
    """petr_transformer.py:37-177 (identical to mmcv's MultiheadAttention wrapper): nn.MultiheadAttention
    with positional encodings and an identity connection.  Used for the 900x900 self-attention."""

    def __init__(self, embed_dims, num_heads, attn_drop=0., proj_drop=0.,
                 dropout_layer=dict(type="Dropout", drop_prob=0.), init_cfg=None, batch_first=False, **kwargs):
        super().__init__()
        attn_drop, dropout_layer = _dropout_cfg(dropout_layer, kwargs, attn_drop)
        self.embed_dims = embed_dims
        self.num_heads = num_heads
        self.batch_first = batch_first
        self.attn = nn.MultiheadAttention(embed_dims, num_heads, attn_drop, **kwargs)
        self.proj_drop = nn.Dropout(proj_drop)
        self.dropout_layer = nn.Dropout(dropout_layer["drop_prob"]) if dropout_layer else nn.Identity()

    def forward(self, query, key=None, value=None, identity=None, query_pos=None, key_pos=None,
                attn_mask=None, key_padding_mask=None, **kwargs):
        key, value, identity, key_pos = _resolve_pos(query, key, value, identity, query_pos, key_pos,
                                                     self.__class__.__name__)
        if query_pos is not None:
            query = query + query_pos
        if key_pos is not None:
            key = key + key_pos
        if self.batch_first:
            query, key, value = query.transpose(0, 1), key.transpose(0, 1), value.transpose(0, 1)
        out = self.attn(query=query, key=key, value=value, attn_mask=attn_mask,
                        key_padding_mask=key_padding_mask, need_weights=False)[0]
        if self.batch_first:
            out = out.transpose(0, 1)
        return identity + self.dropout_layer(self.proj_drop(out))


@ATTENTION.register_module()
class PETRMultiheadFlashAttention(nn.Module):
    """petr_transformer.py:182-321.  Sequence-first in / out like the reference; inner FlashMHA is
    batch-first.  Note the reference's constructor quirk: `FlashMHA(embed_dims, num_heads, attn_drop, ...)`
    passes attn_drop positionally into `bias` (petr_transformer.py:226 vs attention.py:97), i.e. bias on,
    attention dropout 0 -- reproduced here.

    Extra keyword arguments (flow through **kwargs exactly like mmcv's layer loop forwards them):
      kv_cache, layer_index : hoisted all-layer K/V projection built by CmtTransformer."""

    def __init__(self, embed_dims, num_heads, attn_drop=0., proj_drop=0.,
                 dropout_layer=dict(type="Dropout", drop_prob=0.), init_cfg=None, batch_first=True, **kwargs):
        super().__init__()
        attn_drop, dropout_layer = _dropout_cfg(dropout_layer, kwargs, attn_drop)
        self.embed_dims = embed_dims
        self.num_heads = num_heads
        self.batch_first = True
        self.attn = FlashMHA(embed_dims, num_heads, attn_drop, **kwargs)
        self.proj_drop = nn.Dropout(proj_drop)
        self.dropout_layer = nn.Dropout(dropout_layer["drop_prob"]) if dropout_layer else nn.Identity()

    def forward(self, query, key=None, value=None, identity=None, query_pos=None, key_pos=None,
                attn_mask=None, key_padding_mask=None, kv_cache: KVCache = None, layer_index: int = 0, **kwargs):
        if kv_cache is None:
            key, value, identity, key_pos = _resolve_pos(query, key, value, identity, query_pos, key_pos,
                                                         self.__class__.__name__)
        elif identity is None:
            identity = query
        if query_pos is not None:
            query = query + query_pos
        q = query.transpose(0, 1)
        if kv_cache is None:
            if key_pos is not None:
                key = key + key_pos
            out = self.attn(q=q, k=key.transpose(0, 1), v=value.transpose(0, 1), key_padding_mask=None)[0]
        else:
            # the sensor mask of the cache (None unless a sensor is missing for some frames) is the key_padding_mask
            out = self.attn(q=q, k=None, v=None, key_padding_mask=kv_cache.key_keep, kv_cache=kv_cache,
                            layer_index=layer_index)[0]
        out = out.transpose(0, 1)
        return identity + self.dropout_layer(self.proj_drop(out))


@FEEDFORWARD_NETWORK.register_module()
class FFN(nn.Module):
    """mmcv FFN: layers = Sequential(Sequential(Linear, ReLU, Dropout), Linear, Dropout); out + identity.
    State-dict keys layers.0.0.{weight,bias}, layers.1.{weight,bias}."""

    def __init__(self, embed_dims=256, feedforward_channels=1024, num_fcs=2, act_cfg=dict(type="ReLU", inplace=True),
                 ffn_drop=0., dropout_layer=None, add_identity=True, init_cfg=None, **kwargs):
        super().__init__()
        assert num_fcs >= 2
        self.embed_dims = embed_dims
        layers, c = [], embed_dims
        for _ in range(num_fcs - 1):
            layers.append(nn.Sequential(nn.Linear(c, feedforward_channels), nn.ReLU(inplace=True), nn.Dropout(ffn_drop)))
            c = feedforward_channels
        layers += [nn.Linear(feedforward_channels, embed_dims), nn.Dropout(ffn_drop)]
        self.layers = nn.Sequential(*layers)
        self.dropout_layer = nn.Dropout(dropout_layer["drop_prob"]) if dropout_layer else nn.Identity()
        self.add_identity = add_identity

    def forward(self, x, identity=None):
        out = self.layers(x)
        if not self.add_identity:
            return self.dropout_layer(out)
        return (x if identity is None else identity) + self.dropout_layer(out)


@TRANSFORMER_LAYER.register_module()
class PETRTransformerDecoderLayer(nn.Module):
    """petr_transformer.py:374-487 + the mmcv BaseTransformerLayer behaviour it inherits."""

    def __init__(self, attn_cfgs, feedforward_channels=None, ffn_dropout=0.0, operation_order=None,
                 act_cfg=dict(type="ReLU", inplace=True), norm_cfg=dict(type="LN"), ffn_num_fcs=2, with_cp=True,
                 ffn_cfgs=dict(type="FFN", embed_dims=256, feedforward_channels=1024, num_fcs=2, ffn_drop=0.,
                               act_cfg=dict(type="ReLU", inplace=True)),
                 batch_first=False, init_cfg=None, **kwargs):
        super().__init__()
        assert len(operation_order) == 6
        assert set(operation_order) == set(["self_attn", "norm", "cross_attn", "ffn"])
        ffn_cfgs = copy.deepcopy(dict(ffn_cfgs))
        # mmcv maps the deprecated arguments into ffn_cfgs (the configs still pass feedforward_channels)
        if feedforward_channels is not None:
            ffn_cfgs["feedforward_channels"] = feedforward_channels
        ffn_cfgs["ffn_drop"] = ffn_dropout if "ffn_drop" not in ffn_cfgs else ffn_cfgs["ffn_drop"]
        ffn_cfgs["num_fcs"] = ffn_num_fcs
        self.batch_first = batch_first
        self.operation_order = tuple(operation_order)
        self.pre_norm = operation_order[0] == "norm"
        self.use_checkpoint = with_cp
        num_attn = operation_order.count("self_attn") + operation_order.count("cross_attn")
        if isinstance(attn_cfgs, dict):
            attn_cfgs = [copy.deepcopy(attn_cfgs) for _ in range(num_attn)]
        assert len(attn_cfgs) == num_attn
        self.num_attn = num_attn
        self.attentions = nn.ModuleList()
        for cfg in attn_cfgs:
            cfg = dict(copy.deepcopy(cfg))
            cfg["batch_first"] = batch_first
            self.attentions.append(ATTENTION.build(cfg))
        self.embed_dims = self.attentions[0].embed_dims
        self.ffns = nn.ModuleList()
        for _ in range(operation_order.count("ffn")):
            c = dict(ffn_cfgs)
            c.setdefault("embed_dims", self.embed_dims)
            self.ffns.append(FEEDFORWARD_NETWORK.build(c))
        assert norm_cfg.get("type", "LN") == "LN"
        self.norms = nn.ModuleList(nn.LayerNorm(self.embed_dims, eps=norm_cfg.get("eps", 1e-5))
                                   for _ in range(operation_order.count("norm")))

    def forward(self, query, key=None, value=None, query_pos=None, key_pos=None, attn_masks=None,
                query_key_padding_mask=None, key_padding_mask=None, **kwargs):
        if self.training:
            raise NotImplementedError("libcmtcoop_b200 is forward/inference only (call .eval())")
        norm_i = attn_i = ffn_i = 0
        identity = query
        if attn_masks is None:
            attn_masks = [None] * self.num_attn
        elif isinstance(attn_masks, torch.Tensor):
            attn_masks = [attn_masks.clone() for _ in range(self.num_attn)]
        for op in self.operation_order:
            if op == "self_attn":
                query = self.attentions[attn_i](query, query, query, identity if self.pre_norm else None,
                                                query_pos=query_pos, key_pos=query_pos,
                                                attn_mask=attn_masks[attn_i],
                                                key_padding_mask=query_key_padding_mask, **kwargs)
                attn_i += 1
                identity = query
            elif op == "norm":
                query = self.norms[norm_i](query)
                norm_i += 1
            elif op == "cross_attn":
                query = self.attentions[attn_i](query, key, value, identity if self.pre_norm else None,
                                                query_pos=query_pos, key_pos=key_pos,
                                                attn_mask=attn_masks[attn_i],
                                                key_padding_mask=key_padding_mask, **kwargs)
                attn_i += 1
                identity = query
            elif op == "ffn":
                query = self.ffns[ffn_i](query, identity if self.pre_norm else None)
                ffn_i += 1
        return query


@TRANSFORMER_LAYER_SEQUENCE.register_module()
class PETRTransformerDecoder(nn.Module):
    """petr_transformer.py:324-371: stack of layers, every layer output post-normed and stacked."""

    def __init__(self, transformerlayers=None, num_layers=None, post_norm_cfg=dict(type="LN"),
                 return_intermediate=False, init_cfg=None):
        super().__init__()
        if isinstance(transformerlayers, dict):
            transformerlayers = [copy.deepcopy(transformerlayers) for _ in range(num_layers)]
        assert len(transformerlayers) == num_layers
        self.num_layers = num_layers
        self.layers = nn.ModuleList(TRANSFORMER_LAYER.build(c) for c in transformerlayers)
        self.embed_dims = self.layers[0].embed_dims
        self.pre_norm = self.layers[0].pre_norm
        self.return_intermediate = return_intermediate
        self.post_norm = nn.LayerNorm(self.embed_dims) if post_norm_cfg is not None else None

    def forward(self, query, *args, **kwargs):
        intermediate = []
        for i, layer in enumerate(self.layers):
            query = layer(query, *args, layer_index=i, **kwargs)
            if self.return_intermediate:
                intermediate.append(self.post_norm(query) if self.post_norm is not None else query)
        if not self.return_intermediate:
            if self.post_norm is not None:
                query = self.post_norm(query)[None]
            return query
        return torch.stack(intermediate)


def build_transformer_layer_sequence(cfg):
    return TRANSFORMER_LAYER_SEQUENCE.build(cfg)
