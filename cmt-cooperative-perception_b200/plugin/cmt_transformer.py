"""CmtTransformer / CmtLidarTransformer / CmtImageTransformer with the reference's signatures
(projects/mmdet3d_plugin/models/utils/cmt_transformer.py:48-282).

Where the reference materialises `memory` and `pos_embed` as two [N_kv,B,C] fp32 tensors
(rearrange + cat + repeat, :105-110) and lets every decoder layer redo `key + key_pos` and the K/V
projections, these classes run ONE fused gather kernel (NCHW -> token-major, BEV ++ image concat,
+pos, cast) and ONE pair of all-layer K / V^T projection GEMMs, then hand the decoder a KVCache.
"""
from __future__ import annotations

import torch
import torch.nn as nn

from .. import ops
from . import fused_decoder
from .attention import KVCache
from .petr_transformer import PETRMultiheadFlashAttention, build_transformer_layer_sequence
from .registry import TRANSFORMER


_compute_dtype = ops.compute_dtype


class _CmtTransformerBase(nn.Module):
    def __init__(self, encoder=None, decoder=None, init_cfg=None, cross=False):
        super().__init__()
        self.encoder = build_transformer_layer_sequence(encoder) if encoder is not None else None
        self.decoder = build_transformer_layer_sequence(decoder)
        self.embed_dims = self.decoder.embed_dims
        self.cross = cross
        self.precision = "bf16"
        self.kv_split_group = None
        self.kv_split_peer = False      # True: exchange + merge as one kernel over peer memory instead of NCCL all-gather + merge
        self._peer = None
        self.use_fused_decoder = True  # False: module-by-module path (torch self-attention / LN / FFN)
        self._kv_w = None
        self._xp = None
        self._is_init = False

    def init_weights(self):
        # follow the official DETR init (cmt_transformer.py:77-82): xavier-uniform on every >1-dim weight
        for m in self.modules():
            if hasattr(m, "weight") and isinstance(m.weight, torch.Tensor) and m.weight.dim() > 1:
                nn.init.xavier_uniform_(m.weight)
                if getattr(m, "bias", None) is not None:
                    nn.init.constant_(m.bias, 0.0)
        self._is_init = True

    def set_precision(self, precision):
        _compute_dtype(precision)   # rejects an unknown precision
        self.precision = precision
        for m in self.modules():
            if hasattr(m, "precision"):
                m.precision = precision

    # -- hoisted all-layer K / V projection ---------------------------------------------------
    def _cross_attns(self):
        out = []
        for layer in self.decoder.layers:
            ca = [a for a, op in zip(layer.attentions, [o for o in layer.operation_order if o.endswith("attn")])
                  if op == "cross_attn"]
            assert len(ca) == 1 and isinstance(ca[0], PETRMultiheadFlashAttention), \
                "cross-attention must be PETRMultiheadFlashAttention (as in every reference config)"
            out.append(ca[0].attn)
        return out

    def _stacked_kv_weights(self):
        mhas = self._cross_attns()
        dt = _compute_dtype(self.precision)
        key = (dt,) + tuple((m.in_proj_weight._version, m.in_proj_weight.data_ptr(),
                             None if m.in_proj_bias is None else m.in_proj_bias._version) for m in mhas)
        if self._kv_w is None or self._kv_w[0] != key:
            E = self.embed_dims
            wk = torch.cat([m.in_proj_weight.detach()[E:2 * E] for m in mhas]).to(dt).contiguous()
            wv = torch.cat([m.in_proj_weight.detach()[2 * E:] for m in mhas]).to(dt).contiguous()
            if mhas[0].in_proj_bias is not None:
                bk = torch.cat([m.in_proj_bias.detach()[E:2 * E] for m in mhas]).float().contiguous()
                bv = torch.cat([m.in_proj_bias.detach()[2 * E:] for m in mhas]).float().contiguous()
            else:
                bk = bv = None
            self._kv_w = (key, (wk, bk, wv, bv))
        return self._kv_w[1]

    def kv_token_range(self, n_kv):
        """Token range [lo, hi) of the concatenated BEV ++ image axis this rank gathers, projects and attends:
        everything unless the KV-token split is enabled (then a tile-aligned share, parallel.kv_split_range)."""
        if self.kv_split_group is None:
            return 0, n_kv
        import torch.distributed as dist
        from .. import parallel
        return parallel.kv_split_range(n_kv, dist.get_rank(self.kv_split_group), dist.get_world_size(self.kv_split_group))

    def build_kv_cache(self, x_bev, x_img, bev_pos, rv_pos, B, V, conv=None, rv_rows=None, sensor_valid=None):
        """gather (K4) + all-layer K / V^T projection (K2).  Returns (KVCache, xv [B,n_tok,C]) where n_tok is
        this rank's share of the token axis (all tokens without the KV-token split).
        conv: None, or the folded shared_conv (w [Cout, 9*Cin] tap-major in the compute dtype with the BN scale folded in,
        bias [Cout] fp32); x_bev is then the map BEFORE shared_conv, and the 3x3 convolution runs as a tcgen05 implicit
        GEMM whose epilogue writes the BEV token rows of xk / xv directly (cmt_head.py:280-287,481 fused with
        cmt_transformer.py:105-110 and petr_transformer.py:296-299).
        rv_rows: None, or (a, b) when rv_pos holds rows [a, b) of every frame's V*h*w image tokens only, [B, b-a, C] (a
        rank of the KV-token split runs the rv-PE MLP on its own tokens; a == b: its share holds no image token).
        sensor_valid: optional torch.bool [S, B] device mask, one row per sensor in token order (the BEV map first when
        there is one, then the V cameras).  An absent sensor's tokens become zero rows of xk / xv (the fused shared_conv
        path: zero input rows, hence finite conv rows) and the cache carries the [B, N_kv] key mask that drops them from
        every cross-attention."""
        dt = _compute_dtype(self.precision)
        n_img_tok = V * x_img.shape[2] * x_img.shape[3] if x_img is not None else 0
        n_kv = (x_bev.shape[2] * x_bev.shape[3] if x_bev is not None else 0) + n_img_tok
        lo, hi = self.kv_token_range(n_kv)
        if rv_rows is not None and rv_rows[1] <= rv_rows[0]:
            x_img, rv_pos, rv_rows, V = None, None, None, 0   # this rank's share holds no image token
        group = self.kv_split_group
        L = len(self.decoder.layers)
        H = self.decoder.layers[0].attentions[-1].num_heads
        if hi <= lo:   # more ranks than token tiles: this rank contributes the neutral element of the merge
            return KVCache(None, None, 0, group, peer=self._peer_exchange if self.kv_split_peer else None), None
        # with the split, the gather kernel itself produces only the rank's rows: K1/K4/K2 all shard with the tokens
        if conv is not None:
            Hb, Wb = x_bev.shape[2], x_bev.shape[3]
            n_bev = Hb * Wb
            w, bias = conv
            C = w.shape[0]
            dev = x_bev.device
            xk = torch.empty((B, hi - lo, C), dtype=dt, device=dev)
            xv = torch.empty((B, hi - lo, C), dtype=dt, device=dev)
            key = (tuple(x_bev.shape), str(dev), dt)
            lidar_valid = None if sensor_valid is None else sensor_valid[0]
            if self._xp is None or self._xp[0] != key:   # zero-padded channel-last operand: zeroed once, interior rewritten per call
                self._xp = (key, ops.nchw_to_padded_nhwc(x_bev, dtype=dt, frame_valid=lidar_valid))
            else:
                ops.nchw_to_padded_nhwc(x_bev, self._xp[1], dtype=dt, frame_valid=lidar_valid)
            if lo < n_bev:
                ops.shared_conv_tokens(self._xp[1], w, bias, bev_pos, xk, xv, Hb, Wb, tok_range=(lo, min(hi, n_bev)))
            if x_img is not None and hi > n_bev:
                ops.gather_tokens(None, x_img, None, rv_pos, B, V, out_dtype=dt, tok_range=(lo, hi), n_bev_reserved=n_bev,
                                  out=(xk, xv), rv_rows=rv_rows, sensor_valid=sensor_valid)
        else:
            xk, xv = ops.gather_tokens(x_bev, x_img, bev_pos, rv_pos, B, V, out_dtype=dt,
                                       tok_range=None if group is None else (lo, hi), rv_rows=rv_rows,
                                       sensor_valid=sensor_valid)
        key_keep = None
        if sensor_valid is not None:
            key_keep = ops.sensor_key_keep(sensor_valid, B, n_kv - n_img_tok, V, n_img_tok // V if V else 0)
        wk, bk, wv, bv = self._stacked_kv_weights()
        kn2 = torch.zeros((B, L, H), dtype=torch.float32, device=xk.device) if dt != torch.float32 else None
        k = ops.project_keys(xk, wk, bk, L, H, norm2_max=kn2)
        vt = ops.project_values_t(xv, wv, bv, L, H)
        return KVCache(k, vt, hi - lo, group, k_norm2=kn2, peer=self._peer_exchange if (group is not None and self.kv_split_peer) else None,
                       key_keep=key_keep), xv

    def enable_kv_split(self, group=None, peer_memory=False):
        """Split the K/V token axis across the ranks of `group` (default: the WORLD group); every rank
        must call forward with the SAME frames.  Pass `False` to switch back to frame sharding.
        peer_memory=True: the per-layer exchange of (O | LSE) records and their merge run as ONE kernel that reads the
        other ranks' records through NVLink (parallel.PeerExchange, cmt_lse_merge_peer) -- no NCCL call on the data path;
        False: one NCCL all-gather per layer + cmt_lse_merge."""
        if group is False:
            self.kv_split_group = None
            self.kv_split_peer = False
            self._peer = None
            return self
        import torch.distributed as dist
        self.kv_split_group = group if group is not None else dist.group.WORLD
        self.kv_split_peer = bool(peer_memory)
        return self

    def _peer_exchange(self, B, Nq, H, device):
        """The peer-mapped record buffers for this shape (allocated collectively on first use: every rank of the group
        reaches this point with the same shapes; not inside a CUDA-graph capture -- run one eager forward first)."""
        L = max(2, len(self.decoder.layers))
        if self._peer is None or not self._peer.matches(B, Nq, H, L):
            from .. import parallel
            self._peer = parallel.PeerExchange(self.kv_split_group, device, B, Nq, H, L)
        return self._peer

    def decode(self, caches, query_embed, attn_masks=None):
        """Decoder pass over the frames of a list of KVCaches: query_embed [sum B_i, Nq, C], caches[i] covering the next
        B_i frames.  Returns the stacked outputs [L, sum B_i, Nq, C].  The fused decoder takes every cache in one pass
        when it supports the configuration; otherwise a single cache goes through the module-by-module path and several
        caches give None (the caller then decodes each cache on its own)."""
        if self.training:
            raise NotImplementedError("libcmtcoop_b200 is forward/inference only (call .eval())")
        if self.use_fused_decoder and fused_decoder.supports(self.decoder, attn_masks, caches):
            return fused_decoder.run(self.decoder, query_embed, caches, self.precision)
        if len(caches) > 1:
            return None
        query_embed = query_embed.transpose(0, 1)  # [B,Nq,C] -> [Nq,B,C]
        target = torch.zeros_like(query_embed)
        out_dec = self.decoder(query=target, key=None, value=None, key_pos=None, query_pos=query_embed,
                               key_padding_mask=None, attn_masks=[attn_masks, None], kv_cache=caches[0])
        return out_dec.transpose(1, 2)  # [L,B,Nq,C]


@TRANSFORMER.register_module()
class CmtTransformer(_CmtTransformerBase):
    """cmt_transformer.py:48-127: BEV + image tokens."""

    def forward(self, x, x_img, query_embed, bev_pos_embed, rv_pos_embed, attn_masks=None, reg_branch=None):
        bs = x.shape[0]
        V = x_img.shape[0] // bs
        cache, xv = self.build_kv_cache(x.contiguous(), x_img.contiguous(), bev_pos_embed.contiguous(),
                                        rv_pos_embed.contiguous(), bs, V)
        out_dec = self.decode([cache], query_embed, attn_masks)
        return out_dec, (None if xv is None else xv.transpose(0, 1))  # memory as [N_kv,B,C] (compute dtype)


@TRANSFORMER.register_module()
class CmtLidarTransformer(_CmtTransformerBase):
    """cmt_transformer.py:130-204: BEV tokens only. `mask` is accepted and ignored like the reference's
    all-zero key_padding_mask."""

    def forward(self, x, mask, query_embed, pos_embed, attn_masks=None, reg_branch=None):
        bs = x.shape[0]
        cache, xv = self.build_kv_cache(x.contiguous(), None, pos_embed.contiguous(), None, bs, 0)
        out_dec = self.decode([cache], query_embed, attn_masks)
        return out_dec, (None if xv is None else xv.transpose(0, 1))


@TRANSFORMER.register_module()
class CmtImageTransformer(_CmtTransformerBase):
    """cmt_transformer.py:207-282: image tokens only."""

    def forward(self, x_img, query_embed, rv_pos_embed, attn_masks=None, reg_branch=None, bs=2):
        V = x_img.shape[0] // bs
        cache, xv = self.build_kv_cache(None, x_img.contiguous(), None, rv_pos_embed.contiguous(), bs, V)
        out_dec = self.decode([cache], query_embed, attn_masks)
        return out_dec, (None if xv is None else xv.transpose(0, 1))
