"""FlashAttention / FlashMHA with the reference's constructor and forward signatures
(projects/mmdet3d_plugin/models/utils/attention.py:30-138), backed by libcmtcoop_b200:
in-projection and out-projection run on the tcgen05 GEMM, the attention core on the tcgen05
flash kernel (bf16 and fp16 modes) or on the fp32 CUDA-core kernels (fp32 verification mode).

State-dict keys are the reference's: in_proj_weight [3E,E], in_proj_bias [3E], out_proj.{weight,bias}.
"""
from __future__ import annotations

import math

import torch
import torch.nn as nn

from .. import ops

_Q_SCALE = ops.LOG2E / math.sqrt(ops.HEAD_DIM)  # Q is pre-multiplied by log2(e)/sqrt(d): softmax is a bare exp2
_compute_dtype = ops.compute_dtype


class KVCache:
    """Keys / transposed values of *all* decoder layers, projected once per forward.

    `key + key_pos` and `value` are identical for the six decoder layers
    (models/utils/cmt_transformer.py:116-125 hands the same memory/pos_embed to every layer); only
    W_k / W_v differ, so the twelve per-layer projections of the reference are two wide GEMMs here.
    k:  [B, L, H, N_kv, 32]      vt: [B, L, H, 32, ld]
    k_norm2: [B, L, H] fp32 max_token |k|^2 (written by the K projection's epilogue), or None: with the matching
    query maxima it lets the attention kernel use a static softmax shift (ops.cross_attn).
    key_keep: [B, N_kv] bool, False for the tokens of a sensor that did not deliver the frame (ops.sensor_key_keep), or
    None: every cross-attention of every layer attends the True tokens only.
    """

    def __init__(self, k, vt, n_kv, group=None, k_norm2=None, peer=None, key_keep=None):
        self.peer = peer      # callable (B, Nq, H, device) -> parallel.PeerExchange: the layer's exchange + merge as one kernel over peer memory; None: NCCL all-gather
        self.k = k
        self.vt = vt
        self.k_norm2 = k_norm2
        self.key_keep = key_keep
        self.n_kv = n_kv      # tokens held by THIS rank (all of them unless KV-split)
        self.group = group    # torch.distributed group when the token axis is split across ranks


class FlashAttention(nn.Module):
    """attention.py:30-92.  forward(q [B,T,H,D], kv [B,S,2,H,D]) -> (out [B,T,H,D] fp32, None)."""

    def __init__(self, softmax_scale=None, attention_dropout=0.0, device=None, dtype=None):
        super().__init__()
        self.softmax_scale = softmax_scale
        self.dropout_p = attention_dropout
        self.fp16_enabled = True
        self.precision = "bf16"

    def set_precision(self, precision):
        """'bf16' (default) or 'fp16' (tcgen05 kernel; the reference runs flash-attn in fp16), or 'fp32' (CUDA-core)."""
        _compute_dtype(precision)
        self.precision = precision
        return self

    def forward(self, q, kv, causal=False, key_padding_mask=None):
        assert q.is_cuda and kv.is_cuda, "FlashAttention runs on the GPU only (no CPU fallback)"
        assert q.shape[0] == kv.shape[0] and q.shape[-2] == kv.shape[-2] and q.shape[-1] == kv.shape[-1]
        if causal:
            raise NotImplementedError("causal attention is never used on the CMT path (attention.py:98)")
        if key_padding_mask is not None:
            # attention.py:76-90: unpad_input keeps the keys whose mask entry is True (flash-attn bert_padding
            # convention) and packs them with cu_seqlens_k; masking the dropped keys is the same softmax
            assert key_padding_mask.shape == (q.shape[0], kv.shape[1]), "key_padding_mask must be [B, S]"
        if self.training and self.dropout_p > 0:
            raise NotImplementedError("forward/inference only")
        B, T, H, D = q.shape
        S = kv.shape[1]
        assert D == ops.HEAD_DIM, "head_dim 32 only (256/8 in every reference config)"
        scale = self.softmax_scale if self.softmax_scale is not None else 1.0 / math.sqrt(D)
        dt = _compute_dtype(self.precision)
        qs = (q.float() * (scale * ops.LOG2E)).to(dt).reshape(B, T, H * D).contiguous()
        k = kv[:, :, 0].permute(0, 2, 1, 3).to(dt).contiguous().view(B, 1, H, S, D)
        ld = (S + 7) // 8 * 8
        vt = torch.zeros((B, 1, H, D, ld), dtype=dt, device=q.device)
        vt[:, 0, :, :, :S] = kv[:, :, 1].permute(0, 2, 3, 1).to(dt)   # [B,H,D,S] into the single-layer cache
        o = ops.cross_attn(qs, k, vt, 0, o_dtype=torch.float32,
                           key_keep=None if key_padding_mask is None else key_padding_mask.to(q.device).bool())
        return o.view(B, T, H, D), None


class FlashMHA(nn.Module):
    """attention.py:95-138 (batch-first). forward(q,k,v,key_padding_mask=None) -> (out, None)."""

    def __init__(self, embed_dim, num_heads, bias=True, batch_first=True, attention_dropout=0.0,
                 causal=False, device=None, dtype=None, **kwargs):
        assert batch_first
        if causal:
            # the reference forwards causal=self.causal to the inner attention (attention.py:136); no CMT config sets it
            # and the tcgen05 kernel has no causal mask: refuse instead of silently computing non-causal attention
            raise NotImplementedError("FlashMHA(causal=True): causal attention is not on the CMT path (attention.py:98)")
        super().__init__()
        self.embed_dim = embed_dim
        self.causal = causal
        self.bias = bias
        self.num_heads = num_heads
        assert embed_dim % num_heads == 0, "self.kdim must be divisible by num_heads"
        self.head_dim = embed_dim // num_heads
        assert self.head_dim == ops.HEAD_DIM, "libcmtcoop_b200 implements head_dim 32 (embed 256 / 8 heads)"
        self.in_proj_weight = nn.Parameter(torch.empty((3 * embed_dim, embed_dim)))
        if bias:
            self.in_proj_bias = nn.Parameter(torch.empty(3 * embed_dim))
        else:
            self.register_parameter("in_proj_bias", None)
        self.inner_attn = FlashAttention(attention_dropout=attention_dropout)
        self.out_proj = nn.Linear(embed_dim, embed_dim, bias=bias)
        self.precision = "bf16"
        self._wcache = None
        self._reset_parameters()

    def set_precision(self, precision):
        """'bf16' (default), 'fp16' or 'fp32' for the projections and the attention core."""
        _compute_dtype(precision)
        self.precision = precision
        self.inner_attn.precision = precision
        return self

    def _reset_parameters(self):
        nn.init.xavier_uniform_(self.in_proj_weight)
        if self.in_proj_bias is not None:
            nn.init.constant_(self.in_proj_bias, 0.0)
            nn.init.constant_(self.out_proj.bias, 0.0)

    # -- weights in the compute dtype, refreshed when the parameters change -------------------
    def compute_weights(self):
        dt = _compute_dtype(self.precision)
        key = (dt, self.in_proj_weight._version, self.in_proj_weight.data_ptr(), self.out_proj.weight._version,
               self.out_proj.weight.data_ptr(),
               None if self.in_proj_bias is None else self.in_proj_bias._version,
               None if self.out_proj.bias is None else self.out_proj.bias._version)
        if self._wcache is None or self._wcache[0] != key:
            E = self.embed_dim
            w = self.in_proj_weight.detach()
            b = self.in_proj_bias.detach().float() if self.in_proj_bias is not None else None
            ws = dict(
                wq=w[:E].to(dt).contiguous(), wk=w[E:2 * E].to(dt).contiguous(), wv=w[2 * E:].to(dt).contiguous(),
                bq=None if b is None else b[:E].contiguous(), bk=None if b is None else b[E:2 * E].contiguous(),
                bv=None if b is None else b[2 * E:].contiguous(),
                wo=self.out_proj.weight.detach().to(dt).contiguous(),
                bo=None if self.out_proj.bias is None else self.out_proj.bias.detach().float().contiguous())
            self._wcache = (key, ws)
        return self._wcache[1]

    def project_q(self, q):
        """(q W_q^T + b_q) * log2(e)/sqrt(d), [B,Nq,E] in the compute dtype (attention.py:21-27,131)."""
        ws = self.compute_weights()
        dt = _compute_dtype(self.precision)
        return ops.linear(q.to(dt).contiguous(), ws["wq"], ws["bq"], alpha=_Q_SCALE, out_dtype=dt)

    def attend(self, q, cache: KVCache, layer: int, kv_begin=0, kv_end=None, return_lse=False, o_dtype=None,
               key_keep=None):
        qp = self.project_q(q)
        return ops.cross_attn(qp, cache.k, cache.vt, layer, kv_begin=kv_begin, kv_end=kv_end,
                              return_lse=return_lse, o_dtype=o_dtype, key_keep=key_keep)

    def project_out(self, ctx):
        ws = self.compute_weights()
        return ops.linear(ctx, ws["wo"], ws["bo"], out_dtype=torch.float32)

    def forward(self, q, k, v, key_padding_mask=None, kv_cache: KVCache = None, layer_index: int = 0):
        """q [B,Nq,E], k/v [B,S,E] (batch-first).  With `kv_cache` the K/V projections of this layer are
        taken from the hoisted all-layer projection and `k`/`v` are ignored."""
        if self.training:
            raise NotImplementedError("libcmtcoop_b200 is forward/inference only")
        key_keep = None
        if key_padding_mask is not None:
            # attention.py:131-137 hands the mask to FlashAttention, whose unpad_input keeps the True entries
            # (attention.py:76-90); the CMT wrappers always pass None (petr_transformer.py:312-316)
            if kv_cache is not None and kv_cache.group is not None:
                raise NotImplementedError("key_padding_mask together with the multi-GPU KV-token split")
            key_keep = key_padding_mask.to(q.device).bool()
        if not q.is_cuda:
            raise RuntimeError("FlashMHA needs CUDA tensors: libcmtcoop_b200 has no CPU fallback")
        if kv_cache is None:
            ws = self.compute_weights()
            dt = _compute_dtype(self.precision)
            kk = ops.project_keys(k.to(dt).contiguous(), ws["wk"], ws["bk"], 1, self.num_heads)
            vt = ops.project_values_t(v.to(dt).contiguous(), ws["wv"], ws["bv"], 1, self.num_heads)
            kv_cache, layer_index = KVCache(kk, vt, k.shape[1]), 0
        if kv_cache.group is None:
            ctx = self.attend(q, kv_cache, layer_index, key_keep=key_keep)
        else:
            ctx = self._attend_kv_split(q, kv_cache, layer_index)
        return self.project_out(ctx), None

    def _attend_kv_split(self, q, cache: KVCache, layer: int):
        """KV tokens are split across the ranks of `cache.group`: local partial (normalised O + LSE) ->
        all-gather over NVLink (NCCL) -> log-sum-exp merge.  Queries are replicated."""
        return self._merge_kv_split(self.project_q(q), cache, layer)

    def _merge_kv_split(self, qp, cache: KVCache, layer: int, q_norm2=None):
        """qp: already projected + pre-scaled queries [B,Nq,E]; q_norm2: optional [B,H] query norm maxima (with
        cache.k_norm2, the maxima over THIS rank's keys, they select the static-shift kernel for the local partial)."""
        from .. import parallel
        import torch.distributed as dist
        B, Nq, E = qp.shape
        H = self.num_heads
        # the local partial goes straight into the packed (O | LSE) record this rank contributes to the layer's exchange:
        # a slot of the peer-mapped buffer (fused exchange + merge kernel) or a fresh buffer for the NCCL all-gather
        peer = cache.peer(B, Nq, H, qp.device) if cache.peer is not None else None
        record, o_part, lse = peer.record(layer) if peer is not None else ops.packed_partial(B, Nq, H, qp.device)
        if cache.n_kv > 0:
            ops.cross_attn(qp, cache.k, cache.vt, layer, o_dtype=torch.float32, out=o_part, lse_out=lse,
                           q_norm2=q_norm2, k_norm2=cache.k_norm2 if q_norm2 is not None else None)
        else:  # this rank holds no tokens: neutral element of the merge
            o_part.zero_()
            lse.fill_(float("-inf"))
        if peer is not None:
            return peer.merge(layer, _compute_dtype(self.precision))
        allrec = parallel.gather_packed(record, cache.group)
        ctx = ops.lse_merge_packed(allrec, dist.get_world_size(cache.group), B, Nq, H, o_dtype=_compute_dtype(self.precision))
        return ctx
