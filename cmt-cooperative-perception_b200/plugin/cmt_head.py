"""CmtHead / CmtImageHead / CmtLidarHead and SeparateTaskHead with the reference's class names,
constructor arguments, forward signatures and state-dict keys
(projects/mmdet3d_plugin/models/dense_heads/cmt_head.py:97-1085), inference path only.

What runs where (default bf16 inference path):
  * camera-ray PE lift, re-projection of the reference points, sine/cosine embedding, masked view
    sum, token gather, every PE-MLP / projection GEMM, the cross-attention AND the decoder's small ops
    (900x900 self-attention, LayerNorms, FFN: plugin/fused_decoder.py) run in libcmtcoop_b200 -- bf16
    operands on the tensor cores, fp32 accumulation / residuals / statistics.  The reference computes the
    decoder in fp32 (nn.MultiheadAttention, nn.Linear); the difference is inside the 1e-2 rel-L2 budget of
    the bf16 mode and `set_precision('fp32')` selects the fp32 CUDA-core kernels (<= 1e-4).
    `set_precision('fp16')` runs the same tensor-core kernels with fp16 operands (3 more mantissa bits than bf16).
  * the task heads always compute in fp32 (their logits feed the top-k).
Losses, denoising queries and target assignment are training-only and not part of this package.
"""
from __future__ import annotations

import copy

import numpy as np
import torch
import torch.nn as nn

from .. import ops
from .bbox_coder import build_bbox_coder
from .registry import HEADS, TRANSFORMER, ConfigDict


def inverse_sigmoid(x, eps=1e-5):
    """mmdet.models.utils.transformer.inverse_sigmoid (mmdet 2.28.2)."""
    x = x.clamp(min=0, max=1)
    return torch.log(x.clamp(min=eps) / (1 - x).clamp(min=eps))


def multi_apply(func, *args, **kwargs):
    """mmdet.core.multi_apply."""
    from functools import partial
    pfunc = partial(func, **kwargs) if kwargs else func
    return tuple(map(list, zip(*map(pfunc, *args))))


def pos2embed(pos, num_pos_feats=128, temperature=10000, out_dtype=torch.float32):
    """cmt_head.py:40-50 on the GPU (cmt_pos2embed); `temperature` is accepted and unused, as there."""
    return ops.pos2embed(pos.float().contiguous(), num_pos_feats, out_dtype=out_dtype)


class GroupLayerNorm1d(nn.Module):
    """cmt_head.py:53-94 (forward only)."""

    def __init__(self, channels, groups=1, eps=1e-6):
        super().__init__()
        self.weight = nn.Parameter(torch.ones(channels))
        self.bias = nn.Parameter(torch.zeros(channels))
        self.groups = groups
        self.eps = eps

    def forward(self, x):
        N, C, L = x.shape
        xg = x.view(N, self.groups, C // self.groups, L)
        mu = xg.mean(2, keepdim=True)
        var = (xg - mu).pow(2).mean(2, keepdim=True)
        y = (xg - mu) / (var + self.eps).sqrt()
        return self.weight.view(1, C, 1) * y.view(N, C, L) + self.bias.view(1, C, 1)


@HEADS.register_module()
class SeparateTaskHead(nn.Module):
    """cmt_head.py:97-203: per output name, grouped Conv1d -> group LN -> ReLU -> grouped Conv1d over the
    query axis, one group per decoder layer."""

    def __init__(self, in_channels, heads, groups=1, head_conv=64, final_kernel=1, init_bias=-2.19,
                 init_cfg=None, **kwargs):
        assert init_cfg is None
        super().__init__()
        self.heads = heads
        self.groups = groups
        self.init_bias = init_bias
        self._kernel_size = final_kernel
        self._two_stage = all(v[1] == 2 for v in heads.values())
        for head in self.heads:
            classes, num_conv = self.heads[head]
            layers, c_in = [], in_channels
            for _ in range(num_conv - 1):
                layers += [nn.Conv1d(c_in * groups, head_conv * groups, kernel_size=final_kernel, stride=1,
                                     padding=final_kernel // 2, groups=groups, bias=False),
                           GroupLayerNorm1d(head_conv * groups, groups=groups), nn.ReLU(inplace=True)]
                c_in = head_conv
            layers.append(nn.Conv1d(head_conv * groups, classes * groups, kernel_size=final_kernel, stride=1,
                                    padding=final_kernel // 2, groups=groups, bias=True))
            setattr(self, head, nn.Sequential(*layers))

    def init_weights(self):
        for m in self.modules():
            if isinstance(m, nn.Conv1d):
                nn.init.kaiming_normal_(m.weight, mode="fan_out", nonlinearity="relu")
                if m.bias is not None:
                    nn.init.constant_(m.bias, 0.0)
        for head in self.heads:
            if head == "cls_logits":
                getattr(self, head)[-1].bias.data.fill_(self.init_bias)

    # -- fused inference path: tensor-core first convolution (three-term bf16 split) + one tail kernel -----------------
    _PAIRS = ((0, 0), (0, 1), (1, 0), (0, 2), (1, 1), (2, 0))   # (term of x, term of w): every product down to 2^-24

    def fusable(self, x):
        """True when libcmtcoop_b200 computes this head: CUDA, eval, (conv, GroupLN, ReLU, conv) stacks with
        head_conv = 64, kernel size 1 or 3, 256 input channels, at most 8 heads of at most 32 outputs."""
        if self.training or not x.is_cuda or not self._two_stage or self._kernel_size not in (1, 3) or len(self.heads) > 8:
            return False
        seqs = [getattr(self, n) for n in self.heads]
        return all(s[0].weight.shape[0] == 64 * self.groups and s[0].weight.shape[1] == 256 and
                   s[3].weight.shape[0] // self.groups <= 32 for s in seqs) and x.shape[-1] == 256

    def _fused_weights(self):
        """Stacks the heads: first conv as a segmented-GEMM B operand [L, NH*64, KS*6*C] bf16 (weights split into three
        bf16 terms, six products per tap), LN affine [L,NH,64], second conv [L,NH,cmax,KS,64] (zero padded), bias."""
        names = list(self.heads)
        seqs = [getattr(self, n) for n in names]
        key = tuple((s[0].weight._version, s[0].weight.data_ptr(), s[1].weight._version, s[1].bias._version,
                     s[3].weight._version, s[3].bias._version) for s in seqs)
        hit = self.__dict__.get("_fused_cache")
        if hit is None or hit[0] != key:
            L, KS = self.groups, self._kernel_size
            hc = seqs[0][0].weight.shape[0] // L
            C = seqs[0][0].weight.shape[1]
            NH = len(seqs)
            couts = [s[3].weight.shape[0] // L for s in seqs]
            cmax = max(couts)
            w1 = torch.stack([s[0].weight.detach().float().view(L, hc, C, KS) for s in seqs], 1).reshape(L, NH * hc, C, KS)
            t1 = w1.bfloat16()
            r1 = w1 - t1.float()
            t2 = r1.bfloat16()
            t3 = (r1 - t2.float()).bfloat16()
            terms = (t1, t2, t3)
            segs, acol, shift = [], [], []
            for t in range(KS):
                for xi, wj in self._PAIRS:
                    segs.append(terms[wj][..., t])
                    acol.append(xi * C)
                    shift.append(t - KS // 2)
            bmat = torch.cat(segs, dim=-1).contiguous()                      # [L, NH*hc, KS*6*C]
            g = torch.stack([s[1].weight.detach().float().view(L, hc) for s in seqs], 1).contiguous()
            b = torch.stack([s[1].bias.detach().float().view(L, hc) for s in seqs], 1).contiguous()
            w2 = w1.new_zeros(L, NH, cmax, KS, hc)
            b2 = w1.new_zeros(L, NH, cmax)
            for i, (s, co) in enumerate(zip(seqs, couts)):
                w2[:, i, :co] = s[3].weight.detach().float().view(L, co, hc, KS).permute(0, 1, 3, 2)
                b2[:, i, :co] = s[3].bias.detach().float().view(L, co)
            hit = (key, dict(names=names, couts=couts, hc=hc, C=C, KS=KS, bmat=bmat, acol=acol, shift=shift, g=g, b=b,
                             w2=w2.contiguous(), b2=b2.contiguous(), eps=seqs[0][1].eps, cmax=cmax))
            self.__dict__["_fused_cache"] = hit
        return hit[1]

    def _decode_tables(self, pc_range, device):
        """Per (head, output) reference component / scale / offset of the reference-point decode (cmt_head.py:501-513)."""
        w = self._fused_weights()
        key = (tuple(float(v) for v in pc_range), str(device))
        hit = self.__dict__.get("_dec_cache")
        if hit is None or hit[0] != key:
            NH, cmax = len(w["names"]), w["cmax"]
            comp = torch.full((NH, cmax), -1, dtype=torch.int32)
            scale = torch.ones(NH, cmax)
            off = torch.zeros(NH, cmax)
            pc = [float(v) for v in pc_range]
            for i, n in enumerate(w["names"]):
                if n == "center":
                    for o in range(2):
                        comp[i, o], scale[i, o], off[i, o] = o, pc[3 + o] - pc[o], pc[o]
                elif n == "height":
                    comp[i, 0], scale[i, 0], off[i, 0] = 2, pc[5] - pc[2], pc[2]
            hit = (key, (comp.to(device), scale.to(device), off.to(device)))
            self.__dict__["_dec_cache"] = hit
        return hit[1]

    def forward_split(self, xs, B, Q, ref_logit=None, pc_range=None):
        """xs: ops.split3 of the decoder outputs, [L*B, Q+2, 768] bf16.  Returns {name: [L,B,Q,c_out]} fp32 -- with
        ref_logit [B*Q,3] the center / height outputs are already decoded to metric coordinates."""
        w = self._fused_weights()
        L, C, KS, hc = self.groups, w["C"], w["KS"], w["hc"]
        NH = len(w["names"])
        h = torch.empty((L, B * Q, NH, hc), dtype=torch.float32, device=xs.device)
        ops.gemm_segmented(xs, w["bmat"], None, h, Q, NH * hc, C, w["acol"], w["shift"], a_row_off=1, a_rows=Q + 2,
                           a_cols=3 * C, lda=3 * C, ldb=KS * 6 * C, ldc=NH * hc, batch=L * B, strideA=(Q + 2) * 3 * C,
                           strideB=NH * hc * KS * 6 * C, b_batch_div=B, strideC=Q * NH * hc, tag="task_head_conv1")
        dec = (None, None, None)
        if ref_logit is not None:
            dec = self._decode_tables(pc_range, xs.device)
        outs = ops.task_head_tail(h, w["g"], w["b"], w["w2"], w["b2"], w["eps"], ksize=KS, Nq=Q, ref_logit=ref_logit,
                                  dec_comp=dec[0], dec_scale=dec[1], dec_offset=dec[2], head_couts=w["couts"])
        return {n: o.view(L, B, Q, co) for n, o, co in zip(w["names"], outs, w["couts"])}

    def forward(self, x):
        N, B, Q, C = x.shape
        if self.fusable(x):
            return self.forward_split(ops.split3(x.contiguous().float()), B, Q)   # note: applies nan_to_num like the head does
        x = x.permute(1, 0, 3, 2).reshape(B, N * C, Q)  # "n b q c -> b (n c) q"
        ret = {}
        for head in self.heads:
            y = getattr(self, head)(x)
            ret[head] = y.view(B, N, -1, Q).permute(1, 0, 3, 2)  # "b (n c) q -> n b q c"
        return ret


class _ConvModule(nn.Module):
    """mmcv ConvModule(conv_cfg=Conv2d, norm_cfg=BN2d): conv (no bias) -> bn -> relu; keys conv.*, bn.*."""

    def __init__(self, cin, cout, k, padding):
        super().__init__()
        self.conv = nn.Conv2d(cin, cout, k, padding=padding, bias=False)
        self.bn = nn.BatchNorm2d(cout)
        self.activate = nn.ReLU(inplace=True)

    def forward(self, x):
        return self.activate(self.bn(self.conv(x)))


_compute_dtype = ops.compute_dtype


class _torch_math:
    """fp32 verification mode must be fp32 end to end: the torch ops that stay on the path (cuDNN
    shared_conv / Conv1d task heads, cuBLAS self-attention and FFN) default to TF32 on this GPU."""

    def __init__(self, precision):
        self.strict = precision == "fp32"

    def __enter__(self):
        if self.strict:
            self.prev = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
            torch.backends.cudnn.allow_tf32 = False
            torch.backends.cuda.matmul.allow_tf32 = False

    def __exit__(self, *exc):
        if self.strict:
            torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = self.prev
        return False


class _CmtHeadBase(nn.Module):
    """Everything the six head classes share: construction (cmt_head.py:208-318), position encodings
    (:417-473), per-node decoder pass (:481-499 == cmt_head_coop.py:341-360) and the output tail (:501-547)."""

    _has_bev = True
    _has_img = True

    def __init__(self, in_channels, num_query=900, hidden_dim=128, depth_num=64, norm_bbox=True,
                 downsample_scale=8, scalar=10, noise_scale=1.0, noise_trans=0.0, dn_weight=1.0, split=0.75,
                 train_cfg=None, test_cfg=None,
                 common_heads=dict(center=(2, 2), height=(1, 2), dim=(3, 2), rot=(2, 2), vel=(2, 2)),
                 tasks=None, transformer=None, bbox_coder=None, loss_cls=None, loss_bbox=None, loss_heatmap=None,
                 separate_head=dict(type="SeparateMlpHead", init_bias=-2.19, final_kernel=3), init_cfg=None,
                 **kwargs):
        assert init_cfg is None
        super().__init__()
        tasks = tasks or [dict(num_class=10, class_names=["car"] * 10)]
        self.num_classes = [len(t["class_names"]) for t in tasks]
        self.class_names = [t["class_names"] for t in tasks]
        self.hidden_dim = hidden_dim
        self.train_cfg = train_cfg
        self.test_cfg = test_cfg
        self.num_query = num_query
        self.in_channels = in_channels
        self.depth_num = depth_num
        self.norm_bbox = norm_bbox
        self.downsample_scale = downsample_scale
        self.scalar = scalar
        self.bbox_noise_scale = noise_scale
        self.bbox_noise_trans = noise_trans
        self.dn_weight = dn_weight
        self.split = split
        self.bbox_coder = build_bbox_coder(bbox_coder)
        self.pc_range = self.bbox_coder.pc_range
        self.fp16_enabled = False
        self.precision = "bf16"
        # bench.py times "CmtTransformer+PE" from the post-shared_conv BEV map (SURVEY.md 8(d)); set False then
        self.apply_shared_conv = True
        # bf16 / fp16 modes: shared_conv runs as a tcgen05 implicit GEMM whose epilogue writes the BEV token rows directly
        # (cmt_shared_conv_tokens); False keeps torch's Conv2d + BatchNorm2d + ReLU (always used in fp32 mode)
        self.fuse_shared_conv = True

        self.shared_conv = _ConvModule(in_channels, hidden_dim, 3, 1) if self._has_bev else None
        transformer = ConfigDict(copy.deepcopy(transformer))
        self.transformer = TRANSFORMER.build(transformer)
        self.reference_points = nn.Embedding(num_query, 3)
        self.bev_embedding = nn.Sequential(nn.Linear(hidden_dim * 2, hidden_dim), nn.ReLU(inplace=True),
                                           nn.Linear(hidden_dim, hidden_dim))
        self.rv_embedding = nn.Sequential(nn.Linear(depth_num * 3, hidden_dim * 4), nn.ReLU(inplace=True),
                                          nn.Linear(hidden_dim * 4, hidden_dim)) if self._has_img else None
        self.task_heads = nn.ModuleList()
        for num_cls in self.num_classes:
            heads = copy.deepcopy(dict(common_heads))
            heads.update(dict(cls_logits=(num_cls, 2)))
            sh = dict(copy.deepcopy(separate_head))
            sh.update(in_channels=hidden_dim, heads=heads, num_cls=num_cls, groups=transformer.decoder.num_layers)
            self.task_heads.append(HEADS.build(sh))
        self._cache = {}

    # ------------------------------------------------------------------------------------
    def init_weights(self):
        self.transformer.init_weights()
        for th in self.task_heads:
            th.init_weights()
        nn.init.uniform_(self.reference_points.weight.data, 0, 1)

    def set_precision(self, precision):
        """'bf16' (tcgen05 kernels, default), 'fp16' (tcgen05 kernels with fp16 operands: 3 more mantissa bits, the
        attention core at the reference's flash-attn precision) or 'fp32' (CUDA-core verification mode).  The task heads
        are fp32-grade in every mode."""
        _compute_dtype(precision)   # rejects an unknown precision
        self.precision = precision
        self.transformer.set_precision(precision)
        self._cache.clear()
        return self

    @property
    def coords_bev(self):
        """cmt_head.py:324-337."""
        cfg = self.train_cfg if self.train_cfg else self.test_cfg
        x_size = cfg["grid_size"][1] // self.downsample_scale
        y_size = cfg["grid_size"][0] // self.downsample_scale
        by, bx = torch.meshgrid(torch.linspace(0, x_size - 1, x_size), torch.linspace(0, y_size - 1, y_size),
                                indexing="ij")
        bx = (bx + 0.5) / x_size
        by = (by + 0.5) / y_size
        return torch.cat([bx[None], by[None]], dim=0).view(2, -1).transpose(1, 0)

    def prepare_for_dn(self, batch_size, reference_points, img_metas):
        if self.training:
            raise NotImplementedError("denoising queries are training-only (cmt_head.py:339-408)")
        # eval branch (cmt_head.py:410-413): the learned reference points repeated over the batch -- a function of the
        # parameter only, so the repeated tensor (and everything derived from it alone) is cached per parameter version
        return self._ref_derived(batch_size, reference_points)["ref"], None, None

    def _ref_derived(self, batch_size, reference_points):
        """Tensors that depend on the reference points (and weights) only, cached per parameter version and batch size:
        ref [B,Nq,3]; ref_clamped = inverse_sigmoid(ref).sigmoid() (cmt_head.py:470); ref_logit = inverse_sigmoid(ref)
        [B*Nq,3] (:501); bev_query = bev_embedding(pos2embed(ref_clamped)) [Nq,C] (:435-437, identical for every frame)."""
        key = (reference_points.data_ptr(), reference_points._version, batch_size, str(reference_points.device), self.precision,
               id(self._mlp_weights("bev_embedding")[0]) if reference_points.is_cuda else None)
        hit = self._cache.get("ref")
        if hit is None or hit[0] != key:
            ref = reference_points.detach().unsqueeze(0).repeat(batch_size, 1, 1)
            d = dict(ref=ref, ref_logit=inverse_sigmoid(ref.clone()).reshape(-1, 3).contiguous(),
                     ref_clamped=inverse_sigmoid(ref.clone()).sigmoid())
            if ref.is_cuda:
                d["bev_query"] = self._bev_query_embed(d["ref_clamped"][:1], None)[0].contiguous()
            hit = (key, d)
            self._cache["ref"] = hit
        return hit[1]

    # -- MLPs on the tcgen05 GEMM ---------------------------------------------------------
    def _mlp_weights(self, name):
        seq = getattr(self, name)
        dt = _compute_dtype(self.precision)
        key = (name, dt, seq[0].weight._version, seq[0].weight.data_ptr(), seq[2].weight._version,
               seq[2].weight.data_ptr(), seq[0].bias._version, seq[2].bias._version)
        hit = self._cache.get("w_" + name)
        if hit is None or hit[0] != key:
            hit = (key, (seq[0].weight.detach().to(dt).contiguous(), seq[0].bias.detach().float().contiguous(),
                         seq[2].weight.detach().to(dt).contiguous(), seq[2].bias.detach().float().contiguous()))
            self._cache["w_" + name] = hit
        return hit[1]

    def _mlp(self, name, x, tag=None):
        """Linear -> ReLU -> Linear (cmt_head.py:292-301); hidden activation in the compute dtype, fp32 out."""
        w0, b0, w1, b1 = self._mlp_weights(name)
        dt = _compute_dtype(self.precision)
        h = ops.linear(x.to(dt), w0, b0, relu=True, out_dtype=dt, tag=None if tag is None else tag + ".0")
        return ops.linear(h, w1, b1, out_dtype=torch.float32, tag=None if tag is None else tag + ".2")

    # -- shared_conv (cmt_head.py:280-287, applied :481) -------------------------------------
    def _shared_conv_folded(self):
        """conv weight with the eval-mode BatchNorm scale folded in, tap-major [Cout, 9*Cin] in the compute dtype (bf16 or
        fp16), and the remaining per-channel bias: BN(conv(x)) = conv(x; w * s) + (beta - mean * s), s = gamma / sqrt(var + eps)."""
        conv, bn = self.shared_conv.conv, self.shared_conv.bn
        dt = _compute_dtype(self.precision)
        key = ("conv", dt, conv.weight._version, conv.weight.data_ptr(), bn.weight._version, bn.bias._version,
               bn.running_mean._version, bn.running_var._version, bn.running_mean.data_ptr())
        hit = self._cache.get("shared_conv")
        if hit is None or hit[0] != key:
            s = bn.weight.detach().float() / torch.sqrt(bn.running_var.detach().float() + bn.eps)
            w = conv.weight.detach().float() * s[:, None, None, None]                  # [Cout, Cin, 3, 3]
            w = w.permute(0, 2, 3, 1).reshape(w.shape[0], -1).to(dt).contiguous()   # [Cout, (ky, kx, c)]
            b = (bn.bias.detach().float() - bn.running_mean.detach().float() * s).contiguous()
            hit = (key, (w, b))
            self._cache["shared_conv"] = hit
        return hit[1]

    def _apply_shared_conv_to(self, x):
        """(BEV map, folded shared_conv) for build_kv_cache: (x, None) for the input itself (bench scope), (x, (w, bias))
        for the fused implicit-GEMM path (bf16 and fp16 modes), or (torch's conv + BN + ReLU of x, None) in fp32."""
        if not self.apply_shared_conv:
            return x, None
        conv = self.shared_conv.conv
        if (self.precision in ("bf16", "fp16") and self.fuse_shared_conv and conv.kernel_size == (3, 3) and conv.in_channels % 64 == 0
                and conv.out_channels % 32 == 0):
            return x, self._shared_conv_folded()
        return self.shared_conv(x.float()), None

    # -- position encodings -----------------------------------------------------------------
    def _matrices(self, img_metas, device):
        """Host float64 inverse -> fp32 -> device, as cmt_head.py:428-429,441-444. [B,V,4,4] each.
        A calibration already built on the device (plugin/detector_glue.device_calibration, stored in
        img_metas[0]['calibration']) is used as it is."""
        cal = img_metas[0].get("calibration")
        if cal is not None:
            l2i_d, i2l_d = cal
            if l2i_d.device != torch.device(device) or l2i_d.shape[0] != len(img_metas):
                raise ValueError("img_metas[0]['calibration'] must hold [B,V,4,4] tensors on the head's device")
            return l2i_d, i2l_d
        l2i = np.stack([np.asarray(m["lidar2img"], dtype=np.float64) for m in img_metas])
        # calibration rarely changes between frames: the inverse + upload (a host sync inside the path, SURVEY 8(f)
        # rank 3) is done once per distinct set of matrices, keyed by their bytes
        key = (l2i.shape, l2i.tobytes(), str(device))
        table = self._cache.setdefault("mats", {})   # a few entries: the cooperative heads alternate between two nodes
        hit = table.get(key)
        if hit is None:
            i2l = np.linalg.inv(l2i)
            both = torch.from_numpy(np.stack([l2i, i2l]).astype(np.float32)).pin_memory().to(device, non_blocking=True)
            hit = (both[0].contiguous(), both[1].contiguous())
            if len(table) >= 8:
                table.pop(next(iter(table)))
            table[key] = hit
        return hit

    def _rv_pe(self, img_feats, img_metas, mats=None, n_bev=0):
        """cmt_head.py:417-433 -> ([B*V,H,W,C] fp32, None).  Under the KV-token split a rank needs the encodings of its own
        image tokens only: the MLP (22 GF per frame) then runs on that row range [a, b) of every frame's V*H*W image
        tokens, and ([B, b-a, C], (a, b)) is returned (build_kv_cache's rv_rows), or (None, (0, 0)) when the rank's share
        holds no image token."""
        BN, C, H, W = img_feats.shape
        pad_h, pad_w, _ = img_metas[0]["pad_shape"][0]
        if mats is None:
            mats = self._matrices(img_metas, img_feats.device)
        dt = _compute_dtype(self.precision)
        coords = ops.ray_pe(mats[1].reshape(-1, 4, 4), H, W, self.depth_num, pad_h, pad_w, self.pc_range, out_dtype=dt)
        B = len(img_metas)
        n_img = (BN // B) * H * W
        lo, hi = self.transformer.kv_token_range(n_bev + n_img)
        if (lo, hi) != (0, n_bev + n_img):
            a, b = max(lo - n_bev, 0), max(hi - n_bev, 0)
            if b <= a:
                return None, (0, 0)
            rows = coords.view(B, n_img, -1)[:, a:b].contiguous()
            return self._mlp("rv_embedding", rows, tag="rv_pe_mlp"), (a, b)
        return self._mlp("rv_embedding", coords, tag="rv_pe_mlp"), None

    def _bev_pos_embed(self, device):
        """bev_embedding(pos2embed(coords_bev)) (cmt_head.py:489): input independent -> cached per weights."""
        w = self._mlp_weights("bev_embedding")
        key = (id(w[0]), str(device), self.precision)
        hit = self._cache.get("bev_pos")
        if hit is None or hit[0] != key:
            dt = _compute_dtype(self.precision)
            emb = pos2embed(self.coords_bev.to(device), num_pos_feats=self.hidden_dim, out_dtype=dt)
            hit = (key, self._mlp("bev_embedding", emb))
            self._cache["bev_pos"] = hit
        return hit[1]

    def _bev_query_embed(self, ref_points, img_metas):
        dt = _compute_dtype(self.precision)
        return self._mlp("bev_embedding", pos2embed(ref_points, num_pos_feats=self.hidden_dim, out_dtype=dt))

    def _rv_query_embed(self, ref_points, img_metas, mats=None, base=None, view_valid=None):
        """cmt_head.py:439-467 (+ `base`, the BEV query embedding, added after the view sum: :492).  view_valid: the
        camera rows [V, B] of the sensor mask; an absent camera is left out of the view sum."""
        pad_h, pad_w, _ = img_metas[0]["pad_shape"][0]
        if mats is None:
            mats = self._matrices(img_metas, ref_points.device)
        dt = _compute_dtype(self.precision)
        feats, mask = ops.ray_query_pe(ref_points.contiguous(), mats[0], mats[1], self.depth_num, pad_h, pad_w,
                                       self.pc_range, out_dtype=dt)
        emb = self._mlp("rv_embedding", feats)
        return ops.masked_view_sum(emb, mask, base=base, view_valid=view_valid)

    def query_embed(self, ref_points, img_metas, mats=None, view_valid=None):
        """cmt_head.py:469-473 -> (bev_query_embeds, rv_query_embeds)."""
        ref_points = inverse_sigmoid(ref_points.clone()).sigmoid()
        bev = self._bev_query_embed(ref_points, img_metas)
        rv = self._rv_query_embed(ref_points, img_metas, mats, view_valid=view_valid) if self._has_img else None
        return bev, rv

    def _query_embeds(self, reference_points, img_metas, mats, view_valid=None):
        """bev + rv query embedding [B,Nq,C] (cmt_head.py:491-492) with the weight-only parts taken from the cache.
        view_valid: the camera rows of the sensor mask (_rv_query_embed)."""
        B = reference_points.shape[0]
        d = None
        hit = self._cache.get("ref")
        if hit is not None and hit[1]["ref"] is reference_points:
            d = hit[1]
        if d is None or "bev_query" not in d:   # reference points not from prepare_for_dn: the general path
            bev, rv = self.query_embed(reference_points, img_metas, mats, view_valid)
            return bev if rv is None else bev + rv
        if not self._has_img:
            return d["bev_query"].unsqueeze(0).expand(B, -1, -1)
        return self._rv_query_embed(d["ref_clamped"], img_metas, mats, base=d["bev_query"], view_valid=view_valid)

    # -- one node: shared_conv -> PEs -> transformer -> nan_to_num ---------------------------
    def get_outs_dec(self, x, x_img, img_metas, reference_points, attn_mask):
        """cmt_head_coop.py:341-360 (== cmt_head.py:481-499): stacked decoder outputs of one node, nan_to_num'ed."""
        with _torch_math(self.precision):
            query_embeds, cache = self._node_cache(x, x_img, img_metas, reference_points)
            outs_dec = self.transformer.decode([cache], query_embeds, attn_mask)
        return torch.nan_to_num(outs_dec)

    def _check_sensor_valid(self, sensor_valid, x, x_img, img_metas):
        """Host-side checks of the single-node heads' per-frame sensor mask (torch.bool [S, B] on the features' device,
        one row per sensor in token order: the LiDAR first when the head has BEV tokens, then the cameras in the order of
        the img_feats views).  Returns it contiguous; the values are never read on the host."""
        B = len(img_metas)
        S = (1 if self._has_bev else 0) + (x_img.shape[0] // B if self._has_img else 0)
        dev = (x if x is not None else x_img).device
        sensor_valid = ops.check_node_valid(sensor_valid, B, dev, n_nodes=S, name="sensor_valid")
        if self.transformer.kv_split_group is not None:
            raise NotImplementedError("sensor_valid together with the multi-GPU KV-token split")
        return sensor_valid

    def _node_cache(self, x, x_img, img_metas, reference_points, sensor_valid=None):
        """Everything of one node up to the decoder: (query_embeds [B,Nq,C], KVCache) -- query embedding, position
        encodings, token gather / shared_conv, all-layer K / V^T projection.  sensor_valid: the checked [S, B] sensor mask
        (_check_sensor_valid) or None; its camera rows leave absent views out of the query embedding."""
        dev = (x if x is not None else x_img).device
        if dev.type != "cuda":
            raise RuntimeError("CmtHead needs CUDA tensors: libcmtcoop_b200 has no CPU fallback")
        B = len(img_metas)
        mats = self._matrices(img_metas, dev) if self._has_img else None
        view_valid = None
        if sensor_valid is not None and self._has_img:
            view_valid = sensor_valid[1:] if self._has_bev else sensor_valid
        query_embeds = self._query_embeds(reference_points, img_metas, mats, view_valid)
        x_bev, conv = self._apply_shared_conv_to(x) if self._has_bev else (None, None)
        n_bev = x.shape[2] * x.shape[3] if self._has_bev else 0
        rv_pos, rv_rows = self._rv_pe(x_img, img_metas, mats, n_bev=n_bev) if self._has_img else (None, None)
        bev_pos = self._bev_pos_embed(dev) if self._has_bev else None
        V = (x_img.shape[0] // B) if self._has_img else 0
        cache, _ = self.transformer.build_kv_cache(None if x_bev is None else x_bev.contiguous(),
                                                   None if x_img is None else x_img.contiguous(), bev_pos, rv_pos, B, V,
                                                   conv=conv, rv_rows=rv_rows, sensor_valid=sensor_valid)
        return query_embeds, cache

    # -- task heads + reference-point decode (cmt_head.py:501-547, eval branch) ---------------
    def _finish(self, outs_dec, reference_points, outs_dec_other=None, stacked_nodes=False, node_valid=None):
        """outs_dec: raw stacked decoder outputs [L,B,Nq,C] (nan_to_num not yet applied); outs_dec_other: the second node's
        stack for the cooperative heads -- merged with the element-wise max (cmt_head_coop.py:383-389); stacked_nodes:
        outs_dec is [L,2B,Nq,C] with the first node's frames then the second node's in every layer; node_valid: the
        checked [2, B] device mask of the two nodes, applied per frame by the merge (ops.split3)."""
        if stacked_nodes and not all(t.fusable(outs_dec) for t in self.task_heads):
            B2 = outs_dec.shape[1] // 2
            outs_dec, outs_dec_other, stacked_nodes = outs_dec[:, :B2], outs_dec[:, B2:], False
        if all(t.fusable(outs_dec) for t in self.task_heads):
            # libcmtcoop_b200: nan_to_num (+ V2I max) + three-term split -> tensor-core first conv -> fused tail with the
            # reference-point decode; fp32-grade arithmetic (the logits feed the top-k)
            L, B, Q, C = outs_dec.shape
            if stacked_nodes:
                B //= 2
                xs = ops.split3(outs_dec.contiguous(), stacked_nodes=True, node_valid=node_valid)
            else:
                xs = ops.split3(outs_dec.contiguous(), None if outs_dec_other is None else outs_dec_other.contiguous(),
                                node_valid=node_valid)
            hit = self._cache.get("ref")
            if hit is not None and hit[1]["ref"] is reference_points:
                ref_logit = hit[1]["ref_logit"]
            else:
                ref_logit = inverse_sigmoid(reference_points.clone()).reshape(-1, 3).contiguous()
            return [t.forward_split(xs, B, Q, ref_logit, self.pc_range) for t in self.task_heads]
        if node_valid is not None:
            _, outs_dec = ops.split3(outs_dec.contiguous(), outs_dec_other.contiguous(), want_merged=True,
                                     node_valid=node_valid)
        else:
            outs_dec = torch.nan_to_num(outs_dec)
            if outs_dec_other is not None:
                outs_dec = ops.coop_max(outs_dec.contiguous(), torch.nan_to_num(outs_dec_other).contiguous())
        # torch path (non-standard head shapes): strict fp32 (no TF32), these outputs feed the top-k
        with _torch_math("fp32"):
            return self._finish_impl(outs_dec, reference_points)

    def _finish_impl(self, outs_dec, reference_points):
        reference = inverse_sigmoid(reference_points.clone())
        pc = self.pc_range
        ret_dicts = []
        for task in self.task_heads:
            outs = task(outs_dec)
            center = (outs["center"] + reference[None, :, :, :2]).sigmoid()
            height = (outs["height"] + reference[None, :, :, 2:3]).sigmoid()
            _center, _height = center.new_zeros(center.shape), height.new_zeros(height.shape)
            _center[..., 0:1] = center[..., 0:1] * (pc[3] - pc[0]) + pc[0]
            _center[..., 1:2] = center[..., 1:2] * (pc[4] - pc[1]) + pc[1]
            _height[..., 0:1] = height[..., 0:1] * (pc[5] - pc[2]) + pc[2]
            outs["center"] = _center
            outs["height"] = _height
            ret_dicts.append(outs)
        return ret_dicts

    def get_bboxes(self, preds_dicts, img_metas, img=None, rescale=False):
        """cmt_head.py:905-919."""
        preds_dicts = self.bbox_coder.decode(preds_dicts)
        ret_list = []
        for i in range(len(preds_dicts)):
            preds = preds_dicts[i]
            bboxes = preds["bboxes"]
            bboxes[:, 2] = bboxes[:, 2] - bboxes[:, 5] * 0.5
            box_type = img_metas[i].get("box_type_3d")
            if box_type is not None:
                bboxes = box_type(bboxes, bboxes.size(-1))
            ret_list.append([bboxes, preds["scores"], preds["labels"]])
        return ret_list

    def get_bboxes_batched(self, preds_dicts, img_metas, node_valid=None):
        """Fixed-shape counterpart of `get_bboxes` for CUDA tensors: every frame decoded in one launch with the z shift
        applied, no host synchronisation (can be captured in a CUDA graph).  Returns the device-tensor dict
        {boxes [B,K,9], scores [B,K], labels [B,K], count [B], topk_index [B,K]} of `bbox_coder.decode_batched`;
        detector_glue.batched_to_results turns it into per-frame result dicts.  node_valid: the cooperative heads'
        [2, B] node mask, or the single-node heads' [S, B] sensor mask; frames with no node / sensor present get no
        detections."""
        return self.bbox_coder.decode_batched(preds_dicts, bottom_center=True, node_valid=node_valid)


@HEADS.register_module()
class CmtHead(_CmtHeadBase):
    """cmt_head.py:206-919 (multimodal: BEV + camera tokens)."""

    def forward_single(self, x, x_img, img_metas, sensor_valid=None):
        """sensor_valid: optional torch.bool [S, B] on the features' device, one row per sensor in token order -- row 0
        the LiDAR (heads with BEV tokens), then the cameras in the order of the img_feats views and lidar2img -- False
        where that sensor did not deliver the frame.  Each frame is then computed from its present sensors only, as the
        reference would compute it on that frame alone with the absent views removed (x = None without the LiDAR).  An
        absent sensor's features may hold anything (NaN included) and change no output bit; its lidar2img is not read
        into any output but must stay invertible.  A frame with no sensor gets a zero cross-attention context and finite
        outputs (get_bboxes_batched keeps nothing for it).  Absent sensors still cost their GPU time.  None: every
        sensor is present (unchanged path).  CmtImageHead takes one row per camera ([V, B]), CmtLidarHead the LiDAR row
        only ([1, B])."""
        assert self._has_bev or x is None
        assert self._has_img or x_img is None
        if sensor_valid is not None:
            sensor_valid = self._check_sensor_valid(sensor_valid, x, x_img, img_metas)
        reference_points = self.reference_points.weight
        reference_points, attn_mask, mask_dict = self.prepare_for_dn(len(img_metas), reference_points, img_metas)
        with _torch_math(self.precision):
            query_embeds, cache = self._node_cache(x, x_img, img_metas, reference_points, sensor_valid)
            # without the nan_to_num of get_outs_dec: the fused task-head path applies it inside cmt_split3_bf16
            outs_dec = self.transformer.decode([cache], query_embeds, attn_mask)
        return self._finish(outs_dec, reference_points)

    def forward(self, pts_feats, img_feats=None, img_metas=None, sensor_valid=None):
        """sensor_valid: the per-frame sensor mask of forward_single, shared by every feature level."""
        img_metas = [img_metas for _ in range(len(pts_feats))]
        return multi_apply(self.forward_single, pts_feats, img_feats, img_metas, sensor_valid=sensor_valid)


@HEADS.register_module()
class CmtImageHead(CmtHead):
    """cmt_head.py:922-999 (camera only; shared_conv is None)."""
    _has_bev = False


@HEADS.register_module()
class CmtLidarHead(CmtHead):
    """cmt_head.py:1002-1085 (LiDAR only; rv_embedding is None)."""
    _has_img = False
