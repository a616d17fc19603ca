"""CmtHeadCoop / CmtImageHeadCoop / CmtLidarHeadCoop
(projects/mmdet3d_plugin/models/dense_heads/cmt_head_coop.py:72-1017), inference path.

Cooperative fusion in the reference is NOT a cross-node token concatenation: the same decoder
(shared weights, same queries) runs once per node and the two stacks of decoder outputs are merged
with an element-wise max (cmt_head_coop.py:383-389).  The max (with the nan_to_num of :358 folded in)
is the cmt_coop_max kernel.
"""
from __future__ import annotations

import torch

from .. import ops
from .cmt_head import _CmtHeadBase, _torch_math, multi_apply
from .registry import HEADS


def filter_img_metas(img_meta, prefix="", ignore=""):
    """cmt_head_coop.py:41-57: drop keys starting with `ignore`, strip `prefix` from the others."""
    out = {}
    for k, v in img_meta.items():
        if k.startswith(prefix):
            out[k[len(prefix):]] = v
        elif not k.startswith(ignore):
            out[k] = v
    out["node"] = prefix
    return out


def get_infrastructure_image_metas(img_metas):
    return [filter_img_metas(m, prefix="infrastructure_", ignore="vehicle_") for m in img_metas]


def get_vehicle_image_metas(img_metas):
    return [filter_img_metas(m, prefix="vehicle_", ignore="infrastructure_") for m in img_metas]


@HEADS.register_module()
class CmtHeadCoop(_CmtHeadBase):
    """cmt_head_coop.py:72-444 (multimodal, vehicle + infrastructure)."""

    batch_nodes = True   # decode both nodes' frames in one pass (False: two sequential decoder passes like the reference)

    def forward_single(self, x_vehicle, x_infrastructure, x_img_vehicle, x_img_infrastructure, img_metas, node_valid=None):
        """node_valid: optional torch.bool [2, B] on the features' device, row 0 the vehicle and row 1 the infrastructure:
        False where that node did not deliver the frame.  Such a frame's features of that node may hold anything (NaN
        included) and change no output bit: the frame's merged decoder output is the other node's (nan_to_num'ed), or
        zero rows when neither node delivered it.  The absent node's rows still go through the decoder (same GPU time).
        A node missing for the whole batch is passed as None instead, without a mask."""
        has_v = x_vehicle is not None or x_img_vehicle is not None
        has_i = x_infrastructure is not None or x_img_infrastructure is not None
        if node_valid is not None:
            if not (has_v and has_i):
                raise ValueError("node_valid needs the features of both nodes; pass a node missing from the whole batch "
                                 "as None, without a mask")
            dev = (x_vehicle if x_vehicle is not None else x_img_vehicle).device
            node_valid = ops.check_node_valid(node_valid, len(img_metas), dev)
        reference_points = self.reference_points.weight
        reference_points, attn_mask, mask_dict = self.prepare_for_dn(len(img_metas), reference_points, img_metas)
        nodes = []
        if has_v:
            nodes.append((x_vehicle, x_img_vehicle, get_vehicle_image_metas(img_metas)))
        if has_i:
            nodes.append((x_infrastructure, x_img_infrastructure, get_infrastructure_image_metas(img_metas)))
        stacked = None
        with _torch_math(self.precision):
            built = [self._node_cache(x, x_img, metas, reference_points) for x, x_img, metas in nodes]
            if len(built) == 2 and self.batch_nodes:
                # Both nodes in ONE decoder pass: the reference runs the same decoder (shared weights, same reference
                # points) once per node (cmt_head_coop.py:368-389, :946-1017); frames are independent, so stacking the two
                # nodes' frames changes no arithmetic -- every small op of the decoder runs once over 2B frames, the
                # cross-attention is launched per node (their token counts differ), and the V2I max + nan_to_num ride in
                # the task heads' first kernel.
                stacked = self.transformer.decode([c for _, c in built], torch.cat([q for q, _ in built], 0), attn_mask)
            if stacked is None:
                outs = [self.transformer.decode([c], q, attn_mask) for q, c in built]
        if stacked is not None:
            return self._finish(stacked, reference_points, stacked_nodes=True, node_valid=node_valid)
        # max(stack([veh, infra]), 0) (cmt_head_coop.py:383-389) is folded into the task heads' first kernel
        return self._finish(outs[0], reference_points, outs_dec_other=outs[1] if len(outs) == 2 else None,
                            node_valid=node_valid)

    def forward(self, vehicle_pts_feats, infrastructure_pts_feats, vehicle_img_feats=None,
                infrastructure_img_feats=None, img_metas=None, node_valid=None):
        """node_valid: the per-frame node mask of forward_single, shared by every feature level."""
        img_metas = [img_metas for _ in range(len(vehicle_pts_feats))]
        return multi_apply(self.forward_single, vehicle_pts_feats, infrastructure_pts_feats, vehicle_img_feats,
                           infrastructure_img_feats, img_metas, node_valid=node_valid)


@HEADS.register_module()
class CmtImageHeadCoop(CmtHeadCoop):
    """cmt_head_coop.py:812-911 (camera only)."""
    _has_bev = False

    def forward_single(self, x_vehicle, x_infrastructure, x_img_vehicle, x_img_infrastructure, img_metas, node_valid=None):
        assert x_vehicle is None and x_infrastructure is None
        return super().forward_single(None, None, x_img_vehicle, x_img_infrastructure, img_metas, node_valid)


@HEADS.register_module()
class CmtLidarHeadCoop(CmtHeadCoop):
    """cmt_head_coop.py:914-1017 (LiDAR only): both nodes share queries and BEV PE, so a frame is
    simply two decoder passes followed by the pairwise max."""
    _has_img = False

    def forward_single(self, x_vehicle, x_infrastructure, x_img_vehicle, x_img_infrastructure, img_metas, node_valid=None):
        assert x_img_vehicle is None and x_img_infrastructure is None
        return super().forward_single(x_vehicle, x_infrastructure, None, None, img_metas, node_valid)
