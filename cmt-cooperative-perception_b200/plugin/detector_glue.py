"""Detector-side glue of the hot path: the calls `CmtDetector` / `CmtCoopDetector` make into the head
(projects/mmdet3d_plugin/models/detectors/cmt.py:221-231, cmt_coop.py:549-569) and the calibration handling around
them, so that a detector (or a serving loop without the OpenMMLab detector classes) drives the B200 head exactly like
the reference drives its own.

* `simple_test_pts` / `coop_simple_test_pts`: head forward -> get_bboxes -> bbox3d2result, same argument meaning and
  result dicts as the reference methods (`self` replaced by the head).
* `batched_to_results`: the fixed-shape batched decode (`get_bboxes_batched`) -> the per-frame result dicts of
  `simple_test_pts`, with one device->host copy for the whole batch.
* `device_calibration`: lidar2img -> (lidar2img, img2lidar) fp32 device tensors built ON the device in float64 --
  including the vehicle -> infrastructure fold `lidar2img @ inv(vehicle2infrastructure)` that the reference does in its
  CPU data pipeline (datasets/pipelines/transforms_3d_coop.py:213-222) and the float64 inverse the head does with numpy
  (cmt_head.py:428-429, 441-444).  The head picks the tensors up from `img_metas[0]['calibration']`
  (`'vehicle_calibration'` / `'infrastructure_calibration'` for the cooperative heads), so the per-call host inverse,
  the hashing of the matrices and the upload disappear from the path.
"""
from __future__ import annotations

import numpy as np
import torch


def bbox3d2result(bboxes, scores, labels, attrs=None):
    """mmdet3d.core.bbox3d2result (mmdet3d 1.0.0rc6, third-party, restated): detections of one frame as CPU tensors."""
    result = dict(boxes_3d=bboxes.to("cpu"), scores_3d=scores.cpu(), labels_3d=labels.cpu())
    if attrs is not None:
        result["attrs_3d"] = attrs.cpu()
    return result


def batched_to_results(batched, img_metas):
    """batched: CmtHead.get_bboxes_batched(...) (device tensors).  Returns per frame dict(boxes_3d, scores_3d, labels_3d)
    as CPU tensors, equal to what simple_test_pts returns for the same head outputs (box_type_3d applied when the frame's
    metas carry one).  The boxes, scores, labels and counts of all frames travel in ONE device->host copy."""
    boxes, scores, labels, count = batched["boxes"], batched["scores"], batched["labels"], batched["count"]
    B, K = scores.shape
    parts = [boxes.reshape(B, K * 9), scores, labels, count.reshape(B, 1)]
    host = torch.cat([t.contiguous().view(torch.uint8).reshape(B, -1) for t in parts], 1).cpu()
    widths = [K * 36, K * 4, K * 8, 4]
    results = []
    for i in range(B):
        row = host[i].split(widths)
        n = int(row[3].clone().view(torch.int32))
        bboxes = row[0][:n * 36].clone().view(torch.float32).view(n, 9)
        box_type = img_metas[i].get("box_type_3d")
        if box_type is not None:
            bboxes = box_type(bboxes, bboxes.size(-1))
        results.append(bbox3d2result(bboxes, row[1][:n * 4].clone().view(torch.float32),
                                     row[2][:n * 8].clone().view(torch.int64)))
    return results


def _drop_absent_frames(bbox_list, valid):
    """Empty results for the frames none of whose nodes / sensors is present (valid: a [rows, B] device mask).  Called
    after get_bboxes, which has synchronised already: reading the mask on the host costs nothing more."""
    present = valid.any(0).tolist()
    return [item if present[i] else [t[:0] for t in item] for i, item in enumerate(bbox_list)]


def simple_test_pts(head, x, x_img, img_metas, rescale=False, sensor_valid=None):
    """CmtDetector.simple_test_pts (detectors/cmt.py:221-231). x / x_img: lists of feature levels as the detector's
    extract_feat returns them (`[None]` for a missing modality).  sensor_valid: optional torch.bool [S, B] device mask
    of the sensors that delivered each frame (CmtHead.forward_single); a frame with no sensor gets an empty result."""
    outs = head(x, x_img, img_metas, sensor_valid=sensor_valid)
    bbox_list = head.get_bboxes(outs, img_metas, rescale=rescale)
    if sensor_valid is not None:
        bbox_list = _drop_absent_frames(bbox_list, sensor_valid)
    return [bbox3d2result(bboxes, scores, labels) for bboxes, scores, labels in bbox_list]


def coop_simple_test_pts(head, vehicle_pts_feats, infrastructure_pts_feats, vehicle_img_feats, infrastructure_img_feats,
                         img_metas, rescale=False, node_valid=None):
    """CmtCoopDetector.coop_simple_test_pts (detectors/cmt_coop.py:549-569).  node_valid: optional torch.bool [2, B]
    device mask of the nodes that delivered each frame (CmtHeadCoop.forward_single); a frame with neither node gets an
    empty result."""
    if vehicle_pts_feats is None:
        vehicle_pts_feats = [None]
    if infrastructure_pts_feats is None:
        infrastructure_pts_feats = [None]
    if vehicle_img_feats is None:
        vehicle_img_feats = [None]
    if infrastructure_img_feats is None:
        infrastructure_img_feats = [None]
    outs = head(vehicle_pts_feats, infrastructure_pts_feats, vehicle_img_feats, infrastructure_img_feats, img_metas,
                node_valid=node_valid)
    bbox_list = head.get_bboxes(outs, img_metas, rescale=rescale)
    if node_valid is not None:
        bbox_list = _drop_absent_frames(bbox_list, node_valid)
    return [bbox3d2result(bboxes, scores, labels) for bboxes, scores, labels in bbox_list]


def simple_test(head, pts_feats, img_feats, img_metas, rescale=False, sensor_valid=None):
    """The part of CmtDetector.simple_test after extract_feat (detectors/cmt.py:233-252): per-frame result dicts.
    sensor_valid: as in simple_test_pts."""
    if pts_feats is None:
        pts_feats = [None]
    if img_feats is None:
        img_feats = [None]
    bbox_list = [dict() for _ in range(len(img_metas))]
    for result_dict, pts_bbox in zip(bbox_list, simple_test_pts(head, pts_feats, img_feats, img_metas, rescale=rescale,
                                                                sensor_valid=sensor_valid)):
        result_dict["pts_bbox"] = pts_bbox
    return bbox_list


def coop_simple_test(head, vehicle_pts_feats, infrastructure_pts_feats, vehicle_img_feats, infrastructure_img_feats,
                     img_metas, rescale=False, node_valid=None):
    """The part of CmtCoopDetector.simple_test after the two extract_*_feat calls (detectors/cmt_coop.py:571-594).
    node_valid: as in coop_simple_test_pts."""
    bbox_list = [dict() for _ in range(len(img_metas))]
    bbox_pts = coop_simple_test_pts(head, vehicle_pts_feats, infrastructure_pts_feats, vehicle_img_feats,
                                    infrastructure_img_feats, img_metas, rescale=rescale, node_valid=node_valid)
    for result_dict, pts_bbox in zip(bbox_list, bbox_pts):
        result_dict["pts_bbox"] = pts_bbox
    return bbox_list


@torch.no_grad()
def device_calibration(lidar2img, device, vehicle2infrastructure=None):
    """lidar2img: [B,V,4,4] (nested lists / numpy, float64) -> (lidar2img [B,V,4,4] fp32, img2lidar [B,V,4,4] fp32) on
    `device`, computed there in float64.  vehicle2infrastructure: optional [B,4,4] (or [4,4]); when given, the matrices
    are first folded into infrastructure coordinates, lidar2img @ inv(v2i) (transforms_3d_coop.py:213-222)."""
    l2i = torch.from_numpy(np.asarray(lidar2img, dtype=np.float64)).to(device, non_blocking=True)
    if l2i.dim() != 4 or l2i.shape[-2:] != (4, 4):
        raise ValueError(f"lidar2img must be [B,V,4,4], got {tuple(l2i.shape)}")
    if vehicle2infrastructure is not None:
        v2i = torch.from_numpy(np.asarray(vehicle2infrastructure, dtype=np.float64)).to(device, non_blocking=True)
        if v2i.dim() == 2:
            v2i = v2i.unsqueeze(0).expand(l2i.shape[0], -1, -1)
        l2i = l2i @ torch.linalg.inv(v2i).unsqueeze(1)
    i2l = torch.linalg.inv(l2i)
    return l2i.float().contiguous(), i2l.float().contiguous()


def attach_calibration(img_metas, device, prefix="", fold_vehicle2infrastructure=False):
    """Builds the device calibration of a batch from its metas and stores it in img_metas[0][prefix + 'calibration'] (the
    head reads it from there instead of inverting / uploading per call).  fold_vehicle2infrastructure: the metas carry
    raw vehicle matrices plus 'vehicle2infrastructure' (the TransformLidar2ImgToInfraCoords pipeline step was skipped)."""
    l2i = [m[prefix + "lidar2img"] for m in img_metas]
    v2i = [m["vehicle2infrastructure"] for m in img_metas] if fold_vehicle2infrastructure else None
    img_metas[0][prefix + "calibration"] = device_calibration(l2i, device, v2i)
    return img_metas
