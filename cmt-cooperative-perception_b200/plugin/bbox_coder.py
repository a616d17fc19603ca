"""MultiTaskBBoxCoder (projects/mmdet3d_plugin/core/bbox/coders/multi_task_bbox_coder.py:15-141) and
denormalize_bbox (core/bbox/util.py:37-68).  The flat top-k over sigmoid(cls) and `label = idx % C`,
`query = idx // C` are what "identical top-k query indices" checks.

`decode` is the reference's per-frame torch loop: few FLOPs, but about 30 launches and three `nonzero` host
synchronisations per frame (`boxes[mask]`, ...), so it cannot be captured in a CUDA graph; it also serves CPU tensors.
`decode_batched` computes the same detections for every frame in one library launch (`cmt_bbox_topk_decode`) with no
host synchronisation, into fixed-shape outputs that can live in a graph."""
from __future__ import annotations

import torch

from .. import ops
from .registry import BBOX_CODERS


def denormalize_bbox(nb, pc_range=None):
    cx, cy, cz = nb[..., 0:1], nb[..., 1:2], nb[..., 2:3]
    w, l, h = nb[..., 3:4].exp(), nb[..., 4:5].exp(), nb[..., 5:6].exp()
    rot = torch.atan2(nb[..., 6:7], nb[..., 7:8])
    if nb.size(-1) > 8:
        return torch.cat([cx, cy, cz, w, l, h, rot, nb[..., 8:9], nb[..., 9:10]], dim=-1)
    return torch.cat([cx, cy, cz, w, l, h, rot], dim=-1)


@BBOX_CODERS.register_module()
class MultiTaskBBoxCoder:
    def __init__(self, pc_range, voxel_size=None, post_center_range=None, max_num=100, score_threshold=None,
                 num_classes=10):
        self.pc_range = pc_range
        self.voxel_size = voxel_size
        self.post_center_range = post_center_range
        self.max_num = max_num
        self.score_threshold = score_threshold
        self.num_classes = num_classes

    def encode(self):
        pass

    def decode_single(self, cls_scores, bbox_preds, task_ids):
        num_query = cls_scores.shape[0]
        scores, indexs = cls_scores.sigmoid().view(-1).topk(self.max_num)
        labels = indexs % self.num_classes
        bbox_index = indexs // self.num_classes
        task_index = torch.gather(task_ids, 1, labels.unsqueeze(1)).squeeze()
        bbox_preds = bbox_preds[task_index * num_query + bbox_index]
        boxes = denormalize_bbox(bbox_preds, self.pc_range)
        if self.post_center_range is None:
            raise NotImplementedError("Need to reorganize output as a batch, only support "
                                      "post_center_range is not None for now!")
        pcr = torch.as_tensor(self.post_center_range, device=scores.device, dtype=boxes.dtype)
        mask = (boxes[..., :3] >= pcr[:3]).all(1) & (boxes[..., :3] <= pcr[3:]).all(1)
        if self.score_threshold:
            mask &= scores > self.score_threshold
        return dict(bboxes=boxes[mask], scores=scores[mask], labels=labels[mask], topk_index=indexs)

    def decode(self, preds_dicts):
        bbox_l, logit_l, tid_l = [], [], []
        for task_id in range(len(preds_dicts)):
            d = preds_dicts[task_id][0]
            bbox_l.append(torch.cat((d["center"][-1], d["height"][-1], d["dim"][-1], d["rot"][-1], d["vel"][-1]), -1))
            logits = d["cls_logits"][-1]
            logit_l.append(logits)
            tid_l.append(logits.new_ones(logits.shape).int() * task_id)
        all_logits = torch.cat(logit_l, dim=-1)
        all_bbox = torch.cat(bbox_l, dim=1)
        all_tids = torch.cat(tid_l, dim=-1)
        return [self.decode_single(all_logits[i], all_bbox[i], all_tids[i]) for i in range(all_logits.shape[0])]


    def decode_batched(self, preds_dicts, bottom_center=False, node_valid=None):
        """Fixed-shape counterpart of `decode` on CUDA tensors, one launch for the whole batch (ops.bbox_topk_decode).
        Returns {boxes [B,K,9], scores [B,K], labels [B,K], count [B], topk_index [B,K]}: frame b's detections are
        boxes[b, :count[b]] (= decode(...)[b]["bboxes"]), the remaining slots are zero with label -1.  Boxes are before
        CmtHead.get_bboxes' z shift unless bottom_center (then z -= h / 2 in the kernel).  node_valid: optional
        torch.bool [n_nodes, B] device mask; a frame with no node present gets no detections and topk_index -1."""
        if self.post_center_range is None:
            raise NotImplementedError("Need to reorganize output as a batch, only support "
                                      "post_center_range is not None for now!")
        tasks = [{n: preds_dicts[t][0][n][-1] for n in ops.BOX_DECODE_FIELDS} for t in range(len(preds_dicts))]
        n_cls = sum(int(d["cls_logits"].shape[-1]) for d in tasks)
        if n_cls != self.num_classes:
            raise ValueError(f"MultiTaskBBoxCoder: num_classes {self.num_classes} != {n_cls} classes of the task heads")
        return ops.bbox_topk_decode(tasks, self.num_classes, self.max_num, self.post_center_range, self.score_threshold,
                                    bottom_center, node_valid=node_valid)


def build_bbox_coder(cfg):
    return BBOX_CODERS.build(cfg)
