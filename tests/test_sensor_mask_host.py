"""Host-side checks of the single-node heads' per-frame sensor mask (`sensor_valid`, torch.bool [S, B]): its row count
follows the head class (LiDAR row + one per camera), dtype and device are checked without reading the values, a mask
under the KV-token split is refused, and the cooperative heads do not take it.  No GPU needed."""
import numpy as np
import pytest
import torch

from cmtcoop_b200 import synth
from cmtcoop_b200.plugin import build_head
from cmtcoop_b200.runtime import _head_forward

ROWS = {"CmtHead": 3, "CmtImageHead": 2, "CmtLidarHead": 1}   # mini_case: 2 cameras


def _case(kind):
    cfg, inputs = synth.mini_case(kind)
    head = build_head(cfg).eval()
    x = torch.from_numpy(inputs["pts_feats"]) if inputs.get("pts_feats") is not None else None
    xi = torch.from_numpy(inputs["img_feats"]) if inputs.get("img_feats") is not None else None
    return head, x, xi, inputs["img_metas"]


@pytest.mark.parametrize("kind", list(ROWS))
def test_mask_shape_follows_the_head_class(kind):
    head, x, xi, metas = _case(kind)
    B, S = len(metas), ROWS[kind]
    with torch.no_grad():
        for rows in [r for r in (S - 1, S + 1) if r >= 1]:
            with pytest.raises(ValueError, match=f"sensor_valid must be \\[{S}, {B}\\]"):
                head.forward_single(x, xi, metas, sensor_valid=torch.ones(rows, B, dtype=torch.bool))
        for bad, err in ((torch.ones(S, B + 1, dtype=torch.bool), ValueError), (torch.ones(S * B, dtype=torch.bool), ValueError),
                         (torch.ones(S, B, dtype=torch.uint8), TypeError), (torch.ones(S, B), TypeError),
                         ([[True] * B] * S, TypeError),
                         (torch.ones(S, B, dtype=torch.bool, device="meta"), ValueError)):   # not the features' device
            with pytest.raises(err):
                head.forward_single(x, xi, metas, sensor_valid=bad)
        # a well-formed mask passes the checks; the forward itself then needs CUDA tensors
        with pytest.raises(RuntimeError, match="CUDA"):
            head.forward_single(x, xi, metas, sensor_valid=torch.ones(S, B, dtype=torch.bool))


@pytest.mark.parametrize("kind", list(ROWS))
def test_mask_under_the_kv_split_raises(kind):
    head, x, xi, metas = _case(kind)
    head.transformer.kv_split_group = object()   # enable_kv_split(group) without a process group
    with torch.no_grad(), pytest.raises(NotImplementedError):
        head.forward_single(x, xi, metas, sensor_valid=torch.ones(ROWS[kind], len(metas), dtype=torch.bool))


@pytest.mark.parametrize("kind", ["CmtHeadCoop", "CmtLidarHeadCoop", "CmtImageHeadCoop"])
def test_cooperative_heads_do_not_take_sensor_valid(kind):
    cfg, inputs = synth.mini_case(kind)
    head = build_head(cfg).eval()
    names = ("vehicle_pts_feats", "infrastructure_pts_feats", "vehicle_img_feats", "infrastructure_img_feats")
    feats = {k: torch.from_numpy(inputs[k]) for k in names if isinstance(inputs.get(k), np.ndarray)}
    mask = torch.ones(2, len(inputs["img_metas"]), dtype=torch.bool)
    with torch.no_grad():
        with pytest.raises(TypeError):
            head.forward_single(*[feats.get(k) for k in names], inputs["img_metas"], sensor_valid=mask)
        with pytest.raises(ValueError, match="sensor_valid"):   # the graph / runner inputs dict
            _head_forward(head, True, dict(feats, sensor_valid=mask), inputs["img_metas"], False)


def test_single_node_heads_do_not_take_node_valid():
    head, x, xi, metas = _case("CmtHead")
    with torch.no_grad(), pytest.raises(ValueError, match="node_valid"):
        _head_forward(head, False, dict(pts_feats=x, img_feats=xi, node_valid=torch.ones(2, len(metas), dtype=torch.bool)),
                      metas, False)
