"""Host-side checks of the cooperative heads' per-frame node mask (`node_valid`): shape, dtype and device are checked
without reading the values, and a mask that comes with a missing node is refused.  No GPU needed."""
import numpy as np
import pytest
import torch

from cmtcoop_b200 import ops, synth
from cmtcoop_b200.plugin import build_head

B = 4


def test_check_node_valid_accepts_a_bool_mask():
    m = torch.tensor([[True, False, True, False], [True, True, False, False]])
    assert ops.check_node_valid(m, B, "cpu") is m
    t = torch.ones(B, 2, dtype=torch.bool).t()           # non-contiguous view: a contiguous copy comes back
    got = ops.check_node_valid(t, B, "cpu")
    assert got.is_contiguous() and torch.equal(got, t)
    for n in (1, 3):                                      # the decode takes any number of nodes
        assert ops.check_node_valid(torch.ones(n, B, dtype=torch.bool), B, "cpu", n_nodes=None).shape == (n, B)


@pytest.mark.parametrize("bad,err", [
    ([[True] * B, [True] * B], TypeError),                        # not a tensor
    (torch.ones(2, B, dtype=torch.uint8), TypeError),
    (torch.ones(2, B, dtype=torch.float32), TypeError),
    (torch.ones(2, B + 1, dtype=torch.bool), ValueError),
    (torch.ones(3, B, dtype=torch.bool), ValueError),
    (torch.ones(B, dtype=torch.bool), ValueError),
    (torch.ones(2, 2, B, dtype=torch.bool), ValueError),
])
def test_check_node_valid_rejects(bad, err):
    with pytest.raises(err):
        ops.check_node_valid(bad, B, "cpu")


def test_check_node_valid_rejects_another_device():
    m = torch.ones(2, B, dtype=torch.bool)                # a host mask for features on the GPU
    with pytest.raises(ValueError):
        ops.check_node_valid(m, B, "cuda:0")
    with pytest.raises(ValueError):
        ops.check_node_valid(torch.ones(0, B, dtype=torch.bool), B, "cpu", n_nodes=None)


@pytest.mark.parametrize("kind", ["CmtHeadCoop", "CmtLidarHeadCoop", "CmtImageHeadCoop"])
def test_mask_with_a_missing_node_raises(kind):
    cfg, inputs = synth.mini_case(kind)
    head = build_head(cfg).eval()
    names = ("vehicle_pts_feats", "infrastructure_pts_feats", "vehicle_img_feats", "infrastructure_img_feats")
    feats = [torch.from_numpy(inputs[k]) if isinstance(inputs.get(k), np.ndarray) else None for k in names]
    mask = torch.ones(2, len(inputs["img_metas"]), dtype=torch.bool)
    for drop in ("vehicle", "infrastructure"):
        args = [None if n.startswith(drop) else t for n, t in zip(names, feats)]
        with torch.no_grad(), pytest.raises(ValueError):
            head.forward_single(*args, inputs["img_metas"], node_valid=mask)
