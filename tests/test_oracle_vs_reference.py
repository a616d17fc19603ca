"""Where CMT_REFERENCE_ROOT names a checkout of the original project, run the UNMODIFIED reference live against
the oracle on a shape that is NOT among the committed goldens (B=1, 13x13 BEV map, 60 queries, 3 camera views,
2 vehicle + 1 infrastructure views).  Skipped otherwise: the committed goldens (test_oracle_golden.py) compare with
the reference on the mini case only (B=2, 24x24 BEV map, 96 queries)."""
import numpy as np
import pytest
import torch

from cmtcoop_b200 import synth
from oracle import cmt_oracle as O
from oracle import ref_stub

pytestmark = pytest.mark.skipif(not ref_stub.reference_available(),
                                reason="CMT_REFERENCE_ROOT does not name a checkout of the original project")


@pytest.mark.parametrize("kind", ["CmtHead", "CmtImageHeadCoop"])
def test_oracle_equals_verbatim_reference(kind):
    from oracle.make_golden import run_reference
    cfg = synth.head_cfg(kind, num_query=60, num_layers=2, grid=8 * 13, max_num=30)
    inputs = synth.make_inputs(kind, B=1, bev_hw=13, n_views=3, img_hw=(4, 9), vehicle_views=2, infra_views=1, seed=9)
    head, rets, _ = run_reference(kind, cfg, inputs, seed=5)
    sd = {k: v.detach() for k, v in head.state_dict().items()}
    want, _ = O.head_forward(sd, cfg, inputs)
    for name in want[0]:
        assert O.rel_l2(want[0][name], rets[0][name]) < 2e-5, name
