"""The compute precision switch on the host: one name -> dtype map, `set_precision` reaching every module that carries a
precision, unknown names refused.  No GPU needed."""
import pytest
import torch

from cmtcoop_b200 import ops, synth
from cmtcoop_b200.plugin import FlashAttention, FlashMHA, build_head

BAD = ("fp8", "half", "FP16", "", None)


def test_compute_dtype():
    assert ops.compute_dtype("bf16") == torch.bfloat16
    assert ops.compute_dtype("fp16") == torch.float16
    assert ops.compute_dtype("fp32") == torch.float32
    for bad in BAD:
        with pytest.raises(ValueError):
            ops.compute_dtype(bad)


@pytest.mark.parametrize("kind", synth.HEAD_KINDS)
def test_set_precision_fp16_reaches_every_module(kind):
    cfg, _ = synth.mini_case(kind)
    head = build_head(cfg)
    mods = [m for m in head.modules() if hasattr(m, "precision")]
    assert all(m.precision == "bf16" for m in mods)
    assert any(isinstance(m, FlashMHA) for m in mods) and any(isinstance(m, FlashAttention) for m in mods)
    assert head.set_precision("fp16") is head
    assert all(m.precision == "fp16" for m in mods), [type(m).__name__ for m in mods if m.precision != "fp16"]
    for bad in BAD:
        with pytest.raises(ValueError):
            head.set_precision(bad)
        with pytest.raises(ValueError):
            head.transformer.set_precision(bad)
    assert all(m.precision == "fp16" for m in mods)   # a refused name changes nothing


def test_flash_modules_set_precision():
    mha = FlashMHA(256, 8)
    assert mha.set_precision("fp16") is mha
    assert mha.precision == "fp16" and mha.inner_attn.precision == "fp16"
    fa = FlashAttention()
    assert fa.set_precision("fp16") is fa and fa.precision == "fp16"
    for bad in BAD:
        with pytest.raises(ValueError):
            mha.set_precision(bad)
        with pytest.raises(ValueError):
            fa.set_precision(bad)
    assert mha.precision == "fp16" and fa.precision == "fp16"
