"""CPU: ``oracle/emulate.py``, the stage-by-stage emulation of the device numerics that the stage-level GPU tests
(``test_gpu_stages.py``) and the trained-like coordinate tolerances are derived from."""
import pytest
import torch

from oracle import emulate
from oracle import reference_path as ref
from oracle.convnext import make_model
from spine_vision_b200 import synthetic

SLICES = [(20, 1195, 1195), (21, 640, 650), (22, 900, 700), (23, 512, 512)]


def _inputs(size, slices=SLICES[:2]):
    return torch.stack([ref.preprocess_slice(synthetic.make_iso_slice(*c), size)[1] for c in slices])


@pytest.mark.parametrize("variant,size", [("base", (128, 128)), ("tiny", (96, 160)), ("v2_tiny", (64, 64)), ("v2_base", (32, 32))])
def test_emulator_without_rounding_is_the_fp32_network(variant, size):
    """Rounding off, the folded form (one-pass statistics, LayerNorm folded into fc1, the depthwise conv column by column where the
    tensor-core kernel runs, GRN over the hidden activation) is the oracle's network: every stage within ~1e-5 relative."""
    torch.manual_seed(0)
    om = make_model(variant, seed=0, trained_like=True)
    x = _inputs(size)
    want, want_st = emulate.oracle_stages(om, x)
    got, got_st = emulate.forward_stages(om, x, torch.float16, rounding=False)
    assert len(got_st) == len(want_st) == 4
    for s, (g, w) in enumerate(zip(got_st, want_st)):
        assert g.shape == w.shape == (2, size[0] >> (s + 2), size[1] >> (s + 2), om.backbone.stages[s].blocks[0].norm.weight.numel())
        rel = float((g - w).norm() / w.norm())
        assert rel <= 1e-5, f"stage {s}: relative difference {rel:.2e}"
    assert float((got - want).abs().max()) <= 1e-5


def test_emulator_rounds_where_the_device_stores_16_bits():
    """The stage outputs are 16-bit values, and the tensor-core depthwise selection is the one ``dw_tc2_mode`` makes by default."""
    om = make_model("tiny", seed=0, trained_like=True)
    x = _inputs((64, 64))
    for dt in (torch.float16, torch.bfloat16):
        _, st = emulate.forward_stages(om, x, dt)
        assert all(torch.equal(s, s.to(dt).float()) for s in st)
    assert not emulate.tc_depthwise(torch.float16, 96) and emulate.tc_depthwise(torch.float16, 192)
    assert emulate.tc_depthwise(torch.float16, 2048) and not emulate.tc_depthwise(torch.bfloat16, 128)


def test_emulator_predicts_the_recorded_coordinate_error():
    """fp16 on trained-like ``base`` weights at 512^2 (four slices): the device measured 0.117-0.121 px and the emulator's
    earlier form predicted 0.119-0.176 px (DESIGN.md section 5); bf16 measured 0.83 px."""
    om = make_model("base", seed=0, trained_like=True)
    x = _inputs((512, 512), SLICES)
    want, _ = emulate.oracle_stages(om, x)
    e16 = float((emulate.forward_stages(om, x, torch.float16)[0] - want).abs().max()) * 512
    eb16 = float((emulate.forward_stages(om, x, torch.bfloat16)[0] - want).abs().max()) * 512
    print(f"[emulator] base trained-like 512^2: fp16 {e16:.4f} px, bf16 {eb16:.4f} px")
    assert 0.10 <= e16 <= 0.20
    assert 0.5 <= eb16 <= 1.2
