"""CPU: model_variant = "v2_huge" (convnextv2_huge) is accepted by the configuration and the CLI, and the emulation of the device
numerics (``oracle/emulate.py``) covers its widths: 352 stays on the FP32-pipe depthwise path, 704 and wider take the tensor
cores, and with rounding off the emulated stages are the oracle's."""
from types import SimpleNamespace

import torch

from oracle import emulate
from oracle import reference_path as ref
from oracle.convnext import make_model
from spine_vision_b200 import synthetic


def test_config_and_cli_accept_v2_huge(tmp_path, monkeypatch):
    import spine_vision_b200.__main__ as cli
    from spine_vision_b200 import dataset

    cfg = dataset.ClassificationDatasetConfig(base_path=tmp_path, model_variant="v2_huge")
    assert cfg.model_variant == "v2_huge"
    seen = []
    monkeypatch.setattr(dataset, "create_classification_dataset", lambda config: seen.append(config) or SimpleNamespace(summary="ok"))
    assert cli.main(["dataset", "classification", "--base-path", str(tmp_path), "--model-variant", "v2_huge"]) == 0
    assert seen[0].model_variant == "v2_huge"


def test_emulator_depthwise_path_at_v2_huge_widths():
    assert not emulate.tc_depthwise(torch.float16, 352)
    assert all(emulate.tc_depthwise(torch.float16, c) for c in (704, 1408, 2816))
    assert not any(emulate.tc_depthwise(torch.bfloat16, c) for c in (352, 704, 1408, 2816))


def test_emulator_without_rounding_is_the_fp32_v2_huge_network():
    """Rounding off, every v2_huge stage of the folded form is the oracle's within 1e-5 relative (32 x 32: one token in the
    last stage)."""
    om = make_model("v2_huge", seed=0, trained_like=True)
    x = torch.stack([ref.preprocess_slice(synthetic.make_iso_slice(20 + i, 400, 380), (32, 32))[1] for i in range(2)])
    want, want_st = emulate.oracle_stages(om, x)
    got, got_st = emulate.forward_stages(om, x, torch.float16, rounding=False)
    for s, (g, w) in enumerate(zip(got_st, want_st)):
        assert g.shape == w.shape == (2, 32 >> (s + 2), 32 >> (s + 2), (352, 704, 1408, 2816)[s])
        rel = float((g - w).norm() / w.norm())
        assert rel <= 1e-5, f"stage {s}: relative difference {rel:.2e}"
    assert float((got - want).abs().max()) <= 1e-5
