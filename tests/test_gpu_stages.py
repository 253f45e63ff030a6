"""Stage-level parity of the localizer forward: the residual stream after each of the four stages, read out of the real
forward (``svb_model_forward_stages``: same kernels, micro-batches, dual chain and tail chunk), against the fp32 oracle and
against the emulation of the device numerics (``oracle/emulate.py``), on trained-like weights where every ConvNeXt block
contributes.

Why stages and not only coordinates: global average pooling and two LayerNorms dilute an error in one part of the image, so a
kernel that gets one 128-token GEMM tile wrong by half can still land within 0.5 px.  Per stage the same fault is far above
the 16-bit rounding floor.

Metrics, per stage, of a tensor ``a`` against a reference ``r`` (both ``[B, h, w, C]``):
  * normwise relative error   ||a - r|| / ||r||
  * per-token error           max over tokens of rms_c(a - r), over the rms of ``r`` over the whole stage
Gates (``stage_gate``), per stage:
  * device vs fp32 <= 2 x emulator vs fp32 (normwise) and <= 3 x emulator vs fp32 (per-token): the device rounds no worse
    than the emulated design
  * device vs emulator < sqrt(2) x emulator vs fp32 (normwise): the device follows the emulated rounding points.  The two round
    at the same points but accumulate in different fp32 orders, so values near a rounding tie land on different sides, and those
    flips spread through the blocks: by stage 2 the device's and the emulator's rounding noise are nearly independent draws of
    the same process, which lie sqrt(2) x their size apart (measured on a B200: 0.4-0.7 at stage 0, 0.8-1.0 at stage 1,
    1.0-1.16 at stages 2-3).  A device that rounds elsewhere, or adds an error of its own, moves away from both.
Measured on a B200 for every row below: device vs fp32 / emulator vs fp32 = 0.94-1.02 (normwise), 0.92-1.06 (per-token).
``test_stage_gate_sees_tile_faults`` (CPU) keeps the gates honest: three single-tile faults injected into the emulator, each of
which moves the coordinates by no more than about half a pixel, must each fail them.
"""
import copy

import numpy as np
import pytest
import torch

from gpu_util import dev, fp32
from oracle import emulate
from oracle import reference_path as ref
from oracle.convnext import make_model
from spine_vision_b200 import cropping, synthetic

NORM_X, TOKEN_X, EMU_X = 2.0, 3.0, 2.0 ** 0.5
DTYPES = {"fp16": torch.float16, "bf16": torch.bfloat16}


def stage_metrics(a: torch.Tensor, r: torch.Tensor) -> tuple[float, float]:
    d = a.double() - r.double()
    r = r.double()
    return float(d.norm() / r.norm()), float(d.pow(2).mean(-1).sqrt().max() / r.pow(2).mean().sqrt())


def stage_gate(dev_st, emu_st, ref_st):
    """-> (all stages pass, one printable row per stage)."""
    ok, rows = True, []
    for s, (d, e, r) in enumerate(zip(dev_st, emu_st, ref_st)):
        (dn, dt), (en, et), (de, _) = stage_metrics(d, r), stage_metrics(e, r), stage_metrics(d, e)
        row_ok = dn <= NORM_X * en and dt <= TOKEN_X * et and de < EMU_X * en
        ok &= row_ok
        rows.append(f"stage {s}: dev/fp32 {dn:.2e} tok {dt:.2e} | emu/fp32 {en:.2e} tok {et:.2e} | ratio {dn / en:.2f} tok {dt / et:.2f} | "
                    f"dev/emu {de:.2e} ({de / en:.2f} of emu/fp32) {'ok' if row_ok else 'FAIL'}")
    return ok, rows


def _inputs(size, n, seed0=200):
    shapes = [(seed0 + i, 400 + 37 * i, 380 + 53 * i) for i in range(n)]  # distinct images
    pre = [ref.preprocess_slice(synthetic.make_iso_slice(*c), size) for c in shapes]
    return np.stack([p for p, _ in pre]), torch.stack([t for _, t in pre])


# (variant, dtype, image size): base in both dtypes; tiny (96 wide: a ragged channel chunk, no tensor-core depthwise conv),
# large (192 / 1536), xlarge (2048), v2 (GRN); 32^2 (the last stage is one token, mode A at W = 8), 352 x 288 (mode-B windows),
# 1024 x 512 (non-square)
ROWS = [("base", "fp16", (512, 512)), ("base", "bf16", (512, 512)), ("base", "fp16", (32, 32)), ("base", "fp16", (352, 288)),
        ("base", "fp16", (1024, 512)), ("tiny", "fp16", (512, 512)), ("tiny", "fp16", (32, 32)), ("large", "fp16", (352, 288)),
        ("xlarge", "fp16", (512, 512)), ("v2_tiny", "fp16", (352, 288)), ("v2_base", "fp16", (512, 512)), ("v2_base", "fp16", (32, 32))]


@pytest.mark.gpu
@pytest.mark.parametrize("variant,dtype,size", ROWS)
def test_stages_vs_fp32_and_emulator(variant, dtype, size):
    """Micro-batch 2 over 5 images: chunks on both chains plus a tail chunk of one image."""
    mb, B = 2, 5
    om = make_model(variant, seed=0, trained_like=True)
    planes, x = _inputs(size, B)
    model = cropping.LocalizationModel(om.state_dict(), dev(), dtype=dtype, micro_batch=mb)
    coords, dev_st = model.predict_u8_stages(torch.from_numpy(planes).to(dev()))
    om_d, x_d = copy.deepcopy(om).to(dev()), x.to(dev())
    want, ref_st = fp32(emulate.oracle_stages, om_d, x_d)
    emu, emu_st = fp32(emulate.forward_stages, om_d, x_d, DTYPES[dtype])
    dev_st = [t.float() for t in dev_st]
    ok, rows = stage_gate(dev_st, emu_st, ref_st)
    e_dev = float((coords - want).abs().max()) * 512
    e_emu = float((emu - want).abs().max()) * 512
    print(f"\n[stages] {variant} {dtype} {size[0]}x{size[1]} B={B} micro_batch={mb}: coords dev {e_dev:.4f} px, emulator {e_emu:.4f} px (x 512)")
    for r in rows:
        print("  " + r)
    assert ok, f"{variant} {dtype} {size}: " + "; ".join(r for r in rows if r.endswith("FAIL"))


TILE = 128  # tokens per GEMM M tile


@pytest.mark.parametrize("stage,block,factor", [(0, 2, 1.5), (2, 5, 1.05), (1, 1, 1.2)])
def test_stage_gate_sees_tile_faults(stage, block, factor):
    """CPU power check of ``stage_gate``: scaling the MLP output of ONE 128-token tile of one block (base, trained-like, fp16,
    512^2, two images) moves the coordinates by only 0.2-0.3 px, but must fail the gate at that stage."""
    om = make_model("base", seed=0, trained_like=True)
    _, x = _inputs((512, 512), 2)
    _, ref_st = emulate.oracle_stages(om, x)
    emu, emu_st = emulate.forward_stages(om, x, torch.float16)

    def fault(s, j, o):
        if (s, j) == (stage, block):
            o = o.clone()
            o.view(-1, o.shape[-1])[TILE : 2 * TILE] *= factor  # the second M tile of the block's GEMMs
        return o

    bad, bad_st = emulate.forward_stages(om, x, torch.float16, mlp_hook=fault)
    clean_ok, _ = stage_gate(emu_st, emu_st, ref_st)
    assert clean_ok  # the gate passes a device that IS the emulator
    ok, rows = stage_gate(bad_st, emu_st, ref_st)
    print(f"\n[fault] stage {stage} block {block} one tile x{factor}: coordinates move {float((bad - emu).abs().max()) * 512:.3f} px")
    for r in rows:
        print("  " + r)
    assert not ok and rows[stage].endswith("FAIL")
