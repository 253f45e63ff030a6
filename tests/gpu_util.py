import copy

import pytest
import torch

requires_gpu = pytest.mark.gpu


def dev():
    assert torch.cuda.is_available(), "gpu test selected without a GPU"
    return "cuda:0"


def fp32(fn, *a, **k):
    """Run a reference (oracle / emulator) in true fp32 on whatever device holds its inputs: TF32 off for the call."""
    keep = torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = torch.backends.cudnn.allow_tf32 = False
    try:
        return fn(*a, **k)
    finally:
        torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = keep


def trained_like_gate(om, x, dtype=torch.float16, px=512.0):
    """Coordinate gate for trained-like weights, where every ConvNeXt block counts: 0.5 px at 512^2, or twice the error that the
    emulation of the device numerics (``oracle/emulate.py``) predicts for this variant, size and dtype if that is larger.
    ``om`` the oracle model, ``x`` its ``[B,3,H,W]`` input.  Returns (fp32 oracle coordinates on the CPU, predicted px, gate px)."""
    from oracle import emulate

    om_d, x_d = copy.deepcopy(om).to(dev()), x.to(dev())
    want, _ = fp32(emulate.oracle_stages, om_d, x_d)
    emu, _ = fp32(emulate.forward_stages, om_d, x_d, dtype)
    pred = float((emu - want).abs().max()) * px
    return want.cpu().numpy(), pred, max(0.5, 2.0 * pred)
