"""Predicted coordinate error of the device forward (16-bit storage / GEMM operands, fp32 accumulation) from its CPU
emulation, ``oracle/emulate.py``, against the fp32 oracle, per stage and at the coordinates:

    python scripts/emulate_precision.py [fp16|bf16] [variant] [H W]

Test infrastructure (imports oracle/)."""
import sys
from pathlib import Path

import torch

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
from oracle import emulate  # noqa: E402
from oracle import reference_path as ref  # noqa: E402
from oracle.convnext import make_model  # noqa: E402
from spine_vision_b200 import synthetic  # noqa: E402

DT = torch.float16 if (len(sys.argv) < 2 or sys.argv[1] == "fp16") else torch.bfloat16
VARIANT = sys.argv[2] if len(sys.argv) > 2 else "base"
SIZE = (int(sys.argv[3]), int(sys.argv[4])) if len(sys.argv) > 4 else (512, 512)
torch.set_num_threads(8)

SLICES = [(20, 1195, 1195), (21, 640, 650), (22, 900, 700), (23, 512, 512)]
xs = torch.stack([ref.preprocess_slice(synthetic.make_iso_slice(*c), SIZE)[1] for c in SLICES])
for trained in (False, True):
    m = make_model(VARIANT, seed=0, trained_like=trained)
    want, want_st = emulate.oracle_stages(m, xs)
    got, got_st = emulate.forward_stages(m, xs, DT)
    rel = " ".join(f"{float((g - w).norm() / w.norm()):.2e}" for g, w in zip(got_st, want_st))
    print(f"{DT} {VARIANT} {SIZE} trained_like={trained}: max coordinate error {float((got - want).abs().max()) * 512:.4f} px "
          f"(normalised x 512); stage relative errors {rel}", flush=True)
