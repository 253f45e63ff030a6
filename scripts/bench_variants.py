"""Forward-only rate of the localizer for every ``model_variant``: uint8 [256, 512, 512] -> coordinates, fp16 operands, micro-batch
64 (two micro-batches in flight), random-init weights (the rate does not depend on the values).  Timed with CUDA events over
whole ``predict_u8`` calls after two warm-up calls; the median of five.  GEMM TFLOP/s = the GEMM work ``engine.cost`` counts over
the whole forward's time (depthwise conv, LayerNorms, GRN and head included in the time).  The card's name and power limit are
read in the same run.

    python scripts/bench_variants.py [variant ...]
"""
import json
import subprocess
import sys
from pathlib import Path

import torch

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
from oracle.convnext import VARIANTS, make_model  # noqa: E402
from spine_vision_b200.cropping import LocalizationModel  # noqa: E402

B, S, MB, REPS = 256, 512, 64, 5


def card() -> dict:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True,
                       check=True)
    name, power, clock = q.stdout.strip().splitlines()[0].split(", ")
    return {"card": name, "power_limit": power, "max_sm_clock": clock}


def main() -> None:
    assert torch.cuda.is_available(), "bench_variants.py needs a GPU"
    dev = "cuda:0"
    print(json.dumps(card()), flush=True)
    g = torch.Generator(device=dev).manual_seed(0)
    x = torch.randint(0, 256, (B, S, S), generator=g, device=dev, dtype=torch.uint8)
    out = torch.empty((B, 5, 2), dtype=torch.float32, device=dev)
    for variant in sys.argv[1:] or list(VARIANTS):
        model = LocalizationModel(make_model(variant, seed=0).state_dict(), dev, dtype="fp16", micro_batch=MB)
        flops, launches = model.engine.cost(B, S, S)
        for _ in range(2):
            model.predict_u8(x, out=out)
        torch.cuda.synchronize()
        ts = []
        for _ in range(REPS):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            model.predict_u8(x, out=out)
            e1.record()
            torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1))
        ms = sorted(ts)[REPS // 2]
        print(json.dumps({"variant": variant, "dims": list(model.engine.dims), "depths": list(model.engine.depths), "images": B,
                          "size": S, "micro_batch": MB, "dtype": "fp16", "ms_median": round(ms, 2), "ms_all": [round(t, 2) for t in ts],
                          "img_per_s": round(B / ms * 1e3, 1), "gemm_tflop": round(flops / 1e12, 2),
                          "gemm_tflop_per_s": round(flops / ms / 1e9, 1), "launches": launches,
                          "finite": bool(torch.isfinite(out).all())}), flush=True)
        del model
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
