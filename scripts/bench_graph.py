"""Eager forward against its CUDA-graph replay (``LocalizationModel.graphed``): ConvNeXt-base localizer, fp16, 512^2 uint8 planes,
random-init weights (the time does not depend on the values).  Both run in one process on one GPU, alternating in rounds; each
number is the median over the rounds with the smallest and largest round beside it.

- B = 1 (one series per call, as the drop-in ``predict_ivd_locations`` runs): per call, the host clock around the call and a
  ``torch.cuda.synchronize()`` (wall), and around the call alone (enqueue); the median over CALLS calls per round.
- B = 256, micro-batch 64 (two micro-batches in flight, the forward of bench.py's step): ms per step from CUDA events over STEPS
  back-to-back calls, and the host time to enqueue one step (measured on an idle stream, so that it is not waiting for room in
  the launch queue).

It checks that graph and eager coordinates are bit-identical at both sizes, and reads the card's name and power limit in the same
run.

    python scripts/bench_graph.py [--out FILE]
"""
import argparse
import json
import statistics
import subprocess
import sys
import time
from pathlib import Path

import torch

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
from spine_vision_b200 import _lib, synthetic  # noqa: E402
from spine_vision_b200.cropping import LocalizationModel  # noqa: E402

S, MB, ROUNDS, CALLS, STEPS, ENQ_STEPS = 512, 64, 7, 300, 10, 5


def card() -> dict:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True,
                       check=True)
    name, power, clock = q.stdout.strip().splitlines()[0].split(", ")
    return {"card": name, "power_limit": power, "max_sm_clock": clock}


def per_call_b1(fn, x, out):
    wall, enq = [], []
    for _ in range(CALLS):
        t0 = time.perf_counter()
        fn(x, out)
        t1 = time.perf_counter()
        torch.cuda.synchronize()
        t2 = time.perf_counter()
        enq.append((t1 - t0) * 1e3)
        wall.append((t2 - t0) * 1e3)
    return statistics.median(wall), statistics.median(enq)


def per_step_b256(fn, x, out):
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(STEPS):
        fn(x, out)
    e1.record()
    torch.cuda.synchronize()
    enq = []
    for _ in range(ENQ_STEPS):
        t0 = time.perf_counter()
        fn(x, out)
        enq.append((time.perf_counter() - t0) * 1e3)
        torch.cuda.synchronize()
    return e0.elapsed_time(e1) / STEPS, statistics.median(enq)


def summary(vals):
    return {"median": round(statistics.median(vals), 4), "min": round(min(vals), 4), "max": round(max(vals), 4)}


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", type=Path, default=None, help="also write the result lines to this file")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "bench_graph.py needs a GPU"
    dev = "cuda:0"
    lines = [json.dumps(card())]
    print(lines[-1], flush=True)
    model = LocalizationModel(synthetic.random_state_dict("base", seed=0), dev, dtype="fp16", micro_batch=MB)
    lib = _lib.load()
    gen = torch.Generator(device=dev).manual_seed(0)
    for B in (1, 256):
        x = torch.randint(0, 256, (B, S, S), generator=gen, device=dev, dtype=torch.uint8)
        out_e, out_g = (torch.empty((B, 5, 2), dtype=torch.float32, device=dev) for _ in range(2))
        g = model.graphed(B)
        eager = lambda x, o: model.predict_u8(x, out=o)  # noqa: E731
        graph = lambda x, o: g(x, out=o)  # noqa: E731
        n0 = lib.svb_launch_count(0)
        eager(x, out_e)
        launches = lib.svb_launch_count(0) - n0
        for _ in range(3):
            eager(x, out_e)
            graph(x, out_g)
        torch.cuda.synchronize()
        identical = bool(torch.equal(out_e, out_g))
        res = {"eager": ([], []), "graph": ([], [])}
        for _ in range(ROUNDS):
            for name, fn, out in (("eager", eager, out_e), ("graph", graph, out_g)):
                a, b = (per_call_b1 if B == 1 else per_step_b256)(fn, x, out)
                res[name][0].append(a)
                res[name][1].append(b)
        identical = identical and bool(torch.equal(out_e, out_g))
        timed = "wall_ms_per_call" if B == 1 else "ms_per_step_cuda_events"
        line = {"B": B, "size": S, "micro_batch": min(MB, B), "dtype": "fp16", "variant": "base", "rounds": ROUNDS,
                "calls_per_round": CALLS if B == 1 else STEPS, "eager_launches_per_call": launches, "graph_kernel_nodes": g.kernel_nodes,
                "graph_workspace_bytes": int(lib.svb_model_workspace_bytes(model.engine._h, min(MB, B), S, S)),
                "coords_bit_identical": identical}
        for name in ("eager", "graph"):
            line[f"{name}_{timed}"] = summary(res[name][0])
            line[f"{name}_enqueue_ms"] = summary(res[name][1])
        lines.append(json.dumps(line))
        print(lines[-1], flush=True)
        assert identical, f"graph and eager coordinates differ at B = {B}"
        del g
        torch.cuda.empty_cache()
    if args.out:
        args.out.parent.mkdir(parents=True, exist_ok=True)
        args.out.write_text("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
