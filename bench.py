#!/usr/bin/env python
"""Headline benchmark: series/sec of the localize-and-crop hot path (BASELINE.json).

    python bench.py --gpus 1 --steps K --warmup W          # this repo's sm_100a path
    python bench.py --impl reference ...                   # the reference's CPU path (oracle port) on host cores
    python bench.py ... --dump-outputs DIR                 # also write the last timed step's outputs to DIR/*.npy

One step = one pass of the hot path over one batch of synthetic middle slices:
K1 normalise+resize -> ConvNeXt-base localizer -> K3 crops (128^2 + 256^2).  Workload (N=1):
BASELINE.json configs[1] -- 256 series (15 x 512 x 512 fp32 @ 0.7 mm; middle plane resampled to 0.3 mm = 1195 x 1195),
convnext_base random init, 5 levels, crop_delta_mm 50/20/30/30.  `value` is measured with the isotropic
middle slices resident in HBM (K1 -> model -> K3); `e2e` through the public API from HOST buffers: the two
source planes per series in pinned memory -> H2D -> K0+K1 (fused) -> model -> K3 -> crops/coords back to the
host, every copy inside the timed region.  Prints ONE JSON line on rank 0.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time
from pathlib import Path

JSON_OUT = sys.stdout
ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

CROP_DELTA_MM = (50, 20, 30, 30)
CROP_SIZE = (128, 128)
SECOND_SIZE = (256, 256)
IMAGE_SIZE = (512, 512)
SLICE_HW = (1195, 1195)
TRAFFIC_JSON = os.environ.get("SVB_TRAFFIC_JSON", "r03z_gemm_traffic.json")  # per-shape DRAM bytes of the GEMM launches (ncu --set full), see scripts/summarise_ncu_layers.py
WORKLOAD = ("configs[1]: 256 synthetic sagittal series per GPU (15x512x512 fp32 @0.7mm; middle plane at 0.3mm iso = 1195x1195), "
            "convnext_base random-init localizer @512x512, 5 IVD levels, crop_delta_mm 50/20/30/30, 128x128 crops + 256x256 classifier input")
DUMP_SERIES = 32  # --dump-outputs: 32 series x 5 levels x (128^2 + 256^2) float32 = 52 MB per dump, whatever --batch is


def workload_config(args):
    """The SAME dict in both arms (the reference arm times a bounded sample of this workload; its sample is stated in
    cpu_baseline.sample)."""
    return {"workload": WORKLOAD, "series_per_gpu_per_step": args.batch, "micro_batch": args.micro_batch,
            "l2": "inputs larger than L2 (1.46 GB of fp32 slices per step; ~1.8 GB of activations per micro-batch, two in flight)"}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=256, help="series per GPU per step")
    ap.add_argument("--dtype", default="fp16", choices=["bf16", "fp16"],
                    help="GEMM operand type, fp32 accumulation (both 16-bit, same tensor-pipe rate; fp16 = the package default, it holds the 0.5 px gate on trained-like weights)")
    ap.add_argument("--micro-batch", type=int, default=64, help="images per pass through the network (two passes are in flight)")
    ap.add_argument("--stream-chunk", type=int, default=0, help="series per H2D chunk of the end-to-end path (0 = two micro-batches: both chains of the forward busy)")
    ap.add_argument("--distinct", type=int, default=0, help="distinct synthetic series (tiled to the batch); 0 = every series of the batch is distinct")
    ap.add_argument("--no-eager-baseline", action="store_true", help="skip the informational stock-PyTorch-on-this-GPU leg")
    ap.add_argument("--ref-series", type=int, default=16, help="series per step of the CPU reference arm (--impl reference)")
    ap.add_argument("--cpu-baseline-series", type=int, default=32,
                    help="series per pass of the cpu_baseline leg (N=1, rank 0): BASELINE configs[0]'s batch of 32, one warm-up + two timed passes = about 12 s of CPU work")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step returned (rank 0) as float32 DIR/<name>.npy: coords "
                         f"of every series, crops and crops2 of a fixed seeded sample of {DUMP_SERIES} series")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of --impl b200")
    return args


# ----------------------------------------------------------------------------- CPU reference arm
def cpu_reference_rate(n_series: int, steps: int, warmup: int):
    """The reference's own CPU path (oracle/reference_path.py: NumPy + Pillow + OpenCV + torch fp32,
    batch-1 loop exactly as process_spider runs it) on this box's host cores."""
    import torch

    from oracle import reference_path as ref
    from oracle.convnext import make_model
    from spine_vision_b200 import synthetic

    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    try:
        import cv2

        cv2.setNumThreads(cores)
    except Exception:
        pass
    model = make_model("base", seed=0)
    slices = [synthetic.make_iso_slice(s, *SLICE_HW) for s in range(n_series)]
    times = []
    for it in range(warmup + steps):
        t0 = time.perf_counter()
        ref.localize_and_crop_series(model, slices, CROP_SIZE, CROP_DELTA_MM, IMAGE_SIZE)
        dt = time.perf_counter() - t0
        if it >= warmup:
            times.append(dt)
    mean = sum(times) / len(times)
    return n_series / mean, mean, cores


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    rate, mean, cores = cpu_reference_rate(args.ref_series, args.steps, args.warmup)
    sample = f"{args.ref_series} series/step of the same workload, batch-1 loop (reference-faithful), {args.steps} steps after {args.warmup} warm-up"
    line = {
        "impl": "reference", "metric": "series/sec", "value": rate, "unit": "series/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": mean * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic", "config": workload_config(args),
        "crops_per_sec": rate * 5,
        "cpu_baseline": {"value": rate, "unit": "series/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": rate, "unit": "series/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), file=JSON_OUT, flush=True)


def gpu_eager_rate(dev: str, batch: int = 64, reps: int = 5):
    """Informational (SURVEY 2b: "the bar to beat = PyTorch eager / cuDNN / cuBLAS on the same B200"): the oracle's ConvNeXt-base
    CoordinateRegressor as stock PyTorch runs it on this GPU -- channels_last, bf16 autocast, batch 64, model forward only (no
    preprocessing, no crops).  Not the product path; nothing of this repo's kernels runs here."""
    import torch

    from oracle.convnext import make_model

    m = make_model("base", seed=0).to(dev).eval().to(memory_format=torch.channels_last)
    x = torch.randn(batch, 3, *IMAGE_SIZE, device=dev).contiguous(memory_format=torch.channels_last)
    with torch.no_grad(), torch.autocast("cuda", dtype=torch.bfloat16):
        for _ in range(3):
            m(x)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            m(x)
        e1.record()
        torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    del m, x
    torch.cuda.empty_cache()
    return batch / (ms * 1e-3), ms


def dump_outputs(out_dir: str, batch) -> None:
    """Write a pipeline.CropBatch as float32 .npy files (coords [B,5,2]; crops [S,5,128,128] and crops2 [S,5,256,256] of S =
    min(B, DUMP_SERIES) series drawn with a fixed seed), so that two builds run with the same arguments compare output for output."""
    import numpy as np
    import torch

    B = int(batch.coords.shape[0])
    rows = np.sort(np.random.default_rng(0).choice(B, size=min(B, DUMP_SERIES), replace=False))
    idx = torch.from_numpy(rows).to(batch.coords.device)
    os.makedirs(out_dir, exist_ok=True)
    for name, t in (("coords", batch.coords), ("crops", batch.crops[idx]), ("crops2", batch.crops2[idx])):
        np.save(os.path.join(out_dir, f"{name}.npy"), t.float().cpu().numpy())


# ----------------------------------------------------------------------------- clocks sampler
class ClockSampler(threading.Thread):
    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.stop_flag, self.max_mhz = index, [], set(), False, None

    def run(self):
        try:
            import pynvml as nv

            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
            names = {
                nv.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown",
                nv.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
                nv.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown",
                nv.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap",
            }
            while not self.stop_flag:
                self.samples.append(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
                time.sleep(0.1)
        except Exception as e:  # NVML unavailable: report that rather than invent numbers
            self.reasons.add(f"nvml_unavailable:{type(e).__name__}")

    def summary(self):
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons)}


# ----------------------------------------------------------------------------- B200 arm
def run_b200(args):
    import torch
    import torch.distributed as dist

    from spine_vision_b200 import _lib, ops, pipeline, synthetic
    from spine_vision_b200.cropping import LocalizationModel

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    assert torch.cuda.is_available(), "bench.py (impl b200) needs a GPU; there is no CPU fallback"
    torch.cuda.set_device(local_rank)
    dev = f"cuda:{local_rank}"
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device(dev))

    B = args.batch
    # synthetic data (per-rank seeds: weak scaling, every rank owns its own series): source volumes of config 1; only the
    # plan of each (the two planes around the middle Left-Right index + the K0 descriptor) is kept on the host
    from concurrent.futures import ThreadPoolExecutor

    from spine_vision_b200 import volumes as svb_volumes

    n_distinct = min(args.distinct or B, B)
    with ThreadPoolExecutor(max_workers=min(8, os.cpu_count() or 1)) as ex:
        base = list(ex.map(lambda sd: svb_volumes.plan_midplane(*synthetic.make_volume(sd)), [1000 * rank + k for k in range(n_distinct)]))
    series = svb_volumes.PinnedVolumes.from_plans([base[i % n_distinct] for i in range(B)])  # pinned staging, filled once outside the timed region
    assert all(tuple(hw) == SLICE_HW for hw in series.shapes)
    model = LocalizationModel(synthetic.random_state_dict("base", seed=0), dev, dtype=args.dtype, micro_batch=args.micro_batch)
    n_crops = B * 5
    streamer = pipeline.StreamedLocalizer(model, dev, CROP_DELTA_MM, CROP_SIZE, IMAGE_SIZE, SECOND_SIZE, chunk=args.stream_chunk or 2 * args.micro_batch)

    def step_resident(pool, times=None):
        return pipeline.localize_and_crop(pool, model, CROP_DELTA_MM, CROP_SIZE, IMAGE_SIZE, SECOND_SIZE, times=times)

    def gather(coords, crops):
        if world > 1:  # the path's one exchange: crops + coordinates to every rank (NCCL over NVLink)
            gc = torch.empty((world,) + tuple(coords.shape), dtype=coords.dtype, device=dev)
            gk = torch.empty((world,) + tuple(crops.shape), dtype=crops.dtype, device=dev)
            dist.all_gather_into_tensor(gc, coords)
            dist.all_gather_into_tensor(gk, crops)

    def e2e_steps(steps):
        # public host API: pinned host slices in, pinned host coords + crops out; inside a batch the H2D copy of chunk i+1
        # runs under the kernels of chunk i and results return on a third stream; across batches the next batch is started
        # before the previous one is collected (run_async, two output slots), so no batch begins in front of an idle GPU
        pending = None
        for s in range(steps):
            h = streamer.run_async(series, slot=s & 1)
            if world > 1:
                gather(h.device_coords, h.device_crops)
            if pending is not None:
                pending.result()
            pending = h
        pending.result()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    pool = series.resident_pool(dev)  # the isotropic middle slices of the batch, resident in HBM (K0 run once, outside the timed region)
    torch.cuda.synchronize()

    last = {}

    def resident_step():
        b = step_resident(pool)
        gather(b.coords, b.crops)
        last["batch"] = b

    for _ in range(args.warmup):
        resident_step()
    sampler = ClockSampler(local_rank)
    sampler.start()
    _lib.load().svb_launch_count(1)
    ms_total = timed(resident_step, args.steps)
    gpu_launches = int(_lib.load().svb_launch_count(1))
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last["batch"])
    del last["batch"]
    # roofline pass: same steps with a CUDA event pair around every launch of the model, and around
    # K1 / K3 with their (tiny) index tensors prebuilt so that no host work sits between the events
    times: dict = {}
    k1_ms = k3_ms = 0.0
    dpx = pipeline.mm_to_pixels(CROP_DELTA_MM, (0.3, 0.3))
    k3_idx = torch.arange(B, dtype=torch.int32).repeat_interleave(5).contiguous().to(dev)
    k3_delta = torch.tensor([dpx] * n_crops, dtype=torch.int32).to(dev)
    max_box = (dpx[2] + dpx[3], dpx[0] + dpx[1])
    k3_out = torch.empty((n_crops, *CROP_SIZE), dtype=torch.uint8, device=dev)   # preallocated: no allocator work between the events
    k3_out2 = torch.empty((n_crops, *SECOND_SIZE), dtype=torch.uint8, device=dev)
    k1_out = torch.empty((B, *IMAGE_SIZE), dtype=torch.uint8, device=dev)
    # K4 (classifier-input producer, SURVEY 8f row 4) is not part of series/s; it is timed here on this step's crops so that
    # its roofline sits next to K1 / K3: the crops are paired as (T2, T1) samples -> float32 [P, 3, 256, 256]
    k4_p = n_crops // 2
    k4_t2 = torch.arange(0, k4_p, dtype=torch.int32, device=dev)
    k4_t1 = torch.arange(k4_p, 2 * k4_p, dtype=torch.int32, device=dev)
    k4_out = torch.empty((k4_p, 3, *SECOND_SIZE), dtype=torch.float32, device=dev)
    k4_ms = 0.0
    ops.normalize_resize(pool, IMAGE_SIZE, out=k1_out)  # workspace allocation outside the events
    # K0 (+ the fused K0+K1 call of the end-to-end path) timed alone on resident source planes
    k0_vols = series.host.to(dev)
    k0_desc = series.chunk_descs(0, B).to(dev)
    k0_pool = ops.SlicePool(torch.empty_like(pool.data), pool.offs, pool.hw, list(pool.shapes))
    k0_ms = k01_ms = 0.0
    ops.midplane_resample_into(k0_vols, k0_desc, k0_pool)
    ops.midplane_normalize_resize(k0_vols, k0_desc, k0_pool, IMAGE_SIZE, out=k1_out)
    torch.cuda.synchronize()
    for _ in range(args.steps):
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
        ev[0].record()
        ops.midplane_resample_into(k0_vols, k0_desc, k0_pool)
        ev[1].record()
        ev[2].record()
        ops.midplane_normalize_resize(k0_vols, k0_desc, k0_pool, IMAGE_SIZE, out=k1_out)
        ev[3].record()
        torch.cuda.synchronize()
        k0_ms += ev[0].elapsed_time(ev[1])
        k01_ms += ev[2].elapsed_time(ev[3])
    del k0_vols, k0_desc, k0_pool
    for _ in range(args.steps):
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(6)]
        ev[0].record()
        planes = ops.normalize_resize(pool, IMAGE_SIZE, out=k1_out)
        ev[1].record()
        coords = model.predict_u8(planes, times)
        xy = coords.reshape(n_crops, 2)
        torch.cuda.synchronize()
        ev[2].record()
        ops.crop_resample(pool, k3_idx, xy, k3_delta, max_box, CROP_SIZE, SECOND_SIZE, out=k3_out, out2=k3_out2)
        ev[3].record()
        ev[4].record()
        ops.classifier_input(k3_out2, k4_t2, k4_t1, out=k4_out)
        ev[5].record()
        torch.cuda.synchronize()
        k1_ms += ev[0].elapsed_time(ev[1])
        k3_ms += ev[2].elapsed_time(ev[3])
        k4_ms += ev[4].elapsed_time(ev[5])
    # end-to-end pass through the public API: pinned host -> H2D -> kernels -> D2H
    e2e_steps(max(2, args.warmup))  # at least two: both output slots (pinned buffers) exist before the timed region
    ms_e2e = timed(lambda: e2e_steps(args.steps), 1)
    sampler.stop_flag = True
    sampler.join(timeout=2)

    if rank == 0:
        ms_step = ms_total / args.steps
        value = world * B / (ms_step * 1e-3)
        e2e = world * B / (ms_e2e / args.steps * 1e-3)
        gemm_flops, _ = model.engine.cost(B, *IMAGE_SIZE)
        peaks = {}
        try:
            peaks = json.loads((ROOT / "MEASURED_PEAKS.json").read_text())
        except Exception:
            pass
        peak_tf = float(peaks.get("bf16_tflops_sustained", 1400.0))
        peak_src = "MEASURED_PEAKS.json bf16_tflops_sustained (of measured)" if peaks else "fallback 1.4 PFLOP/s sustained (of fallback)"
        fused_ms = times.get("mlp_fused", 0.0) / args.steps  # mlp_fused_kernel (stages 0-1): timed as its own class, part of the GEMM class below
        gemm_only_ms = times.get("gemm", 0.0) / args.steps
        gemm_ms = gemm_only_ms + fused_ms
        achieved = gemm_flops / (gemm_ms * 1e-3) / 1e12 if gemm_ms > 0 else None
        hbm = float(peaks.get("hbm_gbs", 6650.0))
        traffic = traffic_gemm_only = None
        traffic_file = TRAFFIC_JSON if (ROOT / "profiles" / TRAFFIC_JSON).exists() else "r01e_gemm_traffic.json"
        try:  # DRAM bytes of the GEMM launches of one step, from the committed ncu --set full capture of the same kernels
            tj = json.loads((ROOT / "profiles" / traffic_file).read_text())
            if "gemm_dram_bytes_per_micro_batch" in tj:
                traffic = float(tj["gemm_dram_bytes_per_micro_batch"]) * B / float(tj["micro_batch"])
                # gemm_kernel alone (the capture names the fused-MLP launches)
                traffic_gemm_only = sum(float(e["dram_bytes"]) * e["launches_per_micro_batch"] for e in tj["per_launch"]
                                        if "fused" not in e["layer"]) * B / float(tj["micro_batch"])
            else:
                traffic = float(tj["gemm_dram_bytes_per_micro_batch_37"]) * B / 37.0
        except Exception:
            pass
        # algorithmic HBM bytes of the GEMMs of one step (A + W + out, + the residual read of fc2), 16-bit operands: what `traffic`
        # (measured DRAM bytes) is to be compared with
        gemm_bytes = 0.0
        fused_bytes = 0.0
        fused_flops = 0.0
        hh, ww = IMAGE_SIZE[0] // 4, IMAGE_SIZE[1] // 4
        for si, (cd, nd) in enumerate(zip(model.engine.dims, model.engine.depths)):
            if si > 0:
                hh, ww = hh // 2, ww // 2
                mm, kk = B * hh * ww, 4 * model.engine.dims[si - 1]
                gemm_bytes += 2.0 * (mm * kk + cd * kk + mm * cd)
            mm = B * hh * ww
            if cd in (128, 256) and os.environ.get("SVB_MLP_FUSED", "1") != "0":
                fused_flops += nd * 2.0 * 2.0 * mm * 4 * cd * cd
                # mlp_fused_kernel: the hidden activation never leaves the SM (A + W1 + W2 + residual in + out)
                gemm_bytes += nd * 2.0 * (mm * cd + 8 * cd * cd + 2 * mm * cd)
                fused_bytes += nd * 2.0 * (mm * cd + 8 * cd * cd + 2 * mm * cd)
            else:
                gemm_bytes += nd * 2.0 * ((mm * cd + 4 * cd * cd + mm * 4 * cd) + (mm * 4 * cd + 4 * cd * cd + 2 * mm * cd))
        dw_ms = times.get("dwconv_ln", 0.0) / args.steps
        dw_flops = 2.0 * 49 * B * sum(d * (IMAGE_SIZE[0] >> (2 + i)) * (IMAGE_SIZE[1] >> (2 + i)) * n
                                      for i, (d, n) in enumerate(zip(model.engine.dims, model.engine.depths)))
        dw_bytes = 2.0 * 2 * B * sum(d * (IMAGE_SIZE[0] >> (2 + i)) * (IMAGE_SIZE[1] >> (2 + i)) * n
                                     for i, (d, n) in enumerate(zip(model.engine.dims, model.engine.depths)))
        k1_bytes = B * (SLICE_HW[0] * SLICE_HW[1] * 4 + IMAGE_SIZE[0] * IMAGE_SIZE[1])
        k3_bytes = n_crops * (234 * 200 * 4 + CROP_SIZE[0] * CROP_SIZE[1] + SECOND_SIZE[0] * SECOND_SIZE[1])
        k4_bytes = k4_p * SECOND_SIZE[0] * SECOND_SIZE[1] * (2 + 3 * 4)  # two uint8 planes in, three float32 planes out
        model_ms = sum(times.get(k, 0.0) for k in ("stem", "dwconv_ln", "gemm", "mlp_fused", "ln_patchify", "head")) / args.steps
        dw_gbs = dw_bytes / (dw_ms * 1e-3) / 1e9 if dw_ms else None
        k1_gbs = k1_bytes / (k1_ms / args.steps * 1e-3) / 1e9 if k1_ms else None
        k3_gbs = k3_bytes / (k3_ms / args.steps * 1e-3) / 1e9 if k3_ms else None
        ceiling = peak_tf * 1e12 / (gemm_flops / B)  # series/s if the step were nothing but its GEMMs at the measured tensor peak (SURVEY 8d)
        line = {
            "metric": "series/sec", "value": value, "unit": "series/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": args.dtype,
            "data": f"synthetic ({n_distinct} distinct seeded series per rank; random-init convnext_base)",
            "config": workload_config(args),
            "crops_per_sec": value * 5,
            "clocks": sampler.summary(),
            "e2e": {"value": e2e, "unit": "series/s", "h2d_bytes_per_step": int(series.nbytes),
                    "d2h_bytes_per_step": int(B * 5 * (2 * 4 + CROP_SIZE[0] * CROP_SIZE[1] + SECOND_SIZE[0] * SECOND_SIZE[1])),
                    "ms_per_step": ms_e2e / args.steps,
                    "api": "pipeline.StreamedLocalizer.run_async(volumes.PinnedVolumes).result(): per series the two SOURCE planes (15x512x512 volume, "
                           "planes 7 and 8) + one K0 descriptor row go H2D in chunks on a copy stream, overlapped with K0+K1 (fused) / model / K3 "
                           "of the previous chunk; D2H on a third stream; batch k+1 is started before batch k is collected (two output slots); "
                           "index tables (offsets, shapes, crop deltas: 44 bytes per series) are uploaded once per batch geometry and reused"},
            "gpu_launches": int(gpu_launches),
            # the DOMINANT kernel: gemm_kernel (stage 2-3 MLP GEMMs and the downsample convs: half of the step); the GEMM class as a
            # whole (with the fused fc1-GELU-fc2 kernel of stages 0-1, whose bound is its GELU epilogue) is in `gemm_class`
            "roofline": {"kernel": "gemm_kernel (tcgen05 pointwise / downsample GEMMs, all launches of one step)", "bound": "tensor",
                         "achieved": (gemm_flops - fused_flops) / (gemm_only_ms * 1e-3) / 1e12 if gemm_only_ms else None, "peak": peak_tf,
                         "unit": "TFLOP/s",
                         "frac": (gemm_flops - fused_flops) / (gemm_only_ms * 1e-3) / 1e12 / peak_tf if gemm_only_ms else None,
                         "traffic": traffic_gemm_only, "algorithmic_bytes_per_step": gemm_bytes - fused_bytes,
                         "traffic_source": f"profiles/{traffic_file} (ncu --set full, per-shape dram bytes x launches)",
                         "peak_source": peak_src, "flops_per_step": gemm_flops - fused_flops, "ms_per_step": gemm_only_ms,
                         "timing": "CUDA event pair around every launch, separate pass over the same steps",
                         "whole_step_frac_of_tensor_ceiling": value / world / ceiling, "tensor_ceiling_series_per_s": ceiling,
                         "gemm_class": {"kernels": "gemm_kernel + mlp_fused_kernel", "ms_per_step": gemm_ms, "flops_per_step": gemm_flops,
                                        "achieved": achieved, "frac": (achieved / peak_tf) if achieved else None, "traffic": traffic,
                                        "algorithmic_bytes_per_step": gemm_bytes},
                         "mlp_fused_kernel": {"ms_per_step": fused_ms, "flops_per_step": fused_flops,
                                              "achieved": fused_flops / (fused_ms * 1e-3) / 1e12 if fused_ms else None,
                                              "frac": fused_flops / (fused_ms * 1e-3) / 1e12 / peak_tf if fused_ms else None,
                                              "note": "bound by its GELU epilogue (FMA / MUFU pipes), DESIGN.md section 4"}},
            "kernel_ms_per_step": {**{k: v / args.steps for k, v in times.items()}, "k1_normalize_resize": k1_ms / args.steps,
                                   "k3_crop_resample": k3_ms / args.steps, "k0_midplane_resample (e2e path only)": k0_ms / args.steps,
                                   "k0_k1_fused (e2e path only)": k01_ms / args.steps},
            "depthwise_kernel": {
                "kernel": "dwconv_rawtc_kernel + ln_stat_finalize_kernel (fp16: the 7x7 stencil as row-shifted tcgen05 MMAs, column sum by packed "
                          "shuffles) | dwconv_raw_kernel (bf16: FP32 pipe)",
                "ms_per_step": dw_ms, "useful_flops_per_step": dw_flops, "achieved_useful_tflops": dw_flops / (dw_ms * 1e-3) / 1e12 if dw_ms else None,
                "tensor_flops_issued_per_step": dw_flops / 49 * 7 * 16 * 7 if args.dtype == "fp16" else 0.0,
                "bound": "hbm (SURVEY 8d)", "hbm_bytes_per_step": dw_bytes, "achieved_gbs": dw_gbs, "hbm_peak_gbs": hbm,
                "frac_of_hbm": dw_gbs / hbm if dw_gbs else None,
                "note": "fp16: bound by the tensor core's shared-memory operand feed (7.5 KB per 128 x 112 x 16 MMA at ~87 B/clk) and the epilogue's "
                        "TMEM drain, DESIGN.md section 4; the FP32-pipe kernel it replaces ran at 0.16 of HBM"},
            "hbm_kernels": {
                "k1": {"bytes_per_step": k1_bytes, "achieved_gbs": k1_gbs, "peak_gbs": hbm, "frac": k1_gbs / hbm if k1_gbs else None},
                "k3": {"bytes_per_step": k3_bytes, "achieved_gbs": k3_gbs, "peak_gbs": hbm, "frac": k3_gbs / hbm if k3_gbs else None},
                "k4_classifier_input": {"bytes_per_step": k4_bytes, "ms_per_step": k4_ms / args.steps, "samples": k4_p,
                                        "achieved_gbs": k4_bytes / (k4_ms / args.steps * 1e-3) / 1e9 if k4_ms else None, "peak_gbs": hbm,
                                        "frac": k4_bytes / (k4_ms / args.steps * 1e-3) / 1e9 / hbm if k4_ms else None,
                                        "note": "outside the series/s timed region (its consumer is the classifier's data loader)"},
            },
        }
        if world == 1 and not args.no_eager_baseline:
            try:
                rate, ms = gpu_eager_rate(dev)
                line["gpu_eager_baseline"] = {"value": rate, "unit": "img/s (model forward only)", "ms_per_64": ms,
                                              "ours_img_per_s_model_only": B / (model_ms * 1e-3) if model_ms else None,
                                              "what": "oracle ConvNeXt-base CoordinateRegressor, stock PyTorch eager on this GPU: channels_last, bf16 autocast, batch 64 "
                                                      "(cuDNN depthwise conv + ATen LayerNorm + cuBLAS GEMMs); informational, SURVEY 2b's stated bar"}
            except Exception as e:  # noqa: BLE001 -- informational leg: never take the bench line down
                line["gpu_eager_baseline"] = {"unavailable": f"{type(e).__name__}: {e}"}
        if world == 1 and not args.no_cpu_baseline:
            rate, mean, cores = cpu_reference_rate(args.cpu_baseline_series, 2, 1)
            line["cpu_baseline"] = {"value": rate, "unit": "series/s", "cores": cores, "kind": "port",
                                    "sample": f"{args.cpu_baseline_series} series per pass of the same workload (BASELINE configs[0]: batch 32) through oracle/reference_path.py (batch-1 loop, reference-faithful), 2 timed passes after 1 warm-up"}
        print(json.dumps(line), file=JSON_OUT, flush=True)
    if world > 1:
        dist.destroy_process_group()


def _claim_stdout():
    """The JSON line must be the only thing on stdout: libraries (NCCL prints its version banner there) get stderr."""
    sys.stdout.flush()
    real = os.dup(1)
    os.dup2(2, 1)
    return os.fdopen(real, "w")


if __name__ == "__main__":
    a = parse()
    JSON_OUT = _claim_stdout()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_b200(a)
