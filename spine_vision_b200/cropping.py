"""Host-side mirror of the reference's hot-path module, backed by the sm_100a kernels.

Same names, argument meaning and error behaviour as
``spine_vision/datasets/classification/cropping.py`` and
``spine_vision/io/__init__.py`` (numpy in / numpy out, host memory), so the
reference's drivers (``spider.py:114-152``, ``phenikaa.py:178-208``) can import
these instead.  These per-call wrappers exist for drop-in compatibility; the
throughput path is the batched ``spine_vision_b200.pipeline.localize_and_crop``.

No function here falls back to the CPU: without the CUDA library and a B200
every call raises.
"""

from __future__ import annotations

import math
from dataclasses import dataclass
from pathlib import Path
from typing import Literal

import numpy as np
import torch

from . import ops

CropMode = Literal["horizontal", "rotated"]

ISOTROPIC_SPACING = (0.3, 0.3, 0.3)  # cropping.py:22
DEFAULT_IVD_CENTERS = {0: (0.5, 0.25), 1: (0.5, 0.35), 2: (0.5, 0.45), 3: (0.5, 0.55), 4: (0.5, 0.65)}  # cropping.py:28-34

_DEFAULT_DEVICE = "cuda:0"


def get_center_fallback_locations() -> dict[int, tuple[float, float]]:
    """cropping.py:486-492."""
    return DEFAULT_IVD_CENTERS.copy()


def mm_to_pixels(delta_mm, spacing) -> tuple[int, int, int, int]:
    """cropping.py:149-169 -- pure host arithmetic (Python ``round`` = banker's rounding)."""
    row_spacing, col_spacing = spacing
    left_mm, right_mm, top_mm, bottom_mm = delta_mm
    return (
        int(round(left_mm / col_spacing)),
        int(round(right_mm / col_spacing)),
        int(round(top_mm / row_spacing)),
        int(round(bottom_mm / row_spacing)),
    )


def get_rotation_angles(ivd_locations: dict, image_shape: tuple[int, int], last_disc_angle_boost: float = 1.0) -> dict:
    """cropping.py:172-255 -- host arithmetic on five points (same NumPy calls as the reference): tangent of the disc
    chain by forward / central differences, the lowest disc from a 3-point quadratic fit, negated to flatten the tilt."""
    if len(ivd_locations) < 2:
        return {level: 0.0 for level in ivd_locations}
    h, w = image_shape
    points = sorted(((lvl, nx * w, ny * h) for lvl, (nx, ny) in ivd_locations.items()), key=lambda p: p[2])
    n = len(points)
    angles: dict = {}
    for i, (lvl, px, py) in enumerate(points):
        if i == 0:
            dx, dy = points[1][1] - px, points[1][2] - py
            dxdy = dx / dy if dy != 0 else 0.0
        elif i == n - 1:
            if n >= 3:
                last = points[-3:]
                a, b, _ = np.polyfit(np.array([p[2] for p in last]), np.array([p[1] for p in last]), deg=2)
                dxdy = 2 * a * py + b
            else:
                dx, dy = px - points[i - 1][1], py - points[i - 1][2]
                dxdy = dx / dy if dy != 0 else 0.0
        else:
            dx, dy = points[i + 1][1] - points[i - 1][1], points[i + 1][2] - points[i - 1][2]
            dxdy = dx / dy if dy != 0 else 0.0
        angle_deg = float(np.degrees(np.arctan(dxdy)))
        if i == n - 1:
            angle_deg *= last_disc_angle_boost
        angles[lvl] = -angle_deg
    return angles


def inverse_rotation(cx: int, cy: int, angle_deg: float) -> list[float]:
    """The 2x3 map cv2.warpAffine actually applies for ``cv2.getRotationMatrix2D((cx, cy), angle, 1.0)``
    (cropping.py:289-301): OpenCV builds the forward matrix in double and inverts it in place; the six doubles are
    handed to K3, so the device never evaluates a sine."""
    a = angle_deg * (math.pi / 180.0)  # OpenCV: angle *= CV_PI/180 (one multiply by the constant)
    alpha, beta = math.cos(a), math.sin(a)
    m = [alpha, beta, (1 - alpha) * cx - beta * cy, -beta, alpha, beta * cx + (1 - alpha) * cy]
    d = m[0] * m[4] - m[1] * m[3]
    d = 1.0 / d if d != 0 else 0.0
    a11, a22 = m[4] * d, m[0] * d
    m[0] = a11
    m[1] *= -d
    m[3] *= -d
    m[4] = a22
    b1 = -m[0] * m[2] - m[1] * m[5]
    b2 = -m[3] * m[2] - m[4] * m[5]
    m[2], m[5] = b1, b2
    return m


def normalize_to_uint8(arr: np.ndarray, device: str = _DEFAULT_DEVICE) -> np.ndarray:
    """io/__init__.py:15-30 on the GPU (K1 with an identity resize).

    Min-max is global and the map is elementwise, so the array is processed as a flat
    ``[rows, 4096]`` sheet padded with copies of its first element (which cannot move
    the minimum or the maximum)."""
    a = np.asarray(arr)
    if a.size == 0:
        raise ValueError("zero-size array to reduction operation minimum which has no identity")  # numpy's error
    flat = a.astype(np.float32).ravel()
    cols = 4096 if flat.size >= 4096 else (flat.size + 3) // 4 * 4
    rows = (flat.size + cols - 1) // cols
    sheet = np.full(rows * cols, flat[0], dtype=np.float32)
    sheet[: flat.size] = flat
    pool = ops.SlicePool.from_numpy([sheet.reshape(rows, cols)], device)
    out = ops.normalize_resize(pool, (rows, cols))
    return out.cpu().numpy().ravel()[: flat.size].reshape(a.shape)


def resize_with_padding(image: np.ndarray, target_size: tuple[int, int], device: str = _DEFAULT_DEVICE) -> np.ndarray:
    """cropping.py:104-146 for uint8 input: letterboxed cv2-compatible INTER_LINEAR resize (K3 on
    the whole image with the per-crop normalisation switched off)."""
    img = np.asarray(image)
    if img.dtype != np.uint8:
        raise TypeError("resize_with_padding: the GPU path takes uint8 images (the reference's own call site, "
                        "cropping.py:354, always passes uint8)")
    h, w = img.shape[:2]
    pool = ops.SlicePool.from_numpy([img.astype(np.float32)], device)
    dev = pool.data.device
    idx = torch.zeros(1, dtype=torch.int32, device=dev)
    xy = torch.zeros((1, 2), dtype=torch.float32, device=dev)
    delta = torch.tensor([[0, w, 0, h]], dtype=torch.int32, device=dev)
    crops, _, _ = ops.crop_resample(pool, idx, xy, delta, (h, w), target_size, None, normalize=False)
    return crops[0].cpu().numpy()


def crop_region_horizontal(image, center_x, center_y, crop_size, crop_delta, device: str = _DEFAULT_DEVICE) -> np.ndarray:
    """cropping.py:316-354."""
    ctx = CropContext(np.asarray(image), {0: (center_x, center_y)}, tuple(crop_size), tuple(crop_delta), "horizontal", device=device)
    return ctx.crop(0)


@dataclass
class CropContext:
    """cropping.py:357-404.  The image is staged to the device once; ``crop`` is one K3 launch,
    ``crop_all`` cuts every requested level in a single launch."""

    image: np.ndarray
    ivd_locations: dict
    crop_size: tuple
    crop_delta_px: tuple
    mode: CropMode = "horizontal"
    last_disc_angle_boost: float = 1.0
    rotation_angles: dict | None = None
    device: str = _DEFAULT_DEVICE

    def __post_init__(self) -> None:
        if self.mode not in ("horizontal", "rotated"):
            raise ValueError(f"unknown crop mode {self.mode!r}")
        if self.mode == "rotated" and self.rotation_angles is None:  # cropping.py:369-375
            h, w = np.asarray(self.image).shape[:2]
            self.rotation_angles = get_rotation_angles(self.ivd_locations, (h, w), self.last_disc_angle_boost)
        self._pool = None

    def _ensure_pool(self):
        if self._pool is None:
            self._pool = ops.SlicePool.from_numpy([np.asarray(self.image)], self.device)
        return self._pool

    def crop_all(self, level_indices) -> dict[int, np.ndarray]:
        levels = [i for i in level_indices if i in self.ivd_locations]
        if not levels:
            return {}
        pool = self._ensure_pool()
        dev = pool.data.device
        h, w = pool.shapes[0]
        xy_host = [[float(self.ivd_locations[i][0]), float(self.ivd_locations[i][1])] for i in levels]
        xy = torch.tensor(xy_host, dtype=torch.float64).to(dev)  # the Python floats the caller gave: int(x * w) sees the same double
        idx = torch.zeros(len(levels), dtype=torch.int32, device=dev)
        l, r, t, b = (int(v) for v in self.crop_delta_px)
        delta = torch.tensor([[l, r, t, b]] * len(levels), dtype=torch.int32).to(dev)
        inv = None
        if self.mode == "rotated" and self.rotation_angles:  # cropping.py:390-399
            # centre as the reference computes it: int(x * w) on the Python floats it was given
            rows = [inverse_rotation(int(self.ivd_locations[i][0] * w), int(self.ivd_locations[i][1] * h),
                                     self.rotation_angles.get(i, 0.0)) for i in levels]
            inv = torch.tensor(rows, dtype=torch.float64).to(dev)
        crops, _, _ = ops.crop_resample(pool, idx, xy, delta, (min(h, max(t + b, 1)), min(w, max(l + r, 1))),
                                        self.crop_size, None, inv_affine=inv)
        host = crops.cpu().numpy()
        return {lvl: host[k] for k, lvl in enumerate(levels)}

    def crop(self, level_idx: int) -> np.ndarray | None:
        if level_idx not in self.ivd_locations:
            return None
        return self.crop_all([level_idx])[level_idx]


class LocalizationModel:
    """What ``load_localization_model`` returns: the reference hands back an ``nn.Module`` in eval
    mode; this is its inference-only device twin (``eval()`` / ``to()`` are accepted no-ops)."""

    def __init__(self, state_dict, device: str = _DEFAULT_DEVICE, dtype: str | None = None, micro_batch: int = 64):
        import os

        # fp16 operands are the default: they hold the 0.5 px gate on trained-like weights (0.18 px; bf16 measures 1.0 px), at the
        # same tensor-pipe rate.  The reference trains under fp16 autocast (trainers/base.py:229-237), so a real checkpoint's
        # activations are in fp16 range by construction; conversions saturate.  dtype="bf16" / SPINE_B200_DTYPE=bf16 opt in.
        dtype = dtype or os.environ.get("SPINE_B200_DTYPE", "fp16")
        self.device = device
        self.engine = ops.LocalizationEngine(state_dict, device, dtype, micro_batch)
        self.num_levels = self.engine.num_levels

    def eval(self):
        return self

    def to(self, *_a, **_k):
        return self

    def predict_u8(self, planes_u8: torch.Tensor, times: dict | None = None, out: torch.Tensor | None = None) -> torch.Tensor:
        return self.engine.forward(planes_u8, times, out)

    def predict_u8_stages(self, planes_u8: torch.Tensor) -> tuple[torch.Tensor, list[torch.Tensor]]:
        """``predict_u8`` plus the residual stream after each of the four stages, ``[B, H / 2^(s+2), W / 2^(s+2), C_s]`` in the
        model's 16-bit dtype (stage-level parity tests and profiling)."""
        e = self.engine
        B, H, W = planes_u8.shape
        dt = torch.float16 if e.dtype in ("fp16", "float16", "half") else torch.bfloat16
        stages = [torch.empty((B, H >> (s + 2), W >> (s + 2), e.dims[s]), dtype=dt, device=planes_u8.device) for s in range(4)]
        return e.forward(planes_u8, stage_out=stages), stages

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        """``CoordinateRegressor.forward`` (generic.py:380-391) for callers that build the input themselves:
        ``x`` = ``[B,3,H,W]`` float, /255 and ImageNet-normalised (any device / float dtype) -> ``[B, num_levels, 2]`` float32
        on the model's device.  Inference only (no autograd graph)."""
        if x.dim() != 4 or x.shape[1] != 3:
            raise ValueError(f"expected a [B,3,H,W] tensor, got {tuple(x.shape)}")
        xd = x.detach().to(self.device, torch.float32).contiguous()
        return self.engine.forward_tensor(xd)

    __call__ = forward

    def predict(self, x: torch.Tensor) -> torch.Tensor:
        """``BaseModel.predict`` (base.py:80-81 / generic.py:393-395): same as ``forward`` in eval mode."""
        return self.forward(x)


def load_localization_model(model_path: Path, variant: str, device: str, dtype: str | None = None) -> LocalizationModel:
    """cropping.py:407-441 -- same checkpoint format (``torch.save`` dict whose
    ``"model_state_dict"`` holds the 348 ``backbone.*`` / ``head.*`` tensors,
    trainers/base.py:695-706), strict key check, weights repacked for the tensor cores."""
    checkpoint = torch.load(model_path, map_location="cpu", weights_only=False)
    return LocalizationModel(checkpoint["model_state_dict"], device, dtype)


def predict_ivd_locations(model: LocalizationModel, image: np.ndarray, device: str, image_size: tuple[int, int]):
    """cropping.py:444-483 -- one series, batch 1 (drop-in signature).  K1 then the model, one D2H."""
    pool = ops.SlicePool.from_numpy([np.asarray(image)], device)
    planes = ops.normalize_resize(pool, image_size)
    out = model.predict_u8(planes).cpu().numpy()[0]
    return {i: (float(out[i, 0]), float(out[i, 1])) for i in range(out.shape[0])}
