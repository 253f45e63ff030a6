"""Batched device operators over ``libspine_b200.so``.

PyTorch is plumbing here (device memory, streams, pinned staging); every
operator is one C-ABI call into hand-written sm_100a kernels.  Nothing in this
module computes on the CPU and nothing imports ``oracle/``.
"""

from __future__ import annotations

import ctypes as C
from dataclasses import dataclass

import numpy as np
import torch

from . import _lib


def _require_cuda(device) -> torch.device:
    dev = torch.device(device)
    if dev.type != "cuda" or not torch.cuda.is_available():
        raise RuntimeError(
            f"spine_vision_b200 needs a CUDA (B200, sm_100) device, got {device!r}; there is no CPU fallback"
        )
    return dev


def _device_of(args, kwargs):
    for a in list(args) + list(kwargs.values()):
        if isinstance(a, torch.Tensor) and a.is_cuda:
            return a.device
        d = getattr(a, "data", None)
        if isinstance(d, torch.Tensor) and d.is_cuda:  # a SlicePool
            return d.device
        d = getattr(a, "device", None)
        if isinstance(d, torch.device) and d.type == "cuda":  # a LocalizationEngine
            return d
    return None


def _on_device(fn):
    """Run ``fn`` with the CUDA device of its data current: the library launches on the CURRENT device's current stream and keeps
    per-device kernel attributes, so an op on ``cuda:1`` tensors must not run while ``cuda:0`` is current (ADVICE r01)."""
    import functools

    @functools.wraps(fn)
    def wrapper(*args, **kwargs):
        dev = _device_of(args, kwargs)
        if dev is None or dev.index is None or dev.index == torch.cuda.current_device():
            return fn(*args, **kwargs)
        with torch.cuda.device(dev):
            return fn(*args, **kwargs)

    return wrapper


@dataclass
class SlicePool:
    """A ragged batch of float32 slices resident in HBM: one flat pool plus
    per-slice element offsets and (H, W).  Offsets are 4-element aligned so each
    slice starts on a 16-byte boundary (128-bit loads)."""

    data: torch.Tensor  # float32 [total]
    offs: torch.Tensor  # int64 [B] (device)
    hw: torch.Tensor  # int32 [B,2] (device)
    shapes: list  # host copy [(h, w)]
    h2d_bytes: int = 0
    pixel_kind: torch.Tensor | None = None  # int32 [B] (device) SVB_PIXEL_* per slice, None = all float32 (rotated crop mode only)

    @property
    def n(self) -> int:
        return len(self.shapes)

    @property
    def max_hw(self) -> tuple[int, int]:
        return max(s[0] for s in self.shapes), max(s[1] for s in self.shapes)

    @staticmethod
    def layout(shapes):
        offs, o = [], 0
        for h, w in shapes:
            offs.append(o)
            o += (h * w + 3) // 4 * 4
        return offs, o

    @classmethod
    def pin(cls, slices):
        """Stage host slices into one pinned float32 buffer (done once; outside any timed region)."""
        shapes = [tuple(int(v) for v in s.shape) for s in slices]
        offs, total = cls.layout(shapes)
        host = torch.empty(max(total, 4), dtype=torch.float32).pin_memory()
        hv = host.numpy()
        for s, o in zip(slices, offs):
            # spine_vision/io/__init__.py:26: arr.astype(np.float32) happens on the host, exactly as the reference
            hv[o : o + s.size] = np.asarray(s).astype(np.float32, copy=False).ravel()
        return host, offs, shapes

    @classmethod
    def from_pinned(cls, host: torch.Tensor, offs, shapes, device="cuda:0") -> "SlicePool":
        dev = _require_cuda(device)
        data = host.to(dev, non_blocking=True)
        meta = torch.tensor(offs, dtype=torch.int64).pin_memory().to(dev, non_blocking=True)
        hw = torch.tensor(shapes, dtype=torch.int32).reshape(-1, 2).pin_memory().to(dev, non_blocking=True)
        return cls(data, meta, hw, list(shapes), h2d_bytes=host.numel() * 4 + meta.numel() * 8 + hw.numel() * 4)

    @staticmethod
    def kind_of(dtype) -> int:
        """SVB_PIXEL_* of a NumPy dtype: how ``cv2.warpAffine`` treats a slice of that type (cropping.py:292-301)."""
        dt = np.dtype(dtype)
        return {np.dtype(np.int16): _lib.PIXEL_INT16, np.dtype(np.uint16): _lib.PIXEL_UINT16,
                np.dtype(np.uint8): _lib.PIXEL_UINT8}.get(dt, _lib.PIXEL_FLOAT)

    def set_pixel_kinds(self, kinds) -> "SlicePool":
        kinds = [int(k) for k in kinds]
        assert len(kinds) == self.n
        self.pixel_kind = torch.tensor(kinds, dtype=torch.int32).to(self.data.device) if any(kinds) else None
        return self

    @classmethod
    def from_numpy(cls, slices, device="cuda:0") -> "SlicePool":
        """Slices keep what the reference's rotated crop mode needs of their dtype (int16 / uint16 / uint8 slices are warped
        in that type by OpenCV); the values themselves travel as float32 (io/__init__.py:26)."""
        _require_cuda(device)
        host, offs, shapes = cls.pin(slices)
        return cls.from_pinned(host, offs, shapes, device).set_pixel_kinds([cls.kind_of(np.asarray(s).dtype) for s in slices])

    @classmethod
    def from_device_batch(cls, batch: torch.Tensor) -> "SlicePool":
        """Uniform batch already on the device: float32 [B,H,W] (H*W % 4 == 0 or B == 1)."""
        assert batch.is_cuda and batch.dtype == torch.float32 and batch.dim() == 3 and batch.is_contiguous()
        b, h, w = batch.shape
        assert (h * w) % 4 == 0 or b == 1, "uniform device batches need H*W % 4 == 0"
        offs = torch.arange(b, dtype=torch.int64, device=batch.device) * (h * w)
        hw = torch.tensor([[h, w]] * b, dtype=torch.int32, device=batch.device)
        return cls(batch.reshape(-1), offs, hw, [(h, w)] * b)


class _Workspace:
    """Grow-only device scratch, one per (device, tag)."""

    _bufs: dict = {}

    @classmethod
    def get(cls, tag: str, nbytes: int, device) -> torch.Tensor:
        key = (tag, str(device))
        buf = cls._bufs.get(key)
        if buf is None or buf.numel() < nbytes:
            buf = torch.empty(max(nbytes, 1024) + 1024, dtype=torch.uint8, device=device)
            cls._bufs[key] = buf
        return buf


class PinnedCache:
    """Grow-only pinned host staging buffers by tag: ``cudaHostAlloc`` costs milliseconds per call, more than the kernels a
    chunk of a dataset run feeds.  A buffer is handed out again only by the same tag, so a caller that double-buffers uses
    two tags.  Not thread-safe per tag (each pipeline stage owns its tags)."""

    _bufs: dict = {}

    @classmethod
    def get(cls, tag: str, nelem: int, dtype=torch.float32) -> torch.Tensor:
        buf = cls._bufs.get(tag)
        if buf is None or buf.numel() < nelem or buf.dtype != dtype:
            buf = torch.empty(max(int(nelem), 4), dtype=dtype)
            if torch.cuda.is_available():
                buf = buf.pin_memory()
            cls._bufs[tag] = buf
        return buf[: max(int(nelem), 4)]


def _aligned_ptr(buf: torch.Tensor, align: int = 1024) -> tuple[int, int]:
    p = buf.data_ptr()
    a = (p + align - 1) // align * align
    return a, buf.numel() - (a - p)


@_on_device
def normalize_resize(pool: SlicePool, out_hw=(512, 512), out: torch.Tensor | None = None, return_minmax: bool = False):
    """K1: per-slice global min-max -> uint8 (truncating) -> Pillow antialiased bilinear resize.
    Device mirror of ``normalize_to_uint8`` (io/__init__.py:15-30) + ``transforms.Resize``
    (cropping.py:463-472).  Returns uint8 ``[B, out_h, out_w]`` (one plane; R=G=B)."""
    lib = _lib.load()
    dev = pool.data.device
    B = pool.n
    oh, ow = int(out_hw[0]), int(out_hw[1])
    if out is None:
        out = torch.empty((B, oh, ow), dtype=torch.uint8, device=dev)
    minmax = torch.empty((B, 2), dtype=torch.float32, device=dev) if return_minmax else None
    if B == 0:
        return (out, minmax) if return_minmax else out
    mh, mw = pool.max_hw
    need = lib.svb_k1_workspace_bytes(B, mh, mw, oh, ow)
    ws = _Workspace.get("k1", need, dev)
    wp, wn = _aligned_ptr(ws, 256)
    _lib.check(lib.svb_k1_normalize_resize(pool.data.data_ptr(), pool.offs.data_ptr(), pool.hw.data_ptr(), B, mh, mw, oh, ow,
                                           out.data_ptr(), _lib.ptr(minmax), wp, wn, _lib.current_stream()))
    return (out, minmax) if return_minmax else out


@_on_device
def midplane_normalize_resize(vols_d: torch.Tensor, desc_d: torch.Tensor, pool: SlicePool, out_hw=(512, 512),
                              out: torch.Tensor | None = None, return_minmax: bool = False):
    """K0 + K1 in one call (``svb_k01_midplane_normalize_resize``): ``vols_d`` float32 source planes and ``desc_d`` the
    ``svb_k0_series`` rows (both on the device, see ``volumes.PinnedVolumes``); ``pool`` is the EMPTY destination pool of the
    isotropic middle planes (offsets / shapes from the plans), filled here and kept for K3.  Returns the uint8 model planes."""
    lib = _lib.load()
    dev = pool.data.device
    B = pool.n
    oh, ow = int(out_hw[0]), int(out_hw[1])
    if out is None:
        out = torch.empty((B, oh, ow), dtype=torch.uint8, device=dev)
    minmax = torch.empty((B, 2), dtype=torch.float32, device=dev) if return_minmax else None
    if B == 0:
        return (out, minmax) if return_minmax else out
    assert out.is_cuda and out.dtype == torch.uint8 and out.is_contiguous() and out.numel() == B * oh * ow
    mh, mw = pool.max_hw
    need = lib.svb_k01_workspace_bytes(B, mh, mw, oh, ow)
    ws = _Workspace.get("k01", need, dev)
    wp, wn = _aligned_ptr(ws, 256)
    _lib.check(lib.svb_k01_midplane_normalize_resize(vols_d.data_ptr(), desc_d.data_ptr(), B, mh, mw, pool.data.data_ptr(),
                                                     pool.offs.data_ptr(), pool.hw.data_ptr(), oh, ow, out.data_ptr(), _lib.ptr(minmax),
                                                     wp, wn, _lib.current_stream()))
    return (out, minmax) if return_minmax else out


@_on_device
def midplane_resample_into(vols_d: torch.Tensor, desc_d: torch.Tensor, pool: SlicePool) -> SlicePool:
    """K0 alone (``svb_k0_midplane_resample``) into an existing pool -- the no-model (centre fallback) branch of the streamed
    driver."""
    lib = _lib.load()
    if pool.n == 0:
        return pool
    mh, mw = pool.max_hw
    need = lib.svb_k0_workspace_bytes(pool.n, mh, mw)
    ws = _Workspace.get("k0", need, pool.data.device)
    _lib.check(lib.svb_k0_midplane_resample(vols_d.data_ptr(), desc_d.data_ptr(), pool.n, mh, mw, pool.data.data_ptr(), ws.data_ptr(),
                                            ws.numel(), _lib.current_stream()))
    return pool


@_on_device
def normalize_u8(pool: SlicePool, out: torch.Tensor | None = None, return_minmax: bool = False):
    """``normalize_to_uint8`` (io/__init__.py:15-30) over a ragged batch without resizing: returns a flat uint8 pool with the
    same element offsets as ``pool`` (slice b = ``out[offs[b] : offs[b] + h*w].view(h, w)``).  Device mirror of the
    localization dataset builder's per-image normalisation (datasets/localization.py:147-151, 262-267)."""
    lib = _lib.load()
    dev = pool.data.device
    B = pool.n
    if out is None:
        out = torch.empty(pool.data.numel(), dtype=torch.uint8, device=dev)
    assert out.dtype == torch.uint8 and out.is_contiguous() and out.numel() >= pool.data.numel()
    minmax = torch.empty((B, 2), dtype=torch.float32, device=dev) if return_minmax else None
    if B == 0:
        return (out, minmax) if return_minmax else out
    mh, mw = pool.max_hw
    need = lib.svb_normalize_u8_workspace_bytes(B)
    ws = _Workspace.get("norm", need, dev)
    _lib.check(lib.svb_normalize_u8(pool.data.data_ptr(), pool.offs.data_ptr(), pool.hw.data_ptr(), B, mh, mw, out.data_ptr(),
                                    _lib.ptr(minmax), ws.data_ptr(), ws.numel(), _lib.current_stream()))
    return (out, minmax) if return_minmax else out


@_on_device
def crop_resample(pool: SlicePool, slice_idx: torch.Tensor, xy: torch.Tensor, delta_px: torch.Tensor, max_box_hw,
                  crop_size=(128, 128), second_size=(256, 256), return_geom: bool = False, normalize: bool = True,
                  out: torch.Tensor | None = None, out2: torch.Tensor | None = None, inv_affine: torch.Tensor | None = None):
    """K3: one crop per (slice_idx, xy, delta_px) row.  Device mirror of
    ``CropContext.crop`` -> ``crop_region_horizontal`` (cropping.py:316-404) and, for the
    second output, the classifier's ``Resize`` (training/datasets/classification.py:247-278).
    ``xy`` is float32 (model output) or float64 (centres that are Python floats in the reference: the fallback table).
    ``inv_affine`` (float64 ``[N,6]`` on the device, from ``cropping.inverse_rotation``) switches on the rotated crop
    mode (``crop_region_rotated``, cropping.py:258-313).
    Returns ``(crops u8 [N,ch,cw], crops2 u8 [N,oh2,ow2] | None, geom int32 [N,8] | None)``."""
    lib = _lib.load()
    dev = pool.data.device
    N = int(xy.shape[0])
    ch, cw = int(crop_size[0]), int(crop_size[1])
    crops = out if out is not None else torch.empty((N, ch, cw), dtype=torch.uint8, device=dev)
    assert crops.is_contiguous() and crops.dtype == torch.uint8 and crops.numel() == N * ch * cw
    crops2 = None
    oh2 = ow2 = 0
    if second_size is not None:
        oh2, ow2 = int(second_size[0]), int(second_size[1])
        crops2 = out2 if out2 is not None else torch.empty((N, oh2, ow2), dtype=torch.uint8, device=dev)
        assert crops2.is_contiguous() and crops2.dtype == torch.uint8 and crops2.numel() == N * oh2 * ow2
    geom = torch.empty((N, 8), dtype=torch.int32, device=dev) if return_geom else None
    if N == 0:
        return crops, crops2, geom
    assert slice_idx.dtype == torch.int32 and xy.dtype in (torch.float32, torch.float64) and delta_px.dtype == torch.int32
    flags = (0 if normalize else 1) | (2 if xy.dtype == torch.float64 else 0)  # SVB_K3_NO_NORMALIZE, SVB_K3_XY_F64
    assert slice_idx.is_contiguous() and xy.is_contiguous() and delta_px.is_contiguous()
    need = lib.svb_k3_workspace_bytes(ch, cw, oh2, ow2)
    ws = _Workspace.get("k3", need, dev)
    wp, wn = _aligned_ptr(ws, 256)
    if inv_affine is not None:
        assert inv_affine.dtype == torch.float64 and inv_affine.is_contiguous() and tuple(inv_affine.shape) == (N, 6)
    _lib.check(lib.svb_k3_crop_resample_rotated(pool.data.data_ptr(), pool.offs.data_ptr(), pool.hw.data_ptr(), slice_idx.data_ptr(),
                                                xy.data_ptr(), delta_px.data_ptr(), _lib.ptr(inv_affine),
                                                _lib.ptr(pool.pixel_kind) if inv_affine is not None else None, N, int(max_box_hw[0]),
                                                int(max_box_hw[1]), ch, cw, crops.data_ptr(), oh2, ow2, _lib.ptr(crops2),
                                                _lib.ptr(geom), flags, wp, wn, _lib.current_stream()))
    return crops, crops2, geom


_OUT_DTYPES = {torch.float32: _lib.SVB_F32, torch.bfloat16: _lib.SVB_BF16, torch.float16: _lib.SVB_FP16}


@_on_device
def classifier_input(planes: torch.Tensor, t2_idx: torch.Tensor, t1_idx: torch.Tensor, normalize: bool = True,
                     dtype: torch.dtype = torch.float32, mean=None, std=None, out: torch.Tensor | None = None) -> torch.Tensor:
    """K4: ``[T2, T1, T2]`` stack + ``ToTensor`` + ``Normalize`` for a batch of (patient, level) samples from the resized
    uint8 planes K3 produced.  Device mirror of ``construct_3channel`` + the non-augmenting transform of
    ``ClassificationDataset`` (training/datasets/classification.py:40-68, 247-278).
    ``planes`` uint8 ``[N,H,W]``; ``t2_idx`` / ``t1_idx`` int32 ``[P]`` (-1 = series missing).  Returns ``[P,3,H,W]``."""
    lib = _lib.load()
    dev = planes.device
    assert planes.dtype == torch.uint8 and planes.dim() == 3 and planes.is_contiguous()
    assert t2_idx.dtype == torch.int32 and t1_idx.dtype == torch.int32 and t2_idx.shape == t1_idx.shape
    P, H, W = int(t2_idx.shape[0]), int(planes.shape[1]), int(planes.shape[2])
    if out is None:
        out = torch.empty((P, 3, H, W), dtype=dtype, device=dev)
    assert out.is_contiguous() and out.dtype == dtype and out.numel() == P * 3 * H * W
    mean_c = (C.c_float * 3)(*mean) if mean is not None else None
    std_c = (C.c_float * 3)(*std) if std is not None else None
    for p0 in range(0, P, 65535):  # grid.y limit of one launch
        n = min(65535, P - p0)
        _lib.check(lib.svb_k4_classifier_input(planes.data_ptr(), t2_idx[p0:].data_ptr(), t1_idx[p0:].data_ptr(), n, H, W,
                                               C.addressof(mean_c) if mean_c is not None else None,
                                               C.addressof(std_c) if std_c is not None else None, int(bool(normalize)),
                                               _OUT_DTYPES[dtype], out[p0:].data_ptr(), _lib.current_stream()))
    return out


class LocalizationEngine:
    """Owns one ``svb_model`` handle: the ``CoordinateRegressor`` forward
    (training/models/generic.py:389-391) as sm_100a kernels.  Input is the K1 output
    (uint8 ``[B,H,W]``); /255 and ImageNet mean/std live in the folded stem."""

    def __init__(self, state_dict, device="cuda:0", dtype: str = "bf16", micro_batch: int = 32):
        self.device = _require_cuda(device)
        self.dtype = dtype
        self.micro_batch = int(micro_batch)
        lib = _lib.load()
        keep, descs = [], (_lib.WeightDesc * len(state_dict))()
        for i, (name, t) in enumerate(state_dict.items()):
            a = t.detach().to("cpu", torch.float32).contiguous()
            keep.append(a)
            descs[i].name = name.encode()
            descs[i].data = a.data_ptr()
            descs[i].ndim = a.dim()
            for k in range(4):
                descs[i].shape[k] = a.shape[k] if k < a.dim() else 1
        handle = C.c_void_p()
        with torch.cuda.device(self.device):
            _lib.check(lib.svb_model_create(C.byref(handle), descs, len(state_dict), _lib.DTYPES[dtype]))
        self._h = handle
        info = (C.c_int32 * 10)()
        _lib.check(lib.svb_model_info(self._h, C.byref(info)))
        self.num_levels, self.num_outputs = int(info[0]), int(info[1])
        self.dims, self.depths = tuple(info[2:6]), tuple(info[6:10])

    def __del__(self):
        h, self._h = getattr(self, "_h", None), None
        if h:
            try:
                _lib.load().svb_model_destroy(h)
            except Exception:
                pass

    def cost(self, B: int, H: int, W: int) -> tuple[float, int]:
        fl, n = C.c_double(), C.c_int64()
        _lib.check(_lib.load().svb_model_cost(self._h, B, H, W, C.byref(fl), C.byref(n)))
        return fl.value, n.value

    @_on_device
    def forward(self, u8: torch.Tensor, times: dict | None = None, out: torch.Tensor | None = None,
                stage_out: list[torch.Tensor] | None = None) -> torch.Tensor:
        """uint8 [B,H,W] on the device -> float32 [B, num_levels, 2] in [0,1].  ``stage_out`` (tests, profiling): up to four
        device tensors ``[B, H / 2^(s+2), W / 2^(s+2), dims[s]]`` of the model dtype that receive the residual stream after the
        last block of stage s (``svb_model_forward_stages``: the same kernels and schedule as without it)."""
        assert u8.is_cuda and u8.dtype == torch.uint8 and u8.dim() == 3 and u8.is_contiguous()
        lib = _lib.load()
        B, H, W = u8.shape
        coords = out if out is not None else torch.empty((B, self.num_levels, self.num_outputs), dtype=torch.float32, device=u8.device)
        assert coords.is_contiguous() and coords.dtype == torch.float32 and coords.numel() == B * self.num_levels * self.num_outputs
        if B == 0:
            return coords
        mb = min(self.micro_batch, B)
        need = lib.svb_model_workspace_bytes(self._h, mb, H, W)
        ws = _Workspace.get("model", need, u8.device)
        wp, wn = _aligned_ptr(ws, 1024)
        if stage_out is not None:
            assert times is None, "per-stage readout is not timed"
            want = torch.float16 if _lib.DTYPES[self.dtype] == _lib.SVB_FP16 else torch.bfloat16
            for s, t in enumerate(stage_out):
                assert t.device == u8.device and t.dtype == want and t.is_contiguous(), f"stage {s}: {want} on {u8.device}"
                assert tuple(t.shape) == (B, H >> (s + 2), W >> (s + 2), self.dims[s]), f"stage {s}: shape {tuple(t.shape)}"
            ptrs = (C.c_void_p * len(stage_out))(*[t.data_ptr() for t in stage_out])
            _lib.check(lib.svb_model_forward_stages(self._h, u8.data_ptr(), B, H, W, coords.data_ptr(), mb, wp, wn, _lib.current_stream(),
                                                    ptrs, len(stage_out)))
            return coords
        tbuf = (C.c_float * len(_lib.KERNEL_CLASSES))() if times is not None else None
        _lib.check(lib.svb_model_forward(self._h, u8.data_ptr(), B, H, W, coords.data_ptr(), mb, wp, wn, _lib.current_stream(),
                                         C.cast(tbuf, C.c_void_p) if tbuf is not None else None))
        if times is not None:
            for k, name in enumerate(_lib.KERNEL_CLASSES):
                times[name] = times.get(name, 0.0) + float(tbuf[k])
        return coords


    def forward_tensor(self, x: torch.Tensor, out: torch.Tensor | None = None) -> torch.Tensor:
        """float32 NCHW ``[B,3,H,W]`` (already /255 and ImageNet-normalised, cropping.py:463-472) on the device -> float32
        ``[B, num_levels, 2]``: what ``model(tensor)`` computes in the reference (generic.py:389-391), through the un-folded stem."""
        assert x.is_cuda and x.dtype == torch.float32 and x.dim() == 4 and x.shape[1] == 3 and x.is_contiguous()
        lib = _lib.load()
        B, _, H, W = x.shape
        coords = out if out is not None else torch.empty((B, self.num_levels, self.num_outputs), dtype=torch.float32, device=x.device)
        if B == 0:
            return coords
        mb = min(self.micro_batch, B)
        with torch.cuda.device(x.device):
            need = lib.svb_model_workspace_bytes(self._h, mb, H, W)
            ws = _Workspace.get("model", need, x.device)
            wp, wn = _aligned_ptr(ws, 1024)
            _lib.check(lib.svb_model_forward_f32(self._h, x.data_ptr(), B, H, W, coords.data_ptr(), mb, wp, wn,
                                                 torch.cuda.current_stream(x.device).cuda_stream, None))
        return coords


@_on_device
def gemm(a: torch.Tensor, w: torch.Tensor, bias: torch.Tensor, mode: int, resid: torch.Tensor | None = None,
         gamma: torch.Tensor | None = None, out: torch.Tensor | None = None) -> torch.Tensor:
    """Standalone tcgen05 GEMM (unit tests / profiling): ``epilogue(a @ w.T)``; a [M,K], w [N,K]."""
    lib = _lib.load()
    assert a.dtype == w.dtype and a.dtype in (torch.bfloat16, torch.float16) and a.is_contiguous() and w.is_contiguous()
    M, K = a.shape
    N = w.shape[0]
    if out is None:
        out = torch.empty((M, N), dtype=a.dtype, device=a.device)
    dt = _lib.SVB_BF16 if a.dtype == torch.bfloat16 else _lib.SVB_FP16
    _lib.check(lib.svb_gemm(a.data_ptr(), w.data_ptr(), out.data_ptr(), _lib.ptr(resid), bias.data_ptr(), _lib.ptr(gamma), M, N, K,
                            mode, dt, _lib.current_stream()))
    return out


@_on_device
def mlp_fused(a: torch.Tensor, w1: torch.Tensor, b1: torch.Tensor, w2: torch.Tensor, b2: torch.Tensor, gamma: torch.Tensor,
              x: torch.Tensor) -> torch.Tensor:
    """Standalone fused MLP (tests / profiling): ``x += gamma * (gelu(a @ w1.T + b1) @ w2.T + b2)`` in place."""
    assert a.dtype == w1.dtype == w2.dtype == x.dtype and a.is_contiguous() and x.is_contiguous()
    M, Cc = a.shape
    _lib.check(_lib.load().svb_mlp_fused(a.data_ptr(), w1.data_ptr(), b1.data_ptr(), w2.data_ptr(), b2.data_ptr(), gamma.data_ptr(),
                                         x.data_ptr(), M, Cc, _dt(a), _lib.current_stream()))
    return x


@_on_device
def mlp_fused_ln(a: torch.Tensor, w1g: torch.Tensor, t: torch.Tensor, s: torch.Tensor, rowstat: torch.Tensor, w2: torch.Tensor, b2: torch.Tensor,
                 gamma: torch.Tensor, x: torch.Tensor) -> torch.Tensor:
    """Fused MLP with the LayerNorm folded into fc1 (``svb_mlp_fused_ln``): ``a`` is the raw depthwise output, ``rowstat`` its
    (rstd, -mean * rstd) per token; ``x += gamma * (gelu(rstd * (a @ w1g.T) - rstd * mean * s + t) @ w2.T + b2)`` in place."""
    assert a.dtype == w1g.dtype == w2.dtype == x.dtype and a.is_contiguous() and x.is_contiguous()
    M, Cc = a.shape
    _lib.check(_lib.load().svb_mlp_fused_ln(a.data_ptr(), w1g.data_ptr(), t.data_ptr(), s.data_ptr(), rowstat.data_ptr(), w2.data_ptr(),
                                            b2.data_ptr(), gamma.data_ptr(), x.data_ptr(), M, Cc, _dt(a), _lib.current_stream()))
    return x


# ------------------------------------------------------------------ standalone layers (tests / ncu)
def _dt(t: torch.Tensor) -> int:
    assert t.dtype in (torch.bfloat16, torch.float16)
    return _lib.SVB_BF16 if t.dtype == torch.bfloat16 else _lib.SVB_FP16


@_on_device
def stem_ln(u8: torch.Tensor, wf: torch.Tensor, bf: torch.Tensor, lnw: torch.Tensor, lnb: torch.Tensor, dtype=torch.bfloat16):
    """u8 [B,H,W] -> [B,H/4,W/4,C0] with the folded stem (wf [C0,16], bf [C0])."""
    B, H, W = u8.shape
    C0 = wf.shape[0]
    out = torch.empty((B, H // 4, W // 4, C0), dtype=dtype, device=u8.device)
    _lib.check(_lib.load().svb_stem_ln(u8.data_ptr(), wf.data_ptr(), bf.data_ptr(), lnw.data_ptr(), lnb.data_ptr(), out.data_ptr(),
                                       B, H, W, C0, _dt(out), _lib.current_stream()))
    return out


@_on_device
def dwconv_ln(x: torch.Tensor, taps: torch.Tensor, bias: torch.Tensor, lnw: torch.Tensor, lnb: torch.Tensor, out: torch.Tensor | None = None):
    """x NHWC 16-bit [B,H,W,C]; taps fp32 [49,C] (tap-major) -> LayerNorm(dwconv7x7(x)+bias) [B,H,W,C]."""
    B, H, W, Cc = x.shape
    if out is None:
        out = torch.empty_like(x)
    _lib.check(_lib.load().svb_dwconv_ln(x.data_ptr(), taps.data_ptr(), bias.data_ptr(), lnw.data_ptr(), lnb.data_ptr(),
                                         out.data_ptr(), B, H, W, Cc, _dt(x), _lib.current_stream()))
    return out


@_on_device
def dwconv_raw(x: torch.Tensor, taps: torch.Tensor, bias: torch.Tensor, out: torch.Tensor | None = None):
    """Depthwise 7x7 + bias, LayerNorm folded into fc1 (``svb_dwconv_raw``): x NHWC 16-bit [B,H,W,C] -> (raw convolution
    [B,H,W,C] 16-bit, row statistics float32 [B*H*W, 2] = (rstd, -mean * rstd) of each token's rounded values).  The fc1 that
    consumes them is ``gemm(a, w_g, t, mode=3, resid=rowstat, gamma=s)``."""
    B, H, W, Cc = x.shape
    if out is None:
        out = torch.empty_like(x)
    stat = torch.empty((B * H * W, 2), dtype=torch.float32, device=x.device)
    _lib.check(_lib.load().svb_dwconv_raw(x.data_ptr(), taps.data_ptr(), bias.data_ptr(), out.data_ptr(), stat.data_ptr(), B, H, W, Cc,
                                          _dt(x), _lib.current_stream()))
    return out, stat


def dwconv_tc_pack(taps: torch.Tensor, dtype: torch.dtype) -> torch.Tensor:
    """taps fp32 [49, C] -> the B operands of ``dwconv_raw_tc`` ([C/64, 7, 112, 64] 16-bit of ``dtype``, on the taps' device);
    packed on the host by ``svb_dwconv_tc_pack`` (what ``svb_model_create`` does once per block)."""
    Cc = taps.shape[1]
    host = taps.detach().to("cpu", torch.float32).contiguous()
    out = torch.empty((Cc // 64, 7, 112, 64), dtype=dtype)
    _lib.check(_lib.load().svb_dwconv_tc_pack(host.data_ptr(), out.data_ptr(), Cc, _dt(out)))
    return out.to(taps.device)


@_on_device
def dwconv_raw_tc(x: torch.Tensor, wtc: torch.Tensor, bias: torch.Tensor, out: torch.Tensor | None = None, part: torch.Tensor | None = None):
    """``dwconv_raw`` on the tensor cores (``svb_dwconv_raw_tc``): x NHWC 16-bit [B,H,W,C], wtc from ``dwconv_tc_pack`` ->
    (raw convolution [B,H,W,C] 16-bit, row statistics float32 [B*H*W, 2] = (rstd, -mean * rstd)), as ``dwconv_raw`` returns.
    ``part`` (scratch, float32 [B*H*W, C/64, 2]) holds the per-chunk partial sums the statistics are added up from."""
    B, H, W, Cc = x.shape
    if out is None:
        out = torch.empty_like(x)
    if part is None:
        part = torch.empty((B * H * W, Cc // 64, 2), dtype=torch.float32, device=x.device)
    stat = torch.empty((B * H * W, 2), dtype=torch.float32, device=x.device)
    _lib.check(_lib.load().svb_dwconv_raw_tc(x.data_ptr(), wtc.data_ptr(), bias.data_ptr(), out.data_ptr(), stat.data_ptr(), part.data_ptr(),
                                             B, H, W, Cc, _dt(x), _lib.current_stream()))
    return out, stat


@_on_device
def dwconv_ln_tc(x: torch.Tensor, taps: torch.Tensor, bias: torch.Tensor, lnw: torch.Tensor, lnb: torch.Tensor):
    """Same operator as ``dwconv_ln`` on the tensor cores (taps are rounded to the activation dtype)."""
    B, H, W, Cc = x.shape
    out = torch.empty_like(x)
    taps16 = taps.to(x.dtype).contiguous()
    _lib.check(_lib.load().svb_dwconv_ln_tc(x.data_ptr(), taps16.data_ptr(), bias.data_ptr(), lnw.data_ptr(), lnb.data_ptr(),
                                            out.data_ptr(), B, H, W, Cc, _dt(x), _lib.current_stream()))
    return out


@_on_device
def ln_patchify(x: torch.Tensor, lnw: torch.Tensor, lnb: torch.Tensor):
    B, H, W, Cc = x.shape
    out = torch.empty((B, H // 2, W // 2, 4 * Cc), dtype=x.dtype, device=x.device)
    _lib.check(_lib.load().svb_ln_patchify(x.data_ptr(), lnw.data_ptr(), lnb.data_ptr(), out.data_ptr(), B, H, W, Cc, _dt(x),
                                           _lib.current_stream()))
    return out


@_on_device
def head(x: torch.Tensor, n0w, n0b, n1w, n1b, w1, b1, w2, b2):
    """x [B,tokens,C] 16-bit -> sigmoid coords fp32 [B,NOUT]."""
    B, tokens, Cc = x.shape
    hid, nout = w1.shape[0], w2.shape[0]
    out = torch.empty((B, nout), dtype=torch.float32, device=x.device)
    _lib.check(_lib.load().svb_head(x.data_ptr(), B, tokens, Cc, n0w.data_ptr(), n0b.data_ptr(), n1w.data_ptr(), n1b.data_ptr(),
                                    w1.data_ptr(), b1.data_ptr(), hid, w2.data_ptr(), b2.data_ptr(), nout, out.data_ptr(), _dt(x),
                                    _lib.current_stream()))
    return out
