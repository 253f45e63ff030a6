"""ctypes binding of ``libspine_b200.so`` (the C ABI in ``include/spine_b200.h``).

There is no CPU fallback: if the shared library is missing or a call fails the
caller gets an exception, never a silently different code path.
"""

from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

_PKG = Path(__file__).resolve().parent
LIB_PATH = Path(os.environ.get("SPINE_B200_LIB", _PKG / "libspine_b200.so"))

SVB_BF16, SVB_FP16, SVB_F32 = 0, 1, 2
PIXEL_FLOAT, PIXEL_INT16, PIXEL_UINT16, PIXEL_UINT8 = 0, 1, 2, 3  # SVB_PIXEL_*: the file's pixel type of a slice (rotated crops)
DTYPES = {"bf16": SVB_BF16, "bfloat16": SVB_BF16, "fp16": SVB_FP16, "float16": SVB_FP16, "half": SVB_FP16}
GRAPH_INPUT_U8, GRAPH_INPUT_F32 = 0, 1  # SVB_GRAPH_INPUT_*: what a captured forward reads
KERNEL_CLASSES = ("stem", "dwconv_ln", "gemm", "ln_patchify", "head", "mlp_fused")

# every symbol include/spine_b200.h declares
EXPORTS = (
    "svb_version", "svb_last_error", "svb_device_check", "svb_launch_count",
    "svb_k0_workspace_bytes", "svb_k0_midplane_resample",
    "svb_k01_workspace_bytes", "svb_k01_midplane_normalize_resize",
    "svb_k1_workspace_bytes", "svb_k1_normalize_resize", "svb_normalize_u8_workspace_bytes", "svb_normalize_u8",
    "svb_k3_workspace_bytes", "svb_k3_crop_resample", "svb_k3_crop_resample_rotated",
    "svb_model_create", "svb_model_destroy", "svb_model_workspace_bytes", "svb_model_forward", "svb_model_forward_f32",
    "svb_model_forward_stages", "svb_model_graph_create", "svb_model_graph_launch", "svb_model_graph_info", "svb_model_graph_destroy",
    "svb_model_info", "svb_model_cost", "svb_gemm", "svb_mlp_fused", "svb_mlp_fused_ln",
    "svb_stem_ln", "svb_dwconv_ln", "svb_dwconv_raw", "svb_dwconv_tc_pack", "svb_dwconv_raw_tc", "svb_ln_patchify", "svb_head",
    "svb_k4_classifier_input",
    "svb_png_bound", "svb_png_encode_gray8", "svb_png_write_gray8_batch", "svb_png_write_gray8_ragged",
    "svb_mha_read_header", "svb_mha_read_f32", "svb_mha_read_batch_f32", "svb_mha_read_batch_slab_f32",
    "svb_dicom_read_headers", "svb_dicom_read_slices_f32",
)


class SvbError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"libspine_b200 error {code}: {msg}")
        self.code = code


class MhaInfo(C.Structure):
    """``svb_mha_info`` (include/spine_b200.h)."""

    _fields_ = [("ndim", C.c_int32), ("dim", C.c_int32 * 3), ("spacing", C.c_double * 3), ("origin", C.c_double * 3),
                ("direction", C.c_double * 9), ("element_type", C.c_int32), ("element_bytes", C.c_int32), ("channels", C.c_int32),
                ("compressed", C.c_int32), ("big_endian", C.c_int32), ("has_spacing", C.c_int32), ("data_offset", C.c_int64),
                ("header_size", C.c_int64), ("compressed_size", C.c_int64), ("data_file", C.c_char * 1024)]


class DicomInfo(C.Structure):
    """``svb_dicom_info`` (include/spine_b200.h)."""

    _fields_ = [("rows", C.c_int32), ("cols", C.c_int32), ("bits_allocated", C.c_int32), ("pixel_representation", C.c_int32),
                ("samples_per_pixel", C.c_int32), ("monochrome1", C.c_int32), ("instance_number", C.c_int32), ("big_endian", C.c_int32),
                ("has_position", C.c_int32), ("has_orientation", C.c_int32), ("has_spacing", C.c_int32), ("encapsulation", C.c_int32),
                ("pixel_spacing", C.c_double * 2), ("position", C.c_double * 3), ("orientation", C.c_double * 6),
                ("rescale_slope", C.c_double), ("rescale_intercept", C.c_double), ("slice_thickness", C.c_double),
                ("spacing_between_slices", C.c_double), ("pixel_offset", C.c_int64), ("pixel_bytes", C.c_int64),
                ("bits_stored", C.c_int32), ("pad", C.c_int32), ("series_uid", C.c_char * 72)]


class WeightDesc(C.Structure):
    _fields_ = [("name", C.c_char_p), ("data", C.c_void_p), ("ndim", C.c_int32), ("shape", C.c_int64 * 4)]


_lib = None


def load() -> C.CDLL:
    """Load the shared library (once).  Raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        raise FileNotFoundError(
            f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(or `make -C spine_vision_b200/csrc`). There is no CPU fallback."
        )
    lib = C.CDLL(str(LIB_PATH))
    vp, i32, sz = C.c_void_p, C.c_int, C.c_size_t
    lib.svb_version.restype = C.c_int
    lib.svb_last_error.restype = C.c_char_p
    lib.svb_device_check.restype = C.c_int
    lib.svb_launch_count.restype = C.c_longlong
    lib.svb_launch_count.argtypes = [C.c_int]
    lib.svb_k0_workspace_bytes.restype = sz
    lib.svb_k0_workspace_bytes.argtypes = [i32] * 3
    lib.svb_k0_midplane_resample.restype = C.c_int
    lib.svb_k0_midplane_resample.argtypes = [vp, vp, i32, i32, i32, vp, vp, sz, vp]
    lib.svb_k01_workspace_bytes.restype = sz
    lib.svb_k01_workspace_bytes.argtypes = [i32] * 5
    lib.svb_k01_midplane_normalize_resize.restype = C.c_int
    lib.svb_k01_midplane_normalize_resize.argtypes = [vp, vp, i32, i32, i32, vp, vp, vp, i32, i32, vp, vp, vp, sz, vp]
    lib.svb_k1_workspace_bytes.restype = sz
    lib.svb_k1_workspace_bytes.argtypes = [i32] * 5
    lib.svb_k1_normalize_resize.restype = C.c_int
    lib.svb_k1_normalize_resize.argtypes = [vp, vp, vp, i32, i32, i32, i32, i32, vp, vp, vp, sz, vp]
    lib.svb_k3_workspace_bytes.restype = sz
    lib.svb_k3_workspace_bytes.argtypes = [i32] * 4
    lib.svb_k3_crop_resample.restype = C.c_int
    lib.svb_k3_crop_resample.argtypes = [vp, vp, vp, vp, vp, vp, i32, i32, i32, i32, i32, vp, i32, i32, vp, vp, i32, vp, sz, vp]
    lib.svb_k3_crop_resample_rotated.restype = C.c_int
    lib.svb_k3_crop_resample_rotated.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp, i32, i32, i32, i32, i32, vp, i32, i32, vp, vp, i32, vp, sz, vp]
    lib.svb_model_create.restype = C.c_int
    lib.svb_model_create.argtypes = [C.POINTER(vp), C.POINTER(WeightDesc), i32, i32]
    lib.svb_model_destroy.restype = C.c_int
    lib.svb_model_destroy.argtypes = [vp]
    lib.svb_model_workspace_bytes.restype = sz
    lib.svb_model_workspace_bytes.argtypes = [vp, i32, i32, i32]
    lib.svb_model_forward.restype = C.c_int
    lib.svb_model_forward.argtypes = [vp, vp, i32, i32, i32, vp, i32, vp, sz, vp, vp]
    lib.svb_model_forward_f32.restype = C.c_int
    lib.svb_model_forward_f32.argtypes = [vp, vp, i32, i32, i32, vp, i32, vp, sz, vp, vp]
    lib.svb_model_forward_stages.restype = C.c_int
    lib.svb_model_forward_stages.argtypes = [vp, vp, i32, i32, i32, vp, i32, vp, sz, vp, C.POINTER(vp), i32]
    lib.svb_model_graph_create.restype = C.c_int
    lib.svb_model_graph_create.argtypes = [vp, i32, i32, i32, i32, i32, vp, sz, vp, C.POINTER(vp)]
    lib.svb_model_graph_launch.restype = C.c_int
    lib.svb_model_graph_launch.argtypes = [vp, vp, vp, vp]
    lib.svb_model_graph_info.restype = C.c_int
    lib.svb_model_graph_info.argtypes = [vp, C.POINTER(C.c_int32 * 4)]
    lib.svb_model_graph_destroy.restype = C.c_int
    lib.svb_model_graph_destroy.argtypes = [vp]
    lib.svb_model_info.restype = C.c_int
    lib.svb_model_info.argtypes = [vp, C.POINTER(C.c_int32 * 10)]
    lib.svb_model_cost.restype = C.c_int
    lib.svb_model_cost.argtypes = [vp, i32, i32, i32, C.POINTER(C.c_double), C.POINTER(C.c_int64)]
    lib.svb_gemm.restype = C.c_int
    lib.svb_gemm.argtypes = [vp, vp, vp, vp, vp, vp, i32, i32, i32, i32, i32, vp]
    lib.svb_mlp_fused.restype = C.c_int
    lib.svb_mlp_fused.argtypes = [vp, vp, vp, vp, vp, vp, vp, i32, i32, i32, vp]
    lib.svb_mlp_fused_ln.restype = C.c_int
    lib.svb_mlp_fused_ln.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp, vp, i32, i32, i32, vp]
    lib.svb_stem_ln.restype = C.c_int
    lib.svb_stem_ln.argtypes = [vp, vp, vp, vp, vp, vp, i32, i32, i32, i32, i32, vp]
    lib.svb_dwconv_ln.restype = C.c_int
    lib.svb_dwconv_ln.argtypes = [vp, vp, vp, vp, vp, vp, i32, i32, i32, i32, i32, vp]
    lib.svb_dwconv_raw.restype = C.c_int
    lib.svb_dwconv_raw.argtypes = [vp, vp, vp, vp, vp, i32, i32, i32, i32, i32, vp]
    lib.svb_dwconv_tc_pack.restype = C.c_int
    lib.svb_dwconv_tc_pack.argtypes = [vp, vp, i32, i32]
    lib.svb_dwconv_raw_tc.restype = C.c_int
    lib.svb_dwconv_raw_tc.argtypes = [vp, vp, vp, vp, vp, vp, i32, i32, i32, i32, i32, vp]
    lib.svb_ln_patchify.restype = C.c_int
    lib.svb_ln_patchify.argtypes = [vp, vp, vp, vp, i32, i32, i32, i32, i32, vp]
    lib.svb_head.restype = C.c_int
    lib.svb_head.argtypes = [vp, i32, i32, i32, vp, vp, vp, vp, vp, vp, i32, vp, vp, i32, vp, i32, vp]
    lib.svb_k4_classifier_input.restype = C.c_int
    lib.svb_k4_classifier_input.argtypes = [vp, vp, vp, i32, i32, i32, vp, vp, i32, i32, vp, vp]
    lib.svb_png_bound.restype = sz
    lib.svb_png_bound.argtypes = [i32, i32]
    lib.svb_png_encode_gray8.restype = C.c_int
    lib.svb_png_encode_gray8.argtypes = [vp, i32, i32, i32, vp, sz, C.POINTER(sz)]
    lib.svb_png_write_gray8_batch.restype = C.c_int
    lib.svb_png_write_gray8_batch.argtypes = [vp, i32, i32, i32, C.POINTER(C.c_char_p), i32, i32, vp]
    lib.svb_mha_read_header.restype = C.c_int
    lib.svb_mha_read_header.argtypes = [C.c_char_p, C.POINTER(MhaInfo)]
    lib.svb_mha_read_f32.restype = C.c_int
    lib.svb_mha_read_f32.argtypes = [C.c_char_p, C.POINTER(MhaInfo), vp, sz]
    lib.svb_mha_read_batch_f32.restype = C.c_int
    lib.svb_mha_read_batch_f32.argtypes = [C.POINTER(C.c_char_p), i32, C.POINTER(MhaInfo), C.POINTER(vp), C.POINTER(sz), i32, vp]
    lib.svb_mha_read_batch_slab_f32.restype = C.c_int
    lib.svb_mha_read_batch_slab_f32.argtypes = [C.POINTER(C.c_char_p), i32, C.POINTER(MhaInfo), C.POINTER(vp), C.POINTER(sz),
                                                C.POINTER(C.c_int32), C.POINTER(C.c_int32), i32, vp]
    lib.svb_normalize_u8_workspace_bytes.restype = sz
    lib.svb_normalize_u8_workspace_bytes.argtypes = [i32]
    lib.svb_normalize_u8.restype = C.c_int
    lib.svb_normalize_u8.argtypes = [vp, vp, vp, i32, i32, i32, vp, vp, vp, sz, vp]
    lib.svb_png_write_gray8_ragged.restype = C.c_int
    lib.svb_png_write_gray8_ragged.argtypes = [vp, vp, vp, i32, C.POINTER(C.c_char_p), i32, i32, vp]
    lib.svb_dicom_read_headers.restype = C.c_int
    lib.svb_dicom_read_headers.argtypes = [C.POINTER(C.c_char_p), i32, C.POINTER(DicomInfo), i32, vp]
    lib.svb_dicom_read_slices_f32.restype = C.c_int
    lib.svb_dicom_read_slices_f32.argtypes = [C.POINTER(C.c_char_p), i32, C.POINTER(DicomInfo), C.POINTER(vp), C.POINTER(sz), i32, vp]
    _lib = lib
    return lib


def check(rc: int) -> None:
    if rc != 0:
        raise SvbError(rc, load().svb_last_error().decode("utf-8", "replace"))


def ptr(t) -> int | None:
    """Device/host pointer of a torch tensor (None passes NULL)."""
    return None if t is None else t.data_ptr()


def current_stream() -> int:
    import torch

    return torch.cuda.current_stream().cuda_stream
