"""GPU: the C ABI's error behaviour -- bad arguments come back as a negative svb_status with a message in svb_last_error(),
never as a crash, a silent no-op or a fallback; empty batches are successful no-ops (include/spine_b200.h, conventions)."""
import ctypes as C

import numpy as np
import pytest
import torch

from gpu_util import dev, requires_gpu
from spine_vision_b200 import _lib, ops, synthetic

INVALID, WS_SMALL, BOX, MISSING, UNSUPPORTED_MODEL = -1, -4, -5, -6, -7


def _err():
    return _lib.load().svb_last_error().decode()


@requires_gpu
def test_null_and_size_arguments():
    lib = _lib.load()
    d = dev()
    st = torch.cuda.current_stream().cuda_stream
    assert lib.svb_device_check() == 0
    sl = torch.zeros(64 * 64, dtype=torch.float32, device=d)
    offs = torch.zeros(1, dtype=torch.int64, device=d)
    hw = torch.tensor([[64, 64]], dtype=torch.int32, device=d)
    out = torch.zeros(32 * 32, dtype=torch.uint8, device=d)
    ws = torch.zeros(1 << 20, dtype=torch.uint8, device=d)
    # K1
    assert lib.svb_k1_normalize_resize(None, offs.data_ptr(), hw.data_ptr(), 1, 64, 64, 32, 32, out.data_ptr(), None, ws.data_ptr(), ws.numel(), st) == INVALID
    assert "k1" in _err()
    assert lib.svb_k1_normalize_resize(sl.data_ptr(), offs.data_ptr(), hw.data_ptr(), 1, 64, 64, 0, 32, out.data_ptr(), None, ws.data_ptr(), ws.numel(), st) == INVALID
    assert lib.svb_k1_normalize_resize(sl.data_ptr(), offs.data_ptr(), hw.data_ptr(), 1, 64, 64, 32, 32, out.data_ptr(), None, ws.data_ptr(), 16, st) == WS_SMALL
    assert lib.svb_k1_normalize_resize(sl.data_ptr(), offs.data_ptr(), hw.data_ptr(), 0, 64, 64, 32, 32, out.data_ptr(), None, ws.data_ptr(), ws.numel(), st) == 0
    # normalise only
    assert lib.svb_normalize_u8(sl.data_ptr(), offs.data_ptr(), hw.data_ptr(), 1, 64, 64, None, None, ws.data_ptr(), ws.numel(), st) == INVALID
    assert lib.svb_normalize_u8(sl.data_ptr(), offs.data_ptr(), hw.data_ptr(), 1, 64, 64, out.data_ptr(), None, ws.data_ptr(), 8, st) == WS_SMALL
    # K3: crop width must be a multiple of 4; a box that cannot fit on chip is refused, not truncated
    idx = torch.zeros(1, dtype=torch.int32, device=d)
    xy = torch.full((1, 2), 0.5, dtype=torch.float32, device=d)
    delta = torch.tensor([[10, 10, 10, 10]], dtype=torch.int32, device=d)
    crops = torch.zeros(130 * 130, dtype=torch.uint8, device=d)
    args = lambda mbh, mbw, ch, cw: (sl.data_ptr(), offs.data_ptr(), hw.data_ptr(), idx.data_ptr(), xy.data_ptr(), delta.data_ptr(), 1, mbh, mbw, ch, cw,  # noqa: E731
                                     crops.data_ptr(), 0, 0, None, None, 0, ws.data_ptr(), ws.numel(), st)
    assert lib.svb_k3_crop_resample(*args(20, 20, 128, 126)) == INVALID and "multiple of 4" in _err()
    assert lib.svb_k3_crop_resample(*args(2000, 2000, 128, 128)) == BOX and "shared memory" in _err()
    assert lib.svb_k3_crop_resample(*args(20, 20, 128, 128)) == 0
    # K4
    planes = torch.zeros((2, 4, 4), dtype=torch.uint8, device=d)
    o4 = torch.zeros((1, 3, 4, 4), dtype=torch.float32, device=d)
    assert lib.svb_k4_classifier_input(planes.data_ptr(), idx.data_ptr(), idx.data_ptr(), 1, 4, 4, None, None, 1, 7, o4.data_ptr(), st) == INVALID
    assert "out_dtype" in _err()
    assert lib.svb_k4_classifier_input(planes.data_ptr(), idx.data_ptr(), idx.data_ptr(), 1, 4, 4, None, None, 1, 2, None, st) == INVALID
    torch.cuda.synchronize()


@requires_gpu
def test_model_create_rejects_incomplete_or_unsupported_checkpoints():
    sd = synthetic.random_state_dict("base", seed=0)
    bad = dict(sd)
    del bad["backbone.stages.2.blocks.13.mlp.fc1.weight"]
    with pytest.raises(_lib.SvbError) as e:
        ops.LocalizationEngine(bad, dev())
    assert e.value.code == MISSING and "fc1" in str(e.value)
    wrong = dict(sd)
    wrong["head.5.weight"] = torch.zeros(7, 256)  # odd number of outputs: not (x, y) pairs
    with pytest.raises(_lib.SvbError):
        ops.LocalizationEngine(wrong, dev())
    eng = ops.LocalizationEngine(sd, dev())
    with pytest.raises((_lib.SvbError, AssertionError, ValueError)):
        eng.forward(torch.zeros((1, 500, 512), dtype=torch.uint8, device=dev()))  # H not a multiple of 32
    out = eng.forward(torch.zeros((0, 512, 512), dtype=torch.uint8, device=dev()))
    assert tuple(out.shape) == (0, 5, 2)


@requires_gpu
def test_model_forward_stages_rejects_bad_stage_buffers():
    lib = _lib.load()
    eng = ops.LocalizationEngine(synthetic.random_state_dict("tiny", seed=0), dev(), "fp16", micro_batch=2)
    u8 = torch.zeros((3, 64, 64), dtype=torch.uint8, device=dev())
    coords = torch.zeros((3, 5, 2), dtype=torch.float32, device=dev())
    ws = torch.zeros(lib.svb_model_workspace_bytes(eng._h, 2, 64, 64) + 1024, dtype=torch.uint8, device=dev())
    wp = (ws.data_ptr() + 1023) // 1024 * 1024
    stages = [torch.zeros((3, 64 >> (s + 2), 64 >> (s + 2), eng.dims[s]), dtype=torch.float16, device=dev()) for s in range(4)]
    st = torch.cuda.current_stream().cuda_stream

    def call(bufs, n):
        arr = (C.c_void_p * max(1, len(bufs)))(*bufs) if bufs else None
        return lib.svb_model_forward_stages(eng._h, u8.data_ptr(), 3, 64, 64, coords.data_ptr(), 2, wp, ws.numel() - 1024, st, arr, n)

    ptrs = [t.data_ptr() for t in stages]
    assert call([], 4) == INVALID and "null" in _err()
    assert call(ptrs, 0) == INVALID and "stage buffers" in _err()
    assert call(ptrs, 5) == INVALID and "stage buffers" in _err()
    assert call(ptrs[:2] + [None] + ptrs[3:], 4) == INVALID and "stage buffer 2 is null" in _err()
    assert call(ptrs[:2], 2) == 0  # the first stages only
    torch.cuda.synchronize()
    assert stages[1].abs().sum() > 0 and stages[2].abs().sum() == 0
    with pytest.raises(AssertionError):  # wrong shape caught before the call
        eng.forward(u8, stage_out=[stages[1]])
