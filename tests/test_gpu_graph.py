"""GPU: the localizer forward captured as a CUDA graph (svb_model_graph_*, LocalizationModel.graphed) and under torch.cuda.graph.

A graph holds the kernels of svb_model_forward with the same arguments, so every coordinate check is bit equality with the
eager forward on the same input (eager runs are bit-reproducible).  Inputs change on every replay to exercise the rebinding of
the input and coordinate arguments."""
import ctypes as C
import subprocess
import sys
import textwrap
from pathlib import Path

import pytest
import torch

from gpu_util import dev, requires_gpu
from oracle.convnext import make_model
from spine_vision_b200 import _lib, cropping, ops

INVALID, WS_SMALL = -1, -4
ROOT = Path(__file__).resolve().parent.parent


def _err():
    return _lib.load().svb_last_error().decode()


def _u8(seed, B, H=512, W=512):
    g = torch.Generator(device=dev()).manual_seed(seed)
    return torch.randint(0, 256, (B, H, W), dtype=torch.uint8, device=dev(), generator=g)


def _f32(seed, B, H=512, W=512):
    g = torch.Generator(device=dev()).manual_seed(seed)
    return torch.randn((B, 3, H, W), dtype=torch.float32, device=dev(), generator=g)


def _model(variant="base", dtype="fp16", micro_batch=64):
    return cropping.LocalizationModel(make_model(variant, seed=0, trained_like=True).state_dict(), dev(), dtype=dtype, micro_batch=micro_batch)


@pytest.fixture(scope="module")
def base():
    return _model()


def _launches():
    return int(_lib.load().svb_launch_count(0))


@requires_gpu
@pytest.mark.parametrize("B", [256, 70, 1])  # two chains over four micro-batches; a tail micro-batch of 6; one image, one chain
def test_graph_replays_match_eager_base_fp16(base, B):
    xs = [_u8(100 + k, B) for k in range(3)]
    n0 = _launches()
    want = [base.predict_u8(x) for x in xs]
    eager_launches = (_launches() - n0) // 3
    g = base.graphed(B)
    assert g.kernel_nodes == eager_launches, (g.kernel_nodes, eager_launches)
    n0 = _launches()
    got = [g(x) for x in xs]
    assert _launches() - n0 == 3 * g.kernel_nodes
    out = torch.full_like(want[0], -1.0)
    assert g(xs[1], out=out) is out
    torch.cuda.synchronize()
    for k in range(3):
        assert torch.equal(got[k], want[k]), f"replay {k}: {(got[k] - want[k]).abs().max().item()}"
    assert torch.equal(out, want[1])


@requires_gpu
@pytest.mark.parametrize("variant,dtype,H,W", [
    ("base", "bf16", 512, 512),    # dwconv_raw_kernel instead of the tensor-core depthwise kernel
    ("v2_tiny", "fp16", 512, 512),  # GRN launches
    ("tiny", "fp16", 352, 288),
])
def test_graph_other_paths_and_f32_input(variant, dtype, H, W):
    m = _model(variant, dtype, micro_batch=2)  # 5 images: two chains, a tail micro-batch of 1
    g8, g32 = m.graphed(5, (H, W)), m.graphed(5, (H, W), normalised_input=True)
    for seed in (1, 2):
        x8, x32 = _u8(seed, 5, H, W), _f32(seed, 5, H, W)
        assert torch.equal(g8(x8), m.predict_u8(x8))
        assert torch.equal(g32(x32), m.engine.forward_tensor(x32))


def _torch_graph(fn, static):
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        fn(static)
    torch.cuda.current_stream().wait_stream(s)
    tg = torch.cuda.CUDAGraph()
    with torch.cuda.graph(tg):
        out = fn(static)
    return tg, out


@requires_gpu
def test_torch_cuda_graph_capture_of_predict_u8_and_model_call(base):
    static8, static32 = _u8(0, 70), _f32(0, 70)
    tg8, out8 = _torch_graph(base.predict_u8, static8)
    tg32, out32 = _torch_graph(base, static32)
    for seed in (5, 6, 7):
        static8.copy_(_u8(seed, 70))
        static32.copy_(_f32(seed, 70))
        tg8.replay()
        tg32.replay()
        assert torch.equal(out8, base.predict_u8(static8)), seed
        assert torch.equal(out32, base(static32)), seed


@requires_gpu
def test_replays_survive_plan_cache_churn_and_workspace_growth(base):
    key = ("model", str(torch.device(dev())))
    ops._Workspace._bufs.pop(key, None)  # start small, so that the larger batch below has to grow the shared workspace
    static = _u8(10, 4)
    g = base.graphed(4)
    tg, tout = _torch_graph(base.predict_u8, static)
    want = base.predict_u8(static)
    tg.replay()
    assert torch.equal(g(static), want) and torch.equal(tout, want)
    old = ops._Workspace._bufs[key]
    old_n = old.numel()
    del old
    # five other shapes: more (workspace, micro-batch, H, W) plans than the handle's four-entry cache holds
    for B, H, W in [(3, 256, 256), (5, 512, 384), (2, 384, 640), (1, 1024, 512), (70, 512, 512)]:
        base.predict_u8(_u8(B + H, B, H, W))
    assert ops._Workspace._bufs[key].numel() > old_n
    guard = torch.full((old_n,), 7, dtype=torch.uint8, device=dev())  # most likely the freed workspace's memory
    for seed in (11, 12):
        static.copy_(_u8(seed, 4))
        got = g(static)
        tg.replay()
        want = base.predict_u8(static)
        assert torch.equal(got, want) and torch.equal(tout, want), seed
    assert bool((guard == 7).all()), "a replay wrote into memory it does not own"


_FRESH = textwrap.dedent("""
    import sys, torch
    sys.path.insert(0, {root!r})
    from spine_vision_b200 import cropping, synthetic
    m = cropping.LocalizationModel(synthetic.random_state_dict("base", seed=0, trained_like=True), "cuda:0", dtype="fp16", micro_batch=4)
    x = torch.randint(0, 256, (9, 512, 512), dtype=torch.uint8, device="cuda:0")
    if {mode!r} == "torch":
        tg = torch.cuda.CUDAGraph()
        with torch.cuda.graph(tg):  # global capture mode, and the first forward of the process
            out = m.predict_u8(x)
        tg.replay()
    else:
        out = m.graphed(9)(x)
    assert torch.equal(out, m.predict_u8(x))
    print("fresh ok")
""")


@requires_gpu
@pytest.mark.parametrize("mode", ["torch", "graphed"])
def test_capture_as_first_forward_of_a_process(mode):
    """Every lazily made set-up of the forward (kernel attributes, plans) happens inside the capture here."""
    r = subprocess.run([sys.executable, "-c", _FRESH.format(root=str(ROOT), mode=mode)], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "fresh ok" in r.stdout, r.stdout[-2000:] + r.stderr[-4000:]


@requires_gpu
@pytest.mark.filterwarnings("ignore:The CUDA Graph is empty")  # the refused captures record nothing
def test_graph_abi_errors(base):
    lib = _lib.load()
    h = base.engine._h
    side = torch.cuda.Stream()
    st = side.cuda_stream
    need = lib.svb_model_workspace_bytes(h, 2, 512, 512)
    ws = torch.empty(need + 2048, dtype=torch.uint8, device=dev())
    wp, wn = ops._aligned_ptr(ws, 1024)
    out = C.c_void_p()
    U8 = _lib.GRAPH_INPUT_U8
    assert lib.svb_model_graph_create(None, U8, 2, 512, 512, 2, wp, wn, st, C.byref(out)) == INVALID and "null" in _err()
    assert lib.svb_model_graph_create(h, U8, 2, 512, 512, 2, wp, wn, st, None) == INVALID
    assert lib.svb_model_graph_create(h, 7, 2, 512, 512, 2, wp, wn, st, C.byref(out)) == INVALID and "input_kind" in _err()
    assert lib.svb_model_graph_create(h, U8, 0, 512, 512, 2, wp, wn, st, C.byref(out)) == INVALID
    assert lib.svb_model_graph_create(h, U8, 2, 500, 512, 2, wp, wn, st, C.byref(out)) == INVALID and "multiple of 32" in _err()
    assert lib.svb_model_graph_create(h, U8, 2, 512, 512, 2, wp, need // 4, st, C.byref(out)) == WS_SMALL
    assert lib.svb_model_graph_create(h, U8, 2, 512, 512, 2, wp + 256, wn - 256, st, C.byref(out)) == INVALID and "aligned" in _err()
    assert out.value is None
    # the legacy default stream cannot capture: refused, and the stream still runs an eager forward
    assert lib.svb_model_graph_create(h, U8, 2, 512, 512, 2, wp, wn, 0, C.byref(out)) < 0 and "capture" in _err()
    x = _u8(3, 2)
    want = base.predict_u8(x)
    # a stream that is already capturing (torch.cuda.graph) is refused, and so is per-launch timing inside a capture
    tg = torch.cuda.CUDAGraph()
    with pytest.raises(_lib.SvbError) as e:
        with torch.cuda.graph(tg):
            cur = torch.cuda.current_stream().cuda_stream
            assert lib.svb_model_graph_create(h, U8, 2, 512, 512, 2, wp, wn, cur, C.byref(out)) == INVALID and "capturing" in _err()
            base.predict_u8(x, times={})
    assert e.value.code == INVALID and "capturing" in str(e.value)
    assert torch.equal(base.predict_u8(x), want)  # eager on the same (default) stream after the refused captures
    # launch / info / destroy
    g = base.graphed(2)
    coords = torch.empty((2, 5, 2), dtype=torch.float32, device=dev())
    info = (C.c_int32 * 4)()
    assert lib.svb_model_graph_launch(None, x.data_ptr(), coords.data_ptr(), 0) == INVALID
    assert lib.svb_model_graph_launch(g._h, None, coords.data_ptr(), 0) == INVALID
    assert lib.svb_model_graph_launch(g._h, x.data_ptr(), None, 0) == INVALID
    assert lib.svb_model_graph_info(None, C.byref(info)) == INVALID
    assert lib.svb_model_graph_info(g._h, C.byref(info)) == 0 and tuple(info) == (g.kernel_nodes, 2, 512, 512)
    assert lib.svb_model_graph_destroy(None) == 0
    # GraphedForward refuses what it was not captured for, before any launch
    n0 = _launches()
    for bad in (x[:1], x.to(torch.float32), x.transpose(1, 2), x.cpu(), x.view(-1)):
        with pytest.raises(ValueError):
            g(bad)
    with pytest.raises(ValueError):
        g(x, out=torch.empty((2, 5, 2), dtype=torch.float64, device=dev()))
    assert _launches() == n0
    assert torch.equal(g(x), want)
