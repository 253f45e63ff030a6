"""GPU parity: the CoordinateRegressor forward and the whole localize-and-crop path vs the fp32 oracle."""
import numpy as np
import pytest
import torch

from conftest import GOLDEN
from gpu_util import dev, trained_like_gate
from oracle import reference_path as ref
from oracle.convnext import make_model
from spine_vision_b200 import cropping, ops, pipeline, synthetic

pytestmark = pytest.mark.gpu
PX = 512.0
SLICES = [(20, 1195, 1195), (21, 640, 650), (22, 900, 700), (23, 512, 512)]


def _oracle_coords(model, slices):
    out = []
    for sl in slices:
        _, t = ref.preprocess_slice(sl, (512, 512))
        with torch.no_grad():
            out.append(model(t.unsqueeze(0))[0].numpy())
    return np.stack(out)


# tolerance stated by BASELINE.json north_star: 0.5 px at 512^2 on random-init weights; SURVEY 8d asks the same of the
# "trained-like" weights (layer-scale U(0.1,1)), which make 36 blocks of 16-bit rounding visible.  The DEFAULT dtype (None ->
# fp16, what load_localization_model hands every real checkpoint) holds 0.5 px on both weight sets.  dtype="bf16" is an
# explicit opt-in: 0.22 px on random-init weights, 1.0 px on trained-like ones (8 mantissa bits through 75 GEMMs -- the same
# figure a PyTorch bf16-rounded emulation of the network gives, DESIGN.md section 5); that row is reported, held to 1.5 px,
# and is NOT the shipped configuration.
@pytest.mark.parametrize("dtype,trained,tol_px", [(None, False, 0.5), (None, True, 0.5), ("fp16", False, 0.5), ("fp16", True, 0.5),
                                                  ("bf16", False, 0.5), ("bf16", True, 1.5)])
def test_model_coords_vs_oracle(dtype, trained, tol_px):
    torch.set_num_threads(max(1, torch.get_num_threads()))
    om = make_model("base", seed=0, trained_like=trained)
    slices = [synthetic.make_iso_slice(*c) for c in SLICES]
    want = _oracle_coords(om, slices)
    model = cropping.LocalizationModel(om.state_dict(), dev(), dtype=dtype, micro_batch=3)  # 3 + 1: exercises the tail chunk
    pool = ops.SlicePool.from_numpy(slices, dev())
    planes = ops.normalize_resize(pool, (512, 512))
    got = model.predict_u8(planes).cpu().numpy()
    err_px = np.abs(got - want).max() * PX
    assert got.shape == (4, 5, 2) and np.isfinite(got).all()
    print(f"[coords] dtype={dtype} trained_like={trained}: max error {err_px:.4f} px at 512^2 (tolerance {tol_px})")
    assert err_px <= tol_px, f"{dtype} trained={trained}: max coordinate error {err_px:.3f} px (tolerance {tol_px})"
    # golden coordinates frozen from the reference's own predict_ivd_locations
    g = np.load(GOLDEN / "model_coords.npz")
    tag = "trained" if trained else "init"
    for i, (seed, h, w) in enumerate(SLICES[:2]):
        gerr = np.abs(got[i] - g[f"coords_{tag}_{seed}_{h}_{w}"]).max() * PX
        assert gerr <= tol_px, f"vs reference golden: {gerr:.3f} px"


def test_unfolded_layernorm_path_still_agrees(monkeypatch):
    """SVB_LN_FOLD=0 at model creation keeps the round-1 block (dwconv_ln_kernel writes the normalised fc1 operand): both
    forms of the block hold the gate on trained-like weights, and agree with each other to well inside it."""
    om = make_model("base", seed=0, trained_like=True)
    slices = [synthetic.make_iso_slice(*c) for c in SLICES[:2]]
    want = _oracle_coords(om, slices)
    pool = ops.SlicePool.from_numpy(slices, dev())
    planes = ops.normalize_resize(pool, (512, 512))
    folded = cropping.LocalizationModel(om.state_dict(), dev()).predict_u8(planes).cpu().numpy()
    monkeypatch.setenv("SVB_LN_FOLD", "0")
    plain = cropping.LocalizationModel(om.state_dict(), dev()).predict_u8(planes).cpu().numpy()
    e_f, e_p = np.abs(folded - want).max() * PX, np.abs(plain - want).max() * PX
    print(f"[coords] trained-like fp16: folded LayerNorm {e_f:.4f} px, separate LayerNorm {e_p:.4f} px")
    assert e_f <= 0.5 and e_p <= 0.5 and np.abs(folded - plain).max() * PX <= 0.5


@pytest.mark.parametrize("env", [{"SVB_DWCONV_TC2": "0"}, {"SVB_MLP_FUSED": "0"}, {"SVB_TC2_MODEB": "0"}, {"SVB_DWCONV_TC2": "0", "SVB_MLP_FUSED": "0"},
                                 {"SVB_TC2_PAIR": "1"},
                                 {"SVB_DWCONV_TC2": "2", "dtype": "bf16"}])
def test_alternative_block_kernels_still_agree(monkeypatch, env):
    """The A/B switches of the block (read at model creation): FP32-pipe depthwise kernel instead of the tensor-core one, two GEMMs
    instead of the fused MLP, tensor-core depthwise kernel only where a warp holds whole image rows, its cta_group::2 variant, and the
    tensor-core depthwise kernel with bf16 taps (opt-in) -- each holds the gate on trained-like weights and stays close to the default path."""
    env = dict(env)
    dtype = env.pop("dtype", None)
    om = make_model("base", seed=0, trained_like=True)
    slices = [synthetic.make_iso_slice(*c) for c in SLICES[:2]]
    want = _oracle_coords(om, slices)
    pool = ops.SlicePool.from_numpy(slices, dev())
    planes = ops.normalize_resize(pool, (512, 512))
    default = cropping.LocalizationModel(om.state_dict(), dev(), dtype=dtype).predict_u8(planes).cpu().numpy()
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    other = cropping.LocalizationModel(om.state_dict(), dev(), dtype=dtype).predict_u8(planes).cpu().numpy()
    e_d, e_o = np.abs(default - want).max() * PX, np.abs(other - want).max() * PX
    print(f"[coords] trained-like {dtype or 'fp16'}: default {e_d:.4f} px, {env} {e_o:.4f} px, apart {np.abs(default - other).max() * PX:.4f} px")
    tol = 0.5 if dtype is None else 1.5
    assert e_o <= tol and np.abs(default - other).max() * PX <= tol


def test_default_dtype_is_fp16():
    """Real checkpoints run what holds the 0.5 px gate on trained-like weights (VERDICT r01, weak #1)."""
    om = make_model("base", seed=0)
    assert cropping.LocalizationModel(om.state_dict(), dev()).engine.dtype == "fp16"


@pytest.mark.parametrize("trained", [False, True])
def test_end_to_end_crop_agreement_config1(trained):
    """BASELINE configs[0] (32 series of 1195 x 1195, seeds 0..31): how often is the END-TO-END crop -- device coordinates ->
    int(x*w), int(y*h) -> box -> normalise -> letterbox (cropping.py:338-354) -- the very crop the fp32 reference produces?
    A 0.2-0.5 px error at 512^2 is 0.5-1.2 px at 1195^2, so a centre can fall on the other side of an integer and the whole box
    moves by one pixel.  Reported per dtype: fraction of (series, level) boxes equal to the fp32 oracle's, bit-exactness of the
    crops of those, and the size of the shift of the rest.  Gate: every equal-box crop is bit-exact; no centre moves by more than
    2 px at 1195^2 for the default dtype (fp16) and for bf16 on random-init weights."""
    om = make_model("base", seed=0, trained_like=trained)
    slices = [synthetic.make_iso_slice(s, 1195, 1195) for s in range(32)]
    want = _oracle_coords(om, slices)
    dpx = ref.mm_to_pixels((50, 20, 30, 30), (0.3, 0.3))
    want_crops = [[ref.crop_region_horizontal(sl, float(want[i, l, 0]), float(want[i, l, 1]), (128, 128), dpx) for l in range(5)]
                  for i, sl in enumerate(slices)]
    pool = ops.SlicePool.from_numpy(slices, dev())
    for dtype in ("fp16", "bf16"):
        model = cropping.LocalizationModel(om.state_dict(), dev(), dtype=dtype)
        batch = pipeline.localize_and_crop(pool, model, (50, 20, 30, 30), (128, 128))
        coords, crops, _ = batch.to_host()
        same = exact = 0
        shifts = []
        for i in range(32):
            for l in range(5):
                cx, cy = int(float(coords[i, l, 0]) * 1195), int(float(coords[i, l, 1]) * 1195)
                wx, wy = int(float(want[i, l, 0]) * 1195), int(float(want[i, l, 1]) * 1195)
                if (cx, cy) == (wx, wy):
                    same += 1
                    exact += int(np.array_equal(crops[i, l], want_crops[i][l]))
                else:
                    shifts.append(max(abs(cx - wx), abs(cy - wy)))
                    near = ref.crop_region_horizontal(slices[i], float(coords[i, l, 0]), float(coords[i, l, 1]), (128, 128), dpx)
                    assert np.array_equal(crops[i, l], near)  # still the reference arithmetic on the device's own centre
        err_px = np.abs(coords - want).max() * PX
        print(f"[crop agreement] weights={'trained-like' if trained else 'random-init'} dtype={dtype}: coords max err {err_px:.3f} px @512; "
              f"{same}/160 boxes equal the fp32 oracle's ({100.0 * same / 160:.1f} %), {exact}/{same} of those crops bit-exact; "
              f"shifted boxes: {len(shifts)} (max shift {max(shifts) if shifts else 0} px at 1195^2)")
        assert exact == same
        if dtype == "fp16" or not trained:
            assert err_px <= 0.5 and (not shifts or max(shifts) <= 2)


def test_model_call_on_reference_tensor():
    """SURVEY 8b "model plug points": callers other than predict_ivd_locations run ``model(tensor)`` on the [B,3,H,W] float
    tensor they normalised themselves (generic.py:389-391; notebooks, BaseModel.test_inference).  The un-folded stem gives the
    coordinates of the folded one-plane stem (same planes) and of the fp32 oracle within the gate, for CPU and CUDA inputs,
    and for a tensor that is NOT three copies of one plane."""
    om = make_model("base", seed=0)
    model = cropping.LocalizationModel(om.state_dict(), dev())
    slices = [synthetic.make_iso_slice(40, 640, 650), synthetic.make_iso_slice(41, 1195, 1195), synthetic.make_iso_slice(42, 512, 600)]
    tensors = torch.stack([ref.preprocess_slice(sl, (512, 512))[1] for sl in slices])
    with torch.no_grad():
        want = om(tensors).numpy()
    got = model(tensors)  # CPU tensor in, as the reference's callers hold it before .to(device)
    assert got.is_cuda and tuple(got.shape) == (3, 5, 2) and got.dtype == torch.float32
    assert np.abs(got.cpu().numpy() - want).max() * PX <= 0.5
    pool = ops.SlicePool.from_numpy(slices, dev())
    folded = model.predict_u8(ops.normalize_resize(pool, (512, 512))).cpu().numpy()
    assert np.abs(got.cpu().numpy() - folded).max() * PX <= 0.1  # same network, stem weights folded vs not
    rgb = torch.randn(2, 3, 256, 384, generator=torch.Generator().manual_seed(3))
    with torch.no_grad():
        want_rgb = om(rgb).numpy()
    got_rgb = model(rgb.to(dev()).half()).cpu().numpy()
    assert np.abs(got_rgb - want_rgb).max() <= 1.0 / PX
    assert model.eval() is model and model.to("cuda:0") is model and torch.equal(model.predict(rgb), model(rgb))
    with pytest.raises(ValueError):
        model(torch.zeros(2, 1, 64, 64))


def test_checkpoint_roundtrip_and_predict_api(tmp_path):
    om = make_model("base", seed=0)
    ck = tmp_path / "best_model.pt"
    torch.save({"epoch": 3, "model_state_dict": om.state_dict(), "optimizer_state_dict": {}, "scheduler_state_dict": None,
                "best_metric": 0.0, "best_epoch": 3, "history": {}, "config": {}}, ck)  # trainers/base.py:695-706
    model = cropping.load_localization_model(ck, "base", dev())
    img = synthetic.make_iso_slice(21, 640, 650)
    locs = cropping.predict_ivd_locations(model, img, dev(), (512, 512))
    want = ref.predict_ivd_locations(om, img, "cpu", (512, 512))
    assert set(locs) == {0, 1, 2, 3, 4} and all(isinstance(v[0], float) for v in locs.values())
    assert max(abs(locs[i][k] - want[i][k]) for i in range(5) for k in range(2)) * PX <= 0.5
    bad = dict(om.state_dict())
    bad.pop("backbone.stages.1.blocks.0.gamma")
    with pytest.raises(Exception, match="gamma|stage"):
        cropping.LocalizationModel(bad, dev())


def test_pipeline_end_to_end_vs_oracle():
    om = make_model("base", seed=0)
    slices = [synthetic.make_iso_slice(30 + i, h, w) for i, (h, w) in enumerate([(1195, 1195), (640, 650), (880, 1000)])]
    model = cropping.LocalizationModel(om.state_dict(), dev(), dtype="bf16")
    pool = ops.SlicePool.from_numpy(slices, dev())
    batch = pipeline.localize_and_crop(pool, model, (50, 20, 30, 30), (128, 128), keep_planes=True)
    coords, crops, crops2 = batch.to_host()
    planes = batch.planes.cpu().numpy()
    dpx = ref.mm_to_pixels((50, 20, 30, 30), (0.3, 0.3))
    for i, sl in enumerate(slices):
        plane, _ = ref.preprocess_slice(sl, (512, 512))
        assert np.array_equal(planes[i], plane)
        for lvl in range(5):
            # crops are bit-exact given the coordinates the device produced
            want = ref.crop_region_horizontal(sl, float(coords[i, lvl, 0]), float(coords[i, lvl, 1]), (128, 128), dpx)
            assert np.array_equal(crops[i, lvl], want)
    want_c = _oracle_coords(om, slices)
    assert np.abs(coords - want_c).max() * PX <= 0.5
    # centre-crop fallback when no model is given (__init__.py:194-197)
    fb = pipeline.localize_and_crop(pool, None, (50, 20, 30, 30), (128, 128))
    c0 = fb.crops.cpu().numpy()
    for lvl, (x, y) in cropping.get_center_fallback_locations().items():
        assert np.array_equal(c0[0, lvl], ref.crop_region_horizontal(slices[0], x, y, (128, 128), dpx))


def test_streamed_driver_equals_resident_path():
    """pipeline.StreamedLocalizer (chunked H2D under compute, D2H on a third stream) is a schedule, not
    different arithmetic: identical coordinates and crops to localize_and_crop over a resident pool,
    on a ragged batch with a tail chunk, twice in a row (buffer reuse)."""
    om = make_model("base", seed=0)
    shapes = [(30, 640, 650), (31, 512, 700), (32, 900, 512), (33, 1195, 1195), (34, 350, 420), (35, 600, 600), (36, 777, 333)]
    slices = [synthetic.make_iso_slice(*c) for c in shapes]
    model = cropping.LocalizationModel(om.state_dict(), dev(), dtype="bf16", micro_batch=3)
    pool = ops.SlicePool.from_numpy(slices, dev())
    want = pipeline.localize_and_crop(pool, model, (50, 20, 30, 30), (128, 128), (512, 512), (256, 256))
    wc, wk, wk2 = want.to_host()
    series = pipeline.PinnedSeries(slices)
    streamer = pipeline.StreamedLocalizer(model, dev(), (50, 20, 30, 30), (128, 128), (512, 512), (256, 256), chunk=3)
    for _ in range(2):
        gc, gk, gk2 = streamer.run(series)
        assert np.array_equal(gc.numpy(), wc)
        assert np.array_equal(gk.numpy(), wk)
        assert np.array_equal(gk2.numpy(), wk2)
    # batches in flight: the next one is started before the previous one is collected (two output slots, shared staging)
    other = pipeline.PinnedSeries(slices[::-1])
    want_o = pipeline.localize_and_crop(ops.SlicePool.from_numpy(slices[::-1], dev()), model, (50, 20, 30, 30), (128, 128), (512, 512), (256, 256)).to_host()
    handles = [streamer.run_async(series, slot=0), streamer.run_async(other, slot=1), None]
    a = [t.numpy().copy() for t in handles[0].result()]
    handles[2] = streamer.run_async(series, slot=0)  # slot 0 again: waits for its previous D2H by itself
    b = [t.numpy().copy() for t in handles[1].result()]
    c = [t.numpy().copy() for t in handles[2].result()]
    for got, want_t in ((a, (wc, wk, wk2)), (b, want_o), (c, (wc, wk, wk2))):
        assert all(np.array_equal(g, w) for g, w in zip(got, want_t))
    # centre-crop fallback (no model, __init__.py:194-197)
    fb = pipeline.StreamedLocalizer(None, dev(), (50, 20, 30, 30), (128, 128), (512, 512), None, chunk=4)
    fc, fk, fk2 = fb.run(series)
    ref_fb = pipeline.localize_and_crop(pool, None, (50, 20, 30, 30), (128, 128), (512, 512), None)
    assert fk2 is None and np.array_equal(fk.numpy(), ref_fb.crops.cpu().numpy()) and np.allclose(fc.numpy(), ref_fb.coords.cpu().numpy())


@pytest.mark.parametrize("image_size", [(768, 768), (512, 768), (640, 384)])
def test_model_other_input_sizes_config5(image_size):
    """BASELINE config 5 runs the localizer at 768x768; image_size is a config field (config.py:53-54), so any multiple
    of 32 must work, square or not.  Same normalised tolerance as the 512^2 gate (0.5 px / 512).  The random-init weights
    (layer scale 1e-6) test the stem, the downsample layers and the head; the trained-like fp16 row, gated by what the emulation
    of the device numerics predicts for the size, tests the ConvNeXt blocks."""
    om = make_model("base", seed=0)
    slices = [synthetic.make_iso_slice(50, 1195, 1195), synthetic.make_iso_slice(51, 700, 900)]
    want = []
    for sl in slices:
        _, t = ref.preprocess_slice(sl, image_size)
        with torch.no_grad():
            want.append(om(t.unsqueeze(0))[0].numpy())
    want = np.stack(want)
    model = cropping.LocalizationModel(om.state_dict(), dev(), dtype="bf16")
    pool = ops.SlicePool.from_numpy(slices, dev())
    planes = ops.normalize_resize(pool, image_size)
    for i, sl in enumerate(slices):
        plane, _ = ref.preprocess_slice(sl, image_size)
        assert np.array_equal(planes[i].cpu().numpy(), plane)
    got = model.predict_u8(planes).cpu().numpy()
    err = np.abs(got - want).max()
    print(f"[coords] image_size={image_size}: max normalised error {err:.2e} ({err * 512:.3f} px at 512)")
    assert err <= 0.5 / 512
    tm = make_model("base", seed=0, trained_like=True)
    want_t, pred, gate = trained_like_gate(tm, torch.stack([ref.preprocess_slice(sl, image_size)[1] for sl in slices]))
    got_t = cropping.LocalizationModel(tm.state_dict(), dev(), dtype="fp16").predict_u8(planes).cpu().numpy()
    err_t = np.abs(got_t - want_t).max() * PX
    print(f"[coords] image_size={image_size} trained-like fp16: {err_t:.4f} px (x 512), emulator predicts {pred:.4f}, gate {gate:.3f}")
    assert err_t <= gate


def test_config3_ragged_volumes_with_their_own_spacing():
    """BASELINE config 3 in miniature: series of different in-plane size AND spacing (so different iso sizes and the same
    0.3 mm crop box), from the volume on, against the oracle chain itk_resample -> preprocess -> fp32 model -> crop."""
    from oracle import itk_resample as itk

    om = make_model("base", seed=0)
    model = cropping.LocalizationModel(om.state_dict(), dev(), dtype="bf16")
    rng = np.random.default_rng(3)
    vols, sps, dirs = [], [], []
    for k in range(4):
        h, w = int(rng.integers(320, 700)), int(rng.integers(320, 700))
        sp = float(rng.uniform(0.30, 0.95))
        v, _, d = synthetic.make_volume(60 + k, int(rng.integers(11, 24)), h, w, (sp, sp, float(rng.uniform(3.3, 4.8))))
        vols.append(v); sps.append((sp, sp, 4.0)); dirs.append(d)
    batch = pipeline.localize_and_crop_volumes(vols, sps, dirs, model, dev(), crop_delta_mm=(50, 20, 30, 30), crop_size=(128, 128))
    coords, crops, _ = batch.to_host()
    for i in range(4):
        sl, sp2 = itk.resample_middle_sagittal(vols[i], sps[i], dirs[i])
        _, t = ref.preprocess_slice(sl, (512, 512))
        with torch.no_grad():
            want_c = om(t.unsqueeze(0))[0].numpy()
        assert np.abs(coords[i] - want_c).max() * PX <= 0.5
        dpx = ref.mm_to_pixels((50, 20, 30, 30), sp2)
        for lvl in range(5):
            want = ref.crop_region_horizontal(sl, float(coords[i, lvl, 0]), float(coords[i, lvl, 1]), (128, 128), dpx)
            assert np.array_equal(crops[i, lvl], want)


def test_model_batch_composition_invariance_at_bench_size():
    """Size-independent property at BASELINE config-2 scale (256 slices, micro-batch 37 -> 6 full chunks + a tail of 34): an
    image's coordinates do not depend on where it sits in the batch or on the micro-batch size (every kernel is
    deterministic and per-image), so a permuted batch gives the permuted result bit for bit."""
    om = make_model("base", seed=0)
    g = torch.Generator().manual_seed(5)
    distinct = torch.randint(0, 256, (6, 512, 512), generator=g, dtype=torch.uint8)
    idx = torch.randint(0, 6, (256,), generator=g)
    planes = distinct[idx].contiguous().to(dev())
    perm = torch.randperm(256, generator=g)
    m37 = cropping.LocalizationModel(om.state_dict(), dev(), dtype="bf16", micro_batch=37)
    a = m37.predict_u8(planes).cpu()
    b = m37.predict_u8(planes[perm.to(dev())].contiguous()).cpu()
    assert torch.equal(b, a[perm])
    for k in range(6):  # identical inputs -> identical outputs, wherever they sit
        rows = a[idx == k]
        assert (rows == rows[0]).all()
    m5 = cropping.LocalizationModel(om.state_dict(), dev(), dtype="bf16", micro_batch=5)
    assert torch.equal(m5.predict_u8(planes[:23].contiguous()).cpu(), a[:23])


def test_model_config5_scale_768_batch():
    """BASELINE config 5 geometry (768 x 768 input) over more than one micro-batch: finite, in (0, 1), permutation-consistent."""
    om = make_model("base", seed=0)
    g = torch.Generator().manual_seed(6)
    distinct = torch.randint(0, 256, (3, 768, 768), generator=g, dtype=torch.uint8)
    idx = torch.randint(0, 3, (80,), generator=g)
    planes = distinct[idx].contiguous().to(dev())
    model = cropping.LocalizationModel(om.state_dict(), dev(), dtype="bf16", micro_batch=37)
    out = model.predict_u8(planes).cpu()
    assert out.shape == (80, 5, 2) and torch.isfinite(out).all() and (out > 0).all() and (out < 1).all()
    for k in range(3):
        rows = out[idx == k]
        assert (rows == rows[0]).all()


@pytest.mark.parametrize("variant,dims", [("xlarge", (256, 512, 1024, 2048)), ("large", (192, 384, 768, 1536)),
                                          ("small", (96, 192, 384, 768)), ("tiny", (96, 192, 384, 768))])
def test_model_other_variants(variant, dims):
    """config.model_variant (config.py:27-39) beyond "base": every other ConvNeXt-v1 size -- tiny / small (96-channel stem: one
    and a half 64-channel chunks), large (multiples of 64 only), xlarge.  Same gate as base: 0.5 px at 512^2 vs the fp32 oracle.
    Random-init weights (layer scale 1e-6) hide every block, so they test the stem, the downsample layers and the head at these
    widths; the trained-like fp16 row tests the blocks, gated by what the emulation of the device numerics predicts."""
    om = make_model(variant, seed=0)
    slices = [synthetic.make_iso_slice(80, 700, 640), synthetic.make_iso_slice(81, 512, 512)]
    want = _oracle_coords(om, slices)
    model = cropping.LocalizationModel(om.state_dict(), dev(), dtype="bf16")
    assert tuple(model.engine.dims) == dims
    pool = ops.SlicePool.from_numpy(slices, dev())
    got = model.predict_u8(ops.normalize_resize(pool, (512, 512))).cpu().numpy()
    err_px = np.abs(got - want).max() * PX
    print(f"[coords] {variant} bf16: max error {err_px:.4f} px")
    assert np.isfinite(got).all() and err_px <= 0.5
    tm = make_model(variant, seed=0, trained_like=True)
    want_t, pred, gate = trained_like_gate(tm, torch.stack([ref.preprocess_slice(sl, (512, 512))[1] for sl in slices]))
    got_t = cropping.LocalizationModel(tm.state_dict(), dev(), dtype="fp16").predict_u8(ops.normalize_resize(pool, (512, 512))).cpu().numpy()
    err_t = np.abs(got_t - want_t).max() * PX
    print(f"[coords] {variant} trained-like fp16: max error {err_t:.4f} px, emulator predicts {pred:.4f} px, gate {gate:.3f} px")
    assert np.isfinite(got_t).all() and err_t <= gate


@pytest.mark.parametrize("variant,dims,tol_px", [("v2_base", (128, 256, 512, 1024), 0.5), ("v2_tiny", (96, 192, 384, 768), 0.5),
                                                 ("v2_large", (192, 384, 768, 1536), 0.5)])
def test_model_convnext_v2_grn(variant, dims, tol_px):
    """config.model_variant = v2_* (config.py:27-39): timm convnextv2 -- GlobalResponseNorm inside every block's MLP, no layer
    scale.  The GRN weights are zero at init (identity), so the oracle model gets random ones; fp16 operands, 0.5 px gate
    (without the 1e-6 layer scale every block contributes, like the "trained-like" v1 case)."""
    om = make_model(variant, seed=0, trained_like=True)
    slices = [synthetic.make_iso_slice(90, 640, 600), synthetic.make_iso_slice(91, 512, 512), synthetic.make_iso_slice(92, 700, 512)]
    want = _oracle_coords(om, slices)
    model = cropping.LocalizationModel(om.state_dict(), dev(), dtype="fp16", micro_batch=2)  # 2 + 1: the per-image norm must not mix images
    assert tuple(model.engine.dims) == dims
    pool = ops.SlicePool.from_numpy(slices, dev())
    planes = ops.normalize_resize(pool, (512, 512))
    got = model.predict_u8(planes).cpu().numpy()
    err_px = np.abs(got - want).max() * PX
    print(f"[coords] {variant} fp16 (GRN): max error {err_px:.4f} px")
    assert np.isfinite(got).all() and err_px <= tol_px
    # per-image statistic: an image's coordinates do not depend on its neighbours in the batch
    solo = model.predict_u8(planes[1:2].contiguous()).cpu().numpy()
    assert np.array_equal(solo[0], got[1])
    # a small input (the last stage has 2 x 3 tokens): the per-stage scratch of the response norm is sized by its largest stage
    small = ops.normalize_resize(pool, (64, 96))
    want_s = []
    for sl in slices:
        _, t = ref.preprocess_slice(sl, (64, 96))
        with torch.no_grad():
            want_s.append(om(t.unsqueeze(0))[0].numpy())
    got_s = model.predict_u8(small).cpu().numpy()
    assert np.abs(got_s - np.stack(want_s)).max() <= tol_px / PX
