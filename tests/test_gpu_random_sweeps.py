"""GPU parity: seeded random sweeps of K1 and K3 against the port of the reference (NumPy + Pillow + OpenCV themselves).
The fixed cases elsewhere were picked by hand; these walk shapes nobody picked: 1-pixel and few-pixel slices, widths that are
not multiples of 4, strips, slices full of exact ties with the minimum, integer-valued and negative data, crop boxes hanging
over every border, non-square crop sizes, zero deltas on one side."""
import numpy as np
import pytest
import torch
from PIL import Image

from gpu_util import dev, trained_like_gate
from oracle import fixedpoint as fx
from oracle import reference_path as ref
from spine_vision_b200 import cropping, ops, synthetic

pytestmark = pytest.mark.gpu


def _random_slice(rng, h, w):
    kind = int(rng.integers(0, 6))
    if kind == 0:  # MRI-like: exact-zero background (ties with the minimum), smooth foreground
        a = synthetic.make_iso_slice(int(rng.integers(0, 1 << 30)), h, w)
    elif kind == 1:  # integer-valued (what a DICOM decodes to), narrow range: many exact products k/range*255
        a = rng.integers(0, int(rng.integers(2, 700)), size=(h, w)).astype(np.float32)
    elif kind == 2:  # negative and positive, wide range
        a = (rng.standard_normal((h, w)) * 1e4).astype(np.float32)
    elif kind == 3:  # tiny range around a large offset (rounding of x - min matters)
        a = (1000.0 + rng.random((h, w)) * 1e-2).astype(np.float32)
    elif kind == 4:  # constant: the reference casts instead of scaling
        a = np.full((h, w), float(rng.integers(-300, 600)), dtype=np.float32)
    else:  # values that land exactly on the 0..255 grid after scaling
        a = rng.integers(0, 256, size=(h, w)).astype(np.float32) * 4.0
        a.flat[0], a.flat[-1] = 0.0, 1020.0
    return np.ascontiguousarray(a, dtype=np.float32)


def _random_shape(rng, big):
    pick = int(rng.integers(0, 5))
    if pick == 0:
        return int(rng.integers(1, 9)), int(rng.integers(1, 9))
    if pick == 1:
        return int(rng.integers(1, 40)), int(rng.integers(200, 900))
    if pick == 2:
        return int(rng.integers(200, 900)), int(rng.integers(1, 40))
    if pick == 3 and big:
        return int(rng.integers(900, 2600)), int(rng.integers(900, 2600))
    return int(rng.integers(9, 900)), int(rng.integers(9, 900))


@pytest.mark.parametrize("out_hw,big,seed", [((512, 512), True, 0), ((512, 512), True, 1), ((256, 384), False, 2), ((64, 96), False, 3),
                                             ((768, 768), True, 4)])
def test_k1_random_ragged_batches_vs_reference_chain(out_hw, big, seed):
    """normalize_to_uint8 -> PIL -> Resize (io/__init__.py:15-30, cropping.py:463-472) on 24 random slices per batch."""
    rng = np.random.default_rng(1000 + seed)
    slices = []
    for _ in range(24):
        h, w = _random_shape(rng, big)
        slices.append(_random_slice(rng, h, w))
    pool = ops.SlicePool.from_numpy(slices, dev())
    out, mm = ops.normalize_resize(pool, out_hw, return_minmax=True)
    out, mm = out.cpu().numpy(), mm.cpu().numpy()
    for i, a in enumerate(slices):
        u8 = ref.normalize_to_uint8(a)
        if a.shape[0] > 100 * a.shape[1] and out_hw[0] < a.shape[0]:
            # the installed Pillow 12.2.0 resizes such slivers vertically first (Image.py, resize); the reference pins Pillow 10.2.0
            # (uv.lock:2563-2564), which has the one order K1 implements: horizontal, then vertical (tests/test_oracle.py
            # pins both statements)
            want = fx.pillow_resize_u8(u8, out_hw)
        else:
            want = np.asarray(Image.fromarray(u8).resize((out_hw[1], out_hw[0]), Image.BILINEAR))
        assert mm[i, 0] == a.min() and mm[i, 1] == a.max()
        assert np.array_equal(out[i], want), f"slice {i} {a.shape} -> {out_hw}: {(out[i] != want).sum()} px differ"
    only = ops.normalize_u8(pool)  # the no-resize entry of the localization dataset builder on the same batch
    flat = only.cpu().numpy()
    offs = pool.offs.cpu().numpy()
    for i, a in enumerate(slices):
        got = flat[offs[i] : offs[i] + a.size].reshape(a.shape)
        assert np.array_equal(got, ref.normalize_to_uint8(a)), f"normalize_u8 slice {i} {a.shape}"


@pytest.mark.parametrize("crop_size,second,seed", [((128, 128), (256, 256), 0), ((256, 256), None, 1), ((96, 160), (224, 224), 2),
                                                   ((64, 32), (128, 64), 3), ((224, 224), (224, 224), 4)])
def test_k3_random_boxes_vs_reference(crop_size, second, seed):
    """crop_region_horizontal (cropping.py:316-354) on 160 random (slice, centre, deltas) rows in one launch; the second output
    against Pillow's resize of the first (training/datasets/classification.py:247-278)."""
    rng = np.random.default_rng(2000 + seed)
    slices = []
    for _ in range(10):
        h, w = _random_shape(rng, False)
        slices.append(_random_slice(rng, h, w))
    pool = ops.SlicePool.from_numpy(slices, dev())
    n = 160
    idx = rng.integers(0, len(slices), size=n).astype(np.int32)
    xy = rng.random((n, 2)).astype(np.float32)
    xy[rng.random(n) < 0.15] = 0.0
    xy[rng.random(n) < 0.15, 0] = np.float32(0.99999)
    delta = np.stack([rng.integers(0, 150, size=n), rng.integers(1, 150, size=n), rng.integers(0, 120, size=n),
                      rng.integers(1, 120, size=n)], axis=1).astype(np.int32)
    max_box = (int((delta[:, 2] + delta[:, 3]).max()), int((delta[:, 0] + delta[:, 1]).max()))
    crops, crops2, geom = ops.crop_resample(pool, torch.from_numpy(idx).to(dev()), torch.from_numpy(xy).to(dev()),
                                            torch.from_numpy(delta).to(dev()), max_box, crop_size, second, return_geom=True)
    crops = crops.cpu().numpy()
    crops2 = None if crops2 is None else crops2.cpu().numpy()
    checked = raised = 0
    for k in range(n):
        a = slices[idx[k]]
        try:
            want = ref.crop_region_horizontal(a, float(xy[k, 0]), float(xy[k, 1]), crop_size, tuple(int(v) for v in delta[k]))
        except Exception:  # noqa: BLE001 -- the reference raises (cv2.resize to a zero-sized target); its drivers skip the series
            raised += 1
            assert crops[k].max() == 0, f"row {k}: the reference raises here, K3 must hand back an empty canvas"
            continue
        assert np.array_equal(crops[k], want), f"row {k} slice {a.shape} xy {xy[k]} delta {delta[k]}: {(crops[k] != want).sum()} px differ"
        if crops2 is not None:
            up = np.asarray(Image.fromarray(want).resize((second[1], second[0]), Image.BILINEAR))
            assert np.array_equal(crops2[k], up), f"row {k}: second output"
        checked += 1
    assert checked >= 120, (checked, raised)


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_k3_random_rotated_vs_reference(seed):
    """CropContext(mode="rotated") (cropping.py:172-313, 357-404) on random slices and random five-point spines -- including
    nearly vertical, zig-zag and coincident points -- against the reference arithmetic (np.polyfit angles + cv2.warpAffine)."""
    rng = np.random.default_rng(3000 + seed)
    total = 0
    for _ in range(6):
        h, w = int(rng.integers(60, 1000)), int(rng.integers(60, 1000))
        img = _random_slice(rng, h, w)
        xs = np.clip(0.5 + np.cumsum(rng.normal(0, 0.05, 5)), 0.02, 0.98)
        ys = np.sort(rng.random(5)) if rng.random() < 0.8 else rng.random(5)
        if rng.random() < 0.2:
            xs[2], ys[2] = xs[1], ys[1]  # two coincident discs
        locs = {i: (float(np.float32(xs[i])), float(np.float32(ys[i]))) for i in range(5)}
        dpx = tuple(int(v) for v in (rng.integers(20, 170), rng.integers(10, 80), rng.integers(20, 110), rng.integers(20, 110)))
        boost = float(rng.choice([1.0, 1.5, 2.0]))
        cs = (128, 128) if rng.random() < 0.7 else (96, 160)
        want_ctx = ref.CropContext(img, locs, cs, dpx, "rotated", boost)
        got_ctx = cropping.CropContext(img, locs, cs, dpx, "rotated", last_disc_angle_boost=boost, device=dev())
        assert [got_ctx.rotation_angles[i] for i in range(5)] == [want_ctx.rotation_angles[i] for i in range(5)]
        got = got_ctx.crop_all(range(5))
        for i in range(5):
            want = want_ctx.crop(i)
            assert np.array_equal(got[i], want), f"slice {(h, w)} level {i} angle {want_ctx.rotation_angles[i]:.2f}: {(got[i] != want).sum()} px differ"
            total += 1
    assert total == 30


@pytest.mark.parametrize("image_size", [(32, 32), (64, 32), (32, 96), (96, 160), (224, 224), (352, 288), (1024, 512)])
def test_localizer_unusual_image_sizes_vs_fp32_oracle(image_size):
    """``image_size`` is a config field (config.py:53-54): every multiple of 32 must work, down to 32 x 32 where the last stage
    is a single token and every depthwise window hangs over all four borders.  Same normalised gate as at 512^2 (0.5 px / 512).
    Random-init weights (layer scale 1e-6) test the stem, the downsample layers and the head; the trained-like fp16 row tests the
    ConvNeXt blocks (depthwise windows over the borders, tensor-core depthwise modes A and B), gated by what the emulation of the
    device numerics predicts for the size."""
    from oracle.convnext import make_model

    om = make_model("base", seed=0)
    slices = [synthetic.make_iso_slice(300, 400, 380), synthetic.make_iso_slice(301, 333, 517), synthetic.make_iso_slice(302, 640, 650)]
    model = cropping.LocalizationModel(om.state_dict(), dev(), dtype="bf16", micro_batch=2)
    pool = ops.SlicePool.from_numpy(slices, dev())
    planes = ops.normalize_resize(pool, image_size)
    want = []
    for i, sl in enumerate(slices):
        plane, t = ref.preprocess_slice(sl, image_size)
        assert np.array_equal(planes[i].cpu().numpy(), plane)
        with torch.no_grad():
            want.append(om(t.unsqueeze(0))[0].numpy())
    got = model.predict_u8(planes).cpu().numpy()
    err = float(np.abs(got - np.stack(want)).max())
    print(f"[coords] image_size={image_size}: max normalised error {err:.2e}")
    assert np.isfinite(got).all() and err <= 0.5 / 512
    tm = make_model("base", seed=0, trained_like=True)
    want_t, pred, gate = trained_like_gate(tm, torch.stack([ref.preprocess_slice(sl, image_size)[1] for sl in slices]))
    got_t = cropping.LocalizationModel(tm.state_dict(), dev(), dtype="fp16", micro_batch=2).predict_u8(planes).cpu().numpy()
    err_t = float(np.abs(got_t - want_t).max()) * 512
    print(f"[coords] image_size={image_size} trained-like fp16: {err_t:.4f} px (x 512), emulator predicts {pred:.4f}, gate {gate:.3f}")
    assert np.isfinite(got_t).all() and err_t <= gate


def _k0_random_cases(seed, n):
    """Volumes in every axis-aligned orientation (signed permutations), a few oblique ones, random sizes down to a single slice,
    random anisotropic spacings, float and integer pixel types."""
    import itertools

    rng = np.random.default_rng(seed)
    perms = list(itertools.permutations(range(3)))
    cases = []
    for k in range(n):
        shape = (int(rng.integers(1, 12)), int(rng.integers(2, 60)), int(rng.integers(2, 60)))  # z, y, x
        sp = (float(rng.uniform(0.25, 2.5)), float(rng.uniform(0.25, 2.5)), float(rng.uniform(0.3, 5.0)))
        if k % 4 == 3:  # oblique: a random rotation close to a signed permutation
            q, _ = np.linalg.qr(np.eye(3)[list(perms[int(rng.integers(0, 6))])] * rng.choice([-1.0, 1.0], size=3) + rng.normal(0, 0.08, (3, 3)))
            d = tuple(float(v) for v in q.ravel())
        else:
            m = np.eye(3)[list(perms[(k // 8) % 6])] * np.array([1.0 if (k >> b) & 1 else -1.0 for b in range(3)])
            d = tuple(float(v) for v in m.T.ravel())
        kind = k % 3
        if kind == 0:
            v = (rng.random(shape) * 1500).astype(np.float32)
        elif kind == 1:
            v = rng.integers(-500, 3000, size=shape).astype(np.int16)
        else:
            v = rng.integers(0, 256, size=shape).astype(np.uint8)
        cases.append((v, sp, d))
    return cases


@pytest.mark.parametrize("seed", [0, 1])
def test_k0_random_orientations_sizes_types_vs_itk_restatement(seed):
    """K0 against oracle/itk_resample.py (parity unpinned: SimpleITK absent) on 48 random volumes per seed."""
    from oracle import itk_resample as itk
    from spine_vision_b200 import volumes

    cases = _k0_random_cases(4000 + seed, 48)
    want = [itk.resample_middle_sagittal(v, sp, d) for v, sp, d in cases]
    pool, spacings = volumes.midplane_resample([c[0] for c in cases], [c[1] for c in cases], [c[2] for c in cases], dev())
    flat, offs = pool.data.cpu().numpy(), pool.offs.cpu().numpy()
    for i, (w, wsp) in enumerate(want):
        h_, w_ = pool.shapes[i]
        assert (h_, w_) == w.shape and spacings[i] == wsp, (i, (h_, w_), w.shape, spacings[i], wsp)
        got = flat[offs[i] : offs[i] + h_ * w_].reshape(h_, w_)
        assert np.array_equal(got, w.astype(np.float32)), f"case {i} {cases[i][0].shape} {cases[i][0].dtype} dir {cases[i][2]}: max diff {np.abs(got - w).max()}"


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_dwconv_tensor_core_random_shapes_vs_torch_and_fp32_pipe(seed):
    """The tensor-core depthwise kernel (``svb_dwconv_raw_tc``) on shapes nobody picked: heights and widths 1 .. 70 (mode A for
    widths 8 / 16 / 32, windows otherwise; images smaller than the stencil; one-row and one-column images), channel counts
    128 .. 512, batches 1 .. 5, activations with outliers.  Against (a) PyTorch's fp32 depthwise convolution with the taps rounded to
    fp16 (the kernel's operands) within the packed-shuffle budget, (b) the FP32-pipe kernel ``svb_dwconv_raw`` on the same input:
    statistics agree to 2e-3 relative."""
    import torch.nn.functional as F
    rng = np.random.default_rng(1000 + seed)
    g = torch.Generator().manual_seed(seed)
    for _ in range(14):
        B, C = int(rng.integers(1, 6)), int(rng.choice([128, 192, 256, 384, 512]))  # widths both kernels are built for
        H = int(rng.choice([1, 2, 3, 5, 7, 8, 9, 16, 17, 31, 32, 33, 40, 64, 70]))
        W = int(rng.choice([1, 2, 4, 6, 8, 9, 16, 20, 26, 27, 32, 33, 52, 53, 64, 70]))
        x = torch.randn(B, H, W, C, generator=g)
        x[torch.rand(B, H, W, C, generator=g) < 0.01] *= 30.0  # outliers
        x = x.to(torch.float16)
        wt = torch.randn(C, 1, 7, 7, generator=g) * 0.15
        bias = torch.randn(C, generator=g) * 0.2
        y = F.conv2d(x.float().permute(0, 3, 1, 2), wt.to(torch.float16).float(), bias, padding=3, groups=C).permute(0, 2, 3, 1)
        taps = wt.reshape(C, 49).t().contiguous()
        xd, td, bd = x.to(dev()), taps.to(dev()), bias.to(dev())
        raw, stat = ops.dwconv_raw_tc(xd, ops.dwconv_tc_pack(td, torch.float16), bd)
        ref_raw, ref_stat = ops.dwconv_raw(xd, td, bd)
        torch.cuda.synchronize()
        err = (raw.float().cpu() - y).abs()
        # output rounding + six fp16-rounded column partial sums; partial sums can exceed the total when columns cancel, so the
        # budget is taken against the magnitude sum of one column's terms
        mag = F.conv2d(x.float().abs().permute(0, 3, 1, 2), wt.abs(), None, padding=3, groups=C).permute(0, 2, 3, 1)
        tol = 2.0 ** -11 * (y.abs() + 3.0 * mag + 1.0)
        assert int((err > tol).sum()) == 0, f"B={B} H={H} W={W} C={C}: max err {err.max().item():.4g}"
        assert torch.isfinite(stat).all()
        rs, rr = stat.cpu(), ref_stat.cpu()
        assert torch.allclose(rs[:, 0], rr[:, 0], rtol=4e-3, atol=1e-6), f"B={B} H={H} W={W} C={C}: rstd {(rs[:, 0] - rr[:, 0]).abs().max()}"
        assert torch.allclose(rs[:, 1], rr[:, 1], rtol=4e-3, atol=4e-3), f"B={B} H={H} W={W} C={C}: -mu rstd {(rs[:, 1] - rr[:, 1]).abs().max()}"
