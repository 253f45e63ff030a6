"""GPU: model_variant = "v2_huge" (timm convnextv2_huge: depths 3 / 3 / 27 / 3, widths 352 / 704 / 1408 / 2816, GRN in every
block, no layer scale) through the whole localizer forward.  Its widths reach kernels at shapes no other variant has: a
352-wide stem (11 channels per lane), LayerNorm + patchify at 352 / 704 / 1408, the FP32-pipe depthwise kernel at 352 (5.5
channel chunks), the tensor-core depthwise kernel at 44 chunks, GEMMs with K = 352 and N up to 11264, GRN at 4C = 11264 and the
head at 2816 channels."""
import copy

import numpy as np
import pytest
import torch
from PIL import Image

from gpu_util import dev, fp32, trained_like_gate
from oracle import emulate
from oracle import reference_path as ref
from oracle.convnext import make_model
from spine_vision_b200 import _lib, cropping, ops, synthetic
from test_gpu_gemm import test_dwconv_raw_and_folded_layernorm_vs_torch as check_dwconv_raw
from test_gpu_gemm import test_dwconv_raw_tc_and_folded_layernorm_vs_torch as check_dwconv_raw_tc
from test_gpu_gemm import test_stem_patchify_other_widths as check_stem_patchify
from test_gpu_stages import DTYPES, NORM_X, _inputs, stage_gate, stage_metrics

pytestmark = pytest.mark.gpu
PX = 512.0
DIMS = (352, 704, 1408, 2816)
SLICES = [(90, 640, 600), (91, 512, 512), (92, 700, 512)]
UNSUPPORTED_MODEL = -7


@pytest.fixture(scope="module")
def trained():
    return make_model("v2_huge", seed=0, trained_like=True)


@pytest.fixture(scope="module")
def random_init():
    return make_model("v2_huge", seed=3)


@pytest.fixture(scope="module")
def checkpoint(tmp_path_factory, random_init):
    """A LocalizationTrainer-format checkpoint (trainers/base.py:695-706) of a v2_huge model: about 2.6 GB of fp32."""
    path = tmp_path_factory.mktemp("v2_huge") / "best_model.pt"
    torch.save({"epoch": 1, "model_state_dict": random_init.state_dict()}, path)
    return path


def _planes(slices, size=(512, 512)):
    pool = ops.SlicePool.from_numpy(slices, dev())
    return ops.normalize_resize(pool, size)


def _oracle_coords(om, slices, size=(512, 512)):
    x = torch.stack([ref.preprocess_slice(sl, size)[1] for sl in slices])
    return fp32(emulate.oracle_stages, copy.deepcopy(om).to(dev()), x.to(dev()))[0].cpu().numpy()


def _stages(om, dtype, size, mb=2, B=5):
    planes, x = _inputs(size, B)
    model = cropping.LocalizationModel(om.state_dict(), dev(), dtype=dtype, micro_batch=mb)
    assert tuple(model.engine.dims) == DIMS
    coords, dev_st = model.predict_u8_stages(torch.from_numpy(planes).to(dev()))
    om_d, x_d = copy.deepcopy(om).to(dev()), x.to(dev())
    want, ref_st = fp32(emulate.oracle_stages, om_d, x_d)
    emu, emu_st = fp32(emulate.forward_stages, om_d, x_d, DTYPES[dtype])
    return coords, [t.float() for t in dev_st], want, ref_st, emu, emu_st


# fp16 at 512^2, 352 x 288 (mode-B windows of the tensor-core depthwise kernel) and 32^2 (one token in the last stage); bf16 at
# 256^2 puts the FP32-pipe depthwise kernel at every width
@pytest.mark.parametrize("dtype,size", [("fp16", (512, 512)), ("fp16", (352, 288)), ("fp16", (32, 32)), ("bf16", (256, 256))])
def test_v2_huge_stages_vs_fp32_and_emulator(trained, dtype, size):
    """Micro-batch 2 over 5 images (chunks on both chains plus a tail chunk of one image), the gates of test_gpu_stages.py."""
    coords, dev_st, want, ref_st, emu, emu_st = _stages(trained, dtype, size)
    ok, rows = stage_gate(dev_st, emu_st, ref_st)
    e_dev = float((coords - want).abs().max()) * PX
    e_emu = float((emu - want).abs().max()) * PX
    print(f"\n[stages] v2_huge {dtype} {size[0]}x{size[1]} B=5 micro_batch=2: coords dev {e_dev:.4f} px, emulator {e_emu:.4f} px (x 512)")
    for r in rows:
        print("  " + r)
    assert ok, f"v2_huge {dtype} {size}: " + "; ".join(r for r in rows if r.endswith("FAIL"))


def test_v2_huge_raw_depthwise_switch(trained, monkeypatch):
    """SVB_DWCONV_TC2=0 puts the FP32-pipe depthwise kernel at 704 / 1408 / 2816 too.  The emulator rounds as the tensor-core
    kernel does there, so the device-vs-emulator gate does not apply: per stage the device stays within NORM_X of the emulator's
    distance to fp32, and the coordinates stay within 0.5 px of the default path, the bound of
    test_alternative_block_kernels_still_agree.  (Measured on a B200: 0.29 px from fp32 against the default path's 0.36, the
    two 0.16 px apart -- two draws of 16-bit rounding noise; per stage 0.87-1.00 of the emulator's distance to fp32.)"""
    size = (512, 512)
    planes, _ = _inputs(size, 5)
    default = cropping.LocalizationModel(trained.state_dict(), dev(), dtype="fp16", micro_batch=2)
    c_default = default.predict_u8(torch.from_numpy(planes).to(dev())).cpu()
    del default
    monkeypatch.setenv("SVB_DWCONV_TC2", "0")
    coords, dev_st, want, ref_st, emu, emu_st = _stages(trained, "fp16", size)
    apart = float((coords.cpu() - c_default).abs().max()) * PX
    print(f"\n[stages] v2_huge fp16 SVB_DWCONV_TC2=0 512x512: coords {float((coords - want).abs().max()) * PX:.4f} px vs fp32, "
          f"{apart:.4f} px from the default path")
    ok = True
    for s, (d, e, r) in enumerate(zip(dev_st, emu_st, ref_st)):
        (dn, _), (en, _) = stage_metrics(d, r), stage_metrics(e, r)
        print(f"  stage {s}: dev/fp32 {dn:.2e} | emu/fp32 {en:.2e} | ratio {dn / en:.2f}")
        ok &= dn <= NORM_X * en
    assert ok and apart <= 0.5


def test_v2_huge_coords_random_init_vs_oracle(random_init):
    """Random-init weights, slices through K1 and predict_u8: 0.5 px at 512^2.  An image alone gives the same bits as the same
    image in a batch (GRN is a per-image statistic)."""
    slices = [synthetic.make_iso_slice(*c) for c in SLICES]
    want = _oracle_coords(random_init, slices)
    model = cropping.LocalizationModel(random_init.state_dict(), dev(), micro_batch=2)
    assert tuple(model.engine.dims) == DIMS and model.engine.dtype == "fp16"
    planes = _planes(slices)
    got = model.predict_u8(planes).cpu().numpy()
    err = np.abs(got - want).max() * PX
    print(f"[coords] v2_huge random-init fp16: max error {err:.4f} px")
    assert np.isfinite(got).all() and err <= 0.5
    solo = model.predict_u8(planes[1:2].contiguous()).cpu().numpy()
    assert np.array_equal(solo[0], got[1])


def test_v2_huge_coords_trained_like_vs_oracle(trained):
    """Trained-like weights (every block counts), slices through K1: 0.5 px, or twice what the emulator predicts."""
    slices = [synthetic.make_iso_slice(*c) for c in SLICES]
    x = torch.stack([ref.preprocess_slice(sl, (512, 512))[1] for sl in slices])
    want, pred, gate = trained_like_gate(trained, x)
    got = cropping.LocalizationModel(trained.state_dict(), dev(), micro_batch=2).predict_u8(_planes(slices)).cpu().numpy()
    err = np.abs(got - want).max() * PX
    print(f"[coords] v2_huge trained-like fp16: max error {err:.4f} px, emulator predicts {pred:.4f} px, gate {gate:.3f} px")
    assert np.isfinite(got).all() and err <= gate


def test_v2_huge_model_call_on_tensor(random_init):
    """model(tensor) on a [B,3,H,W] float tensor (the un-folded stem at 352 channels) vs the fp32 oracle, and vs the folded stem
    on the same planes."""
    slices = [synthetic.make_iso_slice(*c) for c in SLICES[:2]]
    tensors = torch.stack([ref.preprocess_slice(sl, (512, 512))[1] for sl in slices])
    want = _oracle_coords(random_init, slices)
    model = cropping.LocalizationModel(random_init.state_dict(), dev())
    got = model(tensors)
    assert got.is_cuda and tuple(got.shape) == (2, 5, 2)
    err = np.abs(got.cpu().numpy() - want).max() * PX
    folded = model.predict_u8(_planes(slices)).cpu().numpy()
    print(f"[coords] v2_huge model(tensor): {err:.4f} px vs fp32, {np.abs(got.cpu().numpy() - folded).max() * PX:.4f} px from the folded stem")
    assert err <= 0.5 and np.abs(got.cpu().numpy() - folded).max() * PX <= 0.1


# ---------------------------------------------------------------------------------------------------- layers vs torch fp32
@pytest.mark.parametrize("dtype", ["bf16", "fp16"])
@pytest.mark.parametrize("C", [352, 704, 1408])
def test_v2_huge_stem_and_patchify(dtype, C):
    """The stem at 352 channels (CPL = 12, one part-filled lane) and LayerNorm + patchify at the stage 0-2 widths."""
    check_stem_patchify(dtype, 352, C)


@pytest.mark.parametrize("dtype", ["bf16", "fp16"])
@pytest.mark.parametrize("B,H,W,C", [(2, 33, 40, 352), (4, 128, 64, 352), (1, 9, 13, 2816), (2, 16, 16, 2816), (2, 17, 32, 1408), (1, 15, 23, 704)])
def test_v2_huge_dwconv_raw(B, H, W, C, dtype):
    """FP32-pipe depthwise + folded LayerNorm (TH = 4 tiles, and TH = 8 at 4 x 128 x 64 x 352; TH = 4 always at 704 and wider)."""
    check_dwconv_raw(B, H, W, C, dtype)


@pytest.mark.parametrize("dtype", ["fp16", "bf16"])
@pytest.mark.parametrize("B,H,W,C", [(1, 9, 13, 2816), (2, 16, 16, 2816), (3, 32, 32, 704)])
def test_v2_huge_dwconv_raw_tc(B, H, W, C, dtype):
    """Tensor-core depthwise + folded LayerNorm at 44 channel chunks (partial statistics [token][44]) and at 11."""
    check_dwconv_raw_tc(B, H, W, C, dtype)


@pytest.mark.parametrize("dtype", ["bf16", "fp16"])
def test_v2_huge_head(dtype):
    """Pool + head at 2816 channels: 111 KB of shared memory per CTA of the cluster."""
    C, g, d = 2816, torch.Generator().manual_seed(7), dev()
    xs = torch.randn(3, 64, C, generator=g).to(DTYPES[dtype])
    p = [1 + 0.1 * torch.randn(C, generator=g), 0.1 * torch.randn(C, generator=g), 1 + 0.1 * torch.randn(C, generator=g),
         0.1 * torch.randn(C, generator=g), torch.randn(256, C, generator=g) / C ** 0.5, 0.1 * torch.randn(256, generator=g),
         torch.randn(10, 256, generator=g) / 16, 0.1 * torch.randn(10, generator=g)]
    f = xs.float().mean(1)
    f = torch.nn.functional.layer_norm(f, (C,), p[0], p[1], 1e-6)
    f = torch.nn.functional.layer_norm(f, (C,), p[2], p[3], 1e-5)
    want = torch.sigmoid(torch.nn.functional.gelu(f @ p[4].t() + p[5]) @ p[6].t() + p[7])
    got = ops.head(xs.to(d), *[t.to(d) for t in p]).cpu()
    assert (got - want).abs().max() < 2e-5


# ---------------------------------------------------------------------------------------------------- checkpoint and dataset
def test_v2_huge_checkpoint_loads(checkpoint, random_init):
    model = cropping.load_localization_model(checkpoint, "v2_huge", dev())
    planes = _planes([synthetic.make_iso_slice(*c) for c in SLICES])
    direct = cropping.LocalizationModel(random_init.state_dict(), dev())
    assert torch.equal(model.predict_u8(planes), direct.predict_u8(planes))


def test_v2_huge_dataset_with_checkpoint(checkpoint, tmp_path):
    """create_classification_dataset(model_variant="v2_huge") on a synthetic SPIDER tree: its PNGs equal the module-level
    mirrors called one series at a time (the reference's call sequence)."""
    from spine_vision_b200 import dataset, hostio, volumes

    pids = synthetic.make_spider_tree(tmp_path, n_patients=1, seed=5, in_plane=(160, 150), missing_t1=())
    cfg = dataset.ClassificationDatasetConfig(base_path=tmp_path, output_name="m", localization_model_path=checkpoint, model_variant="v2_huge",
                                              crop_size=(128, 128), crop_delta_mm=(20.0, 8.0, 9.0, 10.0), include_phenikaa=False, device=dev())
    res = dataset.create_classification_dataset(cfg)
    assert res.num_samples > 0
    model = cropping.load_localization_model(checkpoint, "v2_huge", dev())
    checked = 0
    for seq in ("t1", "t2"):
        vol = hostio.read_medical_image(tmp_path / "raw" / "SPIDER" / "images" / f"{pids[0]}_{seq}.mha")
        pool, sp = volumes.midplane_resample([vol.array], [vol.spacing], [vol.direction], dev(), integer_pixels=[True])
        sl = pool.data[: pool.shapes[0][0] * pool.shapes[0][1]].reshape(pool.shapes[0]).cpu().numpy()
        locs = cropping.predict_ivd_locations(model, sl, dev(), (512, 512))
        ctx = cropping.CropContext(sl, locs, (128, 128), cropping.mm_to_pixels(cfg.crop_delta_mm, sp[0]), device=dev())
        for lvl in range(1, 6):
            png = cfg.output_path / "images" / f"spider_{pids[0]}_sag_{seq}_L{lvl}.png"
            if png.exists():
                assert np.array_equal(np.asarray(Image.open(png)), ctx.crop(lvl - 1)), png.name
                checked += 1
    assert checked == res.num_samples


# ---------------------------------------------------------------------------------------------------- C ABI
def _skeleton(dims):
    """The keys svb_model_create reads before it checks the widths (depth 1 per stage)."""
    sd = {"backbone.stem.0.weight": torch.zeros(dims[0], 3, 4, 4)}
    for s, c in enumerate(dims):
        sd[f"backbone.stages.{s}.blocks.0.conv_dw.weight"] = torch.zeros(c, 1, 7, 7)
        sd[f"backbone.stages.{s}.blocks.0.norm.weight"] = torch.ones(c)
    return sd


@pytest.mark.parametrize("dims,word", [((352, 704, 1408, 3072), "width 3072"), ((320, 640, 1280, 2560), "stem width 320")])
def test_model_create_rejects_widths_beyond_v2_huge(dims, word):
    with pytest.raises(_lib.SvbError) as e:
        ops.LocalizationEngine(_skeleton(dims), dev())
    assert e.value.code == UNSUPPORTED_MODEL and word in str(e.value) and "v2_huge" in str(e.value)


def test_model_create_refuses_v2_huge_without_the_folded_layernorm(monkeypatch):
    monkeypatch.setenv("SVB_LN_FOLD", "0")
    with pytest.raises(_lib.SvbError) as e:
        ops.LocalizationEngine(_skeleton(DIMS), dev())
    assert e.value.code == UNSUPPORTED_MODEL and "SVB_LN_FOLD=0" in str(e.value)
