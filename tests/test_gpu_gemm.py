"""GPU numerics: the tcgen05 GEMM and the other ConvNeXt layer kernels vs plain PyTorch fp32 references."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from gpu_util import dev
from spine_vision_b200 import ops

pytestmark = pytest.mark.gpu
DT = {"bf16": torch.bfloat16, "fp16": torch.float16}


def _ref_gemm(a, w, bias, mode, resid=None, gamma=None):
    acc = a.float() @ w.float().t() + bias
    if mode == 0:
        return F.gelu(acc)
    if mode == 1:
        return resid.float() + gamma * acc
    return acc


@pytest.mark.parametrize("dtype", ["bf16", "fp16"])
@pytest.mark.parametrize("M,N,K,mode", [
    (128, 128, 64, 2), (128, 256, 128, 2), (256, 512, 128, 0), (1000, 256, 512, 2), (4096, 128, 512, 1),
    (2048, 1024, 256, 0), (640, 256, 1024, 1), (128 * 150, 512, 128, 0), (3000, 2048, 512, 0), (3000, 512, 2048, 1),
    (512, 1024, 4096, 1), (777, 4096, 1024, 0), (128 * 300 + 5, 128, 512, 1),
    (1000, 768, 192, 0), (1000, 192, 768, 1), (640, 1536, 384, 0), (300, 384, 1536, 1), (512, 384, 768, 2),  # convnext_large: N, K multiples of 64 only
    (1000, 384, 96, 0), (1000, 96, 384, 1), (300, 192, 384, 2),  # convnext_tiny / small: K = 96 is one and a half k-blocks
])
def test_gemm_vs_torch(M, N, K, mode, dtype):
    g = torch.Generator(device="cpu").manual_seed(M * 7 + N * 3 + K + mode)
    a = (torch.randn(M, K, generator=g)).to(DT[dtype]).to(dev())
    w = (torch.randn(N, K, generator=g) / K ** 0.5).to(DT[dtype]).to(dev())
    bias = torch.randn(N, generator=g).to(dev())
    gamma = (torch.rand(N, generator=g) + 0.1).to(dev())
    resid = torch.randn(M, N, generator=g).to(DT[dtype]).to(dev())
    want = _ref_gemm(a, w, bias, mode, resid, gamma)
    if mode == 1:
        out = resid.clone()
        got = ops.gemm(a, w, bias, 1, resid=out, gamma=gamma, out=out)  # in place, as the model runs it
    else:
        got = ops.gemm(a, w, bias, mode)
    torch.cuda.synchronize()
    err = (got.float() - want).abs()
    tol = (2.0 ** -8 if dtype == "bf16" else 2.0 ** -11) * (want.abs() + 1.0)  # output rounding to 16 bits
    bad = int((err > tol).sum())
    assert bad == 0, f"{bad} of {err.numel()} beyond tolerance; max err {err.max().item():.4g} at {np.unravel_index(int(err.argmax()), err.shape)}"


@pytest.mark.parametrize("dtype", ["bf16", "fp16"])
@pytest.mark.parametrize("B,H,W,C", [(2, 16, 16, 128), (1, 37, 21, 128), (2, 64, 64, 256), (3, 32, 32, 512), (2, 16, 16, 1024),
                                     (1, 15, 23, 1024), (1, 128, 128, 128), (2, 16, 16, 2048), (1, 9, 13, 2048),
                                     (2, 40, 24, 192), (2, 32, 32, 384), (2, 17, 32, 768), (3, 16, 16, 1536),  # + convnext_large widths
                                     (2, 33, 40, 96), (1, 128, 128, 96)])  # + convnext_tiny / small stage 0 (1.5 channel chunks)
def test_dwconv_ln_vs_torch(B, H, W, C, dtype):
    g = torch.Generator().manual_seed(B + H + W + C)
    x = torch.randn(B, H, W, C, generator=g).to(DT[dtype])
    wt = torch.randn(C, 1, 7, 7, generator=g) * 0.1
    bias = torch.randn(C, generator=g) * 0.1
    lnw = 1 + 0.2 * torch.randn(C, generator=g)
    lnb = 0.1 * torch.randn(C, generator=g)
    y = F.conv2d(x.float().permute(0, 3, 1, 2), wt, bias, padding=3, groups=C).permute(0, 2, 3, 1)
    want = F.layer_norm(y, (C,), lnw, lnb, 1e-6)
    taps = wt.reshape(C, 49).t().contiguous()
    got = ops.dwconv_ln(x.to(dev()), taps.to(dev()), bias.to(dev()), lnw.to(dev()), lnb.to(dev())).float().cpu()
    err = (got - want).abs()
    tol = (2.0 ** -8 if dtype == "bf16" else 2.0 ** -11) * (want.abs() + 1.0)
    assert int((err > tol).sum()) == 0, f"max err {err.max().item():.4g}"


@pytest.mark.parametrize("dtype", ["bf16", "fp16"])
@pytest.mark.parametrize("B,H,W,C", [(2, 16, 16, 128), (1, 37, 21, 128), (2, 64, 64, 256), (3, 32, 32, 512), (2, 16, 16, 1024), (1, 15, 23, 1024),
                                     (1, 128, 128, 128), (1, 9, 13, 2048), (2, 40, 24, 192), (2, 17, 32, 768), (2, 33, 40, 96), (1, 7, 5, 384)])
def test_dwconv_raw_and_folded_layernorm_vs_torch(B, H, W, C, dtype):
    """The default block: ``svb_dwconv_raw`` (raw depthwise convolution in 16 bits + per-token (rstd, -mean * rstd)) followed by the
    fc1 GEMM with the LayerNorm folded in (``svb_gemm`` mode 3) equals GELU(fc1(LayerNorm(conv(x)))) of plain PyTorch fp32:
    (a) the raw output is the convolution to 16-bit rounding; (b) the statistics are those of the fp32 convolution (taken before
    the rounding); (c) the composite is within the output rounding of the un-folded reference."""
    g = torch.Generator().manual_seed(B + H + W + C)
    x = torch.randn(B, H, W, C, generator=g).to(DT[dtype])
    wt = torch.randn(C, 1, 7, 7, generator=g) * 0.1
    bias = torch.randn(C, generator=g) * 0.1 + 0.3  # a non-zero token mean: the subtraction in the epilogue has something to cancel
    lnw = 1 + 0.2 * torch.randn(C, generator=g)
    lnb = 0.1 * torch.randn(C, generator=g)
    N = 4 * C if C <= 512 else 512
    w1 = torch.randn(N, C, generator=g) / C ** 0.5
    b1 = 0.1 * torch.randn(N, generator=g)
    y = F.conv2d(x.float().permute(0, 3, 1, 2), wt, bias, padding=3, groups=C).permute(0, 2, 3, 1)
    taps = wt.reshape(C, 49).t().contiguous()
    raw, stat = ops.dwconv_raw(x.to(dev()), taps.to(dev()), bias.to(dev()))
    torch.cuda.synchronize()
    rawf = raw.float().cpu()
    eps16 = 2.0 ** -8 if dtype == "bf16" else 2.0 ** -11
    assert int(((rawf - y).abs() > eps16 * (y.abs() + 1.0)).sum()) == 0, f"raw conv: max err {(rawf - y).abs().max().item():.4g}"
    mu = y.mean(-1)
    var = y.var(-1, unbiased=False)
    rstd = torch.rsqrt(var + 1e-6)
    st = stat.cpu().view(B, H, W, 2)
    assert torch.allclose(st[..., 0], rstd, rtol=2e-4, atol=1e-6), (st[..., 0] - rstd).abs().max()
    assert torch.allclose(st[..., 1], -mu * rstd, rtol=2e-4, atol=2e-4), (st[..., 1] + mu * rstd).abs().max()
    wg = (w1 * lnw[None, :]).to(DT[dtype])
    s_n = wg.float().sum(1)
    t_n = (w1.double() @ lnb.double()).float() + b1
    got = ops.gemm(raw.view(-1, C), wg.to(dev()), t_n.to(dev()), 3, resid=stat, gamma=s_n.to(dev())).float().cpu()
    want = F.gelu(F.layer_norm(y, (C,), lnw, lnb, 1e-6).reshape(-1, C) @ w1.t() + b1)
    err = (got - want).abs()
    # the reference rounds nothing; the device rounds the conv output and W1 * g to 16 bits and accumulates in fp32: the bound is
    # the operand rounding through a C-term dot product of O(1) terms (same budget as the un-folded pair: LN output + W1 rounded)
    tol = 4 * eps16 * (want.abs() + 1.0)
    assert int((err > tol).sum()) == 0, f"{int((err > tol).sum())} beyond tolerance, max err {err.max().item():.4g}"


@pytest.mark.parametrize("dtype", ["fp16", "bf16"])
@pytest.mark.parametrize("B,H,W,C", [(3, 32, 32, 512), (2, 16, 16, 1024), (5, 32, 32, 128), (1, 8, 8, 64), (2, 20, 32, 192), (3, 12, 16, 64),
                                     (2, 64, 64, 256), (1, 128, 128, 128), (2, 37, 21, 128), (1, 15, 23, 1024), (1, 9, 13, 2048), (2, 33, 40, 64),
                                     (1, 7, 5, 384), (40, 32, 32, 512)])
def test_dwconv_raw_tc_and_folded_layernorm_vs_torch(B, H, W, C, dtype):
    """``svb_dwconv_raw_tc`` (the depthwise stencil on the tensor cores: mode A for W in {8, 16, 32}, mode B windows otherwise)
    + the fc1 GEMM with the folded LayerNorm: (a) the raw output is the convolution WITH THE TAPS ROUNDED TO 16 BITS (the
    kernel's operands; activation x tap products are exact, accumulation fp32) to output rounding; (b) the statistics (per-chunk
    partial sums added up by the finalize launch) are those of the fp32 convolution; (c) the composite equals
    GELU(fc1(LayerNorm(conv))) of plain PyTorch within the same budget as the FP32-pipe pair; (d) a second launch gives identical
    bits (fixed summation order, no atomics)."""
    g = torch.Generator().manual_seed(B + H + W + C + 1)
    x = torch.randn(B, H, W, C, generator=g).to(DT[dtype])
    wt = torch.randn(C, 1, 7, 7, generator=g) * 0.1
    bias = torch.randn(C, generator=g) * 0.1 + 0.3
    lnw = 1 + 0.2 * torch.randn(C, generator=g)
    lnb = 0.1 * torch.randn(C, generator=g)
    N = 4 * C if C <= 512 else 512
    w1 = torch.randn(N, C, generator=g) / C ** 0.5
    b1 = 0.1 * torch.randn(N, generator=g)
    wt16 = wt.to(DT[dtype]).float()
    y = F.conv2d(x.float().permute(0, 3, 1, 2), wt16, bias, padding=3, groups=C).permute(0, 2, 3, 1)
    taps = wt.reshape(C, 49).t().contiguous()
    wtc = ops.dwconv_tc_pack(taps.to(dev()), DT[dtype])
    xd, bd = x.to(dev()), bias.to(dev())
    raw, stat = ops.dwconv_raw_tc(xd, wtc, bd)
    torch.cuda.synchronize()
    rawf = raw.float().cpu()
    eps16 = 2.0 ** -8 if dtype == "bf16" else 2.0 ** -11
    # fp16: the six off-centre stencil columns' partial sums cross lanes as fp16 (packed shuffles), so the bound is their half-ulp
    # roundings (|partial| <= sum |x| |w| of one column) on top of the output rounding; bf16 keeps fp32 shuffles
    slack = 1.01 if dtype == "bf16" else 3.0
    bad = (rawf - y).abs() > eps16 * (y.abs() + 1.0) * slack
    assert int(bad.sum()) == 0, f"raw conv: {int(bad.sum())} off, max err {(rawf - y).abs().max().item():.4g} at {bad.nonzero()[:4].tolist()}"
    assert float((rawf - y).abs().mean()) < 0.6 * eps16 * float(y.abs().mean() + 1.0)
    mu = y.mean(-1)
    var = y.var(-1, unbiased=False)
    rstd = torch.rsqrt(var + 1e-6)
    st = stat.cpu().view(B, H, W, 2)
    assert torch.allclose(st[..., 0], rstd, rtol=2e-4, atol=1e-6), (st[..., 0] - rstd).abs().max()
    assert torch.allclose(st[..., 1], -mu * rstd, rtol=2e-4, atol=2e-4), (st[..., 1] + mu * rstd).abs().max()
    wg = (w1 * lnw[None, :]).to(DT[dtype])
    s_n = wg.float().sum(1)
    t_n = (w1.double() @ lnb.double()).float() + b1
    got = ops.gemm(raw.view(-1, C), wg.to(dev()), t_n.to(dev()), 3, resid=stat, gamma=s_n.to(dev())).float().cpu()
    want = F.gelu(F.layer_norm(y, (C,), lnw, lnb, 1e-6).reshape(-1, C) @ w1.t() + b1)
    err = (got - want).abs()
    tol = 4 * eps16 * (want.abs() + 1.0)
    assert int((err > tol).sum()) == 0, f"{int((err > tol).sum())} beyond tolerance, max err {err.max().item():.4g}"
    r2, s2 = ops.dwconv_raw_tc(xd, wtc, bd)
    torch.cuda.synchronize()
    assert torch.equal(r2, raw) and torch.equal(s2, stat)
    # the cta_group::2 variant (CTA pairs, half of every B matrix per CTA; SVB_TC2_PAIR is read per call here): identical bits
    import os
    os.environ["SVB_TC2_PAIR"] = "1"
    try:
        r3, s3 = ops.dwconv_raw_tc(xd, wtc, bd)
        torch.cuda.synchronize()
    finally:
        del os.environ["SVB_TC2_PAIR"]
    assert torch.equal(r3, raw) and torch.equal(s3, stat)


@pytest.mark.parametrize("dtype", ["bf16", "fp16"])
@pytest.mark.parametrize("C0,C", [(192, 192), (192, 384), (256, 768), (96, 96)])
def test_stem_patchify_other_widths(dtype, C0, C):
    """The widths of convnext_large / xlarge: stem at 192 / 256 channels, LayerNorm + patchify at 192 (a half-empty last lane
    group), 384, 768."""
    g = torch.Generator().manual_seed(C0 + C)
    d = dev()
    u8 = torch.randint(0, 256, (2, 32, 64), generator=g, dtype=torch.uint8)
    wf, bf = torch.randn(C0, 16, generator=g) * 0.01, torch.randn(C0, generator=g) * 0.1
    lnw, lnb = 1 + 0.1 * torch.randn(C0, generator=g), 0.1 * torch.randn(C0, generator=g)
    y = F.conv2d(u8.float().unsqueeze(1), wf.view(C0, 1, 4, 4), bf, stride=4).permute(0, 2, 3, 1)
    want = F.layer_norm(y, (C0,), lnw, lnb, 1e-6)
    got = ops.stem_ln(u8.to(d), wf.to(d), bf.to(d), lnw.to(d), lnb.to(d), DT[dtype]).float().cpu()
    tol = (2.0 ** -8 if dtype == "bf16" else 2.0 ** -11) * (want.abs() + 1.0)
    assert int(((got - want).abs() > tol).sum()) == 0
    x = torch.randn(2, 6, 10, C, generator=g).to(DT[dtype])
    lw, lb = 1 + 0.1 * torch.randn(C, generator=g), 0.1 * torch.randn(C, generator=g)
    n = F.layer_norm(x.float(), (C,), lw, lb, 1e-6)
    want = n.view(2, 3, 2, 5, 2, C).permute(0, 1, 3, 2, 4, 5).reshape(2, 3, 5, 4 * C)
    got = ops.ln_patchify(x.to(d), lw.to(d), lb.to(d)).float().cpu()
    tol = (2.0 ** -8 if dtype == "bf16" else 2.0 ** -11) * (want.abs() + 1.0)
    assert int(((got - want).abs() > tol).sum()) == 0


@pytest.mark.parametrize("dtype", ["bf16", "fp16"])
def test_stem_patchify_head_vs_torch(dtype):
    g = torch.Generator().manual_seed(5)
    d = dev()
    # stem: folded single-channel conv4x4/s4 + LayerNorm2d
    u8 = torch.randint(0, 256, (2, 64, 96), generator=g, dtype=torch.uint8)
    wf = torch.randn(128, 16, generator=g) * 0.01
    bf = torch.randn(128, generator=g) * 0.1
    lnw, lnb = 1 + 0.1 * torch.randn(128, generator=g), 0.1 * torch.randn(128, generator=g)
    y = F.conv2d(u8.float().unsqueeze(1), wf.view(128, 1, 4, 4), bf, stride=4).permute(0, 2, 3, 1)
    want = F.layer_norm(y, (128,), lnw, lnb, 1e-6)
    got = ops.stem_ln(u8.to(d), wf.to(d), bf.to(d), lnw.to(d), lnb.to(d), DT[dtype]).float().cpu()
    tol = (2.0 ** -8 if dtype == "bf16" else 2.0 ** -11) * (want.abs() + 1.0)
    assert int(((got - want).abs() > tol).sum()) == 0
    # LayerNorm2d + 2x2 patchify
    x = torch.randn(2, 8, 12, 256, generator=g).to(DT[dtype])
    lw, lb = 1 + 0.1 * torch.randn(256, generator=g), 0.1 * torch.randn(256, generator=g)
    n = F.layer_norm(x.float(), (256,), lw, lb, 1e-6)
    want = n.view(2, 4, 2, 6, 2, 256).permute(0, 1, 3, 2, 4, 5).reshape(2, 4, 6, 1024)
    got = ops.ln_patchify(x.to(d), lw.to(d), lb.to(d)).float().cpu()
    tol = (2.0 ** -8 if dtype == "bf16" else 2.0 ** -11) * (want.abs() + 1.0)
    assert int(((got - want).abs() > tol).sum()) == 0
    # pool + head
    xs = torch.randn(3, 256, 1024, generator=g).to(DT[dtype])
    p = [1 + 0.1 * torch.randn(1024, generator=g), 0.1 * torch.randn(1024, generator=g),
         1 + 0.1 * torch.randn(1024, generator=g), 0.1 * torch.randn(1024, generator=g),
         torch.randn(256, 1024, generator=g) / 32, 0.1 * torch.randn(256, generator=g),
         torch.randn(10, 256, generator=g) / 16, 0.1 * torch.randn(10, generator=g)]
    f = xs.float().mean(1)
    f = F.layer_norm(f, (1024,), p[0], p[1], 1e-6)
    f = F.layer_norm(f, (1024,), p[2], p[3], 1e-5)
    want = torch.sigmoid(F.gelu(f @ p[4].t() + p[5]) @ p[6].t() + p[7])
    got = ops.head(xs.to(d), *[t.to(d) for t in p]).cpu()
    assert (got - want).abs().max() < 2e-5


@pytest.mark.parametrize("dtype", ["bf16", "fp16"])
@pytest.mark.parametrize("M,C", [(256, 128), (1000, 128), (256 * 80 + 37, 128), (512, 256), (256 * 75 + 130, 256), (128, 256)])
def test_fused_mlp_vs_torch(M, C, dtype):
    """mlp_fused_kernel (fc1 -> GELU -> fc2 -> gamma, +residual with the hidden activation on chip) against fp32 torch
    with the hidden activation rounded to the operand dtype (what the un-fused pair stores between its two GEMMs)."""
    g = torch.Generator().manual_seed(M + C)
    dt = DT[dtype]
    a = torch.randn(M, C, generator=g).to(dt)
    w1 = (torch.randn(4 * C, C, generator=g) / C ** 0.5).to(dt)
    w2 = (torch.randn(C, 4 * C, generator=g) / (4 * C) ** 0.5).to(dt)
    b1, b2 = torch.randn(4 * C, generator=g) * 0.2, torch.randn(C, generator=g) * 0.2
    gamma = torch.rand(C, generator=g) + 0.1
    x = torch.randn(M, C, generator=g).to(dt)
    h = F.gelu(a.float() @ w1.float().t() + b1).to(dt).float()
    want = x.float() + gamma * (h @ w2.float().t() + b2)
    d = dev()
    got = ops.mlp_fused(a.to(d), w1.to(d), b1.to(d), w2.to(d), b2.to(d), gamma.to(d), x.to(d).clone()).float().cpu()
    err = (got - want).abs()
    # output rounding + the propagated rounding of the hidden operand (one 16-bit ulp of h through a 4C-term dot product)
    tol = (2.0 ** -8 if dtype == "bf16" else 2.0 ** -11) * (want.abs() + 1.0) * 1.5
    bad = int((err > tol).sum())
    assert bad == 0, f"{bad} of {err.numel()} beyond tolerance; max err {err.max().item():.4g}"


@pytest.mark.parametrize("dtype", ["bf16", "fp16"])
@pytest.mark.parametrize("M,C", [(256, 128), (1000, 128), (256 * 80 + 17, 128), (512, 256), (3000, 256)])
def test_fused_mlp_folded_layernorm_vs_torch(M, C, dtype):
    """``svb_mlp_fused_ln`` (what stages 0 / 1 of the model run): the raw depthwise output + per-token statistics in, the block's
    residual update out -- against x + gamma * fc2(GELU(fc1(LayerNorm(y)))) of plain PyTorch fp32 with the hidden activation rounded
    to the operand dtype."""
    g = torch.Generator().manual_seed(M + C + 3)
    dt = DT[dtype]
    y = (torch.randn(M, C, generator=g) * 0.7 + 0.3).to(dt)  # raw conv output (16-bit), non-zero token mean
    lnw = 1 + 0.2 * torch.randn(C, generator=g)
    lnb = 0.1 * torch.randn(C, generator=g)
    w1 = torch.randn(4 * C, C, generator=g) / C ** 0.5
    b1 = 0.1 * torch.randn(4 * C, generator=g)
    w2 = (torch.randn(C, 4 * C, generator=g) / (4 * C) ** 0.5).to(dt)
    b2 = torch.randn(C, generator=g) * 0.2
    gamma = torch.rand(C, generator=g) + 0.1
    x = torch.randn(M, C, generator=g).to(dt)
    yf = y.float()
    mu, var = yf.mean(-1), yf.var(-1, unbiased=False)
    rstd = torch.rsqrt(var + 1e-6)
    stat = torch.stack([rstd, -mu * rstd], -1).contiguous()
    wg = (w1 * lnw[None, :]).to(dt)
    s_n = wg.float().sum(1)
    t_n = (w1.double() @ lnb.double()).float() + b1
    h = F.gelu(F.layer_norm(yf, (C,), lnw, lnb, 1e-6) @ w1.t() + b1).to(dt).float()
    want = x.float() + gamma * (h @ w2.float().t() + b2)
    d = dev()
    got = ops.mlp_fused_ln(y.to(d), wg.to(d), t_n.to(d), s_n.to(d), stat.to(d), w2.to(d), b2.to(d), gamma.to(d), x.to(d).clone()).float().cpu()
    err = (got - want).abs()
    # output rounding + the hidden operand's rounding + W1 * g rounded to 16 bits (the un-folded reference rounds nothing there)
    tol = (2.0 ** -8 if dtype == "bf16" else 2.0 ** -11) * (want.abs() + 1.0) * 3.0
    bad = int((err > tol).sum())
    assert bad == 0, f"{bad} of {err.numel()} beyond tolerance; max err {err.max().item():.4g}"
