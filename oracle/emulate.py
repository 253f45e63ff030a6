"""CPU (or any torch device) emulation of the device numerics of the localizer forward, stage by stage.

TEST INFRASTRUCTURE ONLY (see ``oracle/__init__.py``).

It follows the default LayerNorm-folded path of ``svb_convnext.cu`` (``forward_chunk``) and rounds where the kernels round
(16-bit storage and GEMM operands, fp32 accumulation):

* stem: fp32 conv + LayerNorm, stored in 16 bits; downsample: LayerNorm2d -> 16-bit A operand, 16-bit weights, 16-bit output
* depthwise 7x7: fp32 taps (``dwconv_raw_kernel``), or where ``dwconv_rawtc_kernel`` runs (``dw_tc2_mode``: fp16 and
  C % 64 == 0, both of its modes) 16-bit taps with every off-centre stencil column's partial sum rounded to fp16 before the
  cross-lane sum; the raw result y is stored in 16 bits
* LayerNorm statistics from the UNROUNDED y, one pass in fp32: mu = E[y], var = max(E[y^2] - mu^2, 0), rstd = 1 / sqrt(var + eps)
* fc1 with the LayerNorm folded in: W1 * g rounded once, s_n = sum_k r16(W1 * g)[n, k], t_n = W1 @ b_ln + b1;
  h = r16(GELU(rstd * (r16(y) @ r16(W1 g)^T) - mu rstd * s + t))
* v2: GlobalResponseNorm over the 16-bit hidden activation, result rounded again
* fc2: x = r16(x + gamma * (h @ r16(W2)^T + b2)), the residual stream rounded after every block
* head: fp32 from the last 16-bit residual stream

With ``rounding=False`` every rounding is the identity and the result is the fp32 network in the folded form.
"""

from __future__ import annotations

import torch
import torch.nn.functional as F

from oracle.convnext import LN_EPS


def tc_depthwise(dtype: torch.dtype, C: int) -> bool:
    """Does the default forward run the stage's depthwise conv on the tensor cores (``dw_tc2_mode``)?  fp16 only (bf16 needs
    SVB_DWCONV_TC2=2), channel counts that are whole 64-channel chunks (not 96); mode A or B covers every H and W."""
    return dtype == torch.float16 and C % 64 == 0


def _ln(x, w, b):
    return F.layer_norm(x, (x.shape[-1],), w, b, LN_EPS)


def _depthwise(x, w, b, r16, tc):
    """x [B,H,W,C] -> y [B,H,W,C] (fp32, unrounded)."""
    xc = x.permute(0, 3, 1, 2)
    C = xc.shape[1]
    if not tc:
        return F.conv2d(xc, w, b, padding=3, groups=C).permute(0, 2, 3, 1)
    # every stencil column's partial sum over the 7 rows: output channel 7c + dx is column dx of channel c's taps, run as a
    # 7 x 1 conv over the input padded by 3 columns; column dx of output x reads padded column x + dx
    Wd = xc.shape[3]
    cols = F.conv2d(F.pad(xc, (3, 3, 0, 0)), r16(w).permute(0, 3, 2, 1).reshape(7 * C, 1, 7, 1), None, padding=(3, 0), groups=C)
    cols = cols.view(xc.shape[0], C, 7, xc.shape[2], Wd + 6)
    y = b.view(1, -1, 1, 1) + cols[:, :, 3, :, 3 : 3 + Wd]
    for dx in (0, 1, 2, 4, 5, 6):
        y = y + r16(cols[:, :, dx, :, dx : dx + Wd])
    return y.permute(0, 2, 3, 1)


@torch.no_grad()
def forward_stages(model, x: torch.Tensor, dtype: torch.dtype = torch.float16, rounding: bool = True, mlp_hook=None):
    """``model`` a ``CoordinateRegressor`` (``oracle.convnext.make_model``), ``x`` its ``[B,3,H,W]`` fp32 input.
    Returns (coords ``[B, levels, 2]``, [four stage tensors ``[B, h_s, w_s, C_s]`` fp32 holding 16-bit values]).
    ``mlp_hook(stage, block, o) -> o``, if given, may alter a block's MLP output ``[B, h, w, C]`` before the residual add
    (fault injection for tests of the stage-level gates)."""
    r16 = (lambda t: t.to(dtype).float()) if rounding else (lambda t: t)
    bb = model.backbone
    x = bb.stem[0](x).permute(0, 2, 3, 1)
    x = r16(_ln(x, bb.stem[1].weight, bb.stem[1].bias))
    stages = []
    for s, st in enumerate(bb.stages):
        if not isinstance(st.downsample, torch.nn.Identity):
            a = r16(_ln(x, st.downsample[0].weight, st.downsample[0].bias))
            w = r16(st.downsample[1].weight)
            x = r16(F.conv2d(a.permute(0, 3, 1, 2), w, st.downsample[1].bias, stride=2).permute(0, 2, 3, 1))
        C = x.shape[-1]
        tc = rounding and tc_depthwise(dtype, C)
        for j, blk in enumerate(st.blocks):
            y = _depthwise(x, blk.conv_dw.weight, blk.conv_dw.bias, r16, tc)
            mu = y.mean(-1, keepdim=True)
            var = ((y * y).mean(-1, keepdim=True) - mu * mu).clamp_min(0.0)
            rstd = 1.0 / torch.sqrt(var + LN_EPS)
            W1, b1 = blk.mlp.fc1.weight, blk.mlp.fc1.bias
            Wg = r16(W1 * blk.norm.weight[None, :])
            sn = Wg.double().sum(1).float()
            tn = (W1.double() @ blk.norm.bias.double() + b1.double()).float()
            h = rstd * (r16(y) @ Wg.t()) + (-mu * rstd) * sn + tn
            h = r16(F.gelu(h))
            if blk.mlp.use_grn:
                g = blk.mlp.grn
                gx = torch.sqrt((h * h).sum(dim=(1, 2), keepdim=True))
                n = gx / (gx.mean(dim=-1, keepdim=True) + g.eps)
                h = r16(h * (1.0 + g.weight * n) + g.bias)
            o = h @ r16(blk.mlp.fc2.weight).t() + blk.mlp.fc2.bias
            if blk.gamma is not None:
                o = blk.gamma * o
            if mlp_hook is not None:
                o = mlp_hook(s, j, o)
            x = r16(x + o)
        stages.append(x)
    f = _ln(x.mean(dim=(1, 2)), bb.head.norm.weight, bb.head.norm.bias)
    return model.head(f).view(-1, model._num_levels, model._num_outputs), stages


@torch.no_grad()
def oracle_stages(model, x: torch.Tensor):
    """The fp32 oracle's coordinates and its residual stream after each stage (forward hooks on ``backbone.stages[s]``),
    channels-last ``[B, h_s, w_s, C_s]`` like ``forward_stages``."""
    outs = []
    hooks = [st.register_forward_hook(lambda _m, _i, o: outs.append(o.permute(0, 2, 3, 1).contiguous())) for st in model.backbone.stages]
    try:
        coords = model(x)
    finally:
        for h in hooks:
            h.remove()
    return coords, outs
