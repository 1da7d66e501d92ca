"""Layer-level autograd nodes on the B200 kernels for the Residual / Attention / Trans U-Net variants
(reference: models/res_unet.py, models/attention_unet.py, models/trans_unet.py).

Activations travel between nodes as NHWC bf16 tensors ``[N, H, W, C]``; 1-channel tensors (network input
and output, attention logits) are fp32 planes ``[N, H, W]``, and 2-4 channel network inputs / outputs are fp32 NCHW
plane stacks ``[N, C, H, W]``.  Parameters are the fp32 tensors of the
drop-in ``nn.Module`` tree in the reference's layouts.  Every node's forward AND backward is a kernel of
libpai_b200.so; there is no PyTorch-op implementation behind them.
"""
from __future__ import annotations

import torch
import torch.nn as nn

from . import ops
from .engine import BN_EPS, BN_MOMENTUM, _packs
from .ops import ACT_LEAKY, ACT_NONE, ACT_RELU, ACT_TANH  # noqa: F401


def _need(flag_list, i):
    return flag_list[i]


# ------------------------------------------------------------------------------------------ convolutions
def _pad64(c):
    return 64 * ((c + 63) // 64)


def _pack_c1_f_padded(w):    # rows padded to a multiple of 64 so the padded output can be a GEMM K dimension
    cout, cin = w.shape[0], w.shape[1]
    out = torch.zeros(_pad64(cout), cin, dtype=torch.bfloat16, device=w.device)
    out[:cout].copy_(w.reshape(cout, cin))
    return out


def _pack_c1_d_padded(w):    # [cin, pad64(cout)]
    cout, cin = w.shape[0], w.shape[1]
    out = torch.zeros(ops.padded_cout(cin), _pad64(cout), dtype=torch.bfloat16, device=w.device)
    out[:cin, :cout].copy_(w.reshape(cout, cin).t())
    return out


class _Conv1x1(torch.autograd.Function):
    """nn.Conv2d(cin, cout, 1) / nn.Linear on the tensor-core pointwise GEMM.  cin must be a multiple of 64; a
    cout that is not (the 32-channel attention gate) is computed in a zero-padded 64-channel buffer."""

    @staticmethod
    def forward(ctx, x, weight, bias):
        cout = weight.shape[0]
        cp = _pad64(cout)
        wp = _packs.get("c1_f", weight, _pack_c1_f_padded)
        b = None
        if bias is not None:
            b = bias.detach()
            if cp != cout:
                b = torch.cat([b, b.new_zeros(cp - cout)])
        y = ops.pointwise_gemm(x, wp, cp, bias=b)
        ctx.save_for_backward(x, weight)
        ctx.has_bias = bias is not None
        return y if cp == cout else y[..., :cout]

    @staticmethod
    def backward(ctx, gy):
        x, weight = ctx.saved_tensors
        cout, cin = weight.shape[0], weight.shape[1]
        cp = _pad64(cout)
        if cp != cout:
            full = torch.zeros(*gy.shape[:-1], cp, dtype=torch.bfloat16, device=gy.device)
            full[..., :cout].copy_(gy)
            gy = full
        else:
            gy = gy.contiguous()
        gx = gw = gb = None
        if ctx.needs_input_grad[0]:
            wt = _packs.get("c1_d", weight, _pack_c1_d_padded)
            gx = ops.pointwise_gemm(gy, wt, cin)
        if ctx.needs_input_grad[1]:
            gw = ops.pointwise_wgrad(gy, x)[:cout].reshape(weight.shape)
        if ctx.has_bias and ctx.needs_input_grad[2]:
            gb = ops.colsum(gy)[:cout].clone()
        return gx, gw, gb


class _Conv3x3(torch.autograd.Function):
    """nn.Conv2d(cin, cout, 3, padding=1) on the implicit-GEMM kernel (cin, cout multiples of 64)."""

    @staticmethod
    def forward(ctx, x, weight, bias):
        cout = weight.shape[0]
        wp = _packs.get("c3_f", weight, ops.pack_conv3x3_weight)
        y = ops.conv3x3_fprop(x, wp, cout, bias=None if bias is None else bias.detach())
        ctx.save_for_backward(x, weight)
        ctx.has_bias = bias is not None
        return y

    @staticmethod
    def backward(ctx, gy):
        x, weight = ctx.saved_tensors
        gy = gy.contiguous()
        cout, cin = weight.shape[0], weight.shape[1]
        gx = gw = gb = None
        if ctx.needs_input_grad[0]:
            wd = _packs.get("c3_d", weight, ops.pack_conv3x3_weight_dgrad)
            gx = ops.conv3x3_fprop(gy, wd, cin)
        if ctx.needs_input_grad[1]:
            gw = ops.conv3x3_wgrad(x, gy).permute(1, 2, 0).reshape(cout, cin, 3, 3)
        if ctx.has_bias and ctx.needs_input_grad[2]:
            gb = ops.colsum(gy).clone()
        return gx, gw, gb


def _gw_fwd(w):      # [C, 4, 3, 3] -> fp32 [C, 9, 4]
    return w.permute(0, 2, 3, 1).reshape(w.shape[0], 9, 4).contiguous()


def _gw_bwd(w):      # data-gradient weights: taps flipped, (co, j) transposed inside each group of 4
    c = w.shape[0]
    g = w.view(c // 4, 4, 4, 3, 3).flip(3, 4).permute(0, 2, 1, 3, 4).reshape(c, 4, 3, 3)
    return _gw_fwd(g)


def _g4_dense_blocks(w):
    """Grouped weight ``[C, 4, 3, 3]`` (groups of 4 channels) -> dense block-diagonal weights ``[C/64, 64, 64, 3, 3]``:
    each 64-channel block holds its 16 groups on the diagonal, zeros elsewhere."""
    c = w.shape[0]
    nb = c // 64
    dense = torch.zeros(nb, 16, 4, 16, 4, 3, 3, dtype=w.dtype, device=w.device)
    ar = torch.arange(16, device=w.device)
    dense[:, ar, :, ar] = w.view(nb, 16, 4, 4, 3, 3).permute(1, 0, 2, 3, 4, 5)      # [g][nb, co, ci, ky, kx]
    return dense.view(nb, 64, 64, 3, 3)


def _g4_pack_f(w):      # -> bf16 [C/64, 64, 9*64] fprop operands of the 64-channel blocks
    return torch.stack([ops.pack_conv3x3_weight(d) for d in _g4_dense_blocks(w)])


def _g4_pack_d(w):      # -> bf16 [C/64, 64, 9*64] dgrad operands (taps flipped, in/out transposed)
    return torch.stack([ops.pack_conv3x3_weight_dgrad(d) for d in _g4_dense_blocks(w)])


class _GroupedConv3x3(torch.autograd.Function):
    """nn.Conv2d(c, c, 3, padding=1, groups=c/4) (ResNeXt cardinality 32 x bottleneck 4, res_unet.py:150-156) on the
    tensor cores: every 64-channel slice of the NHWC tensor is a dense 3x3 implicit GEMM whose weight matrix is
    block-diagonal (16 groups of 4x4).  15/16 of the MACs multiply zeros, but the tcgen05 kernel still runs the layer
    an order of magnitude faster than a CUDA-core kernel can (5.4 ms -> ~0.5 ms at 32 x 256 x 256 x 128)."""

    @staticmethod
    def forward(ctx, x, weight, bias):
        n, h, w, c = x.shape
        wp = _packs.get("g4_dense_f", weight, _g4_pack_f)
        y = torch.empty(n, h, w, c, dtype=torch.bfloat16, device=x.device)
        b = None if bias is None else bias.detach()
        for k in range(c // 64):
            sl = slice(64 * k, 64 * k + 64)
            ops.conv3x3_fprop(x[..., sl], wp[k], 64, bias=None if b is None else b[sl], out=y[..., sl])
        ctx.save_for_backward(x, weight)
        ctx.has_bias = bias is not None
        return y

    @staticmethod
    def backward(ctx, gy):
        x, weight = ctx.saved_tensors
        gy = gy.contiguous()
        n, h, w, c = x.shape
        gx = gw = gb = None
        if ctx.needs_input_grad[0]:
            wd = _packs.get("g4_dense_d", weight, _g4_pack_d)
            gx = torch.empty(n, h, w, c, dtype=torch.bfloat16, device=x.device)
            for k in range(c // 64):
                sl = slice(64 * k, 64 * k + 64)
                ops.conv3x3_fprop(gy[..., sl], wd[k], 64, out=gx[..., sl])
        if ctx.needs_input_grad[1]:
            # weight gradient: the dense 64 x 64 wgrad blocks would spend 16x the MACs on off-diagonal entries that are
            # thrown away and measured slower (5.1 ms per Res U-Net step) than the direct kernel that only forms the
            # 4 x 4 group blocks (4.0 ms) -- unlike fprop / dgrad, where the tensor cores win by 10x
            gw = ops.gconv4_3x3_wgrad(x, gy).view(-1, 3, 3, 4).permute(0, 3, 1, 2).contiguous()
        if ctx.has_bias and ctx.needs_input_grad[2]:
            gb = ops.colsum(gy).clone()
        return gx, gw, gb


class _PlaneToWide(torch.autograd.Function):
    """nn.Conv2d(1, c, k, padding=k//2) on an fp32 plane (the network input: no data gradient)."""

    @staticmethod
    def forward(ctx, plane, weight, bias, act):
        c, k = weight.shape[0], weight.shape[2]
        y = ops.conv_plane_to_wide(plane, weight.detach().reshape(c, k * k), None if bias is None else bias.detach(), k,
                                   k // 2, act)
        ctx.save_for_backward(plane, y)
        ctx.k, ctx.act, ctx.has_bias = k, act, bias is not None
        return y

    @staticmethod
    def backward(ctx, gy):
        plane, y = ctx.saved_tensors
        gy = gy.contiguous()
        if ctx.act != ACT_NONE:
            g2 = torch.empty_like(gy)
            ops.act_bwd(y, gy, ctx.act, None, ACT_NONE, g2)
            gy = g2
        c, k = gy.shape[3], ctx.k
        gw = ops.conv_plane_wide_wgrad(plane, gy, k, k // 2).view(c, 1, k, k)
        gb = ops.colsum(gy).clone() if ctx.has_bias else None
        return None, gw, gb, None


class _WideToPlane(torch.autograd.Function):
    """nn.Conv2d(c, 1, k, padding=k//2) (+ Tanh) -> fp32 plane (network output, attention logits)."""

    @staticmethod
    def forward(ctx, x, weight, bias, act):
        c, k = weight.shape[1], weight.shape[2]
        wt = weight.detach().reshape(c, k * k).t().contiguous()           # [taps, c]
        y = ops.conv_wide_to_plane(x, wt, None if bias is None else bias.detach(), k, k // 2, act)
        ctx.save_for_backward(x, weight, y)
        ctx.k, ctx.act, ctx.has_bias = k, act, bias is not None
        return y

    @staticmethod
    def backward(ctx, gy):
        x, weight, y = ctx.saved_tensors
        c, k = weight.shape[1], ctx.k
        g = gy.float().contiguous()
        if ctx.act == ACT_TANH:
            g = g * (1.0 - y * y)
        gx = gw = gb = None
        if ctx.needs_input_grad[0]:
            gx = ops.conv_plane_to_wide(g, weight.detach().reshape(c, k * k), None, k, k // 2, flip=True)
        if ctx.needs_input_grad[1]:
            gw = ops.conv_plane_wide_wgrad(g, x, k, k // 2, flip=True).view(1, c, k, k)
        if ctx.has_bias and ctx.needs_input_grad[2]:
            gb = g.sum().reshape(1)
        return gx, gw, gb, None


class _Conv4x4s2(torch.autograd.Function):
    """nn.Conv2d(cin, cout, 4, 2, 1) (models/pix2pix.py:63-69) on the implicit-GEMM kernel; the packs share the
    fused engine's cache tags, so FusedAdam rewrites them in the optimizer step."""

    @staticmethod
    def forward(ctx, x, weight, bias):
        from . import engine
        y = ops.conv4x4_fprop(x, engine._fprop_pack(weight), weight.shape[0], stride=2,
                              bias=None if bias is None else bias.detach())
        ctx.save_for_backward(x, weight)
        ctx.has_bias = bias is not None
        return y

    @staticmethod
    def backward(ctx, gy):
        from . import engine
        x, weight = ctx.saved_tensors
        gy = gy.contiguous()
        cout, cin = weight.shape[0], weight.shape[1]
        gx = gw = gb = None
        if ctx.needs_input_grad[0]:
            gx = ops.convT4x4s2_fprop(gy, engine._dgrad_pack(weight), cin)
        if ctx.needs_input_grad[1]:
            gw = ops.conv4x4_wgrad(x, gy, stride=2).permute(1, 2, 0).reshape(cout, cin, 4, 4)
        if ctx.has_bias and ctx.needs_input_grad[2]:
            gb = ops.colsum(gy).clone()
        return gx, gw, gb


class _ConvT4x4s2(torch.autograd.Function):
    """nn.ConvTranspose2d(cin, cout, 4, 2, 1) (models/pix2pix.py:99-105), 4 sub-pixel phases."""

    @staticmethod
    def forward(ctx, x, weight, bias):
        from . import engine
        y = ops.convT4x4s2_fprop(x, engine._fpropT_pack(weight), weight.shape[1],
                                 bias=None if bias is None else bias.detach())
        ctx.save_for_backward(x, weight)
        ctx.has_bias = bias is not None
        return y

    @staticmethod
    def backward(ctx, gy):
        from . import engine
        x, weight = ctx.saved_tensors
        gy = gy.contiguous()
        cin, cout = weight.shape[0], weight.shape[1]
        gx = gw = gb = None
        if ctx.needs_input_grad[0]:
            gx = ops.conv4x4_fprop(gy, engine._dgradT_pack(weight), cin, stride=2)
        if ctx.needs_input_grad[1]:
            gw = ops.convT4x4s2_wgrad(x, gy).permute(1, 2, 0).reshape(cin, cout, 4, 4)
        if ctx.has_bias and ctx.needs_input_grad[2]:
            gb = ops.colsum(gy).clone()
        return gx, gw, gb


class _Conv4x4s2In(torch.autograd.Function):
    """nn.Conv2d(1, c, 4, 2, 1) on the fp32 input plane: im2col of the plane + one pointwise GEMM."""

    @staticmethod
    def forward(ctx, plane, weight, bias):
        from . import engine
        n, h, w = plane.shape
        xcol = ops.im2col4x4([plane], h // 2, w // 2, stride=2)
        y = ops.pointwise_gemm(xcol, engine._thin_in_pack(weight), weight.shape[0],
                               bias=None if bias is None else bias.detach(), k_valid=16)
        ctx.save_for_backward(xcol)
        ctx.has_bias = bias is not None
        return y

    @staticmethod
    def backward(ctx, gy):
        (xcol,) = ctx.saved_tensors
        gy = gy.contiguous()
        c = gy.shape[-1]
        gw = ops.pointwise_wgrad(gy, xcol)[:, :16].reshape(c, 1, 4, 4)
        gb = ops.colsum(gy).clone() if ctx.has_bias else None
        return None, gw, gb


class _ConvT4x4s2Out(torch.autograd.Function):
    """nn.ConvTranspose2d(c, 1, 4, 2, 1) + Tanh -> fp32 plane: 16 per-tap partial products per input pixel
    (one GEMM over the wide input) + col2im with bias and Tanh."""

    @staticmethod
    def forward(ctx, x, weight, bias):
        from . import engine
        part = ops.pointwise_gemm(x, engine._thin_out_fprop_pack(weight), 16, out_f32=True)
        y = ops.col2im4x4s2(part, None if bias is None else bias.detach(), ACT_TANH)
        ctx.save_for_backward(x, weight, y)
        ctx.has_bias = bias is not None
        return y

    @staticmethod
    def backward(ctx, g):
        from . import engine
        x, weight, y = ctx.saved_tensors
        n, h2, w2 = y.shape
        g_pre = (g.float() * (1.0 - y * y)).contiguous()
        cin = weight.shape[0]
        gcol = ops.im2col4x4([g_pre], h2 // 2, w2 // 2, stride=2)
        gx = gw = gb = None
        if ctx.needs_input_grad[0]:
            gx = ops.pointwise_gemm(gcol, engine._thin_out_dgrad_pack(weight), cin, k_valid=16)
        if ctx.needs_input_grad[1]:
            gw = ops.pointwise_wgrad(x, gcol)[:, :16].reshape(cin, 1, 4, 4)
        if ctx.has_bias and ctx.needs_input_grad[2]:
            gb = g_pre.sum().reshape(1)
        return gx, gw, gb


# ------------------------------------------------------------------------------------------ 1-4 image planes
# Multi-channel images (RGB, RGBA, ...) enter and leave the networks as fp32 NCHW plane stacks [N, C, H, W] (what the
# model receives and returns, no permute).  C = 1 keeps the 1-plane nodes above; C = 2..4 run the multi-plane kernels.
MAX_PLANES = 4


def _check_planes(c: int, what: str):
    if not 1 <= c <= MAX_PLANES:
        raise RuntimeError(f"pai_b200: {what}={c}: the B200 path takes 1 to {MAX_PLANES} image channels "
                           f"(grayscale, RGB, RGBA); no fallback exists")


def check_image_channels(in_channels: int, out_channels: int):
    """Raises before any launch when a network's image channel counts are outside 1..4."""
    _check_planes(in_channels, "in_channels")
    _check_planes(out_channels, "out_channels")


class _PlanesToWide(torch.autograd.Function):
    """nn.Conv2d(C, c, k, padding=k//2) on fp32 planes ``[N, C, H, W]`` (the network input: no data gradient)."""

    @staticmethod
    def forward(ctx, planes, weight, bias, act):
        c, np_, k = weight.shape[0], weight.shape[1], weight.shape[2]
        y = ops.conv_planes_to_wide(planes, weight.detach().reshape(c, np_ * k * k), None if bias is None else bias.detach(),
                                    k, k // 2, act)
        ctx.save_for_backward(planes, y)
        ctx.k, ctx.act, ctx.has_bias = k, act, bias is not None
        return y

    @staticmethod
    def backward(ctx, gy):
        planes, y = ctx.saved_tensors
        gy = gy.contiguous()
        if ctx.act != ACT_NONE:
            g2 = torch.empty_like(gy)
            ops.act_bwd(y, gy, ctx.act, None, ACT_NONE, g2)
            gy = g2
        c, np_, k = gy.shape[3], planes.shape[1], ctx.k
        gw = ops.conv_planes_wide_wgrad(planes, gy, k, k // 2).view(c, np_, k, k)
        gb = ops.colsum(gy).clone() if ctx.has_bias else None
        return None, gw, gb, None


class _WideToPlanes(torch.autograd.Function):
    """nn.Conv2d(c, C, k, padding=k//2) (+ Tanh) -> fp32 planes ``[N, C, H, W]``, all C from one read of the input."""

    @staticmethod
    def forward(ctx, x, weight, bias, act):
        np_, c, k = weight.shape[0], weight.shape[1], weight.shape[2]
        wt = weight.detach().permute(0, 2, 3, 1).reshape(np_, k * k, c).contiguous()     # [C, taps, c]
        y = ops.conv_wide_to_planes(x, wt, None if bias is None else bias.detach(), k, k // 2, act)
        ctx.save_for_backward(x, weight, y)
        ctx.k, ctx.act, ctx.has_bias = k, act, bias is not None
        return y

    @staticmethod
    def backward(ctx, gy):
        x, weight, y = ctx.saved_tensors
        np_, c, k = weight.shape[0], weight.shape[1], ctx.k
        g = gy.float().contiguous()
        if ctx.act == ACT_TANH:
            g = g * (1.0 - y * y)
        gx = gw = gb = None
        if ctx.needs_input_grad[0]:      # sum over the C gradient planes of the flipped convolution
            wd = weight.detach().transpose(0, 1).reshape(c, np_ * k * k).contiguous()     # [c, C, taps]
            gx = ops.conv_planes_to_wide(g, wd, None, k, k // 2, flip=True)
        if ctx.needs_input_grad[1]:
            dw = ops.conv_planes_wide_wgrad(g, x, k, k // 2, flip=True)                   # [c, C, taps]
            gw = dw.transpose(0, 1).reshape(np_, c, k, k).contiguous()
        if ctx.has_bias and ctx.needs_input_grad[2]:
            gb = g.sum((0, 2, 3))
        return gx, gw, gb, None


class _Conv4x4s2InPlanes(torch.autograd.Function):
    """nn.Conv2d(C, c, 4, 2, 1) on fp32 planes ``[N, C, H, W]``: tap-major im2col (16*C columns) + one pointwise GEMM."""

    @staticmethod
    def forward(ctx, planes, weight, bias):
        from . import engine
        n, np_, h, w = planes.shape
        xcol = ops.im2col4x4_planes(planes, h // 2, w // 2, stride=2)
        y = ops.pointwise_gemm(xcol, engine._thin_in_pack(weight), weight.shape[0],
                               bias=None if bias is None else bias.detach(), k_valid=16 * np_)
        ctx.save_for_backward(xcol)
        ctx.np, ctx.has_bias = np_, bias is not None
        return y

    @staticmethod
    def backward(ctx, gy):
        (xcol,) = ctx.saved_tensors
        gy = gy.contiguous()
        c, np_ = gy.shape[-1], ctx.np
        gw = ops.pointwise_wgrad(gy, xcol)[:, :16 * np_].reshape(c, 4, 4, np_).permute(0, 3, 1, 2).contiguous()
        gb = ops.colsum(gy).clone() if ctx.has_bias else None
        return None, gw, gb


class _ConvT4x4s2OutPlanes(torch.autograd.Function):
    """nn.ConvTranspose2d(c, C, 4, 2, 1) + Tanh -> fp32 planes ``[N, C, 2h, 2w]``: 16*C plane-major per-tap partial
    products per input pixel (one GEMM over the wide input) + col2im with per-plane bias and Tanh."""

    @staticmethod
    def forward(ctx, x, weight, bias):
        from . import engine
        np_ = weight.shape[1]
        part = ops.pointwise_gemm(x, engine._planes_out_fprop_pack(weight), 16 * np_, out_f32=True)
        y = ops.col2im4x4s2_planes(part, np_, None if bias is None else bias.detach(), ACT_TANH)
        ctx.save_for_backward(x, weight, y)
        ctx.has_bias = bias is not None
        return y

    @staticmethod
    def backward(ctx, g):
        from . import engine
        x, weight, y = ctx.saved_tensors
        n, np_, h2, w2 = y.shape
        g_pre = (g.float() * (1.0 - y * y)).contiguous()
        cin = weight.shape[0]
        gcol = ops.im2col4x4_planes(g_pre, h2 // 2, w2 // 2, stride=2)
        gx = gw = gb = None
        if ctx.needs_input_grad[0]:
            gx = ops.pointwise_gemm(gcol, engine._planes_out_dgrad_pack(weight), cin, k_valid=16 * np_)
        if ctx.needs_input_grad[1]:
            gw = ops.pointwise_wgrad(x, gcol)[:, :16 * np_].reshape(cin, 4, 4, np_).permute(0, 3, 1, 2).contiguous()
        if ctx.has_bias and ctx.needs_input_grad[2]:
            gb = g_pre.sum((0, 2, 3))
        return gx, gw, gb


def conv4x4s2(x, mod: nn.Conv2d):
    if x.dim() == 3:
        if mod.in_channels != 1:
            raise RuntimeError("pai_b200: the B200 path takes 1-channel (grayscale PAI) inputs; no fallback exists")
        return _Conv4x4s2In.apply(x, mod.weight, mod.bias)
    if mod.in_channels % 64 or mod.out_channels % 64:
        raise RuntimeError(f"pai_b200: channel counts must be multiples of 64 ({mod})")
    return _Conv4x4s2.apply(x, mod.weight, mod.bias)


def convT4x4s2(x, mod: nn.ConvTranspose2d):
    if mod.in_channels % 64 or mod.out_channels % 64:
        raise RuntimeError(f"pai_b200: channel counts must be multiples of 64 ({mod})")
    return _ConvT4x4s2.apply(x, mod.weight, mod.bias)


def convT4x4s2_out_tanh(x, mod: nn.ConvTranspose2d):
    if mod.out_channels != 1:
        raise RuntimeError("pai_b200: the B200 path produces 1-channel outputs; no fallback exists")
    return _ConvT4x4s2Out.apply(x, mod.weight, mod.bias)


def conv4x4s2_in_planes(planes, mod: nn.Conv2d):
    """First layer of the Attention U-Net on ``to_planes`` output ``[N, C, H, W]``, C = 1..4 (C = 1: use ``conv4x4s2``
    on the ``to_plane`` plane)."""
    _check_planes(mod.in_channels, "in_channels")
    return _Conv4x4s2InPlanes.apply(planes, mod.weight, mod.bias)


def convT4x4s2_out_planes_tanh(x, mod: nn.ConvTranspose2d):
    """Last layer of the Attention U-Net -> fp32 ``[N, C, 2h, 2w]``, C = 1..4."""
    _check_planes(mod.out_channels, "out_channels")
    return _ConvT4x4s2OutPlanes.apply(x, mod.weight, mod.bias)


class _ZeroGradFor(torch.autograd.Function):
    """Identity on ``y``; hands ``param`` an exactly-zero gradient.  Used for a convolution bias in front of a
    train-mode BatchNorm: the BatchNorm backward removes the per-channel mean of the gradient, so the bias gradient is
    mathematically zero (the reference computes ~1e-6 of rounding noise, SURVEY Q11) and the pass over the output
    gradient that would sum it is skipped."""

    @staticmethod
    def forward(ctx, y, param):
        ctx.meta = (param.shape, param.device)
        return y.view_as(y)

    @staticmethod
    def backward(ctx, gy):
        shape, dev = ctx.meta
        return gy, torch.zeros(shape, dtype=torch.float32, device=dev)


class _NoBias:
    """View of an ``nn.Conv2d`` whose bias is detached (no bias-gradient pass in the convolution's backward)."""

    def __init__(self, mod):
        self.mod = mod
        self.bias = None if mod.bias is None else mod.bias.detach()

    def __getattr__(self, name):
        return getattr(self.mod, name)


def conv2d(x, mod: nn.Conv2d, before_train_bn: bool = False, padded: bool = False):
    """Dispatch of an ``nn.Conv2d`` parameter holder onto the kernels (NHWC bf16 in / out).  ``before_train_bn``: the
    output feeds a BatchNorm2d in training mode, whose backward makes the bias gradient exactly zero.  ``padded``:
    channel counts that are not multiples of 64 travel in zero-padded 64-channel carriers (input and output)."""
    if before_train_bn and mod.bias is not None and mod.bias.requires_grad:
        return _ZeroGradFor.apply(conv2d(x, _NoBias(mod), padded=padded), mod.bias)
    k, cin, cout, groups = mod.kernel_size[0], mod.in_channels, mod.out_channels, mod.groups
    if padded and groups == 1 and k in (1, 3) and x.shape[-1] == _pad64(cin) and (cin % 64 or cout % 64):
        if mod.stride != (1, 1) or mod.padding != (k // 2, k // 2) or mod.dilation != (1, 1):
            raise RuntimeError(f"pai_b200: unsupported convolution geometry {mod}")
        # ResNet-50 style bottlenecks of 16 / 32 channels (res_unet.py:84-95)
        return _ConvPadded.apply(x, mod.weight, mod.bias)
    if mod.stride != (1, 1) or mod.padding != (k // 2, k // 2) or mod.dilation != (1, 1):
        raise RuntimeError(f"pai_b200: unsupported convolution geometry {mod}")
    if groups == 1 and cin % 64 == 0 and k == 1 and cout % 8 == 0:
        return _Conv1x1.apply(x, mod.weight, mod.bias)
    if groups == 1 and cin % 64 == 0 and cout % 64 == 0 and k == 3:
        return _Conv3x3.apply(x, mod.weight, mod.bias)
    if k == 3 and groups > 1 and cin == cout and cin // groups == 4 and cin % 64 == 0:
        return _GroupedConv3x3.apply(x, mod.weight, mod.bias)
    raise RuntimeError(f"pai_b200: no B200 kernel for {mod} (channel counts must be multiples of 64, or the "
                       "ResNeXt 4-channel groups); there is no fallback")


def conv_in(plane, mod: nn.Conv2d, act=ACT_NONE):
    if mod.in_channels != 1:
        raise RuntimeError("pai_b200: the B200 path takes 1-channel (grayscale PAI) inputs; got "
                           f"in_channels={mod.in_channels}. No fallback exists.")
    return _PlaneToWide.apply(plane, mod.weight, mod.bias, act)


def conv_out(x, mod: nn.Conv2d, act=ACT_NONE):
    if mod.out_channels != 1:
        raise RuntimeError("pai_b200: the B200 path produces 1-channel outputs; got "
                           f"out_channels={mod.out_channels}. No fallback exists.")
    return _WideToPlane.apply(x, mod.weight, mod.bias, act)


def conv_in_planes(planes, mod: nn.Conv2d, act=ACT_NONE):
    """``conv_in`` for ``to_planes`` output ``[N, C, H, W]``, C = 1..4."""
    _check_planes(mod.in_channels, "in_channels")
    return _PlanesToWide.apply(planes, mod.weight, mod.bias, act)


def conv_out_planes(x, mod: nn.Conv2d, act=ACT_NONE):
    """``conv_out`` -> fp32 ``[N, C, H, W]``, C = 1..4."""
    _check_planes(mod.out_channels, "out_channels")
    return _WideToPlanes.apply(x, mod.weight, mod.bias, act)


# ------------------------------------------------------------------------------------------ BatchNorm (+activation)
class _BatchNormAct(torch.autograd.Function):
    """BatchNorm2d (+ activation) over the first ``c = num_features`` channels of ``raw``; a wider ``raw`` is a
    zero-padded 64-channel carrier (Trans U-Net bottlenecks of 16 / 32 channels) whose tail stays zero."""

    @staticmethod
    def forward(ctx, raw, weight, bias, mod, act):
        training = mod.training or mod.running_mean is None
        c, cfull = weight.shape[0], raw.shape[-1]
        rv = raw if c == cfull else raw[..., :c]
        m = raw.numel() // cfull
        sums = ops.bn_stats(rv) if training else None
        ss = ops.bn_finalize(sums, m, c, weight.detach(), bias.detach(), mod.running_mean, mod.running_var,
                             training=training, eps=mod.eps, momentum=mod.momentum if mod.momentum is not None else 0.1)
        if training and mod.num_batches_tracked is not None:
            mod.num_batches_tracked.add_(1)
        alloc = torch.empty if c == cfull else torch.zeros
        out = alloc(*raw.shape, dtype=torch.bfloat16, device=raw.device)
        ops.bn_apply_act(rv, ss, out if c == cfull else out[..., :c], act)
        ctx.save_for_backward(raw, ss, weight)
        ctx.act, ctx.training = act, training
        return out

    @staticmethod
    def backward(ctx, g):
        raw, ss, weight = ctx.saved_tensors
        g = g.contiguous()
        c, cfull = weight.shape[0], raw.shape[-1]
        if not ctx.training:
            raise RuntimeError("pai_b200: backward through eval-mode BatchNorm is not implemented")
        rv, gv = (raw, g) if c == cfull else (raw[..., :c], g[..., :c])
        sums = ops.bn_bwd_reduce(rv, ss, gv, ctx.act)
        alloc = torch.empty if c == cfull else torch.zeros
        d_raw = alloc(*raw.shape, dtype=torch.bfloat16, device=raw.device)
        ops.bn_bwd_apply(rv, ss, gv, ctx.act, None, ACT_NONE, sums, weight.detach(), d_raw if c == cfull else d_raw[..., :c])
        return d_raw, sums[c:], sums[:c], None, None


def batchnorm_act(raw, mod: nn.BatchNorm2d, act=ACT_NONE):
    if abs(mod.eps - BN_EPS) > 0 and mod.eps <= 0:
        raise RuntimeError("pai_b200: bad BatchNorm eps")
    return _BatchNormAct.apply(raw, mod.weight, mod.bias, mod, act)


# ------------------------------------------------------------------------------------------ elementwise / resampling
class _AddAct(torch.autograd.Function):
    @staticmethod
    def forward(ctx, a, b, act):
        out = ops.add_act(a, b, act)
        ctx.act = act
        if act != ACT_NONE:
            ctx.save_for_backward(out)
        return out

    @staticmethod
    def backward(ctx, g):
        if ctx.act != ACT_NONE:
            (out,) = ctx.saved_tensors
            g2 = torch.empty(*out.shape, dtype=torch.bfloat16, device=out.device)
            ops.act_bwd(out, g.contiguous(), ctx.act, None, ACT_NONE, g2)
            g = g2
        return g, g, None


class _Act(torch.autograd.Function):
    @staticmethod
    def forward(ctx, a, act):
        out = ops.add_act(a, None, act)
        ctx.act = act
        ctx.save_for_backward(out)
        return out

    @staticmethod
    def backward(ctx, g):
        (out,) = ctx.saved_tensors
        g2 = torch.empty(*out.shape, dtype=torch.bfloat16, device=out.device)
        ops.act_bwd(out, g.contiguous(), ctx.act, None, ACT_NONE, g2)
        return g2, None


class _MaxPool2(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x):
        ctx.save_for_backward(x)
        return ops.maxpool2_fwd(x)

    @staticmethod
    def backward(ctx, g):
        (x,) = ctx.saved_tensors
        return ops.maxpool2_bwd(x, g.contiguous())


class _Upsample2(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x):
        return ops.upsample2_fwd(x)

    @staticmethod
    def backward(ctx, g):
        return ops.upsample2_bwd(g.contiguous())


class _ScaleRows(torch.autograd.Function):
    """``x * s`` with a per-pixel fp32 factor (attention_unet.py:96)."""

    @staticmethod
    def forward(ctx, x, s):
        ctx.save_for_backward(x, s)
        return ops.scale_rows_fwd(x, s)

    @staticmethod
    def backward(ctx, g):
        x, s = ctx.saved_tensors
        gx, gs = ops.scale_rows_bwd(x, s, g.contiguous())
        return gx, gs


def add_act(a, b, act=ACT_NONE):
    return _AddAct.apply(a, b, act)


def activation(a, act):
    return _Act.apply(a, act)


def maxpool2(x):
    return _MaxPool2.apply(x)


def upsample2(x):
    return _Upsample2.apply(x)


def scale_rows(x, s):
    return _ScaleRows.apply(x, s)


class _Dropout2d(torch.autograd.Function):
    """nn.Dropout2d in training mode: whole channels of a sample are zeroed with probability p, the rest scaled by
    1 / (1 - p); the mask is drawn with torch's device generator (the reference's CPU stream cannot be reproduced)."""

    @staticmethod
    def forward(ctx, x, p):
        mask = ops.dropout2d_mask(x.shape[0], x.shape[3], p, x.device)
        ctx.save_for_backward(mask)
        return ops.scale_channels(x, mask)

    @staticmethod
    def backward(ctx, gy):
        (mask,) = ctx.saved_tensors
        return ops.scale_channels(gy.contiguous(), mask), None


def dropout2d(x, mod):
    if isinstance(mod, nn.Identity) or not mod.training or mod.p == 0:
        return x
    return _Dropout2d.apply(x, float(mod.p))


# ------------------------------------------------------------------------------------------ Trans U-Net pieces
def _pack_p1_f(w, cin_p):
    cout, cin = w.shape[0], w.shape[1]
    out = torch.zeros(_pad64(cout), cin_p, dtype=torch.bfloat16, device=w.device)
    out[:cout, :cin].copy_(w.reshape(cout, cin))
    return out


def _pack_p1_d(w, cin_p):
    cout, cin = w.shape[0], w.shape[1]
    out = torch.zeros(cin_p, _pad64(cout), dtype=torch.bfloat16, device=w.device)
    out[:cin, :cout].copy_(w.reshape(cout, cin).t())
    return out


class _Conv1x1Padded(torch.autograd.Function):
    """Bias-free 1x1 convolution between zero-padded 64-channel carriers: x ``[..., pad64(cin)]`` ->
    ``[..., pad64(cout)]`` (trans_unet.py:188-205 bottleneck projections with 16 / 32 channels)."""

    @staticmethod
    def forward(ctx, x, weight):
        cin_p = x.shape[-1]
        wp = _packs.get(f"p1_f{cin_p}", weight, lambda w: _pack_p1_f(w, cin_p))
        y = ops.pointwise_gemm(x, wp, wp.shape[0])
        ctx.save_for_backward(x, weight)
        return y

    @staticmethod
    def backward(ctx, gy):
        x, weight = ctx.saved_tensors
        gy = gy.contiguous()
        cout, cin, cin_p = weight.shape[0], weight.shape[1], x.shape[-1]
        gx = gw = None
        if ctx.needs_input_grad[0]:
            wt = _packs.get(f"p1_d{cin_p}", weight, lambda w: _pack_p1_d(w, cin_p))
            gx = ops.pointwise_gemm(gy, wt, cin_p)
        if ctx.needs_input_grad[1]:
            gw = ops.pointwise_wgrad(gy, x)[:cout, :cin].reshape(weight.shape)
        return gx, gw


def _pad_w(w, cin_p):
    """[cout, cin, k, k] -> zero-padded fp32 [pad64(cout), cin_p, k, k]."""
    cout, cin, k = w.shape[0], w.shape[1], w.shape[2]
    out = torch.zeros(_pad64(cout), cin_p, k, k, dtype=torch.float32, device=w.device)
    out[:cout, :cin].copy_(w)
    return out


def _pad_b(b, cout_p):
    out = torch.zeros(cout_p, dtype=torch.float32, device=b.device)
    out[:b.shape[0]].copy_(b)
    return out


class _ConvPadded(torch.autograd.Function):
    """nn.Conv2d(cin, cout, k in {1, 3}, padding=k//2) with bias between zero-padded 64-channel carriers:
    x ``[..., pad64(cin)]`` -> ``[..., pad64(cout)]``, padded output channels stay exactly zero (zero weights, zero
    bias).  The GEMMs run on the padded shapes (pointwise / 3x3 implicit GEMM); gradients are sliced back."""

    @staticmethod
    def forward(ctx, x, weight, bias):
        k, cin_p = weight.shape[2], x.shape[-1]
        cout_p = _pad64(weight.shape[0])
        bp = None if bias is None else _packs.get("cp_b", bias, lambda b: _pad_b(b, cout_p))
        if k == 1:
            wp = _packs.get(f"p1_f{cin_p}", weight, lambda w: _pack_p1_f(w, cin_p))
            y = ops.pointwise_gemm(x, wp, cout_p, bias=bp)
        else:
            wp = _packs.get(f"cp3_f{cin_p}", weight, lambda w: ops.pack_conv3x3_weight(_pad_w(w, cin_p)))
            y = ops.conv3x3_fprop(x, wp, cout_p, bias=bp)
        ctx.save_for_backward(x, weight)
        ctx.has_bias = bias is not None
        return y

    @staticmethod
    def backward(ctx, gy):
        x, weight = ctx.saved_tensors
        gy = gy.contiguous()
        cout, cin, k, cin_p = weight.shape[0], weight.shape[1], weight.shape[2], x.shape[-1]
        gx = gw = gb = None
        if ctx.needs_input_grad[0]:
            if k == 1:
                wt = _packs.get(f"p1_d{cin_p}", weight, lambda w: _pack_p1_d(w, cin_p))
                gx = ops.pointwise_gemm(gy, wt, cin_p)
            else:
                wd = _packs.get(f"cp3_d{cin_p}", weight, lambda w: ops.pack_conv3x3_weight_dgrad(_pad_w(w, cin_p)))
                gx = ops.conv3x3_fprop(gy, wd, cin_p)
        if ctx.needs_input_grad[1]:
            if k == 1:
                gw = ops.pointwise_wgrad(gy, x)[:cout, :cin].reshape(weight.shape)
            else:
                gw = ops.conv3x3_wgrad(x, gy)[:, :cout, :cin].permute(1, 2, 0).reshape(cout, cin, 3, 3)
        if ctx.has_bias and ctx.needs_input_grad[2]:
            gb = ops.colsum(gy)[:cout].clone()
        return gx, gw, gb


def _w3_as_4x4(w, cin_p):
    """[cout, cin, 3, 3] -> zero-padded [pad64(cout), cin_p, 4, 4]: a 3x3 stride-2 pad-1 convolution reads input
    2*o - 1 + k, exactly taps 0..2 of the 4x4 stride-2 pad-1 convolution."""
    cout, cin = w.shape[0], w.shape[1]
    out = torch.zeros(_pad64(cout), cin_p, 4, 4, dtype=torch.float32, device=w.device)
    out[:cout, :cin, :3, :3].copy_(w)
    return out


class _Conv3x3s2Padded(torch.autograd.Function):
    """Bias-free nn.Conv2d(c, c, 3, stride=2, padding=1) between zero-padded 64-channel carriers, run on the 4x4
    stride-2 implicit-GEMM kernels with a zero 4th kernel row / column (trans_unet.py:191-199)."""

    @staticmethod
    def forward(ctx, x, weight):
        cin_p = x.shape[-1]
        wp = _packs.get(f"c3s2_f{cin_p}", weight, lambda w: ops.pack_conv_weight(_w3_as_4x4(w, cin_p)))
        y = ops.conv4x4_fprop(x, wp, wp.shape[0], stride=2)
        ctx.save_for_backward(x, weight)
        return y

    @staticmethod
    def backward(ctx, gy):
        x, weight = ctx.saved_tensors
        gy = gy.contiguous()
        cout, cin, cin_p = weight.shape[0], weight.shape[1], x.shape[-1]
        gx = gw = None
        if ctx.needs_input_grad[0]:
            wd = _packs.get(f"c3s2_d{cin_p}", weight, lambda w: ops.pack_convT_weight(_w3_as_4x4(w, cin_p)))
            gx = ops.convT4x4s2_fprop(gy, wd, cin_p)
        if ctx.needs_input_grad[1]:
            dw = ops.conv4x4_wgrad(x, gy, stride=2)                      # [16, cout_p, cin_p]
            gw = dw.view(4, 4, dw.shape[1], dw.shape[2])[:3, :3, :cout, :cin].permute(2, 3, 0, 1).contiguous()
        return gx, gw


class _Subsample2(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x):
        return ops.subsample2(x)

    @staticmethod
    def backward(ctx, g):
        return ops.subsample2(g.contiguous(), scatter=True)


class _LayerNorm(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, weight, bias, eps):
        y, mean, rstd = ops.layernorm_fwd(x, weight.detach(), bias.detach(), eps)
        ctx.save_for_backward(x, weight, mean, rstd)
        return y

    @staticmethod
    def backward(ctx, g):
        x, weight, mean, rstd = ctx.saved_tensors
        dx, dgamma, dbeta = ops.layernorm_bwd(x, g.contiguous(), weight.detach(), mean, rstd)
        return dx, dgamma, dbeta, None


class _Gelu(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x):
        ctx.save_for_backward(x)
        return ops.gelu_fwd(x)

    @staticmethod
    def backward(ctx, g):
        (x,) = ctx.saved_tensors
        return ops.gelu_bwd(x, g.contiguous())


class _Attention(torch.autograd.Function):
    """softmax(Q K^T / sqrt(hd)) V per head over the sequence axis of ``qkv [S*B, 3E]``."""

    @staticmethod
    def forward(ctx, qkv, s, b, heads):
        out, probs = ops.attn_fwd(qkv, s, b, heads)
        ctx.save_for_backward(qkv, probs)
        ctx.dims = (s, b, heads)
        return out

    @staticmethod
    def backward(ctx, g):
        qkv, probs = ctx.saved_tensors
        s, b, heads = ctx.dims
        return ops.attn_bwd(qkv, g.contiguous(), probs, s, b, heads), None, None, None


# Train-mode dropout of nn.TransformerEncoderLayer: each node saves the forward's int64 key tensor (never a mask); the
# backward kernels regenerate the mask of their ``site`` from it.
class _AttentionDropout(torch.autograd.Function):
    """softmax(Q K^T / sqrt(hd)) with dropout on the probabilities, times V (site 0 of a layer)."""

    @staticmethod
    def forward(ctx, qkv, s, b, heads, key, site, p):
        out, probs = ops.attn_fwd_dropout(qkv, s, b, heads, key, site, p)
        ctx.save_for_backward(qkv, probs, key)
        ctx.dims = (s, b, heads, site, p)
        return out

    @staticmethod
    def backward(ctx, g):
        qkv, probs, key = ctx.saved_tensors
        s, b, heads, site, p = ctx.dims
        return ops.attn_bwd_dropout(qkv, g.contiguous(), probs, s, b, heads, key, site, p), None, None, None, None, None, None


class _AddDropoutLayerNorm(torch.autograd.Function):
    """LayerNorm(x + dropout(y)): the residual add and norm after the attention (site 1) or feed-forward (site 3) block."""

    @staticmethod
    def forward(ctx, x, y, weight, bias, eps, key, site, p):
        z, out, mean, rstd = ops.add_dropout_layernorm_fwd(x, y, weight.detach(), bias.detach(), eps, key, site, p)
        ctx.save_for_backward(z, weight, mean, rstd, key)
        ctx.site, ctx.p = site, p
        return out

    @staticmethod
    def backward(ctx, g):
        z, weight, mean, rstd, key = ctx.saved_tensors
        dz, dy, dgamma, dbeta = ops.layernorm_bwd_dropout(z, g.contiguous(), weight.detach(), mean, rstd, key, ctx.site, ctx.p)
        return dz, dy, dgamma, dbeta, None, None, None, None


class _GeluDropout(torch.autograd.Function):
    """dropout(GELU(x)) inside the feed-forward block (site 2)."""

    @staticmethod
    def forward(ctx, x, key, site, p):
        ctx.save_for_backward(x, key)
        ctx.site, ctx.p = site, p
        return ops.gelu_dropout_fwd(x, key, site, p)

    @staticmethod
    def backward(ctx, g):
        x, key = ctx.saved_tensors
        return ops.gelu_dropout_bwd(x, g.contiguous(), key, ctx.site, ctx.p), None, None, None


def conv1x1_padded(x, mod: nn.Conv2d):
    if mod.bias is not None or mod.kernel_size != (1, 1) or mod.groups != 1 or x.shape[-1] != _pad64(mod.in_channels):
        raise RuntimeError(f"pai_b200: unexpected bottleneck projection {mod}")
    return _Conv1x1Padded.apply(x, mod.weight)


def conv3x3s2_padded(x, mod: nn.Conv2d):
    if (mod.bias is not None or mod.kernel_size != (3, 3) or mod.stride != (2, 2) or mod.padding != (1, 1)
            or mod.groups != 1 or x.shape[-1] != _pad64(mod.in_channels)):
        raise RuntimeError(f"pai_b200: unexpected strided bottleneck convolution {mod}")
    return _Conv3x3s2Padded.apply(x, mod.weight)


def subsample2(x):
    return _Subsample2.apply(x)


def linear(x2d, weight, bias):
    """nn.Linear on the tensor-core pointwise GEMM; x2d is a dense [m, in] bf16 matrix."""
    if weight.shape[1] % 64 or weight.shape[0] % 8:
        raise RuntimeError(f"pai_b200: Linear {tuple(weight.shape)} needs in % 64 == 0 and out % 8 == 0")
    return _Conv1x1.apply(x2d, weight, bias)


def layernorm(x2d, mod: nn.LayerNorm):
    return _LayerNorm.apply(x2d, mod.weight, mod.bias, mod.eps)


def gelu(x2d):
    return _Gelu.apply(x2d)


def attention(qkv2d, s, b, heads):
    return _Attention.apply(qkv2d, s, b, heads)


def attention_dropout(qkv2d, s, b, heads, key, site, p):
    return _AttentionDropout.apply(qkv2d, s, b, heads, key, site, p)


def add_dropout_layernorm(x2d, y2d, mod: nn.LayerNorm, key, site, p):
    return _AddDropoutLayerNorm.apply(x2d, y2d, mod.weight, mod.bias, mod.eps, key, site, p)


def gelu_dropout(x2d, key, site, p):
    return _GeluDropout.apply(x2d, key, site, p)


def to_plane(x: torch.Tensor) -> torch.Tensor:
    """``[N, 1, H, W]`` network input -> fp32 plane ``[N, H, W]`` on the GPU (the reference's ``x.type(float32)``)."""
    if not x.is_cuda:
        raise RuntimeError("pai_b200: the B200 path needs CUDA tensors; there is no CPU fallback")
    if x.dim() != 4 or x.shape[1] != 1:
        raise RuntimeError(f"pai_b200: expected a [N, 1, H, W] input, got {tuple(x.shape)}")
    return x.float().contiguous().view(x.shape[0], x.shape[2], x.shape[3])


def to_planes(x: torch.Tensor, channels: int) -> torch.Tensor:
    """``[N, C, H, W]`` network input with C == ``channels`` (1..4) -> contiguous fp32 planes ``[N, C, H, W]``."""
    _check_planes(channels, "in_channels")
    if not x.is_cuda:
        raise RuntimeError("pai_b200: the B200 path needs CUDA tensors; there is no CPU fallback")
    if x.dim() != 4 or x.shape[1] != channels:
        raise RuntimeError(f"pai_b200: expected a [N, {channels}, H, W] input, got {tuple(x.shape)}")
    return x.float().contiguous()
