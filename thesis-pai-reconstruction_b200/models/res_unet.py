"""Mirror of /root/reference/models/res_unet.py (``ResUnetGAN``, ``ResUnet`` and the four residual block
flavours "18", "50", "v2", "next") on the B200 kernels.

The module tree (``in_conv``, ``encoders.{i}.encode.0.conv_block.{k}``, ``...conv_skip.{k}``,
``decoders.{j}.decode.0...``, ``out.0``) and constructor signatures are the reference's, so its
``state_dict`` keys, shapes and initial weights (same seed) are reproduced exactly; the ``nn.Conv2d`` /
``nn.BatchNorm2d`` sub-modules only hold parameters.  ``forward`` runs the layer nodes of
``pai_b200.layers`` on NHWC bf16 activations: 1x1 and dense 3x3 convolutions on the tcgen05 implicit
GEMM, the ResNeXt grouped 3x3, BatchNorm(+ReLU), residual add, MaxPool2d(2) and Upsample(x2) as
HBM-bound stream kernels.  There is no PyTorch-op fallback.
"""
from typing import Literal, Sequence

import torch
import torch.nn as nn

from pai_b200 import check, engine, layers as L, lib

from .wrapper import UnetWrapper

ResType = Literal["18", "50", "v2", "next"]


class ResUnetGAN(UnetWrapper):
    """Residual U-net (+ PatchGAN for ``loss_type="gan"``), constructor as models/res_unet.py:28-36."""

    def __init__(
        self,
        in_channels: int = 3,
        out_channels: int = 3,
        res_type: ResType = "18",
        channel_mults: Sequence[int] = (1, 2, 4, 8, 8, 8, 8, 8),
        dropout: float = 0.5,
        loss_type: Literal["gan", "ssim", "psnr", "ssim+psnr", "mse"] = "gan",
    ):
        unet = ResUnet(in_channels, out_channels, res_type, channel_mults=channel_mults, dropout=dropout)
        super().__init__(unet, loss_type=loss_type)
        self.example_input_array = torch.Tensor(2, in_channels, 256, 256)
        self.save_hyperparameters()


def _cba(x, conv, bn, act, padded=False):
    """Conv2d -> BatchNorm2d -> activation (``padded``: bottleneck channels in zero-padded 64-channel carriers)."""
    return L.batchnorm_act(L.conv2d(x, conv, before_train_bn=bn.training, padded=padded), bn, act)


class _SkipMixin:
    def _skip(self, x):
        if isinstance(self.conv_skip, nn.Identity):
            return x
        return self._skip_path(x)


class ResidualBlock18(nn.Module, _SkipMixin):
    """relu(conv3x3-bn-relu-conv3x3-bn (x) + skip(x))   (res_unet.py:53-90)."""

    def __init__(self, in_channels: int, out_channels: int):
        super().__init__()
        self.conv_block = nn.Sequential(
            nn.Conv2d(in_channels, out_channels, kernel_size=3, padding=1),
            nn.BatchNorm2d(out_channels),
            nn.ReLU(),
            nn.Conv2d(out_channels, out_channels, kernel_size=3, padding=1),
            nn.BatchNorm2d(out_channels),
        )
        self.conv_skip = nn.Sequential(
            nn.Conv2d(in_channels, out_channels, kernel_size=1),
            nn.BatchNorm2d(out_channels),
        ) if in_channels != out_channels else nn.Identity()
        self.out = nn.ReLU()

    def _skip_path(self, x):
        return _cba(x, self.conv_skip[0], self.conv_skip[1], L.ACT_NONE)

    def forward(self, x):
        b = self.conv_block
        h = _cba(x, b[0], b[1], L.ACT_RELU)
        h = _cba(h, b[3], b[4], L.ACT_NONE)
        return L.add_act(h, self._skip(x), L.ACT_RELU)


class ResidualBlock50(nn.Module, _SkipMixin):
    """Bottleneck block: 1x1 (cin/4) - 3x3 - 1x1, ReLU after the sum   (res_unet.py:93-130)."""

    def __init__(self, in_channels: int, out_channels: int):
        super().__init__()
        mid = in_channels // 4
        self.conv_block = nn.Sequential(
            nn.Conv2d(in_channels, mid, kernel_size=1),
            nn.BatchNorm2d(mid),
            nn.ReLU(),
            nn.Conv2d(mid, mid, kernel_size=3, padding=1),
            nn.BatchNorm2d(mid),
            nn.ReLU(),
            nn.Conv2d(mid, out_channels, kernel_size=1),
            nn.BatchNorm2d(out_channels),
        )
        self.conv_skip = nn.Sequential(
            nn.Conv2d(in_channels, out_channels, kernel_size=1),
            nn.BatchNorm2d(out_channels),
        ) if in_channels != out_channels else nn.Identity()
        self.out = nn.ReLU()

    def _skip_path(self, x):
        return _cba(x, self.conv_skip[0], self.conv_skip[1], L.ACT_NONE)

    def forward(self, x):
        b = self.conv_block
        pad = b[0].out_channels % 64 != 0           # 16 / 32-channel bottlenecks of the first levels
        h = _cba(x, b[0], b[1], L.ACT_RELU, padded=pad)
        h = _cba(h, b[3], b[4], L.ACT_RELU, padded=pad)
        h = _cba(h, b[6], b[7], L.ACT_NONE, padded=pad)
        return L.add_act(h, self._skip(x), L.ACT_RELU)


class ResidualBlockV2(nn.Module, _SkipMixin):
    """Pre-activation block: bn-relu-conv3x3-bn-relu-conv3x3, raw sum   (res_unet.py:133-171, SURVEY Q10)."""

    def __init__(self, in_channels: int, out_channels: int):
        super().__init__()
        self.conv_block = nn.Sequential(
            nn.BatchNorm2d(in_channels),
            nn.ReLU(),
            nn.Conv2d(in_channels, out_channels, kernel_size=3, padding=1),
            nn.BatchNorm2d(out_channels),
            nn.ReLU(),
            nn.Conv2d(out_channels, out_channels, kernel_size=3, padding=1),
        )
        self.conv_skip = nn.Sequential(
            nn.BatchNorm2d(in_channels),
            nn.ReLU(),
            nn.Conv2d(in_channels, out_channels, kernel_size=1),
        ) if in_channels != out_channels else nn.Identity()

    def _skip_path(self, x):
        return L.conv2d(L.batchnorm_act(x, self.conv_skip[0], L.ACT_RELU), self.conv_skip[2])

    def forward(self, x):
        b = self.conv_block
        h = L.conv2d(L.batchnorm_act(x, b[0], L.ACT_RELU), b[2])
        h = L.conv2d(L.batchnorm_act(h, b[3], L.ACT_RELU), b[5])
        return L.add_act(h, self._skip(x), L.ACT_NONE)


class ResidualBlockNeXt(nn.Module, _SkipMixin):
    """ResNeXt block: 1x1 -> grouped 3x3 (32 groups x 4) -> 1x1, each BN+ReLU; raw sum with the skip
    (res_unet.py:174-235; no activation after the add, SURVEY Q10)."""

    def __init__(self, in_channels: int, out_channels: int, cardinality: int = 32, bottleneck: int = 4):
        super().__init__()
        width = bottleneck * cardinality
        self.conv_block = nn.Sequential(
            nn.Conv2d(in_channels, width, kernel_size=1),
            nn.BatchNorm2d(width),
            nn.ReLU(),
            nn.Conv2d(width, width, kernel_size=3, padding=1, groups=cardinality),
            nn.BatchNorm2d(width),
            nn.ReLU(),
            nn.Conv2d(width, out_channels, kernel_size=1),
            nn.BatchNorm2d(out_channels),
            nn.ReLU(),
        )
        self.conv_skip = nn.Sequential(
            nn.Conv2d(in_channels, out_channels, kernel_size=1),
            nn.BatchNorm2d(out_channels),
        ) if in_channels != out_channels else nn.Identity()

    def _skip_path(self, x):
        return _cba(x, self.conv_skip[0], self.conv_skip[1], L.ACT_NONE)

    def forward(self, x):
        b = self.conv_block
        h = _cba(x, b[0], b[1], L.ACT_RELU)
        h = _cba(h, b[3], b[4], L.ACT_RELU)
        h = _cba(h, b[6], b[7], L.ACT_RELU)
        return L.add_act(h, self._skip(x), L.ACT_NONE)


res_blocks = {
    "18": ResidualBlock18,
    "50": ResidualBlock50,
    "v2": ResidualBlockV2,
    "next": ResidualBlockNeXt,
}


class EncoderBlock(nn.Module):
    """residual block -> MaxPool2d(2)   (res_unet.py:246-262)."""

    def __init__(self, in_channels: int, out_channels: int, res_type: ResType):
        super().__init__()
        self.encode = nn.Sequential(res_blocks[res_type](in_channels, out_channels), nn.MaxPool2d(2))

    def forward(self, x):
        return L.maxpool2(self.encode[0](x))


class DecoderBlock(nn.Module):
    """residual block -> Dropout2d -> Upsample(x2, nearest)   (res_unet.py:265-295)."""

    def __init__(self, in_channels: int, out_channels: int, res_type: ResType, dropout: float = 0.0):
        super().__init__()
        self.decode = nn.Sequential(
            res_blocks[res_type](in_channels, out_channels),
            nn.Dropout2d(dropout) if dropout > 0 else nn.Identity(),
            nn.Upsample(scale_factor=2),
        )

    def forward(self, x):
        return L.upsample2(L.dropout2d(self.decode[0](x), self.decode[1]))


class ResUnet(nn.Module):
    """``[N, in_channels, H, W] -> [N, out_channels, H, W]`` in (-1, 1), 1 to 4 channels each (grayscale, RGB, RGBA);
    H and W divisible by 2^len(channel_mults)."""

    def __init__(self, in_channels: int = 3, out_channels: int = 3, res_type: ResType = "18",
                 channel_mults: Sequence[int] = (1, 2, 4, 8, 8, 8, 8, 8), dropout: float = 0.5):
        super().__init__()
        self.in_conv = nn.Conv2d(in_channels, 64, kernel_size=3, padding=1)
        widths = [64 * m for m in channel_mults]
        depth = len(widths)
        down, cin = [], 64
        for cw in widths:
            down.append(EncoderBlock(cin, cw, res_type))
            cin = cw
        self.encoders = nn.ModuleList(down)

        up, widest = [], max(channel_mults)
        for lvl in range(depth - 2, -1, -1):
            drop = dropout if (channel_mults[lvl] == widest and lvl > depth - 5) else 0
            up.append(DecoderBlock(cin, widths[lvl], res_type, dropout=drop))
            cin = 2 * widths[lvl]
        up.append(DecoderBlock(cin, widths[0], res_type))
        self.decoders = nn.ModuleList(up)
        self.out = nn.Sequential(nn.Conv2d(widths[0], out_channels, kernel_size=3, padding=1), nn.Tanh())

    def forward(self, x):
        with lib.on_device(x):
            return self._forward(x)

    def _forward(self, x):
        if engine.check_path_enabled():                # exact fp32 kernels (pai_b200/check.py)
            return check.res_unet_forward(self, x)
        n, _, hh, ww = x.shape
        depth = len(self.encoders)
        if hh % (1 << depth) or ww % (1 << depth):
            raise RuntimeError(f"pai_b200: input {hh}x{ww} must be divisible by 2^{depth}")
        cin, cout = self.in_conv.in_channels, self.out[0].out_channels
        L.check_image_channels(cin, cout)
        if cin == 1:
            h = L.conv_in(L.to_plane(x), self.in_conv)
        else:
            h = L.conv_in_planes(L.to_planes(x, cin), self.in_conv)
        skips = []
        for enc in self.encoders:
            h = enc(h)
            skips.append(h)
        skips.pop()                       # the deepest map feeds the first decoder directly
        for j, dec in enumerate(self.decoders):
            if j != 0:
                h = torch.cat([h, skips.pop()], dim=-1)      # NHWC: channel concat on the last axis
            h = dec(h)
        if cout == 1:
            y = L.conv_out(h, self.out[0], L.ACT_TANH)
            return y.view(n, 1, hh, ww)
        return L.conv_out_planes(h, self.out[0], L.ACT_TANH)
