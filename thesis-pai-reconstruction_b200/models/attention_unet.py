"""Mirror of /root/reference/models/attention_unet.py (``AttentionUnetGAN``, ``AttentionBlock``,
``AttentionUnet``) on the B200 kernels: the Pix2Pix encoder / decoder (4x4 stride-2 implicit GEMMs) with an
additive attention gate (Oktay et al. 2018) on every skip connection.  Module tree, ``state_dict`` keys and
constructor signatures are the reference's; the sub-modules only hold parameters.

Per gate (attention_unet.py:90-96):  ``x * sigmoid(BN(conv1x1_{A->1}(relu(BN(conv1x1(signal)) + BN(conv1x1(x))))))``
with A = C/2.  The two C->A projections run on the tensor-core pointwise GEMM, the A->1 projection and the
row scaling are stream kernels; only the 1-channel BatchNorm + sigmoid of the [N,H,W] logit plane uses torch ops.
"""
from typing import Literal, Sequence

import torch
import torch.nn as nn
import torch.nn.functional as F

from pai_b200 import check, engine, layers as L, lib

from .pix2pix import DecoderBlock, EncoderBlock
from .wrapper import UnetWrapper

_K = dict(kernel_size=4, stride=2, padding=1)


class AttentionUnetGAN(UnetWrapper):
    """Attention U-net (+ PatchGAN for ``loss_type="gan"``), constructor as models/attention_unet.py:28-35."""

    def __init__(
        self,
        in_channels: int = 3,
        out_channels: int = 3,
        channel_mults: Sequence[int] = (1, 2, 4, 8, 8, 8, 8, 8),
        dropout: float = 0.5,
        loss_type: Literal["gan", "ssim", "psnr", "ssim+psnr", "mse"] = "gan",
    ):
        unet = AttentionUnet(in_channels, out_channels, channel_mults=channel_mults, dropout=dropout)
        super().__init__(unet, loss_type=loss_type)
        self.example_input_array = torch.Tensor(2, in_channels, 256, 256)
        self.save_hyperparameters()


class AttentionBlock(nn.Module):
    """``(x [N,h,w,C], signal [N,h,w,Cs]) -> x * attention`` (NHWC bf16)."""

    def __init__(self, input_channels: int, signal_channels: int, attention_channels: int):
        super().__init__()
        self.input_gate = nn.Sequential(
            nn.Conv2d(input_channels, attention_channels, kernel_size=1),
            nn.BatchNorm2d(attention_channels),
        )
        self.signal_gate = nn.Sequential(
            nn.Conv2d(signal_channels, attention_channels, kernel_size=1),
            nn.BatchNorm2d(attention_channels),
        )
        self.attention = nn.Sequential(
            nn.Conv2d(attention_channels, 1, kernel_size=1),
            nn.BatchNorm2d(1),
            nn.Sigmoid(),
        )
        self.relu = nn.ReLU()

    def forward(self, x, signal):
        h_in = L.batchnorm_act(L.conv2d(x, self.input_gate[0], before_train_bn=self.input_gate[1].training), self.input_gate[1], L.ACT_NONE)
        h_sig = L.batchnorm_act(L.conv2d(signal, self.signal_gate[0], before_train_bn=self.signal_gate[1].training), self.signal_gate[1],
                                 L.ACT_NONE)
        h = L.add_act(h_sig, h_in, L.ACT_RELU)
        logit = L.conv_out(h, self.attention[0])                       # fp32 plane [N, h, w]
        bn = self.attention[1]
        if bn.training and bn.num_batches_tracked is not None:
            bn.num_batches_tracked.add_(1)
        z = F.batch_norm(logit.unsqueeze(1), bn.running_mean, bn.running_var, bn.weight, bn.bias,
                         bn.training, bn.momentum, bn.eps)
        att = torch.sigmoid(z).squeeze(1).contiguous()
        return L.scale_rows(x, att)


class AttentionUnet(nn.Module):
    """``[N, in_channels, H, W] -> [N, out_channels, H, W]`` in (-1, 1), 1 to 4 channels each."""

    def __init__(self, in_channels: int = 3, out_channels: int = 3,
                 channel_mults: Sequence[int] = (1, 2, 4, 8, 8, 8, 8, 8), dropout: float = 0.5):
        super().__init__()
        widths = [64 * m for m in channel_mults]
        depth = len(widths)
        down = [nn.Conv2d(in_channels, widths[0], **_K)]
        for lvl in range(1, depth):
            down.append(EncoderBlock(widths[lvl - 1], widths[lvl], norm=lvl != depth - 1))
        self.encoders = nn.ModuleList(down)

        up, gates, cin = [], [], widths[-1]
        widest = max(channel_mults)
        for lvl in range(depth - 2, -1, -1):
            drop = dropout if (channel_mults[lvl] == widest and lvl > depth - 5) else 0
            up.append(DecoderBlock(cin, widths[lvl], dropout=drop))
            gates.append(AttentionBlock(widths[lvl], widths[lvl], widths[lvl] // 2))
            cin = 2 * widths[lvl]
        up.append(nn.ConvTranspose2d(cin, out_channels, **_K))
        self.decoders = nn.ModuleList(up)
        self.attention_blocks = nn.ModuleList(gates)
        self.out = nn.Tanh()

    @staticmethod
    def _encode(block, h):
        if isinstance(block, nn.Conv2d):
            return L.conv4x4s2(h, block)
        seq = block.encode
        raw = L.conv4x4s2(L.activation(h, L.ACT_LEAKY), seq[1])
        return L.batchnorm_act(raw, seq[2], L.ACT_NONE) if isinstance(seq[2], nn.BatchNorm2d) else raw

    @staticmethod
    def _decode(block, h):
        seq = block.decode
        raw = L.convT4x4s2(L.activation(h, L.ACT_RELU), seq[1])
        return L.dropout2d(L.batchnorm_act(raw, seq[2], L.ACT_NONE), seq[3])

    def forward(self, x):
        with lib.on_device(x):
            return self._forward(x)

    def _forward(self, x):
        if engine.check_path_enabled():                # exact fp32 kernels (pai_b200/check.py)
            return check.attention_unet_forward(self, x)
        n, _, hh, ww = x.shape
        depth = len(self.encoders)
        if hh % (1 << depth) or ww % (1 << depth):
            raise RuntimeError(f"pai_b200: input {hh}x{ww} must be divisible by 2^{depth}")
        cin, cout = self.encoders[0].in_channels, self.decoders[-1].out_channels
        L.check_image_channels(cin, cout)
        if cin == 1:
            h = self._encode(self.encoders[0], L.to_plane(x))
        else:
            h = L.conv4x4s2_in_planes(L.to_planes(x, cin), self.encoders[0])
        feats = [h]
        for enc in self.encoders[1:]:
            h = self._encode(enc, h)
            feats.append(h)
        feats.pop()
        last = len(self.decoders) - 1
        for j, dec in enumerate(self.decoders):
            if j != 0:
                s = self.attention_blocks[j - 1](feats.pop(), h)
                h = torch.cat([h, s], dim=-1)
            if j == last:                                                     # bare ConvTranspose2d: no ReLU before it
                if cout == 1:
                    return L.convT4x4s2_out_tanh(h, dec).view(n, 1, hh, ww)
                return L.convT4x4s2_out_planes_tanh(h, dec)
            h = self._decode(dec, h)
