"""Mirror of /root/reference/models/trans_unet.py (``TransUnetGAN``, ``TransUnet``, ``VisionTransformer``,
``EncoderBlock``, ``DecoderBlock``) on the B200 kernels.  Module tree, ``state_dict`` keys, constructor signatures
and initial weights are the reference's (the torch modules only hold parameters).

* encoders: ResNet-50 style bottleneck with a stride-2 3x3 and a stride-2 1x1 projection, bias-free
  (trans_unet.py:178-222).  The 16 / 32-channel bottlenecks travel in zero-padded 64-channel tensors so every
  convolution is a tensor-core GEMM; the 3x3 stride-2 runs on the 4x4 stride-2 implicit GEMM with a zero 4th
  kernel row / column; the 1x1 stride-2 is a subsampling stream + pointwise GEMM.
* ViT bottleneck (:120-175): patches -> LayerNorm -> Linear -> LayerNorm -> + positional embedding -> 12 post-norm
  ``nn.TransformerEncoderLayer``s.  The reference builds them without ``batch_first`` and feeds [n, patches, d], so
  attention runs over the BATCH axis (SURVEY.md Q4) -- reproduced exactly: sequence = images of this GPU's batch.
  Linear layers run on the pointwise GEMM; LayerNorm, GELU and the attention core are kernels of csrc/transformer.cu.
  Train-mode dropout (the layer's four sites) is fused into those kernels: each forward draws one int64 key from
  torch's CUDA generator and the kernels regenerate their Philox masks from it (csrc/pai_dropout.cuh).
* decoders: 2 x (3x3 conv + BN + ReLU) + nearest upsample on the 9-tap implicit GEMM.
"""
import math
from typing import Literal, Sequence

import torch
import torch.nn as nn
from einops.layers.torch import Rearrange

from pai_b200 import layers as L, lib

from .wrapper import UnetWrapper


class TransUnetGAN(UnetWrapper):
    """Constructor as models/trans_unet.py:27-35 (``image_size`` is fixed to 256 there)."""

    def __init__(
        self,
        in_channels: int = 3,
        out_channels: int = 3,
        channel_mults: Sequence[int] = (1, 2, 2, 4, 4),
        patch_size: int = 2,
        dropout: float = 0.5,
        loss_type: Literal["gan", "ssim", "psnr", "ssim+psnr", "mse"] = "gan",
    ):
        unet = TransUnet(in_channels, out_channels, image_size=256, channel_mults=channel_mults,
                         patch_size=patch_size, num_heads=8, dropout=dropout)
        super().__init__(unet, loss_type=loss_type)
        self.example_input_array = torch.Tensor(2, in_channels, 256, 256)
        self.save_hyperparameters()


class EncoderBlock(nn.Module):
    """relu(bottleneck(x) + projection(x)), both stride 2.  (The reference names the main path ``decode``.)"""

    def __init__(self, in_channels: int, out_channels: int):
        super().__init__()
        mid = in_channels // 4
        self.decode = nn.Sequential(
            nn.Conv2d(in_channels, mid, kernel_size=1, bias=False),
            nn.BatchNorm2d(mid),
            nn.ReLU(),
            nn.Conv2d(mid, mid, kernel_size=3, stride=2, padding=1, bias=False),
            nn.BatchNorm2d(mid),
            nn.ReLU(),
            nn.Conv2d(mid, out_channels, kernel_size=1, bias=False),
            nn.BatchNorm2d(out_channels),
        )
        self.skip = nn.Sequential(
            nn.Conv2d(in_channels, out_channels, kernel_size=1, stride=2, bias=False),
            nn.BatchNorm2d(out_channels),
        )
        self.out = nn.ReLU()

    def forward(self, x):
        d = self.decode
        h = L.batchnorm_act(L.conv1x1_padded(x, d[0]), d[1], L.ACT_RELU)
        h = L.batchnorm_act(L.conv3x3s2_padded(h, d[3]), d[4], L.ACT_RELU)
        h = L.batchnorm_act(L.conv1x1_padded(h, d[6]), d[7], L.ACT_NONE)
        s = L.batchnorm_act(L.conv1x1_padded(L.subsample2(x), self.skip[0]), self.skip[1], L.ACT_NONE)
        return L.add_act(h, s, L.ACT_RELU)


class DecoderBlock(nn.Module):
    """conv3x3-bn-relu, conv3x3-bn-relu, nearest upsample x2 (trans_unet.py:225-255)."""

    def __init__(self, in_channels: int, out_channels: int):
        super().__init__()
        self.decode = nn.Sequential(
            nn.Conv2d(in_channels, out_channels, kernel_size=3, padding=1),
            nn.BatchNorm2d(out_channels),
            nn.ReLU(),
            nn.Conv2d(out_channels, out_channels, kernel_size=3, padding=1),
            nn.BatchNorm2d(out_channels),
            nn.ReLU(),
            nn.Upsample(scale_factor=2),
        )

    def forward(self, x):
        d = self.decode
        h = L.batchnorm_act(L.conv2d(x, d[0], before_train_bn=d[1].training), d[1], L.ACT_RELU)
        h = L.batchnorm_act(L.conv2d(h, d[3], before_train_bn=d[4].training), d[4], L.ACT_RELU)
        return L.upsample2(h)


class VisionTransformer(nn.Module):
    """NHWC bf16 ``[n, s, s, c]`` -> same shape through the patch transformer."""

    def __init__(self, channels: int, input_size: int, patch_size: int = 16, num_heads: int = 8,
                 dropout: float = 0.5, transformer_layers: int = 12):
        super().__init__()
        patch_dim = channels * patch_size * patch_size
        num_patches = (input_size ** 2) // (patch_size ** 2)
        self.to_patch_embedding = nn.Sequential(
            Rearrange("n c (h p1) (w p2) -> n (h w) (p1 p2 c)", p1=patch_size, p2=patch_size),
            nn.LayerNorm(patch_dim),
            nn.Linear(patch_dim, patch_dim),
            nn.LayerNorm(patch_dim),
        )
        self.pos_embedding = nn.Parameter(torch.randn(1, num_patches, patch_dim))
        layer = nn.TransformerEncoderLayer(patch_dim, num_heads, dropout=dropout, activation="gelu")
        self.transformer = nn.TransformerEncoder(layer, transformer_layers)
        side = int(math.sqrt(num_patches))
        self.to_image = Rearrange("n (h w) (p1 p2 c) -> n c (h p1) (w p2)", h=side, w=side, p1=patch_size, p2=patch_size)
        self.patch_size, self.num_heads, self.dropout = patch_size, num_heads, dropout
        self._dropout_key = None     # int64 [1] device tensor: the key of the last train-mode forward with dropout

    def _layer(self, x, lyr, s, b):
        att = lyr.self_attn
        qkv = L.linear(x, att.in_proj_weight, att.in_proj_bias)
        a = L.attention(qkv, s, b, self.num_heads)
        x = L.layernorm(L.add_act(x, L.linear(a, att.out_proj.weight, att.out_proj.bias)), lyr.norm1)
        f = L.linear(L.gelu(L.linear(x, lyr.linear1.weight, lyr.linear1.bias)), lyr.linear2.weight, lyr.linear2.bias)
        return L.layernorm(L.add_act(x, f), lyr.norm2)

    def _layer_dropout(self, x, lyr, s, b, key, site):
        """``_layer`` with the train-mode dropout of nn.TransformerEncoderLayer at sites ``site + 0..3``: attention
        probabilities, attention output (dropout1), after the GELU (dropout), feed-forward output (dropout2)."""
        att, p = lyr.self_attn, self.dropout
        qkv = L.linear(x, att.in_proj_weight, att.in_proj_bias)
        a = L.attention_dropout(qkv, s, b, self.num_heads, key, site, p)
        x = L.add_dropout_layernorm(x, L.linear(a, att.out_proj.weight, att.out_proj.bias), lyr.norm1, key, site + 1, p)
        h = L.gelu_dropout(L.linear(x, lyr.linear1.weight, lyr.linear1.bias), key, site + 2, p)
        f = L.linear(h, lyr.linear2.weight, lyr.linear2.bias)
        return L.add_dropout_layernorm(x, f, lyr.norm2, key, site + 3, p)

    def forward(self, x):
        key = None
        if self.training and self.dropout > 0:
            if self.dropout >= 1:
                raise RuntimeError(f"pai_b200: ViT dropout must be < 1 in training mode, got {self.dropout}")
            # one draw from torch's CUDA generator per forward: seeded by torch.manual_seed, and a new key at every
            # replay of a captured step graph
            key = torch.randint(-2 ** 63, 2 ** 63 - 1, (1,), dtype=torch.int64, device=x.device)
            self._dropout_key = key
        n, hh, ww, c = x.shape
        p = self.patch_size
        gh, gw = hh // p, ww // p
        tokens = gh * gw
        d = p * p * c
        if tokens != self.pos_embedding.shape[1] or d != self.pos_embedding.shape[2]:
            raise RuntimeError(f"pai_b200: bottleneck {hh}x{ww}x{c} does not match the {tuple(self.pos_embedding.shape)} "
                               "positional embedding (TransUnetGAN assumes 256x256 inputs)")
        # "n c (h p1) (w p2) -> n (h w) (p1 p2 c)" on the NHWC tensor
        t = x.view(n, gh, p, gw, p, c).permute(0, 1, 3, 2, 4, 5).reshape(n * tokens, d)
        emb = self.to_patch_embedding
        t = L.layernorm(t, emb[1])
        t = L.linear(t, emb[2].weight, emb[2].bias)
        t = L.layernorm(t, emb[3])
        t = (t.view(n, tokens, d) + self.pos_embedding.to(t.dtype)).reshape(n * tokens, d)
        # no batch_first in the reference: sequence axis = n (batch), "batch" axis = tokens
        for i, lyr in enumerate(self.transformer.layers):
            t = self._layer(t, lyr, n, tokens) if key is None else self._layer_dropout(t, lyr, n, tokens, key, 4 * i)
        return t.view(n, gh, gw, p, p, c).permute(0, 1, 3, 2, 4, 5).reshape(n, hh, ww, c)


class TransUnet(nn.Module):
    """``[N, 1, 256, 256] -> [N, 1, 256, 256]`` in (-1, 1)."""

    def __init__(self, in_channels: int = 3, out_channels: int = 3, image_size: int = 256,
                 channel_mults: Sequence[int] = (1, 2, 4, 8), patch_size: int = 16, num_heads: int = 8,
                 dropout: float = 0.5):
        super().__init__()
        self.in_conv = nn.Conv2d(in_channels, 64, kernel_size=3, padding=1)
        down, cin = [], 64
        for mult in channel_mults:
            down.append(EncoderBlock(cin, mult * 64))
            cin = mult * 64
        self.encoders = nn.ModuleList(down)
        self.vit_bottleneck = VisionTransformer(
            channels=channel_mults[-1] * 64, input_size=image_size // (2 ** len(channel_mults)),
            patch_size=patch_size, num_heads=num_heads, dropout=dropout, transformer_layers=12)
        up = []
        for mult in reversed(list(channel_mults[:-1])):
            up.append(DecoderBlock(cin, mult * 64))
            cin = mult * 64 * 2
        up.append(DecoderBlock(cin, 64))
        self.decoders = nn.ModuleList(up)
        self.out = nn.Sequential(nn.Conv2d(64, out_channels, kernel_size=3, padding=1), nn.Tanh())

    def forward(self, x):
        with lib.on_device(x):
            return self._forward(x)

    def _forward(self, x):
        n, _, hh, ww = x.shape
        h = L.conv_in(L.to_plane(x), self.in_conv)
        skips = []
        for enc in self.encoders:
            h = enc(h)
            skips.append(h)
        skips.pop()
        h = self.vit_bottleneck(h)
        for j, dec in enumerate(self.decoders):
            if j != 0:
                h = torch.cat([h, skips.pop()], dim=-1)
            h = dec(h)
        return L.conv_out(h, self.out[0], L.ACT_TANH).view(n, 1, hh, ww)
