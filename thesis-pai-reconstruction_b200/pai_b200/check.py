"""fp32 check-path forwards of the Residual, Attention and Trans U-Nets (models/res_unet.py, attention_unet.py,
trans_unet.py), taken by their ``_forward`` inside ``engine.check_path()``.

Each forward walks the drop-in's module tree in fp32 NCHW (the reference's own layout) and runs every arithmetic layer
on the exact kernels of csrc/check_f32.cu through the autograd nodes of ``engine`` (``_CheckConv2d``, ``_CheckBN``,
``_CheckAct``, ``_CheckMaxPool2``, ``_CheckUpsample2``, ``_CheckLayerNorm``, ``_CheckLinear``, ``_CheckAttention``), so
``loss.backward()`` on a graph built inside the context gives check-path gradients of every parameter.  Torch only moves
data (``cat``, ``view``, ``permute``, ``reshape``: the skip concatenations and the ViT's two ``Rearrange``s) and adds or
multiplies two fp32 tensors (a residual sum before its activation kernel, the positional embedding, the attention gate
``x * a``).  BatchNorm running statistics and ``num_batches_tracked`` move as in the reference.  Training with Dropout2d
or ViT dropout is refused: the check path is deterministic."""
from __future__ import annotations

import torch
import torch.nn as nn

from . import engine, layers as L
from .ops import ACT_GELU, ACT_LEAKY, ACT_NONE, ACT_RELU, ACT_SIGMOID, ACT_TANH

_NO_DROPOUT = "pai_b200: the fp32 check path has no {} (it is a deterministic forward check)"


def _conv(x, mod):
    """``nn.Conv2d`` or ``nn.ConvTranspose2d`` (square kernel, stride and padding; no output padding)."""
    transposed = isinstance(mod, nn.ConvTranspose2d)
    if (mod.kernel_size[0] != mod.kernel_size[1] or mod.stride[0] != mod.stride[1] or mod.padding[0] != mod.padding[1]
            or mod.dilation != (1, 1) or (transposed and mod.output_padding != (0, 0))):
        raise RuntimeError(f"pai_b200 check path: unexpected convolution {mod}")
    return engine._CheckConv2d.apply(x, mod.weight, mod.bias, mod.stride[0], mod.padding[0], mod.groups, transposed)


def _bn(x, mod: nn.BatchNorm2d):
    return engine._CheckBN.apply(x, mod.weight, mod.bias, mod, mod.training)


def _act(x, act):
    return engine._CheckAct.apply(x, act)


def _cba(x, conv, bn, act):
    """Conv2d -> BatchNorm2d (-> activation)."""
    h = _bn(_conv(x, conv), bn)
    return h if act == ACT_NONE else _act(h, act)


def _images(x, cin, cout):
    L.check_image_channels(cin, cout)
    return L.to_planes(x, cin)


def _check_divisible(x, depth):
    hh, ww = x.shape[2], x.shape[3]
    if hh % (1 << depth) or ww % (1 << depth):
        raise RuntimeError(f"pai_b200: input {hh}x{ww} must be divisible by 2^{depth}")


def _refuse_dropout2d(mod):
    if isinstance(mod, nn.Dropout2d) and mod.training and mod.p > 0:
        raise RuntimeError(_NO_DROPOUT.format("Dropout2d"))


# ------------------------------------------------------------------------------------------ Residual U-Net
def _res_block(blk, x):
    """The four residual blocks of models/res_unet.py ("18", "50", "v2", "next")."""
    b, kind = blk.conv_block, type(blk).__name__
    identity = isinstance(blk.conv_skip, nn.Identity)
    if kind == "ResidualBlockV2":              # pre-activation: bn-relu-conv twice, raw sum
        h = _conv(_act(_bn(x, b[0]), ACT_RELU), b[2])
        h = _conv(_act(_bn(h, b[3]), ACT_RELU), b[5])
        s = x if identity else _conv(_act(_bn(x, blk.conv_skip[0]), ACT_RELU), blk.conv_skip[2])
        return h + s
    s = x if identity else _cba(x, blk.conv_skip[0], blk.conv_skip[1], ACT_NONE)
    if kind == "ResidualBlock18":
        h = _cba(x, b[0], b[1], ACT_RELU)
        return _act(_cba(h, b[3], b[4], ACT_NONE) + s, ACT_RELU)
    if kind == "ResidualBlock50":
        h = _cba(_cba(x, b[0], b[1], ACT_RELU), b[3], b[4], ACT_RELU)
        return _act(_cba(h, b[6], b[7], ACT_NONE) + s, ACT_RELU)
    if kind == "ResidualBlockNeXt":            # 1x1 -> grouped 3x3 -> 1x1, each BN + ReLU; raw sum
        h = _cba(_cba(x, b[0], b[1], ACT_RELU), b[3], b[4], ACT_RELU)
        return _cba(h, b[6], b[7], ACT_RELU) + s
    raise RuntimeError(f"pai_b200 check path: unknown residual block {kind}")


def res_unet_forward(unet, x: torch.Tensor) -> torch.Tensor:
    """``ResUnet.forward``: in_conv -> [block -> MaxPool2d(2)] x depth -> [cat skip -> block -> Upsample] -> conv + Tanh."""
    _check_divisible(x, len(unet.encoders))
    h = _conv(_images(x, unet.in_conv.in_channels, unet.out[0].out_channels), unet.in_conv)
    for dec in unet.decoders:
        _refuse_dropout2d(dec.decode[1])
    skips = []
    for enc in unet.encoders:
        h = engine._CheckMaxPool2.apply(_res_block(enc.encode[0], h))
        skips.append(h)
    skips.pop()
    for j, dec in enumerate(unet.decoders):
        if j != 0:
            h = torch.cat([h, skips.pop()], dim=1)
        h = engine._CheckUpsample2.apply(_res_block(dec.decode[0], h))
    return _act(_conv(h, unet.out[0]), ACT_TANH)


# ------------------------------------------------------------------------------------------ Attention U-Net
def _attention_gate(gate, x, signal):
    """``x * sigmoid(BN(conv1x1(relu(BN(conv1x1(signal)) + BN(conv1x1(x))))))`` (one gate value per pixel)."""
    h = _cba(signal, gate.signal_gate[0], gate.signal_gate[1], ACT_NONE) + _cba(x, gate.input_gate[0], gate.input_gate[1],
                                                                               ACT_NONE)
    a = _cba(_act(h, ACT_RELU), gate.attention[0], gate.attention[1], ACT_SIGMOID)
    return x * a


def attention_unet_forward(unet, x: torch.Tensor) -> torch.Tensor:
    """``AttentionUnet.forward``: the Pix2Pix encoder / decoder (4x4 stride-2 convolutions) with a gate on every skip."""
    _check_divisible(x, len(unet.encoders))
    last = unet.decoders[-1]
    v = _images(x, unet.encoders[0].in_channels, last.out_channels)
    for dec in list(unet.decoders)[:-1]:
        _refuse_dropout2d(dec.decode[3])
    h = _conv(v, unet.encoders[0])
    feats = [h]
    for enc in list(unet.encoders)[1:]:
        seq = enc.encode
        h = _conv(_act(h, ACT_LEAKY), seq[1])
        if isinstance(seq[2], nn.BatchNorm2d):
            h = _bn(h, seq[2])
        feats.append(h)
    feats.pop()
    for j, dec in enumerate(list(unet.decoders)[:-1]):
        if j != 0:
            h = torch.cat([h, _attention_gate(unet.attention_blocks[j - 1], feats.pop(), h)], dim=1)
        seq = dec.decode
        h = _bn(_conv(_act(h, ACT_RELU), seq[1]), seq[2])
    h = torch.cat([h, _attention_gate(unet.attention_blocks[-1], feats.pop(), h)], dim=1)
    # the last decoder is a bare ConvTranspose2d: no ReLU in front of it
    return _act(_conv(h, last), ACT_TANH)


# ------------------------------------------------------------------------------------------ Trans U-Net
def _layernorm(t, mod: nn.LayerNorm):
    return engine._CheckLayerNorm.apply(t, mod.weight, mod.bias, mod.eps)


def _linear(t, weight, bias):
    return engine._CheckLinear.apply(t, weight, bias)


def vit_forward(vit, x: torch.Tensor) -> torch.Tensor:
    """``VisionTransformer.forward`` on NCHW ``[n, c, s, s]``: patches -> LayerNorm -> Linear -> LayerNorm -> + positional
    embedding -> post-norm encoder layers (attention over the batch axis, SURVEY Q4) -> image."""
    if vit.training and vit.dropout > 0:
        raise RuntimeError(_NO_DROPOUT.format("ViT dropout"))
    n, c, hh, ww = x.shape
    p = vit.patch_size
    gh, gw = hh // p, ww // p
    tokens, d = gh * gw, p * p * c
    if tokens != vit.pos_embedding.shape[1] or d != vit.pos_embedding.shape[2]:
        raise RuntimeError(f"pai_b200: bottleneck {hh}x{ww}x{c} does not match the {tuple(vit.pos_embedding.shape)} "
                           "positional embedding (TransUnetGAN assumes 256x256 inputs)")
    # "n c (h p1) (w p2) -> n (h w) (p1 p2 c)"
    t = x.view(n, c, gh, p, gw, p).permute(0, 2, 4, 3, 5, 1).reshape(n * tokens, d)
    emb = vit.to_patch_embedding
    t = _layernorm(_linear(_layernorm(t, emb[1]), emb[2].weight, emb[2].bias), emb[3])
    t = (t.view(n, tokens, d) + vit.pos_embedding).reshape(n * tokens, d)
    for lyr in vit.transformer.layers:
        att = lyr.self_attn
        a = engine._CheckAttention.apply(_linear(t, att.in_proj_weight, att.in_proj_bias), n, tokens, vit.num_heads)
        t = _layernorm(t + _linear(a, att.out_proj.weight, att.out_proj.bias), lyr.norm1)
        f = _linear(_act(_linear(t, lyr.linear1.weight, lyr.linear1.bias), ACT_GELU), lyr.linear2.weight, lyr.linear2.bias)
        t = _layernorm(t + f, lyr.norm2)
    # "n (h w) (p1 p2 c) -> n c (h p1) (w p2)"
    return t.view(n, gh, gw, p, p, c).permute(0, 5, 1, 3, 2, 4).reshape(n, c, hh, ww)


def trans_unet_forward(unet, x: torch.Tensor) -> torch.Tensor:
    """``TransUnet.forward``: in_conv -> bias-free bottleneck encoders (stride 2) -> ViT -> [cat skip -> 2 x (conv3x3 + BN
    + ReLU) -> Upsample] -> conv + Tanh."""
    h = _conv(_images(x, unet.in_conv.in_channels, unet.out[0].out_channels), unet.in_conv)
    skips = []
    for enc in unet.encoders:
        d = enc.decode
        m = _cba(_cba(h, d[0], d[1], ACT_RELU), d[3], d[4], ACT_RELU)
        h = _act(_cba(m, d[6], d[7], ACT_NONE) + _cba(h, enc.skip[0], enc.skip[1], ACT_NONE), ACT_RELU)
        skips.append(h)
    skips.pop()
    h = vit_forward(unet.vit_bottleneck, h)
    for j, dec in enumerate(unet.decoders):
        if j != 0:
            h = torch.cat([h, skips.pop()], dim=1)
        d = dec.decode
        h = engine._CheckUpsample2.apply(_cba(_cba(h, d[0], d[1], ACT_RELU), d[3], d[4], ACT_RELU))
    return _act(_conv(h, unet.out[0]), ACT_TANH)
