"""ORACLE (test infrastructure): dtype-agnostic functional restatement of the Residual, Attention and Trans U-Nets of
the reference (models/res_unet.py, attention_unet.py, trans_unet.py), read from a ``state_dict`` with the wrapper's
``unet.`` prefix -- in the style of ``bf16_sites.fwd`` for the Pix2Pix U-Net.  Any number of image channels.

Evaluated in fp32 it reproduces the reference's golden vectors (tests/golden/variants_ref.npz); evaluated in fp64 it is
the exact answer the fp32 check path (pai_b200/check.py) is held to.  BatchNorm running statistics and
``num_batches_tracked`` of ``sd`` move in place in training mode, as in the reference.  No dropout (the cases use 0).
"""
import math

import torch
import torch.nn.functional as F

BN_EPS, BN_MOMENTUM, LN_EPS = 1e-5, 0.1, 1e-5


def _relu(h):
    """Every ReLU of the three families (a module-level hook, so a test can pin the branch taken at a kink)."""
    return F.relu(h)


def _leaky(h):
    """Every LeakyReLU(0.2) (the Attention U-Net's encoders)."""
    return F.leaky_relu(h, 0.2)


def _has(sd, key):
    return key in sd


def _conv(sd, p, h, stride=1, pad=None, groups=1):
    w = sd[p + ".weight"]
    return F.conv2d(h, w, sd.get(p + ".bias"), stride, w.shape[2] // 2 if pad is None else pad, 1, groups)


def _bn(sd, p, h, training):
    out = F.batch_norm(h, sd[p + ".running_mean"], sd[p + ".running_var"], sd[p + ".weight"], sd[p + ".bias"], training,
                       BN_MOMENTUM, BN_EPS)
    if training:
        sd[p + ".num_batches_tracked"] += 1
    return out


def _cbr(sd, pc, pb, h, training, relu=True, **kw):
    h = _bn(sd, pb, _conv(sd, pc, h, **kw), training)
    return _relu(h) if relu else h


# ------------------------------------------------------------------------------------------ Residual U-Net
def _res_block(sd, p, h, training, res_type):
    b, s = p + ".conv_block", p + ".conv_skip"
    skip = _has(sd, s + ".0.running_mean") or _has(sd, s + ".0.weight")
    if res_type == "v2":
        y = _conv(sd, b + ".2", _relu(_bn(sd, b + ".0", h, training)))
        y = _conv(sd, b + ".5", _relu(_bn(sd, b + ".3", y, training)))
        return y + (_conv(sd, s + ".2", _relu(_bn(sd, s + ".0", h, training))) if skip else h)
    sk = _cbr(sd, s + ".0", s + ".1", h, training, relu=False) if skip else h
    if res_type == "18":
        y = _cbr(sd, b + ".0", b + ".1", h, training)
        return _relu(_cbr(sd, b + ".3", b + ".4", y, training, relu=False) + sk)
    if res_type == "50":
        y = _cbr(sd, b + ".3", b + ".4", _cbr(sd, b + ".0", b + ".1", h, training), training)
        return _relu(_cbr(sd, b + ".6", b + ".7", y, training, relu=False) + sk)
    if res_type == "next":
        y = _cbr(sd, b + ".0", b + ".1", h, training)
        w3 = sd[b + ".3.weight"]
        y = _cbr(sd, b + ".3", b + ".4", y, training, groups=y.shape[1] // w3.shape[1])
        return _cbr(sd, b + ".6", b + ".7", y, training) + sk
    raise ValueError(res_type)


def res_unet(sd, x, training, res_type):
    n_enc = len({k.split(".")[2] for k in sd if k.startswith("unet.encoders.")})
    n_dec = len({k.split(".")[2] for k in sd if k.startswith("unet.decoders.")})
    h = _conv(sd, "unet.in_conv", x)
    skips = []
    for i in range(n_enc):
        h = F.max_pool2d(_res_block(sd, f"unet.encoders.{i}.encode.0", h, training, res_type), 2)
        skips.append(h)
    skips.pop()
    for j in range(n_dec):
        if j:
            h = torch.cat([h, skips.pop()], 1)
        h = F.interpolate(_res_block(sd, f"unet.decoders.{j}.decode.0", h, training, res_type), scale_factor=2,
                          mode="nearest")
    return torch.tanh(_conv(sd, "unet.out.0", h))


# ------------------------------------------------------------------------------------------ Attention U-Net
def _gate(sd, p, x, signal, training):
    a = _cbr(sd, p + ".input_gate.0", p + ".input_gate.1", x, training, relu=False)
    s = _cbr(sd, p + ".signal_gate.0", p + ".signal_gate.1", signal, training, relu=False)
    att = torch.sigmoid(_cbr(sd, p + ".attention.0", p + ".attention.1", _relu(s + a), training, relu=False))
    return x * att


def attention_unet(sd, x, training):
    n_enc = len({k.split(".")[2] for k in sd if k.startswith("unet.encoders.")})
    h = F.conv2d(x, sd["unet.encoders.0.weight"], sd["unet.encoders.0.bias"], 2, 1)
    feats = [h]
    for i in range(1, n_enc):
        p = f"unet.encoders.{i}.encode"
        h = F.conv2d(_leaky(h), sd[p + ".1.weight"], sd[p + ".1.bias"], 2, 1)
        if _has(sd, p + ".2.weight"):
            h = _bn(sd, p + ".2", h, training)
        feats.append(h)
    feats.pop()
    for j in range(n_enc):
        if j:
            h = torch.cat([h, _gate(sd, f"unet.attention_blocks.{j - 1}", feats.pop(), h, training)], 1)
        if j < n_enc - 1:
            p = f"unet.decoders.{j}.decode"
            h = _bn(sd, p + ".2", F.conv_transpose2d(_relu(h), sd[p + ".1.weight"], sd[p + ".1.bias"], 2, 1), training)
        else:
            h = F.conv_transpose2d(h, sd[f"unet.decoders.{j}.weight"], sd[f"unet.decoders.{j}.bias"], 2, 1)
    return torch.tanh(h)


# ------------------------------------------------------------------------------------------ Trans U-Net
def _mha(sd, p, t, s, b, heads):
    """nn.MultiheadAttention of the reference (no batch_first): ``t [s*b, E]`` rows ordered (sequence, batch)."""
    e = t.shape[1]
    hd = e // heads
    qkv = F.linear(t, sd[p + ".in_proj_weight"], sd[p + ".in_proj_bias"])
    q, k, v = (u.reshape(s, b, heads, hd).permute(1, 2, 0, 3) for u in qkv.split(e, dim=1))     # [b, heads, s, hd]
    probs = torch.softmax(q @ k.transpose(-1, -2) / math.sqrt(hd), dim=-1)
    out = (probs @ v).permute(2, 0, 1, 3).reshape(s * b, e)
    return F.linear(out, sd[p + ".out_proj.weight"], sd[p + ".out_proj.bias"])


def _ln(sd, p, t):
    return F.layer_norm(t, (t.shape[-1],), sd[p + ".weight"], sd[p + ".bias"], LN_EPS)


def vit(sd, x, heads=8):
    p = "unet.vit_bottleneck"
    n, c, hh, ww = x.shape
    pos = sd[p + ".pos_embedding"]
    tokens, d = pos.shape[1], pos.shape[2]
    ps = math.isqrt(d // c)
    gh, gw = hh // ps, ww // ps
    t = x.reshape(n, c, gh, ps, gw, ps).permute(0, 2, 4, 3, 5, 1).reshape(n * tokens, d)
    t = _ln(sd, p + ".to_patch_embedding.1", t)
    t = F.linear(t, sd[p + ".to_patch_embedding.2.weight"], sd[p + ".to_patch_embedding.2.bias"])
    t = _ln(sd, p + ".to_patch_embedding.3", t)
    t = (t.reshape(n, tokens, d) + pos).reshape(n * tokens, d)
    n_layers = len({k.split(".")[4] for k in sd if k.startswith(p + ".transformer.layers.")})
    for i in range(n_layers):
        q = f"{p}.transformer.layers.{i}"
        t = _ln(sd, q + ".norm1", t + _mha(sd, q + ".self_attn", t, n, tokens, heads))
        f = F.linear(F.gelu(F.linear(t, sd[q + ".linear1.weight"], sd[q + ".linear1.bias"])), sd[q + ".linear2.weight"],
                     sd[q + ".linear2.bias"])
        t = _ln(sd, q + ".norm2", t + f)
    return t.reshape(n, gh, gw, ps, ps, c).permute(0, 5, 1, 3, 2, 4).reshape(n, c, hh, ww)


def trans_unet(sd, x, training, heads=8):
    n_enc = len({k.split(".")[2] for k in sd if k.startswith("unet.encoders.")})
    n_dec = len({k.split(".")[2] for k in sd if k.startswith("unet.decoders.")})
    h = _conv(sd, "unet.in_conv", x)
    skips = []
    for i in range(n_enc):
        p = f"unet.encoders.{i}"
        y = _cbr(sd, p + ".decode.0", p + ".decode.1", h, training)
        y = _cbr(sd, p + ".decode.3", p + ".decode.4", y, training, stride=2)
        y = _cbr(sd, p + ".decode.6", p + ".decode.7", y, training, relu=False)
        h = _relu(y + _cbr(sd, p + ".skip.0", p + ".skip.1", h, training, relu=False, stride=2, pad=0))
        skips.append(h)
    skips.pop()
    h = vit(sd, h, heads)
    for j in range(n_dec):
        if j:
            h = torch.cat([h, skips.pop()], 1)
        p = f"unet.decoders.{j}.decode"
        h = _cbr(sd, p + ".3", p + ".4", _cbr(sd, p + ".0", p + ".1", h, training), training)
        h = F.interpolate(h, scale_factor=2, mode="nearest")
    return torch.tanh(_conv(sd, "unet.out.0", h))


def forward(sd, x, training, family, res_type="18"):
    """``family``: "res" (with ``res_type`` "18" / "50" / "v2" / "next"), "attention" or "trans"."""
    x = x.to(sd["unet.out.0.weight" if "unet.out.0.weight" in sd else "unet.encoders.0.weight"].dtype)
    if family == "res":
        return res_unet(sd, x, training, res_type)
    if family == "attention":
        return attention_unet(sd, x, training)
    if family == "trans":
        return trans_unet(sd, x, training)
    raise ValueError(family)
