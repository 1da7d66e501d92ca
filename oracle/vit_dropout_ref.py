"""Test-only restatement of the Trans U-Net's train-mode ViT dropout (csrc/pai_dropout.cuh, csrc/transformer.cu).

* ``philox4x32_10`` / ``dropout_keep``: numpy Philox4x32-10 (Salmon et al., SC'11; Random123) and the mask rule the
  kernels use -- element ``idx`` of site ``site`` under the 64-bit ``key`` takes word ``idx & 3`` of
  ``philox(counter=(lo32(idx>>2), hi32(idx>>2), site, 0), key=(lo32(key), hi32(key)))`` and is dropped iff that word is
  below ``min(2^32-1, llround(p * 2^32))`` (p as the fp32 the C-ABI receives).
* ``encoder_layer``: fp32 torch restatement of one post-norm ``nn.TransformerEncoderLayer(d, heads, activation="gelu")``
  forward with explicit masks at its four dropout sites, in the batch-axis layout of the B200 path: tokens are rows
  ``s * B + b`` of a ``[S*B, d]`` matrix and attention runs over the S axis (no ``batch_first`` in the reference).
  Autograd on it gives the backward.
"""
import math

import numpy as np
import torch
import torch.nn.functional as F

_M0, _M1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
_W0, _W1 = np.uint64(0x9E3779B9), np.uint64(0xBB67AE85)
_LO = np.uint64(0xFFFFFFFF)
_32 = np.uint64(32)


def philox4x32_10(c0, c1, c2, c3, k0, k1):
    """Vectorised Philox4x32-10: counters and keys are arrays (or scalars) of 32-bit values -> 4 uint32 arrays."""
    c = [np.asarray(v, dtype=np.uint64) & _LO for v in (c0, c1, c2, c3)]
    k0, k1 = np.uint64(k0) & _LO, np.uint64(k1) & _LO
    for _ in range(10):
        p0, p1 = _M0 * c[0], _M1 * c[2]
        c = [((p1 >> _32) ^ c[1] ^ k0) & _LO, p1 & _LO, ((p0 >> _32) ^ c[3] ^ k1) & _LO, p0 & _LO]
        k0, k1 = (k0 + _W0) & _LO, (k1 + _W1) & _LO
    return [v.astype(np.uint32) for v in c]


def dropout_threshold(p: float) -> int:
    t = math.floor(float(np.float32(p)) * 2.0 ** 32 + 0.5)      # llround of a positive double
    return min(2 ** 32 - 1, t)


def dropout_scale(p: float) -> float:
    return float(np.float32(1.0) / (np.float32(1.0) - np.float32(p)))


def dropout_keep(key: int, site: int, n: int, p: float) -> np.ndarray:
    """bool ``[n]``: True where element ``i`` of ``site`` is kept."""
    key &= 2 ** 64 - 1
    groups = np.arange((n + 3) // 4, dtype=np.uint64)
    words = philox4x32_10(groups & _LO, groups >> _32, np.uint64(site), np.uint64(0), key & 0xFFFFFFFF, key >> 32)
    r = np.stack(words, axis=1).reshape(-1)[:n]
    return r >= np.uint32(dropout_threshold(p))


def layer_masks(key: int, layer: int, s: int, b: int, d: int, heads: int, d_ff: int, p: float):
    """fp32 multipliers (0 or 1/(1-p)) of the four sites of encoder layer ``layer``, shaped as ``encoder_layer`` uses them."""
    scale = dropout_scale(p)
    shapes = [(b * heads, s, s), (s * b, d), (s * b, d_ff), (s * b, d)]
    return [torch.from_numpy(dropout_keep(key, 4 * layer + k, int(np.prod(shp)), p).reshape(shp).astype(np.float32) * scale)
            for k, shp in enumerate(shapes)]


def layer_params(lyr):
    """The tensors ``encoder_layer`` needs, from an ``nn.TransformerEncoderLayer``."""
    att = lyr.self_attn
    return dict(w_in=att.in_proj_weight, b_in=att.in_proj_bias, w_out=att.out_proj.weight, b_out=att.out_proj.bias,
                w1=lyr.linear1.weight, b1=lyr.linear1.bias, w2=lyr.linear2.weight, b2=lyr.linear2.bias,
                g1=lyr.norm1.weight, be1=lyr.norm1.bias, eps1=lyr.norm1.eps,
                g2=lyr.norm2.weight, be2=lyr.norm2.bias, eps2=lyr.norm2.eps)


def encoder_layer(x, prm, s: int, b: int, heads: int, masks=None):
    """One post-norm encoder layer on ``x [s*b, d]``; ``masks`` = four multiplier tensors (``layer_masks``) or None."""
    d = x.shape[1]
    hd = d // heads
    m0, m1, m2, m3 = masks if masks is not None else (1.0, 1.0, 1.0, 1.0)
    qkv = x @ prm["w_in"].t() + prm["b_in"]

    def heads_first(t):       # [s*b, d] -> [b*heads, s, hd]
        return t.reshape(s, b, heads, hd).permute(1, 2, 0, 3).reshape(b * heads, s, hd)

    q, k, v = (heads_first(t) for t in qkv.split(d, dim=1))
    att = torch.softmax(q @ k.transpose(1, 2) / math.sqrt(hd), dim=-1) * m0
    o = (att @ v).reshape(b, heads, s, hd).permute(2, 0, 1, 3).reshape(s * b, d)
    a = o @ prm["w_out"].t() + prm["b_out"]
    x = F.layer_norm(x + a * m1, (d,), prm["g1"], prm["be1"], prm["eps1"])
    f = F.gelu(x @ prm["w1"].t() + prm["b1"]) * m2
    f = f @ prm["w2"].t() + prm["b2"]
    return F.layer_norm(x + f * m3, (d,), prm["g2"], prm["be2"], prm["eps2"])
