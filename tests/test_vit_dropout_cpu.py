"""CPU checks of the Trans U-Net's train-mode ViT dropout: the numpy Philox of oracle/vit_dropout_ref.py against the
Random123 known-answer vectors, the fp32 encoder-layer restatement against torch's own nn.TransformerEncoderLayer,
and argument validation of the new C-ABI entry points (before any CUDA call, so no device is needed)."""
import ctypes
import os
import subprocess

import numpy as np
import pytest
import torch

import vit_dropout_ref as ref

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SO = os.path.join(ROOT, "thesis-pai-reconstruction_b200", "pai_b200", "libpai_b200.so")


@pytest.mark.parametrize("ctr, key, want", [
    ((0, 0, 0, 0), (0, 0), (0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8)),
    ((0xffffffff,) * 4, (0xffffffff,) * 2, (0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd)),
    ((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0xa4093822, 0x299f31d0),
     (0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1)),
])
def test_philox_known_answers(ctr, key, want):
    got = ref.philox4x32_10(*ctr, *key)
    assert tuple(int(w) for w in got) == want


def test_mask_rule_uses_the_element_index_layout():
    key, site, n, p = 0x0123456789ABCDEF, 5, 4099, 0.3
    keep = ref.dropout_keep(key, site, n, p)
    thr = ref.dropout_threshold(p)
    for idx in (0, 3, 4, 1025, 4098):
        g = idx >> 2
        w = ref.philox4x32_10(g & 0xFFFFFFFF, g >> 32, site, 0, key & 0xFFFFFFFF, key >> 32)[idx & 3]
        assert bool(keep[idx]) == (int(w) >= thr)
    assert ref.dropout_threshold(1.0 - 1e-12) == 2 ** 32 - 1
    assert ref.dropout_keep(-1, 0, 8, 0.5).shape == (8,)          # a negative int64 key is its two's complement


@pytest.mark.parametrize("s, b, d, heads", [(5, 3, 64, 8), (2, 4, 128, 8)])
def test_restatement_matches_torch_encoder_layer(s, b, d, heads):
    """All-ones masks: the restatement is torch's post-norm layer (eval mode, fp32), forward and parameter gradients."""
    torch.manual_seed(0)
    lyr = torch.nn.TransformerEncoderLayer(d, heads, dim_feedforward=96, dropout=0.5, activation="gelu").eval()
    x = torch.randn(s, b, d)
    gout = torch.randn(s, b, d)
    # torch's eval-mode fast path needs no_grad; with grad enabled it takes the same math as training without dropout
    want = lyr(x)
    (want * gout).sum().backward()
    want_grads = {k: p.grad.clone() for k, p in lyr.named_parameters()}
    lyr.zero_grad()
    prm = ref.layer_params(lyr)
    masks = [torch.ones(b * heads, s, s), torch.ones(s * b, d), torch.ones(s * b, 96), torch.ones(s * b, d)]
    got = ref.encoder_layer(x.reshape(s * b, d), prm, s, b, heads, masks)
    assert torch.allclose(got.reshape(s, b, d), want, atol=1e-5, rtol=1e-5)
    (got * gout.reshape(s * b, d)).sum().backward()
    for k, p in lyr.named_parameters():
        assert torch.allclose(p.grad, want_grads[k], atol=1e-5, rtol=1e-4), k


@pytest.fixture(scope="module")
def so():
    if not os.path.exists(SO):
        subprocess.check_call([os.path.join(ROOT, "thesis-pai-reconstruction_b200", "csrc", "build.sh")])
    lib = ctypes.CDLL(SO)
    lib.pai_last_error.restype = ctypes.c_char_p
    return lib


def _calls(key, p):
    f32, ll, v = ctypes.c_float(p), ctypes.c_longlong, ctypes.c_void_p(16)
    return {
        "pai_dropout_mask": lambda so: so.pai_dropout_mask(key, 0, ll(16), f32, v, None),
        "pai_attn_fwd_dropout": lambda so: so.pai_attn_fwd_dropout(v, 4, 2, 8, 32, key, 0, f32, v, v, None),
        "pai_attn_bwd_dropout": lambda so: so.pai_attn_bwd_dropout(v, v, 4, 2, 8, 32, key, 0, f32, v, v, v, None),
        "pai_add_dropout_layernorm_fwd": lambda so: so.pai_add_dropout_layernorm_fwd(
            v, v, ll(8), 256, key, 1, f32, v, v, ctypes.c_float(1e-5), v, v, v, v, None),
        "pai_layernorm_bwd_dropout": lambda so: so.pai_layernorm_bwd_dropout(
            v, v, ll(8), 256, v, v, v, key, 1, f32, v, v, v, v, None),
        "pai_gelu_dropout_fwd": lambda so: so.pai_gelu_dropout_fwd(v, ll(16), key, 2, f32, v, None),
        "pai_gelu_dropout_bwd": lambda so: so.pai_gelu_dropout_bwd(v, v, ll(16), key, 2, f32, v, None),
    }


@pytest.mark.parametrize("name", list(_calls(None, 0.5)))
def test_dropout_entry_points_validate_arguments_without_gpu(so, name):
    rc = _calls(None, 0.5)[name](so)
    msg = so.pai_last_error()
    assert rc != 0 and name.encode() in msg and b"null key" in msg, msg
    for p in (0.0, 1.0, float("nan")):
        rc = _calls(ctypes.c_void_p(16), p)[name](so)
        msg = so.pai_last_error()
        assert rc != 0 and name.encode() in msg and b"outside (0, 1)" in msg, msg


def test_vit_rejects_dropout_of_one_in_training():
    import models.trans_unet as tu
    vit = tu.VisionTransformer(channels=64, input_size=8, patch_size=2, dropout=1.0, transformer_layers=1).train()
    with pytest.raises(RuntimeError, match="dropout must be < 1"):
        vit(torch.zeros(2, 8, 8, 64, dtype=torch.bfloat16))
