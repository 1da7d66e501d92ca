"""CPU checks of the 1-4 image-plane entry points and models: argument validation of the multi-plane C-ABI happens
before any CUDA call, and models with more channels than the kernels take still construct with the reference's
``state_dict`` layout (so checkpoints load), refusing only in ``forward``."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SO = os.path.join(ROOT, "thesis-pai-reconstruction_b200", "pai_b200", "libpai_b200.so")

P16 = ctypes.c_void_p(16)          # a non-null, aligned dummy pointer: validation fails before it is dereferenced
LL = ctypes.c_longlong


@pytest.fixture(scope="module")
def so():
    if not os.path.exists(SO):
        subprocess.check_call([os.path.join(ROOT, "thesis-pai-reconstruction_b200", "csrc", "build.sh")])
    lib = ctypes.CDLL(SO)
    lib.pai_last_error.restype = ctypes.c_char_p
    return lib


def _calls(so, planes, np_, other):
    """Each multi-plane entry point with the plane pointer `planes`, plane count `np_` and every other pointer `other`
    (8 x 8 images, 64 channels, k = 3)."""
    f32 = ctypes.c_float
    return {
        "pai_conv_planes_to_wide": lambda: so.pai_conv_planes_to_wide(planes, np_, LL(64), 1, 8, 8, 3, 1, 0, other, None, 64,
                                                                      0, f32(0.2), other, 64, None),
        "pai_conv_wide_to_planes": lambda: so.pai_conv_wide_to_planes(other, 1, 8, 8, 64, 64, 3, 1, other, None, 0, planes,
                                                                      np_, LL(64), None),
        "pai_conv_planes_wide_wgrad": lambda: so.pai_conv_planes_wide_wgrad(planes, np_, LL(64), other, 64, 1, 8, 8, 64, 3, 1,
                                                                            0, other, None),
        "pai_im2col4x4_planes": lambda: so.pai_im2col4x4_planes(planes, np_, LL(64), 1, 8, 8, 4, 4, 2, 0, other, None),
        "pai_col2im4x4s2_planes": lambda: so.pai_col2im4x4s2_planes(other, 64, 1, 4, 4, None, 0, planes, np_, LL(64), None),
    }


@pytest.mark.parametrize("name", ["pai_conv_planes_to_wide", "pai_conv_wide_to_planes", "pai_conv_planes_wide_wgrad",
                                  "pai_im2col4x4_planes", "pai_col2im4x4s2_planes"])
def test_multiplane_entry_points_validate_before_cuda(so, name):
    rc = _calls(so, None, 3, P16)[name]()
    assert rc != 0 and b"null pointer" in so.pai_last_error() and name.encode() in so.pai_last_error()
    rc = _calls(so, P16, 3, None)[name]()
    assert rc != 0 and b"null pointer" in so.pai_last_error()
    for bad in (0, 5):
        rc = _calls(so, P16, bad, P16)[name]()
        msg = so.pai_last_error()
        assert rc != 0 and f"plane count {bad} outside 1..4".encode() in msg, msg
    rc = _calls(so, ctypes.c_void_p(18), 3, P16)[name]()          # a plane pointer that is not 4-byte aligned
    assert rc != 0 and b"alignment" in so.pai_last_error()


def test_five_channel_model_constructs_with_reference_state_dict():
    import torch
    from models.res_unet import ResUnetGAN
    kwargs = dict(res_type="18", channel_mults=(1, 2, 4, 8), dropout=0.0, loss_type="ssim")
    gz = np.load(os.path.join(ROOT, "tests", "golden", "variants_ref.npz"))
    torch.manual_seed(0)
    m5 = ResUnetGAN(in_channels=5, out_channels=5, **kwargs)
    m1 = ResUnetGAN(in_channels=1, out_channels=1, **kwargs)
    sd5, sd1 = m5.state_dict(), m1.state_dict()
    assert sorted(sd5) == list(gz["res_18_small/state_keys"])
    widened = {"unet.in_conv.weight": (64, 5, 3, 3), "unet.out.0.weight": (5, 64, 3, 3), "unet.out.0.bias": (5,)}
    for k, v in sd1.items():
        assert tuple(sd5[k].shape) == widened.get(k, tuple(v.shape)), k
    m1.load_state_dict(sd1)
    m5.load_state_dict({k: v.clone() for k, v in sd5.items()})


def test_channel_limit_is_named():
    from pai_b200 import layers as L
    for cin, cout in ((1, 1), (3, 3), (4, 1), (1, 4)):
        L.check_image_channels(cin, cout)
    for cin, cout in ((5, 3), (3, 5), (0, 1)):
        with pytest.raises(RuntimeError, match="1 to 4 image channels"):
            L.check_image_channels(cin, cout)
