"""CPU checks of the fp32 check path of the Residual / Attention / Trans U-Nets: the new ``pai_check_*`` entry points
validate their arguments before any CUDA call, and the fp32 functional restatement ``oracle/variants_port.py`` (what the
GPU tests hold the check path to, evaluated in fp64) reproduces the UNMODIFIED reference's golden vectors
(tests/golden/variants_ref.npz) within 1e-5, on every case (the largest, ``trans_full``, has 1.03 G parameters: 4 GB in
fp32 on the host)."""
import ctypes
import importlib
import os
import subprocess

import numpy as np
import pytest

import pix2pix_port as port
import variants_port
from test_variants_gpu import CASES      # the cases of the reference fixture (constructing them needs no GPU)

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SO = os.path.join(ROOT, "thesis-pai-reconstruction_b200", "pai_b200", "libpai_b200.so")

P = ctypes.c_void_p(16)            # a non-null dummy pointer: validation fails before it is dereferenced
f32, LL = ctypes.c_float, ctypes.c_longlong

def family(name):
    """-> (family, res_type) arguments of ``variants_port.forward`` for a case."""
    module, _, kwargs, *_ = CASES[name]
    return {"models.res_unet": "res", "models.attention_unet": "attention", "models.trans_unet": "trans"}[module], \
        kwargs.get("res_type", "18")


@pytest.fixture(scope="module")
def so():
    if not os.path.exists(SO):
        subprocess.check_call([os.path.join(ROOT, "thesis-pai-reconstruction_b200", "csrc", "build.sh")])
    lib = ctypes.CDLL(SO)
    lib.pai_last_error.restype = ctypes.c_char_p
    return lib


def _calls(so, a, b, shape_ok=True, groups=2):
    """Every new entry point with pointers ``a`` (first) / ``b`` (the rest); a zero or negative size when not ``shape_ok``."""
    s = 8 if shape_ok else 0
    return {
        "pai_check_conv2d_grouped_f32": lambda: so.pai_check_conv2d_grouped_f32(
            a, 1, 4, s, 8, b, 4, 3, 1, 1, groups, 0, None, 0, f32(0.2), 0, b, None),
        "pai_check_conv2d_wgrad_grouped_f32": lambda: so.pai_check_conv2d_wgrad_grouped_f32(
            a, 1, 4, s, 8, b, 4, 3, 1, 1, groups, 0, 0, f32(0.2), 0, b, None, None),
        "pai_check_maxpool2_f32": lambda: so.pai_check_maxpool2_f32(a, 1, 4, s, 8, b, None),
        "pai_check_maxpool2_bwd_f32": lambda: so.pai_check_maxpool2_bwd_f32(a, b, 1, 4, s, 8, b, None),
        "pai_check_upsample2_f32": lambda: so.pai_check_upsample2_f32(a, 1, 4, s, 8, b, None),
        "pai_check_upsample2_bwd_f32": lambda: so.pai_check_upsample2_bwd_f32(a, 1, 4, s, 8, b, None),
        "pai_check_layernorm_f32": lambda: so.pai_check_layernorm_f32(a, 4, s, b, b, f32(1e-5), b, b, b, None),
        "pai_check_layernorm_bwd_f32": lambda: so.pai_check_layernorm_bwd_f32(a, b, 4, s, b, b, b, b, b, b, None),
        "pai_check_linear_f32": lambda: so.pai_check_linear_f32(a, 4, s, 8, b, None, 0, b, None),
        "pai_check_linear_wgrad_f32": lambda: so.pai_check_linear_wgrad_f32(a, b, 4, s, 8, b, None, None),
        "pai_check_attention_f32": lambda: so.pai_check_attention_f32(a, 2, 4, 8, s, b, b, None),
        "pai_check_attention_bwd_f32": lambda: so.pai_check_attention_bwd_f32(a, b, b, 2, 4, 8, s, b, b, None),
    }


NAMES = list(_calls(None, None, None))


@pytest.mark.parametrize("name", NAMES)
def test_check_entry_points_validate_before_cuda(so, name):
    for a, b in ((None, P), (P, None)):
        rc = _calls(so, a, b)[name]()
        msg = so.pai_last_error()
        assert rc != 0 and b"null pointer" in msg and name.encode() in msg, msg
    rc = _calls(so, P, P, shape_ok=False)[name]()
    msg = so.pai_last_error()
    assert rc != 0 and b"bad shape" in msg and name.encode() in msg, msg


@pytest.mark.parametrize("name", ["pai_check_conv2d_grouped_f32", "pai_check_conv2d_wgrad_grouped_f32"])
@pytest.mark.parametrize("groups", [0, 3, 8])
def test_grouped_entry_points_reject_groups_that_do_not_divide(so, name, groups):
    rc = _calls(so, P, P, groups=groups)[name]()           # 4 input and 4 output channels
    msg = so.pai_last_error()
    assert rc != 0 and f"groups={groups} must divide".encode() in msg, msg


def test_output_padding_only_for_transposed(so):
    rc = so.pai_check_conv2d_grouped_f32(P, 1, 4, 8, 8, P, 4, 3, 2, 1, 1, 1, None, 0, f32(0.2), 0, P, None)
    assert rc != 0 and b"output padding" in so.pai_last_error()
    rc = so.pai_check_conv2d_grouped_f32(P, 1, 4, 8, 8, P, 4, 3, 2, 1, 1, 2, None, 0, f32(0.2), 1, P, None)
    assert rc != 0 and b"output padding" in so.pai_last_error()


def test_linear_transpose_takes_no_bias(so):
    rc = so.pai_check_linear_f32(P, 4, 8, 8, P, P, 1, P, None)
    assert rc != 0 and b"no bias" in so.pai_last_error()


def build(name, in_channels=1, out_channels=1, seed=0):
    """The drop-in of a case, built like tests/test_variants_gpu.py (seed 0 gives the fixture's weights)."""
    import torch
    module, cls, kwargs, _, _, loss_type = CASES[name]
    torch.manual_seed(seed)
    return getattr(importlib.import_module(module), cls)(in_channels=in_channels, out_channels=out_channels, dropout=0.0,
                                                         loss_type=loss_type, **kwargs)


def inputs(name, seed=1234):
    _, _, _, n, res, _ = CASES[name]
    x, t = port.synthetic_pairs(n, seed=seed)
    return x[:, :, :res, :res].contiguous(), t[:, :, :res, :res].contiguous()


@pytest.mark.parametrize("name", list(CASES))
def test_port_reproduces_reference_fixture(name, golden_dir):
    import torch
    torch.set_num_threads(os.cpu_count() or 1)
    gz = np.load(os.path.join(golden_dir, "variants_ref.npz"))
    sd = {k: v.detach().clone() for k, v in build(name).state_dict().items()}
    x, target = inputs(name)
    fam, res_type = family(name)
    with torch.no_grad():
        y = variants_port.forward(sd, x, False, fam, res_type)
        e = np.abs(y[:, :, ::4, ::4].numpy() - gz[f"{name}/eval_sub"])
        assert e.max() < 1e-5, ("eval", e.max())
        y = variants_port.forward(sd, x, True, fam, res_type)
        e = np.abs(y[:, :, ::4, ::4].numpy() - gz[f"{name}/train_sub"])
        assert e.max() < 1e-5, ("train", e.max())
        loss = float(port.generator_loss(sd, CASES[name][5], x, y, target))
    ref = float(gz[f"{name}/loss"])
    assert abs(loss - ref) < 1e-5, (loss, ref)
