"""CPU-only checks of the C-ABI boundary: the shared library loads without a GPU, exports every symbol
that include/pai_b200.h declares, and the ctypes signature table (pai_b200/lib.py) covers the header."""
import ctypes
import os
import re
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "pai_b200.h")
SO = os.path.join(ROOT, "thesis-pai-reconstruction_b200", "pai_b200", "libpai_b200.so")


def _declared():
    text = open(HEADER).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(pai_[a-zA-Z0-9_]+)\s*\(", text)))


@pytest.fixture(scope="module")
def so():
    if not os.path.exists(SO):
        subprocess.check_call([os.path.join(ROOT, "thesis-pai-reconstruction_b200", "csrc", "build.sh")])
    return ctypes.CDLL(SO)


def test_header_declares_entry_points():
    names = _declared()
    assert len(names) >= 15 and "pai_conv4x4_fprop" in names and "pai_ssim_psnr_fwd" in names


def test_library_exports_every_declared_symbol(so):
    for name in _declared():
        assert hasattr(so, name), f"{name} declared in include/pai_b200.h but not exported"


def test_ctypes_table_covers_header():
    from pai_b200 import lib
    bound = set(lib.SIGNATURES) | set(lib.RESTYPES) | {"pai_last_error"}
    assert set(_declared()) <= bound, set(_declared()) - bound


def test_version_and_error_channel_without_gpu(so):
    so.pai_last_error.restype = ctypes.c_char_p
    assert so.pai_version() >= 100
    # argument validation happens before any CUDA call, so it is testable without a device
    rc = so.pai_conv4x4_fprop(None, 1, 8, 8, 64, 64, None, 64, 64, 2, None, 0, ctypes.c_float(0.2), None, 64, 0, 64, None, None)
    assert rc != 0 and b"null pointer" in so.pai_last_error()
    rc = so.pai_ssim_psnr_fwd(ctypes.c_void_p(16), ctypes.c_void_p(16), 0, 1, 8, 8, 0, ctypes.c_void_p(16), None,
                              ctypes.c_void_p(16), None, None)
    assert rc != 0 and b"11x11 window" in so.pai_last_error()


def test_no_cpu_fallback_in_product_metrics(monkeypatch):
    import torch
    from pai_b200 import metrics
    monkeypatch.setattr(torch.cuda, "is_available", lambda: False)     # a machine without a CUDA device
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        metrics.ssim(torch.rand(1, 1, 32, 32), torch.rand(1, 1, 32, 32))


def test_dropin_package_mirrors_reference_interface():
    import inspect
    import models.pix2pix as mp
    import models.utils as mu
    import models.wrapper as mw
    for name in ("Pix2Pix", "Unet", "EncoderBlock", "DecoderBlock"):
        assert hasattr(mp, name)
    for name in ("UnetWrapper", "Discriminator", "DiscriminatorBlock"):
        assert hasattr(mw, name)
    for name in ("denormalize", "to_int", "init_weights", "get_parameter_count", "ssim", "psnr", "rmse"):
        assert hasattr(mu, name)
    sig = inspect.signature(mp.Pix2Pix.__init__)
    assert list(sig.parameters)[1:] == ["in_channels", "out_channels", "channel_mults", "dropout", "loss_type"]
    assert sig.parameters["dropout"].default == 0.5 and sig.parameters["in_channels"].default == 3
    assert inspect.signature(mw.Discriminator.__init__).parameters["in_channels"].default == 3
    for meth in ("forward", "loss", "discriminator_loss", "configure_optimizers", "training_step", "validation_step"):
        assert hasattr(mw.UnetWrapper, meth)
    m = mp.Pix2Pix(1, 1, dropout=0.0, loss_type="ssim")
    assert mu.get_parameter_count(m.unet) == 54_413_313 and m.discriminator is None


def test_new_entry_points_validate_arguments_without_gpu(so):
    """Argument validation of the entry points added for the fused step happens before any CUDA call."""
    so.pai_last_error.restype = ctypes.c_char_p
    f32 = ctypes.c_float
    rc = so.pai_conv4x4_dgrad_act(ctypes.c_void_p(16), 1, 8, 8, 128, 128, ctypes.c_void_p(16), 64, 64, None, f32(0.2),
                                  ctypes.c_void_p(16), 64, 0, None, 0, None)
    assert rc != 0 and b"saved activation" in so.pai_last_error()
    rc = so.pai_conv4x4_fprop_bnstats(ctypes.c_void_p(16), 1, 8, 8, 64, 64, ctypes.c_void_p(16), 64, 64, 2, None,
                                      ctypes.c_void_p(16), 64, 0, None, 0, None)
    assert rc != 0 and b"partial-sum buffer" in so.pai_last_error()
    rc = so.pai_wgrad_finish(None, ctypes.c_longlong(16), ctypes.c_void_p(16), 0, None)
    assert rc != 0 and b"pai_wgrad_finish" in so.pai_last_error()
    rc = so.pai_check_conv2d_f32(None, 1, 1, 8, 8, ctypes.c_void_p(16), 1, 4, 2, 1, None, 0, f32(0.2), 0,
                                 ctypes.c_void_p(16), None)
    assert rc != 0 and b"null pointer" in so.pai_last_error()
    rc = so.pai_pointwise_gemm(ctypes.c_void_p(16), ctypes.c_longlong(128), 128, 128, ctypes.c_void_p(16), 64, 64, None, 0,
                               f32(0.2), ctypes.c_void_p(16), 64, 0, None, 0, 0, 0, 16, None)
    assert rc != 0 and b"k_valid" in so.pai_last_error()       # k_valid needs cin == 64
    rc = so.pai_adam_prepare(None, f32(2e-4), f32(0.5), f32(0.999), None, None)
    assert rc != 0 and b"pai_adam_prepare" in so.pai_last_error()


def test_step_graph_and_check_path_are_exposed_on_the_dropin():
    import models.wrapper as mw
    from pai_b200 import engine, graph
    assert hasattr(mw.UnetWrapper, "enable_step_graph") and hasattr(mw.UnetWrapper, "disable_step_graph")
    assert callable(graph.StepGraph) and not engine.check_path_enabled()
    with engine.check_path():
        assert engine.check_path_enabled()
    assert not engine.check_path_enabled()
