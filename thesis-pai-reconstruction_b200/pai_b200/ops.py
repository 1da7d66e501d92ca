"""Tensor-level wrappers over the C-ABI (pai_b200.lib) and the weight packers.

Activations and gradients are NHWC bf16 ``torch.Tensor``s ``[N, H, W, C]`` (possibly a channel slice
``buf[..., c0:c1]`` of a wider concat buffer -- only the last-dim stride 1 and a uniform pixel stride
are required).  PyTorch owns every buffer; the library only enqueues kernels on the current stream.
"""
from __future__ import annotations

import ctypes
import os

import torch

from . import lib

ACT_NONE, ACT_LEAKY, ACT_RELU, ACT_TANH = 0, 1, 2, 3
BN_SMALL_OFF = os.environ.get("PAI_NO_BN_SMALL", "0") == "1"
# ConvTranspose2d(4,2,1) sub-pixel phases (SURVEY.md Appendix B): T[parity] = ((k, d), (k, d))
_T_K = ((1, 3), (0, 2))


# Optional per-launch timing of the implicit-GEMM kernels (bench.py roofline): a list of
# (name, algorithmic_flops, start_event, end_event) recorded on the launching stream.
_prof = None


def profile_start():
    global _prof
    _prof = []


def profile_stop():
    global _prof
    out, _prof = _prof, None
    return out or []


def _igemm_call(name, flops, *args):
    if _prof is None:
        lib.call(name, *args)
        return
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    lib.call(name, *args)
    e1.record()
    _prof.append((name, flops, e0, e1))


def _ptr(t):
    return ctypes.c_void_p(0 if t is None else t.data_ptr())


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _nhwc(t: torch.Tensor):
    """-> (n, h, w, c, ld) of an NHWC view whose pixels are ``ld`` elements apart."""
    assert t.dim() == 4 and t.stride(3) == 1, "expected an NHWC tensor with unit channel stride"
    n, h, w, c = t.shape
    if w > 1:
        ld = t.stride(2)
    elif h > 1:
        ld = t.stride(1)
    elif n > 1:
        ld = t.stride(0)
    else:
        ld = c
    assert (w == 1 or t.stride(2) == ld) and (h == 1 or t.stride(1) == w * ld) and (n == 1 or t.stride(0) == h * w * ld), \
        f"not a uniformly strided NHWC view: shape {tuple(t.shape)} strides {t.stride()}"
    return n, h, w, c, ld


def padded_cout(cout: int) -> int:
    """Rows of a packed weight matrix: multiples of 64 (16 for the 1-2 channel heads); the library picks the
    output-channel tile (256/128/64/32/16) that divides this."""
    q = 64 if cout >= 64 else 16
    return q * ((cout + q - 1) // q)


# ------------------------------------------------------------------------------------------ packing
def pack_conv_weight(w: torch.Tensor) -> torch.Tensor:
    """Conv2d weight ``[Cout, Cin, 4, 4]`` (any strides) -> bf16 ``[cout_pad, 16*Cin]`` with
    ``out[co, (ky*4+kx)*Cin + ci] = w[co, ci, ky, kx]`` (include/pai_b200.h, pai_conv4x4_fprop)."""
    cout, cin = w.shape[0], w.shape[1]
    cp = padded_cout(cout)
    out = torch.zeros(cp, 16 * cin, dtype=torch.bfloat16, device=w.device)
    out[:cout].view(cout, 4, 4, cin).copy_(w.permute(0, 2, 3, 1))
    return out


def pack_convT_weight(w: torch.Tensor) -> torch.Tensor:
    """ConvTranspose2d weight ``[Cin, Cout, 4, 4]`` -> bf16 ``[4, cout_pad, 4*Cin]`` with
    ``out[py*2+px, co, (ty*2+tx)*Cin + ci] = w[ci, co, T[py][ty].k, T[px][tx].k]``."""
    cin, cout = w.shape[0], w.shape[1]
    cp = padded_cout(cout)
    out = torch.zeros(4, cp, 4 * cin, dtype=torch.bfloat16, device=w.device)
    for py in range(2):
        for px in range(2):
            sub = w[:, :, _T_K[py][0]::2, _T_K[px][0]::2][:, :, :2, :2]      # [ci, co, ty, tx] (taps k, k+2)
            out[py * 2 + px, :cout].view(cout, 2, 2, cin).copy_(sub.permute(1, 2, 3, 0))
    return out


# ------------------------------------------------------------------------------------------ zeroed temporaries
class _ZeroPool:
    """One fill per training step for the SMALL zero-initialised fp32 temporaries (split-K workspaces, BatchNorm partial
    sums, zero bias gradients): ~50 of the step's 88 fill kernels were 2 us launches of a few KB each.  While a pool is
    open, ``zeros_f32`` hands out slices of one buffer sized by the previous step's demand; whatever does not fit falls
    back to ``torch.zeros``.  The buffer is a fresh allocation per step (views keep it alive; nothing is recycled under
    a live tensor), also under CUDA-graph capture.  The weight-gradient accumulators are NOT pooled: their fill right in
    front of the wgrad kernel leaves the lines in L2 for its reductions."""
    MAX_ELEMS = 4 << 20                      # larger requests keep their own fill

    def __init__(self):
        self.capacity = 0
        self.buf = None
        self.cursor = 0
        self.demand = 0
        self.depth = 0


_zero_pools = {}


class zero_pool:
    """``with ops.zero_pool(device):`` around one training step (models/wrapper.py)."""

    def __init__(self, device):
        on = device.type == "cuda" and os.environ.get("PAI_NO_ZERO_POOL", "0") != "1"
        self.pool = _zero_pools.setdefault((device.type, device.index), _ZeroPool()) if on else None
        self.device = device

    def __enter__(self):
        pl = self.pool
        if pl is None:
            return self
        pl.depth += 1
        if pl.depth == 1:
            pl.cursor = pl.demand = 0
            pl.buf = torch.zeros(pl.capacity, dtype=torch.float32, device=self.device) if pl.capacity else None
        return self

    def __exit__(self, *exc):
        pl = self.pool
        if pl is None:
            return False
        pl.depth -= 1
        if pl.depth == 0:
            pl.capacity, pl.buf = pl.demand, None
        return False


def zeros_f32(*shape, device) -> torch.Tensor:
    pl = _zero_pools.get((device.type, device.index))
    n = 1
    for d in shape:
        n *= int(d)
    if pl is None or pl.depth == 0 or n > _ZeroPool.MAX_ELEMS or n == 0:
        return torch.zeros(*shape, dtype=torch.float32, device=device)
    padded = (n + 63) & ~63                  # 256-byte slices
    pl.demand += padded
    if pl.buf is None or pl.cursor + padded > pl.buf.numel():
        return torch.zeros(*shape, dtype=torch.float32, device=device)
    out = pl.buf[pl.cursor:pl.cursor + n].view(*shape)
    pl.cursor += padded
    return out


# ------------------------------------------------------------------------------------------ fprop / dgrad
SPLITK_MAX_PIXELS = 74 * 128     # more output pixels than this always fill the GPU with tiles


def _splitk_ws(pixels: int, cout: int, device):
    """Zeroed fp32 split-K workspace for the small (<= 8x8) layers; None for layers that have enough tiles
    (the library decides the split factor, include/pai_b200.h)."""
    if pixels > SPLITK_MAX_PIXELS or cout < 16:
        return None
    return zeros_f32(pixels, cout, device=device)


def conv4x4_fprop(x, w_packed, cout, stride=2, bias=None, act=ACT_NONE, slope=0.2, out=None, out_f32=False,
                  n_tile=0):
    n, h, w, cin, ld = _nhwc(x)
    cp = w_packed.shape[0]
    ho, wo = (h // 2, w // 2) if stride == 2 else (h - 1, w - 1)
    if out is None:
        out = torch.empty(n, ho, wo, cout, dtype=torch.float32 if out_f32 else torch.bfloat16, device=x.device)
    on, oh, ow, oc, old = _nhwc(out)
    assert (on, oh, ow, oc) == (n, ho, wo, cout)
    ws = _splitk_ws(n * ho * wo, cout, x.device)
    _igemm_call("pai_conv4x4_fprop", 2.0 * n * ho * wo * cout * 16 * cin, _ptr(x), n, h, w, cin, ld, _ptr(w_packed), cout, cp, stride, _ptr(bias), act,
             float(slope), _ptr(out), old, int(out.dtype == torch.float32), n_tile, _ptr(ws), _stream())
    return out


def conv4x4_fprop_dual(x, w_packed, cout, bias, out1, act1, out2, act2, slope=0.2):
    """Stride-2 4x4 convolution with two bf16 outputs of the same accumulator (eval-mode encoder with folded BatchNorm:
    LeakyReLU input of the next encoder + ReLU concat slot of the decoder)."""
    n, h, w, cin, ld = _nhwc(x)
    cp = w_packed.shape[0]
    assert tuple(out1.shape) == tuple(out2.shape) == (n, h // 2, w // 2, cout)
    _igemm_call("pai_conv4x4_fprop_dual", 2.0 * n * (h // 2) * (w // 2) * cout * 16 * cin, _ptr(x), n, h, w, cin, ld,
                _ptr(w_packed), cout, cp, 2, _ptr(bias), act1, float(slope), _ptr(out1), _nhwc(out1)[4], _ptr(out2),
                _nhwc(out2)[4], act2, 0, _stream())


def to_uint8(x):
    """``models.utils.to_int`` (torchvision ConvertImageDtype(torch.uint8), models/utils.py:12) on the device."""
    x = x.contiguous().float()
    out = torch.empty(x.shape, dtype=torch.uint8, device=x.device)
    lib.call("pai_to_uint8", _ptr(x), x.numel(), _ptr(out), _stream())
    return out


def afmhot_uint8(img):
    """``report.output_hot_image`` (report.py:220-233) up to the PNG encoder: ``[n, 1, h, w]`` in [0, 1] -> uint8 ``[n, 3, h, w]``."""
    img = img.contiguous().float()
    n, _, h, w = img.shape
    out = torch.empty(n, 3, h, w, dtype=torch.uint8, device=img.device)
    lib.call("pai_afmhot_u8", _ptr(img), n, h * w, _ptr(out), _stream())
    return out


BN_PART_ROWS = 160          # >= number of SMs (one partial-sum row per persistent CTA)


def bn_fusable(pixels: int, cout: int) -> bool:
    """The statistics can ride on the GEMM epilogue when the layer is not split along K and has whole 64-channel chunks."""
    return pixels > SPLITK_MAX_PIXELS and cout % 64 == 0


def conv4x4_fprop_bnstats(x, w_packed, cout, bias=None):
    """Stride-2 4x4 convolution that also yields the BatchNorm partial sums of its (bf16) output:
    -> (raw ``[n, h/2, w/2, cout]`` bf16, partials ``[BN_PART_ROWS, 2*cout]`` fp32 for ``bn_finalize``)."""
    n, h, w, cin, ld = _nhwc(x)
    cp = w_packed.shape[0]
    out = torch.empty(n, h // 2, w // 2, cout, dtype=torch.bfloat16, device=x.device)
    part = zeros_f32(BN_PART_ROWS, 2 * cout, device=x.device)
    _igemm_call("pai_conv4x4_fprop_bnstats", 2.0 * n * (h // 2) * (w // 2) * cout * 16 * cin, _ptr(x), n, h, w, cin, ld,
                _ptr(w_packed), cout, cp, 2, _ptr(bias), _ptr(out), cout, 0, _ptr(part), BN_PART_ROWS, _stream())
    return out, part


def convT4x4s2_fprop_bnstats(x, w_packed, cout, bias=None):
    n, h, w, cin, ld = _nhwc(x)
    cp = w_packed.shape[1]
    out = torch.empty(n, 2 * h, 2 * w, cout, dtype=torch.bfloat16, device=x.device)
    part = zeros_f32(BN_PART_ROWS, 2 * cout, device=x.device)
    _igemm_call("pai_convT4x4s2_fprop_bnstats", 2.0 * n * h * w * cout * 16 * cin, _ptr(x), n, h, w, cin, ld,
                _ptr(w_packed), cout, cp, _ptr(bias), _ptr(out), cout, 0, _ptr(part), BN_PART_ROWS, _stream())
    return out, part


def conv4x4_dgrad_act(gy, w_packed_dgrad, cin, saved_act, slope=0.2, want_colsum=True):
    """Data gradient of a stride-2 4x4 convolution fused with the LeakyReLU backward of the layer below:
    ``gx = convT(gy) * act'(saved_act)`` -> (gx ``[n, 2h, 2w, cin]`` bf16, per-CTA partial column sums or None)."""
    n, h, w, cout, ld = _nhwc(gy)
    cp = w_packed_dgrad.shape[1]
    sn, sh, sw, sc, sld = _nhwc(saved_act)
    assert (sn, sh, sw, sc) == (n, 2 * h, 2 * w, cin) and sld == cin
    out = torch.empty(n, 2 * h, 2 * w, cin, dtype=torch.bfloat16, device=gy.device)
    part = zeros_f32(BN_PART_ROWS, 2 * cin, device=gy.device) if want_colsum else None
    _igemm_call("pai_conv4x4_dgrad_act", 2.0 * n * h * w * cin * 16 * cout, _ptr(gy), n, h, w, cout, ld,
                _ptr(w_packed_dgrad), cin, cp, _ptr(saved_act), float(slope), _ptr(out), cin, 0, _ptr(part), BN_PART_ROWS,
                _stream())
    return out, part


def convT4x4s2_fprop(x, w_packed, cout, bias=None, act=ACT_NONE, slope=0.2, out=None, out_f32=False, n_tile=0):
    n, h, w, cin, ld = _nhwc(x)
    cp = w_packed.shape[1]
    if out is None:
        out = torch.empty(n, 2 * h, 2 * w, cout, dtype=torch.float32 if out_f32 else torch.bfloat16, device=x.device)
    on, oh, ow, oc, old = _nhwc(out)
    assert (on, oh, ow, oc) == (n, 2 * h, 2 * w, cout)
    ws = _splitk_ws(4 * n * h * w, cout, x.device)
    _igemm_call("pai_convT4x4s2_fprop", 2.0 * n * h * w * cout * 16 * cin, _ptr(x), n, h, w, cin, ld, _ptr(w_packed), cout, cp, _ptr(bias), act,
             float(slope), _ptr(out), old, int(out.dtype == torch.float32), n_tile, _ptr(ws), _stream())
    return out


# ------------------------------------------------------------------------------------------ wgrad
def conv4x4_wgrad(x, gy, stride=2, dw=None, splitk=0):
    """-> fp32 ``[16, Cout, Cin]`` (tap-major); ``dw.permute(1, 2, 0).view(Cout, Cin, 4, 4)`` is the
    gradient in the reference's ``[Cout, Cin, kh, kw]`` layout."""
    n, h, w, cin, ld = _nhwc(x)
    gn, gh, gw, cout, gld = _nhwc(gy)
    if dw is None:
        dw = torch.zeros(16, cout, cin, dtype=torch.float32, device=x.device)
    _igemm_call("pai_conv4x4_wgrad", 2.0 * gn * gh * gw * cout * 16 * cin, _ptr(x), n, h, w, cin, ld, _ptr(gy), cout, gld, stride, _ptr(dw), splitk,
             _stream())
    return dw


def convT4x4s2_wgrad(x, gy, dw=None, splitk=0):
    """-> fp32 ``[16, Cin, Cout]``; ``dw.permute(1, 2, 0).view(Cin, Cout, 4, 4)`` is the reference layout."""
    n, h, w, cin, ld = _nhwc(x)
    gn, gh, gw, cout, gld = _nhwc(gy)
    if dw is None:
        dw = torch.zeros(16, cin, cout, dtype=torch.float32, device=x.device)
    _igemm_call("pai_convT4x4s2_wgrad", 2.0 * n * h * w * cout * 16 * cin, _ptr(x), n, h, w, cin, ld, _ptr(gy), cout, gld, _ptr(dw), splitk, _stream())
    return dw


def dropout2d_mask(n: int, c: int, p: float, device) -> torch.Tensor:
    """fp32 ``[n, c]`` Dropout2d mask: 0 with probability ``p``, else ``1 / (1 - p)`` (torch's device generator)."""
    keep = torch.bernoulli(torch.full((n, c), 1.0 - p, dtype=torch.float32, device=device))
    return keep.mul_(1.0 / (1.0 - p))


def scale_channels(x, mask, out=None):
    """``out[n, h, w, :] = x[n, h, w, :] * mask[n, :]`` (Dropout2d forward, and its backward on the gradient)."""
    n, h, w, c, ld = _nhwc(x)
    assert mask.shape == (n, c) and mask.dtype == torch.float32 and mask.is_contiguous()
    if out is None:
        out = torch.empty(n, h, w, c, dtype=torch.bfloat16, device=x.device)
    lib.call("pai_scale_channels", _ptr(x), ld, _ptr(mask), n, h * w, c, _ptr(out), _nhwc(out)[4], _stream())
    return out


def wgrad_finish(dw: torch.Tensor) -> torch.Tensor:
    """tap-major ``[16, A, B]`` (the wgrad kernels' accumulation layout) -> new ``[A, B, 4, 4]`` gradient in the
    parameter layout, one coalesced pass (instead of a generic strided ``permute().reshape()`` copy)."""
    _, a, b = dw.shape
    grad = torch.empty(a, b, 4, 4, dtype=torch.float32, device=dw.device)
    lib.call("pai_wgrad_finish", _ptr(dw), a * b, _ptr(grad), 0, _stream())
    return grad


# ------------------------------------------------------------------------------------------ BatchNorm / activations
def _mat(t: torch.Tensor):
    """NHWC (or [m, c]) view -> (m, c, ld)."""
    if t.dim() == 4:
        n, h, w, c, ld = _nhwc(t)
        return n * h * w, c, ld
    assert t.dim() == 2 and t.stride(1) == 1
    return t.shape[0], t.shape[1], t.stride(0)


def bn_stats(x, sums=None):
    m, c, ld = _mat(x)
    if sums is None:
        sums = torch.empty(2 * c, dtype=torch.float32, device=x.device)
    lib.call("pai_bn_stats", _ptr(x), m, c, ld, _ptr(sums), _stream())
    return sums


def bn_finalize(sums, m, c, gamma, beta, running_mean, running_var, training=True, eps=1e-5, momentum=0.1, ss=None,
                nparts=1):
    if ss is None:
        ss = torch.empty(4 * c, dtype=torch.float32, device=gamma.device)
    if nparts > 1:
        lib.call("pai_bn_finalize_partials", _ptr(sums), nparts, m, c, _ptr(gamma), _ptr(beta), float(eps),
                 float(momentum), int(training), _ptr(running_mean), _ptr(running_var), _ptr(ss), _stream())
    else:
        lib.call("pai_bn_finalize", _ptr(sums), m, c, _ptr(gamma), _ptr(beta), float(eps), float(momentum),
                 int(training), _ptr(running_mean), _ptr(running_var), _ptr(ss), _stream())
    return ss


def bn_apply_act(x, ss, out1, act1, out2=None, act2=ACT_NONE, slope=0.2):
    m, c, ld = _mat(x)
    m1, c1, ld1 = _mat(out1)
    assert (m1, c1) == (m, c)
    ld2 = 0
    if out2 is not None:
        m2, c2, ld2 = _mat(out2)
        assert (m2, c2) == (m, c)
    lib.call("pai_bn_apply_act", _ptr(x), m, c, ld, _ptr(ss), _ptr(out1), ld1, act1, _ptr(out2), ld2, act2,
             float(slope), _stream())


def bn_bwd_reduce(x, ss, g1, act1, g2=None, act2=ACT_NONE, slope=0.2):
    m, c, ld = _mat(x)
    _, _, ldg1 = _mat(g1)
    ldg2 = _mat(g2)[2] if g2 is not None else 0
    sums = torch.empty(2 * c, dtype=torch.float32, device=x.device)
    lib.call("pai_bn_bwd_reduce", _ptr(x), m, c, ld, _ptr(ss), _ptr(g1), ldg1, act1, _ptr(g2), ldg2, act2,
             float(slope), _ptr(sums), _stream())
    return sums


def bn_bwd_apply(x, ss, g1, act1, g2, act2, sums, gamma, dx, slope=0.2):
    m, c, ld = _mat(x)
    _, _, ldg1 = _mat(g1)
    ldg2 = _mat(g2)[2] if g2 is not None else 0
    _, _, lddx = _mat(dx)
    lib.call("pai_bn_bwd_apply", _ptr(x), m, c, ld, _ptr(ss), _ptr(g1), ldg1, act1, _ptr(g2), ldg2, act2,
             float(slope), _ptr(sums), _ptr(gamma), _ptr(dx), lddx, _stream())
    return dx


def bn_small_ok(x, operands: int = 1) -> bool:
    """Does ``x`` ([m, c] view) fit the one-launch BatchNorm of the small layers (one block per 8 channels holding all
    pixels of ``operands`` bf16 tensors in shared memory)?  [PAI_NO_BN_SMALL=1 switches the path off]"""
    if BN_SMALL_OFF:
        return False
    m, c, _ = _mat(x)
    return bool(lib.load().pai_bn_small_ok(m, c, operands))


def bn_small_fwd(x, gamma, beta, running_mean, running_var, out1, act1, out2=None, act2=ACT_NONE, slope=0.2, mask=None,
                 eps=1e-5, momentum=0.1):
    """Training-mode BatchNorm + activation(s) (+ Dropout2d mask on ``out1``) of a small layer in ONE launch;
    -> scale_shift ``[4c]`` like ``bn_finalize``."""
    m, c, ld = _mat(x)
    _, _, ld1 = _mat(out1)
    ld2 = _mat(out2)[2] if out2 is not None else 0
    ss = torch.empty(4 * c, dtype=torch.float32, device=x.device)
    ppi = m // mask.shape[0] if mask is not None else 0
    lib.call("pai_bn_small_fwd", _ptr(x), m, c, ld, _ptr(gamma), _ptr(beta), float(eps), float(momentum),
             _ptr(running_mean), _ptr(running_var), _ptr(ss), _ptr(out1), ld1, act1, _ptr(out2), ld2, act2, float(slope),
             _ptr(mask), ppi, _stream())
    return ss


def bn_small_bwd(x, ss, g1, act1, g2, act2, gamma, dx, slope=0.2, mask=None):
    """``scale_channels`` (Dropout2d backward on ``g1``) + ``bn_bwd_reduce`` + ``bn_bwd_apply`` of a small layer in ONE
    launch; -> sums ``[2c]`` (dbeta | dgamma)."""
    m, c, ld = _mat(x)
    _, _, ldg1 = _mat(g1)
    ldg2 = _mat(g2)[2] if g2 is not None else 0
    _, _, lddx = _mat(dx)
    sums = torch.empty(2 * c, dtype=torch.float32, device=x.device)
    ppi = m // mask.shape[0] if mask is not None else 0
    lib.call("pai_bn_small_bwd", _ptr(x), m, c, ld, _ptr(ss), _ptr(g1), ldg1, act1, _ptr(g2), ldg2, act2, float(slope),
             _ptr(mask), ppi, _ptr(gamma), _ptr(sums), _ptr(dx), lddx, _stream())
    return sums


def act_bwd(x, g1, act1, g2, act2, dx, slope=0.2):
    """Activation backward of a layer without BatchNorm, fused with the bias gradient:
    ``dx = g1*act1'(x) + g2*act2'(x)``; returns ``sums`` with ``sums[:c] = sum over pixels of dx``."""
    m, c, ld = _mat(x)
    _, _, ldg1 = _mat(g1)
    ldg2 = _mat(g2)[2] if g2 is not None else 0
    _, _, lddx = _mat(dx)
    sums = torch.empty(2 * c, dtype=torch.float32, device=x.device)
    lib.call("pai_act_bwd", _ptr(x), m, c, ld, _ptr(g1), ldg1, act1, _ptr(g2), ldg2, act2, float(slope), _ptr(sums),
             _ptr(dx), lddx, _stream())
    return sums


def colsum(x):
    m, c, ld = _mat(x)
    sums = torch.empty(2 * c, dtype=torch.float32, device=x.device)
    lib.call("pai_colsum", _ptr(x), m, c, ld, _ptr(sums), _stream())
    return sums[:c]


# ------------------------------------------------------------------------------------------ degenerate layers
def smallc_conv_fprop(planes, w, bias, out1, act1=ACT_NONE, out2=None, act2=ACT_NONE, stride=2, flip=False, slope=0.2):
    """planes: 1 or 2 fp32 ``[n, ih, iw]`` tensors; w: fp32 ``[c, 16, cin]``; out: NHWC bf16 ``[n, oh, ow, c]``."""
    p0 = planes[0]
    p1 = planes[1] if len(planes) > 1 else None
    n, ih, iw = p0.shape
    on, oh, ow, c, ld1 = _nhwc(out1)
    assert on == n and w.shape == (c, 16, len(planes)) and w.is_contiguous() and p0.is_contiguous()
    ld2 = _nhwc(out2)[4] if out2 is not None else 0
    lib.call("pai_smallc_conv_fprop", _ptr(p0), _ptr(p1), len(planes), n, ih, iw, oh, ow, stride, int(flip), _ptr(w),
             _ptr(bias), c, _ptr(out1), ld1, act1, _ptr(out2), ld2, act2, float(slope), _stream())
    return out1


def smallc_conv_wgrad(a, planes, stride=2, flip=False):
    """a: NHWC bf16 ``[n, oh, ow, c]``; planes: fp32 ``[n, ih, iw]`` x (1|2) -> fp32 ``[c, 16, cin]``."""
    n, oh, ow, c, lda = _nhwc(a)
    p0 = planes[0]
    p1 = planes[1] if len(planes) > 1 else None
    _, ih, iw = p0.shape
    dw = torch.zeros(c, 16, len(planes), dtype=torch.float32, device=a.device)
    lib.call("pai_smallc_conv_wgrad", _ptr(a), lda, c, _ptr(p0), _ptr(p1), len(planes), n, ih, iw, oh, ow, stride,
             int(flip), _ptr(dw), _stream())
    return dw


# ------------------------------------------------------------------------------------------ thin layers as GEMMs
def im2col4x4(planes, oh, ow, stride=2, flip=False):
    """1|2 fp32 planes ``[n, ih, iw]`` -> bf16 ``[n, oh, ow, 64]`` (channel = tap*cin + j).  Only the first
    ``16 * len(planes)`` channels are written: pass ``k_valid=16 * len(planes)`` to ``pointwise_gemm`` and ignore the
    other columns of a ``pointwise_wgrad`` result."""
    p0 = planes[0]
    p1 = planes[1] if len(planes) > 1 else None
    n, ih, iw = p0.shape
    col = torch.empty(n, oh, ow, 64, dtype=torch.bfloat16, device=p0.device)
    lib.call("pai_im2col4x4", _ptr(p0), _ptr(p1), len(planes), n, ih, iw, oh, ow, stride, int(flip), _ptr(col),
             _stream())
    return col


def pointwise_gemm(x, w_packed, cout, bias=None, act=ACT_NONE, slope=0.2, out=None, out_f32=False, out2=None,
                   act2=ACT_NONE, n_tile=0, k_valid=0):
    """1x1 convolution: ``y[..., co] = act(bias + x[..., :] @ w_packed[co, :])`` over all pixels of an NHWC tensor.
    ``k_valid``: only the first ``k_valid`` of the 64 input columns hold data (``im2col4x4`` output)."""
    m, cin, ld = _mat(x)
    cp = w_packed.shape[0]
    if out is None:
        out = torch.empty(*x.shape[:-1], cout, dtype=torch.float32 if out_f32 else torch.bfloat16, device=x.device)
    mo, co, old = _mat(out)
    assert (mo, co) == (m, cout)
    old2 = 0
    if out2 is not None:
        m2, c2, old2 = _mat(out2)
        assert (m2, c2) == (m, cout)
    _igemm_call("pai_pointwise_gemm", 2.0 * m * cin * cout, _ptr(x), m, cin, ld, _ptr(w_packed), cout, cp, _ptr(bias),
                act, float(slope), _ptr(out), old, int(out.dtype == torch.float32), _ptr(out2), old2, act2, n_tile,
                k_valid, _stream())
    return out


def pointwise_wgrad(u, s, splitk=0):
    """-> fp32 ``[cu, cs]`` = sum over pixels of ``u[pix, :]^T s[pix, :]``."""
    m, cu, uld = _mat(u)
    ms, cs, sld = _mat(s)
    assert ms == m
    dw = torch.zeros(cu, cs, dtype=torch.float32, device=u.device)
    _igemm_call("pai_pointwise_wgrad", 2.0 * m * cu * cs, _ptr(u), m, cu, uld, _ptr(s), cs, sld, _ptr(dw), splitk,
                _stream())
    return dw


def col2im4x4s2(p, bias=None, act=ACT_NONE):
    """fp32 per-tap partial products ``[n, h, w, >=16]`` -> fp32 ``[n, 2h, 2w]`` (transposed conv, 1 output channel)."""
    n, h, w, c = p.shape
    assert p.dtype == torch.float32 and p.stride(3) == 1 and c >= 16
    out = torch.empty(n, 2 * h, 2 * w, dtype=torch.float32, device=p.device)
    lib.call("pai_col2im4x4s2", _ptr(p), p.stride(2), n, h, w, _ptr(bias), act, _ptr(out), _stream())
    return out


# ------------------------------------------------------------------------------------------ thin layers, single pass
def thin_conv_fprop(planes, w_packed, cout, bias, out1, act1=ACT_NONE, out2=None, act2=ACT_NONE, slope=0.2):
    """Conv2d(len(planes), cout, 4, 2, 1) straight from 1|2 fp32 planes ``[n, ih, iw]`` (csrc/thin.cu): the im2col rows
    are built in shared memory.  ``w_packed``: bf16 ``[cout, 64]``, column = tap*cin + j; ``out1`` / ``out2``: NHWC bf16."""
    p0 = planes[0]
    p1 = planes[1] if len(planes) > 1 else None
    n, ih, iw = p0.shape
    assert p0.is_contiguous() and p0.dtype == torch.float32 and (p1 is None or (p1.is_contiguous() and p1.shape == p0.shape))
    on, oh, ow, oc, ld1 = _nhwc(out1)
    assert (on, oh, ow, oc) == (n, ih // 2, iw // 2, cout) and tuple(w_packed.shape) == (cout, 64)
    ld2 = 0
    if out2 is not None:
        assert tuple(out2.shape) == (n, ih // 2, iw // 2, cout)
        ld2 = _nhwc(out2)[4]
    _igemm_call("pai_thin_conv4x4s2_fprop", 2.0 * n * (ih // 2) * (iw // 2) * cout * 16 * len(planes), _ptr(p0), _ptr(p1),
                len(planes), n, ih, iw, _ptr(w_packed), cout, _ptr(bias), _ptr(out1), ld1, act1, _ptr(out2), ld2, act2,
                float(slope), _stream())
    return out1


def thin_wgrad_ok(u, planes) -> bool:
    return u.shape[3] in (64, 128) and planes[0].shape[2] % 128 == 0


def thin_conv_wgrad(u, planes):
    """-> fp32 ``[c, 16*cin]`` = sum over pixels of ``u[pix, c] * plane_j[2*oy-1+ky, 2*ox-1+kx]`` (column = tap*cin + j):
    the weight gradient of a 1|2-input-channel stride-2 4x4 convolution (``u`` = gradient of its output), and of a
    1-output-channel transposed one (``u`` = its input, plane = the output gradient)."""
    n, oh, ow, c, uld = _nhwc(u)
    p0 = planes[0]
    p1 = planes[1] if len(planes) > 1 else None
    pn, ih, iw = p0.shape
    assert (pn, ih, iw) == (n, 2 * oh, 2 * ow) and p0.is_contiguous() and p0.dtype == torch.float32
    dw = torch.zeros(c, 16 * len(planes), dtype=torch.float32, device=u.device)
    _igemm_call("pai_thin_conv4x4s2_wgrad", 2.0 * n * oh * ow * c * 16 * len(planes), _ptr(u), uld, c, _ptr(p0), _ptr(p1),
                len(planes), n, ih, iw, _ptr(dw), _stream())
    return dw


def thin_plane_ok(x) -> bool:
    return x.shape[2] == 128 and x.shape[3] % 64 == 0 and x.shape[3] <= 256


def thin_convT_plane(x, w_taps, bias=None, act=ACT_NONE):
    """ConvTranspose2d(c, 1, 4, 2, 1) (+bias, optional Tanh): NHWC bf16 ``[n, h, 128, c]`` -> fp32 ``[n, 2h, 256]`` in one
    streaming pass; ``w_taps``: bf16 ``[16, c]`` (row = ky*4+kx)."""
    n, h, w, c, ld = _nhwc(x)
    assert tuple(w_taps.shape) == (16, c) and w_taps.is_contiguous()
    out = torch.empty(n, 2 * h, 2 * w, dtype=torch.float32, device=x.device)
    _igemm_call("pai_thin_convT4x4s2_plane", 2.0 * n * h * w * c * 16, _ptr(x), n, h, w, c, ld, _ptr(w_taps), _ptr(bias),
                act, _ptr(out), _stream())
    return out


def col2im4x4s1(p):
    """fp32 per-tap partial products ``[n, h, w, >=16]`` -> fp32 ``[n, h-1, w-1]`` (4x4 conv, stride 1, pad 1, 1 output channel)."""
    n, h, w, c = p.shape
    assert p.dtype == torch.float32 and p.stride(3) == 1 and c >= 16
    out = torch.empty(n, h - 1, w - 1, dtype=torch.float32, device=p.device)
    lib.call("pai_col2im4x4s1", _ptr(p), p.stride(2), n, h, w, _ptr(out), _stream())
    return out


# ------------------------------------------------------------------------------------------ Res / Attention / Trans U-Net layers
def pack_conv1x1_weight(w: torch.Tensor) -> torch.Tensor:
    """Conv2d weight ``[Cout, Cin, 1, 1]`` (or a Linear ``[out, in]``) -> bf16 ``[cout_pad, Cin]``."""
    cout, cin = w.shape[0], w.shape[1]
    out = torch.zeros(padded_cout(cout), cin, dtype=torch.bfloat16, device=w.device)
    out[:cout].copy_(w.reshape(cout, cin))
    return out


def pack_conv1x1_weight_t(w: torch.Tensor) -> torch.Tensor:
    """-> bf16 ``[cin_pad, Cout]``: the data-gradient operand of a 1x1 convolution / Linear."""
    cout, cin = w.shape[0], w.shape[1]
    out = torch.zeros(padded_cout(cin), cout, dtype=torch.bfloat16, device=w.device)
    out[:cin].copy_(w.reshape(cout, cin).t())
    return out


def pack_conv3x3_weight(w: torch.Tensor) -> torch.Tensor:
    """Conv2d weight ``[Cout, Cin, 3, 3]`` -> bf16 ``[cout_pad, 9*Cin]``, column ``(ky*3+kx)*Cin + ci``."""
    cout, cin = w.shape[0], w.shape[1]
    out = torch.zeros(padded_cout(cout), 9 * cin, dtype=torch.bfloat16, device=w.device)
    out[:cout].view(cout, 3, 3, cin).copy_(w.permute(0, 2, 3, 1))
    return out


def pack_conv3x3_weight_dgrad(w: torch.Tensor) -> torch.Tensor:
    """-> bf16 ``[cin_pad, 9*Cout]`` with the taps flipped: conv3x3(dL/dy, this) = dL/dx."""
    cout, cin = w.shape[0], w.shape[1]
    out = torch.zeros(padded_cout(cin), 9 * cout, dtype=torch.bfloat16, device=w.device)
    out[:cin].view(cin, 3, 3, cout).copy_(w.flip(2, 3).permute(1, 2, 3, 0))
    return out


def conv3x3_fprop(x, w_packed, cout, bias=None, act=ACT_NONE, slope=0.2, out=None, out_f32=False):
    n, h, w, cin, ld = _nhwc(x)
    cp = w_packed.shape[0]
    if out is None:
        out = torch.empty(n, h, w, cout, dtype=torch.float32 if out_f32 else torch.bfloat16, device=x.device)
    old = _nhwc(out)[4]
    ws = _splitk_ws(n * h * w, cout, x.device)
    _igemm_call("pai_conv3x3_fprop", 2.0 * n * h * w * cout * 9 * cin, _ptr(x), n, h, w, cin, ld, _ptr(w_packed), cout, cp,
                _ptr(bias), act, float(slope), _ptr(out), old, int(out.dtype == torch.float32), 0, _ptr(ws), _stream())
    return out


def conv3x3_wgrad(x, gy):
    """-> fp32 ``[9, Cout, Cin]``; ``.permute(1, 2, 0).reshape(Cout, Cin, 3, 3)`` is the reference layout."""
    n, h, w, cin, ld = _nhwc(x)
    _, _, _, cout, gld = _nhwc(gy)
    dw = torch.zeros(9, cout, cin, dtype=torch.float32, device=x.device)
    _igemm_call("pai_conv3x3_wgrad", 2.0 * n * h * w * cout * 9 * cin, _ptr(x), n, h, w, cin, ld, _ptr(gy), cout, gld,
                _ptr(dw), _stream())
    return dw


def maxpool2_fwd(x):
    n, h, w, c, ld = _nhwc(x)
    y = torch.empty(n, h // 2, w // 2, c, dtype=torch.bfloat16, device=x.device)
    lib.call("pai_maxpool2_fwd", _ptr(x), n, h, w, c, ld, _ptr(y), c, _stream())
    return y


def maxpool2_bwd(x, gy):
    n, h, w, c, ld = _nhwc(x)
    gx = torch.empty(n, h, w, c, dtype=torch.bfloat16, device=x.device)
    lib.call("pai_maxpool2_bwd", _ptr(x), n, h, w, c, ld, _ptr(gy), _nhwc(gy)[4], _ptr(gx), c, _stream())
    return gx


def upsample2_fwd(x, out=None):
    n, h, w, c, ld = _nhwc(x)
    if out is None:
        out = torch.empty(n, 2 * h, 2 * w, c, dtype=torch.bfloat16, device=x.device)
    lib.call("pai_upsample2_fwd", _ptr(x), n, h, w, c, ld, _ptr(out), _nhwc(out)[4], _stream())
    return out


def upsample2_bwd(gy):
    n, h2, w2, c, ld = _nhwc(gy)
    gx = torch.empty(n, h2 // 2, w2 // 2, c, dtype=torch.bfloat16, device=gy.device)
    lib.call("pai_upsample2_bwd", _ptr(gy), n, h2 // 2, w2 // 2, c, ld, _ptr(gx), c, _stream())
    return gx


def add_act(a, b, act=ACT_NONE, slope=0.2, out=None):
    m, c, lda = _mat(a)
    ldb = _mat(b)[2] if b is not None else 0
    if out is None:
        out = torch.empty(*a.shape, dtype=torch.bfloat16, device=a.device)
    lib.call("pai_add_act", _ptr(a), lda, _ptr(b), ldb, m, c, act, float(slope), _ptr(out), _mat(out)[2], _stream())
    return out


def scale_rows_fwd(x, s, act=ACT_NONE, out=None):
    m, c, ld = _mat(x)
    if out is None:
        out = torch.empty(*x.shape, dtype=torch.bfloat16, device=x.device)
    lib.call("pai_scale_rows_fwd", _ptr(x), ld, _ptr(s), m, c, act, _ptr(out), _mat(out)[2], _stream())
    return out


def scale_rows_bwd(x, s, g, act=ACT_NONE):
    m, c, ld = _mat(x)
    gx = torch.empty(*x.shape, dtype=torch.bfloat16, device=x.device)
    gs = torch.empty(s.shape, dtype=torch.float32, device=x.device)
    lib.call("pai_scale_rows_bwd", _ptr(x), ld, _ptr(s), _ptr(g), _mat(g)[2], m, c, act, _ptr(gx), c, _ptr(gs), _stream())
    return gx, gs


def conv_plane_to_wide(plane, w, bias, k, pad, act=ACT_NONE, slope=0.2, flip=False, out=None):
    """plane fp32 ``[n, h, w]``, w fp32 ``[c, k*k]`` -> NHWC bf16 ``[n, h, w, c]``."""
    n, h, wd = plane.shape
    c = w.shape[0]
    if out is None:
        out = torch.empty(n, h, wd, c, dtype=torch.bfloat16, device=plane.device)
    lib.call("pai_conv_plane_to_wide", _ptr(plane), n, h, wd, k, pad, int(flip), _ptr(w), _ptr(bias), c, act, float(slope),
             _ptr(out), _nhwc(out)[4], _stream())
    return out


def conv_wide_to_plane(x, w, bias, k, pad, act=ACT_NONE):
    """NHWC bf16 ``[n, h, w, c]``, w fp32 ``[k*k, c]`` -> fp32 plane ``[n, h, w]``."""
    n, h, wd, c, ld = _nhwc(x)
    out = torch.empty(n, h, wd, dtype=torch.float32, device=x.device)
    lib.call("pai_conv_wide_to_plane", _ptr(x), n, h, wd, c, ld, k, pad, _ptr(w), _ptr(bias), act, _ptr(out), _stream())
    return out


def conv_plane_wide_wgrad(plane, wide, k, pad, flip=False):
    """-> fp32 ``[c, k*k]`` = sum over pixels of ``wide[p, c] * plane[p + off_t]``."""
    n, h, wd, c, ld = _nhwc(wide)
    dw = torch.zeros(c, k * k, dtype=torch.float32, device=wide.device)
    lib.call("pai_conv_plane_wide_wgrad", _ptr(plane), _ptr(wide), ld, n, h, wd, c, k, pad, int(flip), _ptr(dw), _stream())
    return dw


def gconv4_3x3_fprop(x, w, bias=None):
    """Grouped 3x3 conv, 4 channels per group: x NHWC bf16, w fp32 ``[c, 9, 4]``."""
    n, h, wd, c, ld = _nhwc(x)
    y = torch.empty(n, h, wd, c, dtype=torch.bfloat16, device=x.device)
    lib.call("pai_gconv4_3x3_fprop", _ptr(x), n, h, wd, c, ld, _ptr(w), _ptr(bias), _ptr(y), c, _stream())
    return y


def gconv4_3x3_wgrad(x, gy):
    n, h, wd, c, ld = _nhwc(x)
    dw = torch.zeros(c, 9, 4, dtype=torch.float32, device=x.device)
    lib.call("pai_gconv4_3x3_wgrad", _ptr(x), ld, _ptr(gy), _nhwc(gy)[4], n, h, wd, c, _ptr(dw), _stream())
    return dw


# ------------------------------------------------------------------------------------------ Trans U-Net (ViT bottleneck)
def subsample2(x, scatter=False):
    n, h, w, c, ld = _nhwc(x)
    if not scatter:
        y = torch.empty(n, h // 2, w // 2, c, dtype=torch.bfloat16, device=x.device)
        lib.call("pai_subsample2", _ptr(x), n, h, w, c, ld, _ptr(y), c, 0, _stream())
    else:            # x is the coarse gradient [n, h, w, c]; result is the fine [n, 2h, 2w, c]
        y = torch.zeros(n, 2 * h, 2 * w, c, dtype=torch.bfloat16, device=x.device)
        lib.call("pai_subsample2", _ptr(x), n, 2 * h, 2 * w, c, ld, _ptr(y), c, 1, _stream())
    return y


def layernorm_fwd(x, gamma, beta, eps):
    m, d = x.shape
    y = torch.empty_like(x)
    mean = torch.empty(m, dtype=torch.float32, device=x.device)
    rstd = torch.empty(m, dtype=torch.float32, device=x.device)
    lib.call("pai_layernorm_fwd", _ptr(x), m, d, _ptr(gamma), _ptr(beta), float(eps), _ptr(y), _ptr(mean), _ptr(rstd),
             _stream())
    return y, mean, rstd


def layernorm_bwd(x, g, gamma, mean, rstd):
    m, d = x.shape
    dx = torch.empty_like(x)
    dgamma = torch.empty(d, dtype=torch.float32, device=x.device)
    dbeta = torch.empty(d, dtype=torch.float32, device=x.device)
    lib.call("pai_layernorm_bwd", _ptr(x), _ptr(g), m, d, _ptr(gamma), _ptr(mean), _ptr(rstd), _ptr(dx), _ptr(dgamma),
             _ptr(dbeta), _stream(), kernels=2)
    return dx, dgamma, dbeta


def gelu_fwd(x):
    y = torch.empty_like(x)
    lib.call("pai_gelu_fwd", _ptr(x), x.numel(), _ptr(y), _stream())
    return y


def gelu_bwd(x, g):
    dx = torch.empty_like(x)
    lib.call("pai_gelu_bwd", _ptr(x), _ptr(g), x.numel(), _ptr(dx), _stream())
    return dx


def attn_fwd(qkv, s, b, heads):
    e = qkv.shape[1] // 3
    probs = torch.empty(b * heads, s, s, dtype=torch.float32, device=qkv.device)
    out = torch.empty(s * b, e, dtype=torch.bfloat16, device=qkv.device)
    lib.call("pai_attn_fwd", _ptr(qkv), s, b, heads, e // heads, _ptr(probs), _ptr(out), _stream())
    return out, probs


def attn_bwd(qkv, dout, probs, s, b, heads):
    e = qkv.shape[1] // 3
    work = torch.empty_like(probs)
    dqkv = torch.empty_like(qkv)
    lib.call("pai_attn_bwd", _ptr(qkv), _ptr(dout), s, b, heads, e // heads, _ptr(probs), _ptr(work), _ptr(dqkv), _stream(),
             kernels=2)
    return dqkv


# Train-mode dropout of the encoder layer (csrc/pai_dropout.cuh): ``key`` is a one-element int64 device tensor, the
# masks are regenerated from (element index, site, key) inside the kernels and never stored.
def _key(key):
    assert key.dtype == torch.int64 and key.numel() == 1 and key.is_cuda
    return _ptr(key)


def dropout_mask(key, site, n, p):
    """uint8 ``[n]``: 1 where the fused kernels keep element ``i`` of ``site``, 0 where they drop it."""
    out = torch.empty(n, dtype=torch.uint8, device=key.device)
    lib.call("pai_dropout_mask", _key(key), site, n, float(p), _ptr(out), _stream())
    return out


def attn_fwd_dropout(qkv, s, b, heads, key, site, p):
    e = qkv.shape[1] // 3
    probs = torch.empty(b * heads, s, s, dtype=torch.float32, device=qkv.device)
    out = torch.empty(s * b, e, dtype=torch.bfloat16, device=qkv.device)
    lib.call("pai_attn_fwd_dropout", _ptr(qkv), s, b, heads, e // heads, _key(key), site, float(p), _ptr(probs), _ptr(out),
             _stream())
    return out, probs


def attn_bwd_dropout(qkv, dout, probs, s, b, heads, key, site, p):
    e = qkv.shape[1] // 3
    work = torch.empty_like(probs)
    dqkv = torch.empty_like(qkv)
    lib.call("pai_attn_bwd_dropout", _ptr(qkv), _ptr(dout), s, b, heads, e // heads, _key(key), site, float(p), _ptr(probs),
             _ptr(work), _ptr(dqkv), _stream(), kernels=2)
    return dqkv


def add_dropout_layernorm_fwd(x, y, gamma, beta, eps, key, site, p):
    """-> (z = x + dropout(y), LayerNorm(z), mean, rstd)."""
    m, d = x.shape
    assert y.shape == x.shape and x.is_contiguous() and y.is_contiguous()
    z, out = torch.empty_like(x), torch.empty_like(x)
    mean = torch.empty(m, dtype=torch.float32, device=x.device)
    rstd = torch.empty(m, dtype=torch.float32, device=x.device)
    lib.call("pai_add_dropout_layernorm_fwd", _ptr(x), _ptr(y), m, d, _key(key), site, float(p), _ptr(gamma), _ptr(beta),
             float(eps), _ptr(z), _ptr(out), _ptr(mean), _ptr(rstd), _stream())
    return z, out, mean, rstd


def layernorm_bwd_dropout(z, g, gamma, mean, rstd, key, site, p):
    """-> (dz, dy, dgamma, dbeta): the residual branch's and the dropout branch's gradients."""
    m, d = z.shape
    dz, dy = torch.empty_like(z), torch.empty_like(z)
    dgamma = torch.empty(d, dtype=torch.float32, device=z.device)
    dbeta = torch.empty(d, dtype=torch.float32, device=z.device)
    lib.call("pai_layernorm_bwd_dropout", _ptr(z), _ptr(g), m, d, _ptr(gamma), _ptr(mean), _ptr(rstd), _key(key), site,
             float(p), _ptr(dz), _ptr(dy), _ptr(dgamma), _ptr(dbeta), _stream(), kernels=2)
    return dz, dy, dgamma, dbeta


def gelu_dropout_fwd(x, key, site, p):
    y = torch.empty_like(x)
    lib.call("pai_gelu_dropout_fwd", _ptr(x), x.numel(), _key(key), site, float(p), _ptr(y), _stream())
    return y


def gelu_dropout_bwd(x, g, key, site, p):
    dx = torch.empty_like(x)
    lib.call("pai_gelu_dropout_bwd", _ptr(x), _ptr(g), x.numel(), _key(key), site, float(p), _ptr(dx), _stream())
    return dx


# ------------------------------------------------------------------------------------------ fp32 check path
def check_conv2d(x, w, bias=None, stride=2, pad=1, pre_act=ACT_NONE, slope=0.2, transposed=False):
    """nn.Conv2d / nn.ConvTranspose2d on fp32 NCHW (csrc/check_f32.cu): exact-arithmetic twin of the igemm layers."""
    assert x.dtype == torch.float32 and w.dtype == torch.float32 and x.is_cuda
    x, w = x.contiguous(), w.contiguous()
    n, cin, h, wd = x.shape
    k = w.shape[2]
    cout = w.shape[1] if transposed else w.shape[0]
    assert w.shape[2] == w.shape[3] and (w.shape[0] if transposed else w.shape[1]) == cin
    ho = (h - 1) * stride - 2 * pad + k if transposed else (h + 2 * pad - k) // stride + 1
    wo = (wd - 1) * stride - 2 * pad + k if transposed else (wd + 2 * pad - k) // stride + 1
    y = torch.empty(n, cout, ho, wo, dtype=torch.float32, device=x.device)
    b = None if bias is None else bias.contiguous()
    lib.call("pai_check_conv2d_f32", _ptr(x), n, cin, h, wd, _ptr(w), cout, k, stride, pad, _ptr(b), pre_act, slope,
             1 if transposed else 0, _ptr(y), _stream())
    return y


def check_batchnorm(x, gamma, beta, running_mean, running_var, training, eps=1e-5, momentum=0.1):
    assert x.dtype == torch.float32 and x.is_cuda
    x = x.contiguous()
    n, c = x.shape[0], x.shape[1]
    hw = x.numel() // max(n * c, 1)
    y = torch.empty_like(x)
    lib.call("pai_check_batchnorm_f32", _ptr(x), n, c, hw, _ptr(gamma), _ptr(beta), _ptr(running_mean), _ptr(running_var),
             1 if training else 0, eps, momentum, _ptr(y), _stream())
    return y


def check_act(x, act, slope=0.2):
    x = x.contiguous()
    y = torch.empty_like(x)
    lib.call("pai_check_act_f32", _ptr(x), x.numel(), act, slope, _ptr(y), _stream())
    return y


def check_conv2d_wgrad(x, g, w_shape, stride=2, pad=1, pre_act=ACT_NONE, slope=0.2, transposed=False, want_bias=True):
    """-> (dW in the weight's own layout, dbias or None) of ``y = conv(pre_act(x))`` given ``g = dL/dy`` (fp32 NCHW)."""
    x, g = x.contiguous(), g.contiguous()
    n, cin, h, wd = x.shape
    cout, k = g.shape[1], w_shape[2]
    dw = torch.empty(w_shape, dtype=torch.float32, device=x.device)
    db = torch.empty(cout, dtype=torch.float32, device=x.device) if want_bias else None
    lib.call("pai_check_conv2d_wgrad_f32", _ptr(x), n, cin, h, wd, _ptr(g), cout, k, stride, pad, pre_act, slope,
             1 if transposed else 0, _ptr(dw), _ptr(db), _stream(), kernels=2 if want_bias else 1)
    return dw, db


def check_batchnorm_bwd(x, g, gamma, eps=1e-5):
    x, g = x.contiguous(), g.contiguous()
    n, c = x.shape[0], x.shape[1]
    hw = x.numel() // max(n * c, 1)
    dx = torch.empty_like(x)
    dgamma = torch.empty(c, dtype=torch.float32, device=x.device)
    dbeta = torch.empty(c, dtype=torch.float32, device=x.device)
    lib.call("pai_check_batchnorm_bwd_f32", _ptr(x), _ptr(g), n, c, hw, _ptr(gamma), eps, _ptr(dx), _ptr(dgamma), _ptr(dbeta),
             _stream())
    return dx, dgamma, dbeta


def check_act_bwd(x, g, act, slope=0.2):
    x, g = x.contiguous(), g.contiguous()
    dx = torch.empty_like(x)
    lib.call("pai_check_act_bwd_f32", _ptr(x), _ptr(g), x.numel(), act, slope, _ptr(dx), _stream())
    return dx
