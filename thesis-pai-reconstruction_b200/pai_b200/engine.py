"""Whole-network fused forward / backward of the Pix2Pix U-Net generator and the PatchGAN
discriminator on the B200 kernels, exposed as two ``torch.autograd.Function``s.

Reference semantics (file:line in /root/reference):
* ``Unet.forward``            models/pix2pix.py:198-216 (ctor :130-196): 8x [LeakyReLU -> Conv4x4 s2 -> BN],
  8x [ReLU -> ConvT4x4 s2 -> BN] with skip concat, Tanh; the skips are the *un-activated* BN outputs.
* ``Discriminator.forward``   models/wrapper.py:236-238 (blocks :196-206, :228-234).

Data layout in HBM: activations and gradients NHWC bf16; every decoder input is ONE buffer
``[N, h, w, 2C]`` whose first half is written by the previous decoder's BN+ReLU kernel and whose second
half is written by the matching encoder's BN kernel (zero-copy ``torch.cat``).  Parameters stay fp32 in
the reference's ``state_dict`` layout; bf16 GEMM packs are rebuilt when a parameter's version changes.

What rides on the GEMM epilogues (switchable for A/B measurements by the environment variables in brackets):
* BatchNorm statistics of every layer large enough not to be split along K: per-CTA partial rows from
  ``conv4x4_fprop_bnstats`` / ``convT4x4s2_fprop_bnstats``, summed by ``bn_finalize``  [PAI_NO_BN_FUSION];
* the LeakyReLU backward and the bias gradient of the PatchGAN blocks: ``conv4x4_dgrad_act``  [PAI_NO_ACT_BWD_FUSION];
* bias, activation, second (skip) output and sub-pixel phase placement (always).
The 1- and 2-channel layers (enc0, D0, dec7 and their gradients, the PatchGAN head) run as single-pass kernels that build
the thin GEMM operand in shared memory (csrc/thin.cu) instead of an im2col / col2im carrier in HBM  [PAI_NO_THIN_DIRECT].
Train-mode Dropout2d (decoders 0-2 of the default constructor) is a per-(sample, channel) mask applied to the concat
slot; ``check_path()`` switches the forward to the exact fp32 kernels of csrc/check_f32.cu.
The <= 8x8 levels run their whole training-mode BatchNorm (+ activation, + Dropout2d mask) and its whole backward as ONE
launch each (``ops.bn_small_fwd`` / ``bn_small_bwd``)  [PAI_NO_BN_SMALL]; small zeroed temporaries of a step come from one
pooled fill (``ops.zero_pool``)  [PAI_NO_ZERO_POOL]; eval-mode BatchNorm is folded into the GEMM operands  [PAI_NO_BN_FOLD].
Models with more than one image channel (the reference's default is 3) send the image through a zero-padded 64-channel
carrier and the ordinary implicit-GEMM kernels (``_carrier``).
Library-side switches (read by csrc/): PAI_NO_CTA_PAIR, PAI_NO_PHASE_FUSION, PAI_NO_PHASE_MERGE, PAI_IGEMM_KSUB=1,
PAI_L2_PREFETCH=1, PAI_PDL=1 (the last two are opt-in experiments that measured no gain, DESIGN.md 4.1).
"""
from __future__ import annotations

import os
from typing import List, Optional

import torch

from . import dp, ops
from .ops import ACT_LEAKY, ACT_NONE, ACT_RELU, ACT_TANH

BN_EPS, BN_MOMENTUM, SLOPE = 1e-5, 0.1, 0.2
FUSE_BN_STATS = os.environ.get("PAI_NO_BN_FUSION") is None     # BatchNorm statistics from the GEMM epilogue
FUSE_ACT_BWD = os.environ.get("PAI_NO_ACT_BWD_FUSION") is None  # PatchGAN LeakyReLU backward in the dgrad GEMM epilogue
THIN_DIRECT = os.environ.get("PAI_NO_THIN_DIRECT") is None      # 1-2 channel layers as single-pass kernels (csrc/thin.cu)


# ------------------------------------------------------------------------------------------ pack cache
class _PackCache:
    """bf16 GEMM operand packs of fp32 master weights.  The packs live ON the parameter object (so they die
    with it -- ``id()`` of a freed tensor can be reused) and are rebuilt when its version counter or storage
    changes (optimizer step, ``load_state_dict``, ``.cuda()``)."""

    def get(self, tag: str, p: torch.Tensor, fn):
        store = p.__dict__.setdefault("_pai_packs", {})
        stamp = (p._version, p.data_ptr())
        ent = store.get(tag)
        if ent is None or ent[0] != stamp:
            with torch.no_grad():
                ent = (stamp, fn(p.detach()))
            store[tag] = ent
        return ent[1]


_packs = _PackCache()

_P1_TAGS, _P2_TAGS = ("conv_f", "convT_d"), ("conv_d", "convT_f")


def fused_pack_targets(p: torch.Tensor):
    """-> (pack1, pack2, b_pad) of a ``[A, B, 4, 4]`` weight whose cached packs are the two big GEMM operands
    (``pai_adam_pack_conv4x4`` rewrites them in the optimizer step), or None when the parameter has no packs
    or thin-layer packs (those are rebuilt lazily by the Python packers)."""
    store = p.__dict__.get("_pai_packs")
    if not store or p.dim() != 4 or tuple(p.shape[2:]) != (4, 4):
        return None
    p1 = p2 = None
    for tag, ent in store.items():
        if tag in _P1_TAGS:
            p1 = ent[1]
        elif tag in _P2_TAGS:
            p2 = ent[1]
        else:
            return None
    if p1 is None and p2 is None:
        return None
    return p1, p2, (p2.shape[1] if p2 is not None else 0)


def restamp_packs(p: torch.Tensor) -> None:
    """Marks the cached packs of ``p`` as current (called after a kernel rewrote them in place)."""
    store = p.__dict__["_pai_packs"]
    stamp = (p._version, p.data_ptr())
    for tag in store:
        store[tag] = (stamp, store[tag][1])


def repack_in_place(p: torch.Tensor) -> None:
    """Rewrites the packs that FusedAdam refreshes in place (see ``fused_pack_targets``) from the current values of
    ``p``, into the same buffers: for a parameter overwritten in place while a captured step graph keeps reading them.
    The other packs need nothing: the graph rebuilds them from the parameter at every replay."""
    if fused_pack_targets(p) is None:
        return
    fns = {"conv_f": ops.pack_conv_weight, "convT_d": ops.pack_conv_weight,
           "conv_d": ops.pack_convT_weight, "convT_f": ops.pack_convT_weight}
    with torch.no_grad():
        for tag, (_, buf) in p.__dict__["_pai_packs"].items():
            buf.copy_(fns[tag](p.detach()))
    restamp_packs(p)


def _fprop_pack(w):      # Conv2d weight [Cout, Cin, 4, 4]
    return _packs.get("conv_f", w, ops.pack_conv_weight)


def _dgrad_pack(w):      # Conv2d dgrad == ConvT fprop with the weight read as [in=Cout, out=Cin]
    return _packs.get("conv_d", w, ops.pack_convT_weight)


def _fpropT_pack(w):     # ConvTranspose2d weight [Cin, Cout, 4, 4]
    return _packs.get("convT_f", w, ops.pack_convT_weight)


def _dgradT_pack(w):     # ConvT dgrad == Conv fprop with the weight read as [out=Cin, in=Cout]
    return _packs.get("convT_d", w, ops.pack_conv_weight)


def _w_tap_major(w):     # [C, cin, 4, 4] -> fp32 [C, 16, cin] for the direct kernels
    c, cin = w.shape[0], w.shape[1]
    if cin == 1:
        return w.detach().reshape(c, 16, 1)
    return _packs.get("small", w, lambda t: t.permute(0, 2, 3, 1).reshape(c, 16, cin).contiguous())


def _pad_cols(t, cols=64):
    out = torch.zeros(t.shape[0], cols, dtype=torch.bfloat16, device=t.device)
    out[:, :t.shape[1]] = t
    return out


def _thin_in_pack(w):    # Conv2d weight [C, cin<=2, 4, 4] -> bf16 [C, 64]: column = tap*cin + j (im2col order)
    return _packs.get("thin_in", w, lambda t: _pad_cols(t.permute(0, 2, 3, 1).reshape(t.shape[0], -1)))


def _thin_out_fprop_pack(w):   # ConvT weight [Cin, 1, 4, 4] -> bf16 [16, Cin]: row = tap (per-tap partial products)
    return _packs.get("thin_out_f", w, lambda t: t[:, 0].reshape(t.shape[0], 16).t().contiguous().bfloat16())


def _thin_out_dgrad_pack(w):   # ConvT weight [Cin, 1, 4, 4] -> bf16 [Cin, 64]: column = tap
    return _packs.get("thin_out_d", w, lambda t: _pad_cols(t[:, 0].reshape(t.shape[0], 16)))


def _aux_pack(tag: str, p: torch.Tensor, fn):
    """Packs that the fused Adam kernel does not rewrite: kept apart from ``_pai_packs`` (whose tags tell FusedAdam
    which operands to refresh in place) and dropped by FusedAdam after every update of the parameter."""
    store = p.__dict__.setdefault("_pai_aux", {})
    stamp = (p._version, p.data_ptr())
    ent = store.get(tag)
    if ent is None or ent[0] != stamp:
        with torch.no_grad():
            ent = (stamp, fn(p.detach()))
        store[tag] = ent
    return ent[1]


def _head_dgrad_pack(w):       # PatchGAN head Conv2d weight [1, C, 4, 4] -> bf16 [C, 64]: column = tap
    return _aux_pack("head_d", w, lambda t: _pad_cols(t[0].reshape(t.shape[1], 16)))


def _head_fprop_pack(w):       # PatchGAN head Conv2d weight [1, C, 4, 4] -> bf16 [16, C]: row = tap (per-tap partial products)
    return _aux_pack("head_f", w, lambda t: t[0].reshape(t.shape[1], 16).t().contiguous().bfloat16())


def _thin_in_dgrad_pack(w, j):  # Conv2d weight [C, cin, 4, 4] -> bf16 [16, C]: row = tap, for input channel j
    return _packs.get(f"thin_in_d{j}", w, lambda t: t[:, j].reshape(t.shape[0], 16).t().contiguous().bfloat16())


# ---- models with in / out channels != 1 (the reference's own defaults are 3 / 3, models/pix2pix.py:25-27): the few image
# channels travel in a zero-padded 64-channel NHWC carrier and the first / last convolution run on the ordinary
# implicit-GEMM kernels with zero-padded weights.  Functionally complete, not tuned: the BASELINE configurations are
# grayscale and take the thin-layer kernels (csrc/thin.cu).
CARRIER = 64


def _carrier(*images: torch.Tensor) -> torch.Tensor:
    """``[N, C_k, H, W]`` tensors -> bf16 ``[N, H, W, 64]`` with the channels of all tensors side by side, rest zero."""
    n, _, h, w = images[0].shape
    total = sum(t.shape[1] for t in images)
    if total > CARRIER:
        raise RuntimeError(f"pai_b200: at most {CARRIER} image channels per convolution input (got {total})")
    out = torch.zeros(n, h, w, CARRIER, dtype=torch.bfloat16, device=images[0].device)
    c0 = 0
    for t in images:
        out[..., c0:c0 + t.shape[1]] = t.permute(0, 2, 3, 1)
        c0 += t.shape[1]
    return out


def _pad_dim1(t: torch.Tensor) -> torch.Tensor:      # [A, B < 64, 4, 4] -> fp32 [A, 64, 4, 4]
    return torch.nn.functional.pad(t.float(), (0, 0, 0, 0, 0, CARRIER - t.shape[1]))


def _carrier_in_pack(w):         # Conv2d [C, cin, 4, 4] reading a carrier: fprop operand
    return _aux_pack("car_in_f", w, lambda t: ops.pack_conv_weight(_pad_dim1(t)))


def _carrier_in_dgrad_pack(w):   # ... its data gradient (ConvT fprop with the weight read as [in=C, out=64])
    return _aux_pack("car_in_d", w, lambda t: ops.pack_convT_weight(_pad_dim1(t)))


def _carrier_out_pack(w):        # ConvTranspose2d [Cin, cout, 4, 4] writing a carrier: fprop operand
    return _aux_pack("car_out_f", w, lambda t: ops.pack_convT_weight(_pad_dim1(t)))


def _carrier_out_dgrad_pack(w):  # ... its data gradient (Conv fprop with the weight read as [out=Cin, in=64])
    return _aux_pack("car_out_d", w, lambda t: ops.pack_conv_weight(_pad_dim1(t)))


def _carrier_bias(b):            # [cout] -> fp32 [64]
    return _aux_pack("car_b", b, lambda t: torch.nn.functional.pad(t.float(), (0, CARRIER - t.shape[0])))


FOLD_EVAL_BN = os.environ.get("PAI_NO_BN_FOLD") is None      # eval mode: BatchNorm folded into the GEMM operands


def _folded(tag: str, conv, bn: "BNState", transposed: bool):
    """-> (bf16 GEMM pack, fp32 bias) of an eval-mode ``conv -> BatchNorm`` pair folded into one affine convolution
    (report.py:26-43 freezes the model, so BatchNorm is ``y * s + t`` with s = gamma / sqrt(running_var + eps),
    t = beta - running_mean * s): W' = W * s[co], b' = b * s + t.  Cached on the conv weight (FusedAdam drops
    ``_pai_aux`` after every update); the stamp also covers the BatchNorm tensors and the running statistics, which this
    library updates through raw pointers (``_pai_stat_version``)."""
    w = conv.weight
    store = w.__dict__.setdefault("_pai_aux", {})
    m = bn.mod
    stamp = (w._version, w.data_ptr(), conv.bias._version, m.weight._version, m.bias._version, m.running_mean._version,
             m.running_var._version, m.running_mean.data_ptr(), m.__dict__.get("_pai_stat_version", 0))
    ent = store.get(tag)
    if ent is None or ent[0] != stamp:
        with torch.no_grad():
            sc = m.weight.detach().float() * torch.rsqrt(m.running_var.float() + BN_EPS)
            sh = m.bias.detach().float() - m.running_mean.float() * sc
            wf = w.detach().float() * (sc.view(1, -1, 1, 1) if transposed else sc.view(-1, 1, 1, 1))
            bf = (conv.bias.detach().float() * sc + sh).contiguous()
            pack = ops.pack_convT_weight(wf) if transposed else ops.pack_conv_weight(wf)
        ent = (stamp, (pack, bf))
        store[tag] = ent
    return ent[1]


def _bf16(*shape, device):
    return torch.empty(*shape, dtype=torch.bfloat16, device=device)


class BNState:
    """Live view of one nn.BatchNorm2d of the drop-in module tree (attributes are read through the
    module so ``model.cuda()`` / ``load_state_dict`` are picked up)."""

    def __init__(self, mod):
        self.mod = mod

    weight = property(lambda self: self.mod.weight)
    bias = property(lambda self: self.mod.bias)
    running_mean = property(lambda self: self.mod.running_mean)
    running_var = property(lambda self: self.mod.running_var)
    num_batches_tracked = property(lambda self: self.mod.num_batches_tracked)


def _batchnorm(raw, bn: BNState, training: bool, counters=None, partials=None):
    """-> scale_shift [4C] of BN over the pixels of ``raw``; updates running stats when training.  The
    ``num_batches_tracked`` increments of a whole forward are collected in ``counters`` (one foreach launch).
    ``partials``: per-CTA partial sums already produced by the convolution's epilogue (no statistics pass)."""
    m, c, _ = ops._mat(raw)
    if training and partials is not None:
        sums, nparts = partials, partials.shape[0]
    else:
        sums, nparts = (ops.bn_stats(raw) if training else None), 1
    ss = ops.bn_finalize(sums, m, c, bn.weight.detach(), bn.bias.detach(), bn.running_mean, bn.running_var,
                         training=training, eps=BN_EPS, momentum=BN_MOMENTUM, nparts=nparts)
    if training:
        bn.mod.__dict__["_pai_stat_version"] = bn.mod.__dict__.get("_pai_stat_version", 0) + 1   # running stats moved
        if counters is None:
            bn.num_batches_tracked.add_(1)
        else:
            counters.append(bn.num_batches_tracked)
    return ss


def _batchnorm_act(raw, bn: BNState, training, counters, partials, out1, act1, out2=None, act2=ACT_NONE, mask=None):
    """BatchNorm + activation(s) of ``raw`` into ``out1`` (and ``out2``); ``mask`` = Dropout2d scaling of ``out1``.
    Small layers in training mode take ONE launch (``ops.bn_small_fwd``); the rest is statistics (or the partial sums of
    the GEMM epilogue) -> ``bn_finalize`` -> ``bn_apply_act`` (-> ``scale_channels``).  -> scale_shift."""
    if training and partials is None and ops.bn_small_ok(raw):
        ss = ops.bn_small_fwd(raw, bn.weight.detach(), bn.bias.detach(), bn.running_mean, bn.running_var, out1, act1, out2,
                              act2, slope=SLOPE, mask=mask, eps=BN_EPS, momentum=BN_MOMENTUM)
        bn.mod.__dict__["_pai_stat_version"] = bn.mod.__dict__.get("_pai_stat_version", 0) + 1
        if counters is None:
            bn.num_batches_tracked.add_(1)
        else:
            counters.append(bn.num_batches_tracked)
        return ss
    ss = _batchnorm(raw, bn, training, counters, partials)
    ops.bn_apply_act(raw, ss, out1, act1, out2, act2, slope=SLOPE)
    if mask is not None:
        ops.scale_channels(out1, mask, out=out1)
    return ss


# ------------------------------------------------------------------------------------------ fp32 check path
_check = False


class check_path:
    """``with engine.check_path(): y = model(x)`` runs the drop-in generator / PatchGAN on the exact fp32 kernels of
    csrc/check_f32.cu (fp32 NCHW tensors, fp32 FMA accumulation, no bf16 operands) instead of the tcgen05 path -- the
    north star's "1e-5 with the fp32 accumulate check path".  Forward AND backward: ``loss.backward()`` on a graph built
    inside the context gives fp32 check-path gradients of every parameter (wrong index math in a deep wgrad shows up as a
    1e-1 error here, while the bf16 path can only be held to its 8-12 % noise floor)."""

    def __enter__(self):
        global _check
        self.prev, _check = _check, True
        return self

    def __exit__(self, *exc):
        global _check
        _check = self.prev
        return False


def check_path_enabled() -> bool:
    return _check


class _CheckConv(torch.autograd.Function):
    """``y = conv(pre_act(x), w) + b`` (Conv2d or ConvTranspose2d) on the fp32 check kernels, with its exact fp32 backward:
    data gradient = the opposite convolution of ``g`` times ``pre_act'(x)``, weight / bias gradients by
    ``pai_check_conv2d_wgrad_f32`` (double-precision reductions)."""

    @staticmethod
    def forward(ctx, x, w, b, stride, pad, pre_act, transposed):
        y = ops.check_conv2d(x, w, b, stride=stride, pad=pad, pre_act=pre_act, slope=SLOPE, transposed=transposed)
        ctx.save_for_backward(x, w)
        ctx.cfg = (stride, pad, pre_act, transposed, b is not None)
        return y

    @staticmethod
    def backward(ctx, g):
        x, w = ctx.saved_tensors
        stride, pad, pre_act, transposed, has_b = ctx.cfg
        g = g.contiguous().float()
        gx = gw = gb = None
        if ctx.needs_input_grad[0]:
            gx = ops.check_conv2d(g, w, None, stride=stride, pad=pad, pre_act=ACT_NONE, transposed=not transposed)
            if gx.shape != x.shape:          # stride-2 transposed convolution of an odd-sized gradient cannot happen here
                raise RuntimeError(f"pai_b200 check path: data-gradient shape {tuple(gx.shape)} != input {tuple(x.shape)}")
            if pre_act != ACT_NONE:
                gx = ops.check_act_bwd(x, gx, pre_act, SLOPE)
        if ctx.needs_input_grad[1] or (has_b and ctx.needs_input_grad[2]):
            gw, gb = ops.check_conv2d_wgrad(x, g, tuple(w.shape), stride=stride, pad=pad, pre_act=pre_act, slope=SLOPE,
                                            transposed=transposed, want_bias=has_b)
        return gx, gw, gb, None, None, None, None


class _CheckBN(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, gamma, beta, bn, training):
        y = ops.check_batchnorm(x, gamma, beta, bn.running_mean, bn.running_var, training, eps=BN_EPS, momentum=BN_MOMENTUM)
        if training:
            bn.num_batches_tracked.add_(1)
        ctx.save_for_backward(x, gamma)
        ctx.training = training
        return y

    @staticmethod
    def backward(ctx, g):
        if not ctx.training:
            raise RuntimeError("pai_b200 check path: BatchNorm backward is implemented for train mode (batch statistics)")
        x, gamma = ctx.saved_tensors
        dx, dgamma, dbeta = ops.check_batchnorm_bwd(x, g.contiguous().float(), gamma, eps=BN_EPS)
        return dx, dgamma, dbeta, None, None


class _CheckAct(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, act):
        ctx.save_for_backward(x)
        ctx.act = act
        return ops.check_act(x, act)

    @staticmethod
    def backward(ctx, g):
        (x,) = ctx.saved_tensors
        return ops.check_act_bwd(x, g.contiguous().float(), ctx.act, SLOPE), None


def _check_bn(v, bn, training):
    if bn is None:
        return v
    return _CheckBN.apply(v, bn.weight, bn.bias, bn, training)


def unet_forward_check(spec: "UnetSpec", x: torch.Tensor, training: bool) -> torch.Tensor:
    """``Unet.forward`` (models/pix2pix.py:198-216) layer by layer on the fp32 check kernels (differentiable: every
    node has an exact fp32 backward, so ``loss.backward()`` under ``check_path()`` yields check-path gradients)."""
    if training and any(p > 0 for p in spec.dec_dropout):
        raise RuntimeError("pai_b200: the fp32 check path has no Dropout2d (it is a deterministic forward check)")
    L = spec.levels
    skips = []
    v = x.contiguous().float()
    for i in range(L):
        conv = spec.enc_convs[i]
        v = _CheckConv.apply(v, conv.weight, conv.bias, 2, 1, ACT_NONE if i == 0 else ACT_LEAKY, False)
        v = _check_bn(v, spec.enc_bns[i], training)
        skips.append(v)
    for j in range(L):
        conv = spec.dec_convs[j]
        if j > 0:
            v = torch.cat([v, skips[L - 1 - j]], dim=1)            # models/pix2pix.py:212
        # every DecoderBlock starts with a ReLU; the last decoder is a bare ConvTranspose2d (:185-193)
        v = _CheckConv.apply(v, conv.weight, conv.bias, 2, 1, ACT_RELU if j < L - 1 else ACT_NONE, True)
        v = _check_bn(v, spec.dec_bns[j], training)
    return _CheckAct.apply(v, ACT_TANH)


def disc_forward_check(spec: "DiscSpec", x: torch.Tensor, y: torch.Tensor) -> torch.Tensor:
    """``Discriminator.forward`` (models/wrapper.py:236-238): conv -> LeakyReLU blocks, bias-free stride-1 head."""
    v = torch.cat([x.float(), y.float()], dim=1).contiguous()
    K = len(spec.convs)
    for k, conv in enumerate(spec.convs):
        head = k == K - 1
        v = _CheckConv.apply(v, conv.weight, conv.bias, 1 if head else 2, 1, ACT_NONE if k == 0 else ACT_LEAKY, False)
    return v


# ------------------------------------------------------------------------------------------ generator
class UnetSpec:
    """Shapes + parameter holders of a reference-layout Unet (built by models/pix2pix.py:Unet)."""

    def __init__(self, enc_convs, enc_bns, dec_convs, dec_bns, dec_dropout=None):
        # dec_dropout[j]: Dropout2d probability after decoder j's BatchNorm (models/pix2pix.py:107,176-183)
        self.dec_dropout = list(dec_dropout) if dec_dropout is not None else [0.0] * len(dec_convs)
        self.enc_convs, self.enc_bns = enc_convs, [None if b is None else BNState(b) for b in enc_bns]
        self.dec_convs, self.dec_bns = dec_convs, [None if b is None else BNState(b) for b in dec_bns]
        self.levels = len(enc_convs)
        self.enc_ch = [c.weight.shape[0] for c in enc_convs]
        self.in_ch = enc_convs[0].weight.shape[1]
        self.out_ch = dec_convs[-1].weight.shape[1]
        self.dec_out = [c.weight.shape[1] for c in dec_convs]
        if not (1 <= self.in_ch <= CARRIER and 1 <= self.out_ch <= CARRIER):
            raise RuntimeError(f"pai_b200: in / out channels must be in 1..{CARRIER}; got {self.in_ch}/{self.out_ch}. "
                               "No fallback exists.")
        for c in self.enc_ch + self.dec_out[:-1]:
            if c % 64:
                raise RuntimeError(f"pai_b200: channel counts must be multiples of 64 (got {c})")

    def params(self) -> List[torch.Tensor]:
        ps = []
        for conv, bn in list(zip(self.enc_convs, self.enc_bns)) + list(zip(self.dec_convs, self.dec_bns)):
            ps += [conv.weight, conv.bias]
            if bn is not None:
                ps += [bn.weight, bn.bias]
        return ps


class _Saved:
    pass


def unet_forward(spec: UnetSpec, x: torch.Tensor, training: bool, save: bool):
    """x: [N, 1, H, W] fp32 (cuda) -> (y [N, 1, H, W] fp32 in (-1, 1), saved-or-None)."""
    L = spec.levels
    n, _, h, w = x.shape
    if not x.is_cuda or not spec.enc_convs[0].weight.is_cuda:
        raise RuntimeError("pai_b200: the generator runs on the B200 kernels only: input and parameters must be CUDA tensors "
                           "(there is no CPU or PyTorch fallback)")
    if h % (1 << L) or w % (1 << L):
        raise RuntimeError(f"pai_b200: input {h}x{w} must be divisible by 2^{L}")
    dev = x.device
    x = x.contiguous().float()
    if x.shape[1] != spec.in_ch:
        raise RuntimeError(f"pai_b200: the generator takes {spec.in_ch}-channel images, got {x.shape[1]}")
    plane = x.view(n, h, w) if spec.in_ch == 1 else None
    xc = None if spec.in_ch == 1 else _carrier(x)        # multi-channel input: zero-padded 64-channel carrier
    ch = spec.enc_ch
    hs = [h >> (i + 1) for i in range(L)]
    ws = [w >> (i + 1) for i in range(L)]
    s = _Saved()
    counters = []
    # decoder j (>=1) reads cat[j]: [N, hs[L-1-j], ws[L-1-j], 2*C] with C = ch[L-1-j]
    cat = [None] + [_bf16(n, hs[L - 1 - j], ws[L - 1 - j], 2 * ch[L - 1 - j], device=dev) for j in range(1, L)]
    a_in = [None] * (L + 1)                    # a_in[i]: activated input of encoder i (i >= 1)
    raw_e, ss_e = [None] * L, [None] * L
    # ---- encoder 0 (no activation before, no BN after): skip = raw output
    c0 = ch[0]
    a_in[1] = _bf16(n, hs[0], ws[0], c0, device=dev)
    conv0 = spec.enc_convs[0]
    # The last decoder is a bare ConvTranspose2d (models/pix2pix.py:185-193): no ReLU in front of it, so
    # its concat buffer cat[L-1] holds UN-activated values; every other decoder starts with a ReLU.
    # enc0 (1 input channel) = im2col of the plane + one tensor-core GEMM with two fused outputs
    xcol = None
    if xc is not None:
        ops.conv4x4_fprop_dual(xc, _carrier_in_pack(conv0.weight), c0, conv0.bias.detach(), a_in[1], ACT_LEAKY,
                               cat[L - 1][..., c0:], ACT_NONE, slope=SLOPE)
    elif THIN_DIRECT and c0 <= 256:
        # one pass: the 16-tap rows are built in shared memory, both consumers are written by the same epilogue
        ops.thin_conv_fprop([plane], _thin_in_pack(conv0.weight), c0, conv0.bias.detach(), a_in[1], ACT_LEAKY,
                            cat[L - 1][..., c0:], ACT_NONE, slope=SLOPE)
    else:
        xcol = ops.im2col4x4([plane], hs[0], ws[0], stride=2)
        ops.pointwise_gemm(xcol, _thin_in_pack(conv0.weight), c0, bias=conv0.bias.detach(), act=ACT_LEAKY, slope=SLOPE,
                           out=a_in[1], out2=cat[L - 1][..., c0:], act2=ACT_NONE, k_valid=16)
    # ---- encoders 1..L-1
    for i in range(1, L):
        conv, bn = spec.enc_convs[i], spec.enc_bns[i]
        if i < L - 1:
            part = None
            if (bn is not None and not training and not save and FOLD_EVAL_BN and ops.bn_fusable(n * hs[i] * ws[i], ch[i])):
                # eval mode (report.py): BatchNorm folded into the weights, both consumers written by the GEMM epilogue --
                # no raw tensor, no BatchNorm kernels
                wp, bf = _folded("fold_f", conv, bn, transposed=False)
                a_in[i + 1] = _bf16(n, hs[i], ws[i], ch[i], device=dev)
                ops.conv4x4_fprop_dual(a_in[i], wp, ch[i], bf, a_in[i + 1], ACT_LEAKY, cat[L - 1 - i][..., ch[i]:], ACT_RELU,
                                       slope=SLOPE)
                continue
            if bn is not None and training and FUSE_BN_STATS and ops.bn_fusable(n * hs[i] * ws[i], ch[i]):
                # BatchNorm statistics straight from the GEMM epilogue: no separate pass over the raw output
                raw, part = ops.conv4x4_fprop_bnstats(a_in[i], _fprop_pack(conv.weight), ch[i], bias=conv.bias.detach())
            else:
                raw = ops.conv4x4_fprop(a_in[i], _fprop_pack(conv.weight), ch[i], stride=2, bias=conv.bias.detach())
            a_in[i + 1] = _bf16(n, hs[i], ws[i], ch[i], device=dev)
            if bn is not None:
                ss = _batchnorm_act(raw, bn, training, counters, part, a_in[i + 1], ACT_LEAKY, cat[L - 1 - i][..., ch[i]:],
                                    ACT_RELU)
            else:
                ss = None
                ops.bn_apply_act(raw, None, a_in[i + 1], ACT_LEAKY, cat[L - 1 - i][..., ch[i]:], ACT_RELU, slope=SLOPE)
            raw_e[i], ss_e[i] = raw, ss
        else:
            # bottleneck: Identity norm (models/pix2pix.py:157), only consumer is decoder 0's ReLU
            dec_in0 = ops.conv4x4_fprop(a_in[i], _fprop_pack(conv.weight), ch[i], stride=2, bias=conv.bias.detach(),
                                        act=ACT_RELU)
    # ---- decoders 0..L-2 (BN), L-1 (Tanh)
    raw_d, ss_d = [None] * L, [None] * L
    drop_masks = [None] * L
    d_in = dec_in0
    for j in range(L - 1):
        conv, bn = spec.dec_convs[j], spec.dec_bns[j]
        co = spec.dec_out[j]
        part = None
        hj, wj = d_in.shape[1], d_in.shape[2]
        if not training and not save and FOLD_EVAL_BN and ops.bn_fusable(4 * n * hj * wj, co):
            wp, bf = _folded("fold_f", conv, bn, transposed=True)
            ops.convT4x4s2_fprop(d_in, wp, co, bias=bf, act=ACT_RELU if j + 1 < L - 1 else ACT_NONE, out=cat[j + 1][..., :co])
            d_in = cat[j + 1]
            continue
        if training and FUSE_BN_STATS and ops.bn_fusable(4 * n * hj * wj, co):
            raw, part = ops.convT4x4s2_fprop_bnstats(d_in, _fpropT_pack(conv.weight), co, bias=conv.bias.detach())
        else:
            raw = ops.convT4x4s2_fprop(d_in, _fpropT_pack(conv.weight), co, bias=conv.bias.detach())
        slot = cat[j + 1][..., :co]
        if training and spec.dec_dropout[j] > 0:
            # Dropout2d sits between the BatchNorm and the next block's ReLU; the mask is non-negative, so it commutes
            # with the ReLU already applied: relu(mask * z) == mask * relu(z)
            drop_masks[j] = ops.dropout2d_mask(n, co, spec.dec_dropout[j], dev)
        ss = _batchnorm_act(raw, bn, training, counters, part, slot, ACT_RELU if j + 1 < L - 1 else ACT_NONE,
                            mask=drop_masks[j])
        raw_d[j], ss_d[j] = raw, ss
        d_in = cat[j + 1]
    last = spec.dec_convs[L - 1]
    # last decoder (1 output channel): 16 per-tap partial products per input pixel (GEMM, the wide input is
    # read once) + col2im with bias and Tanh
    if spec.out_ch != 1:
        # multi-channel output: ConvT into a 64-channel fp32 carrier (+bias, Tanh; the padding channels give tanh(0) = 0)
        yc = ops.convT4x4s2_fprop(d_in, _carrier_out_pack(last.weight), CARRIER, bias=_carrier_bias(last.bias), act=ACT_TANH,
                                  out_f32=True)
        y = yc[..., :spec.out_ch].permute(0, 3, 1, 2).contiguous()
    elif THIN_DIRECT and ops.thin_plane_ok(d_in):
        y = ops.thin_convT_plane(d_in, _thin_out_fprop_pack(last.weight), last.bias.detach(), ACT_TANH).view(n, 1, h, w)
    else:
        part = ops.pointwise_gemm(d_in, _thin_out_fprop_pack(last.weight), 16, out_f32=True)
        y = ops.col2im4x4s2(part, last.bias.detach(), ACT_TANH).view(n, 1, h, w)
    if counters:
        torch._foreach_add_(counters, 1)
    if not save:
        return y, None
    s.xcol = xcol
    s.drop_masks = drop_masks
    s.plane, s.cat, s.a_in, s.raw_e, s.ss_e, s.raw_d, s.ss_d, s.dec_in0, s.y = plane, cat, a_in, raw_e, ss_e, raw_d, ss_d, dec_in0, y
    s.xc = xc
    return y, s


def unet_backward(spec: UnetSpec, s: _Saved, grad_y: torch.Tensor):
    """-> list of gradients aligned with ``spec.params()`` (reference layouts, fp32)."""
    L = spec.levels
    ch = spec.enc_ch
    y = s.y
    n, _, h, w = y.shape
    dev = y.device
    g_pre = (grad_y.float() * (1.0 - y * y)).contiguous()                       # through Tanh
    grads = {}
    # ---- last decoder: ConvT(2*c0 -> out_ch)
    last = spec.dec_convs[L - 1]
    cin_last = last.weight.shape[0]
    if spec.out_ch != 1:
        gc = _carrier(g_pre)
        dwl = ops.wgrad_finish(ops.convT4x4s2_wgrad(s.cat[L - 1], gc))             # [cin, 64, 4, 4]
        grads[(1, L - 1)] = (dwl[:, :spec.out_ch].contiguous(), g_pre.sum((0, 2, 3)))
        dcat = ops.conv4x4_fprop(gc, _carrier_out_dgrad_pack(last.weight), cin_last, stride=2)
    else:
        g_pre = g_pre.view(n, h, w)
        gcol = None
        if THIN_DIRECT and ops.thin_wgrad_ok(s.cat[L - 1], [g_pre]):
            dw = ops.thin_conv_wgrad(s.cat[L - 1], [g_pre])                      # [cin, 16]
        else:
            gcol = ops.im2col4x4([g_pre], h // 2, w // 2, stride=2)              # [N, h/2, w/2, 64], 16 taps of g
            dw = ops.pointwise_wgrad(s.cat[L - 1], gcol)                         # [cin, 64]
        grads[(1, L - 1)] = (dw[:, :16].reshape(cin_last, 1, 4, 4), g_pre.sum().reshape(1))
        if THIN_DIRECT and cin_last <= 256:
            dcat = _bf16(n, h // 2, w // 2, cin_last, device=dev)
            ops.thin_conv_fprop([g_pre], _thin_out_dgrad_pack(last.weight), cin_last, None, dcat, ACT_NONE)
        else:
            if gcol is None:
                gcol = ops.im2col4x4([g_pre], h // 2, w // 2, stride=2)
            dcat = ops.pointwise_gemm(gcol, _thin_out_dgrad_pack(last.weight), cin_last, k_valid=16)
    # ---- decoders L-2 .. 0
    dskip = [None] * L                          # dskip[i]: grad w.r.t. relu(skip_i) (second half of dcat)
    for j in range(L - 2, -1, -1):
        conv, bn = spec.dec_convs[j], spec.dec_bns[j]
        co = spec.dec_out[j]
        enc_i = L - 2 - j                       # encoder whose skip sits in cat[j+1]
        dskip[enc_i] = dcat[..., co:]
        g1 = dcat[..., :co]
        raw, ss = s.raw_d[j], s.ss_d[j]
        act_out = ACT_RELU if j + 1 < L - 1 else ACT_NONE     # consumer of this decoder's output
        d_raw = _bf16(*raw.shape, device=dev)
        if ops.bn_small_ok(raw, 2):
            # Dropout2d backward + BatchNorm backward (reduce + apply) in one launch
            sums = ops.bn_small_bwd(raw, ss, g1, act_out, None, ACT_NONE, bn.weight.detach(), d_raw, slope=SLOPE,
                                    mask=s.drop_masks[j])
        else:
            if s.drop_masks[j] is not None:
                ops.scale_channels(g1, s.drop_masks[j], out=g1)      # Dropout2d backward, in place on the fresh dgrad
            sums = ops.bn_bwd_reduce(raw, ss, g1, act_out)
            ops.bn_bwd_apply(raw, ss, g1, act_out, None, ACT_NONE, sums, bn.weight.detach(), d_raw)
        d_in = s.cat[j] if j > 0 else s.dec_in0
        cin = conv.weight.shape[0]
        gw = ops.wgrad_finish(ops.convT4x4s2_wgrad(d_in, d_raw))   # [cin, co, 4, 4]
        dp.allreduce_async(gw)                    # data-parallel: the exchange overlaps the rest of the backward
        grads[(1, j)] = (gw, ops.zeros_f32(co, device=dev), sums[co:], sums[:co])
        dcat = ops.conv4x4_fprop(d_raw, _dgradT_pack(conv.weight), cin, stride=2)   # grad w.r.t. decoder input
    # ---- bottleneck encoder L-1: dec_in0 = relu(conv + bias)
    i = L - 1
    conv = spec.enc_convs[i]
    d_raw = _bf16(*s.dec_in0.shape, device=dev)
    sums = ops.act_bwd(s.dec_in0, dcat, ACT_RELU, None, ACT_NONE, d_raw)
    gw = ops.wgrad_finish(ops.conv4x4_wgrad(s.a_in[i], d_raw, stride=2))
    dp.allreduce_async(gw)
    grads[(0, i)] = (gw, sums[:ch[i]].clone())
    d_a = ops.convT4x4s2_fprop(d_raw, _dgrad_pack(conv.weight), ch[i - 1])
    # ---- encoders L-2 .. 1
    for i in range(L - 2, 0, -1):
        conv, bn = spec.enc_convs[i], spec.enc_bns[i]
        raw, ss = s.raw_e[i], s.ss_e[i]
        d_raw = _bf16(*raw.shape, device=dev)
        if bn is not None and ops.bn_small_ok(raw, 3):
            sums = ops.bn_small_bwd(raw, ss, d_a, ACT_LEAKY, dskip[i], ACT_RELU, bn.weight.detach(), d_raw, slope=SLOPE)
        else:
            sums = ops.bn_bwd_reduce(raw, ss, d_a, ACT_LEAKY, dskip[i], ACT_RELU, slope=SLOPE)
            ops.bn_bwd_apply(raw, ss, d_a, ACT_LEAKY, dskip[i], ACT_RELU, sums, None if bn is None else bn.weight.detach(),
                             d_raw, slope=SLOPE)
        gw = ops.wgrad_finish(ops.conv4x4_wgrad(s.a_in[i], d_raw, stride=2))
        dp.allreduce_async(gw)
        if bn is not None:
            grads[(0, i)] = (gw, ops.zeros_f32(ch[i], device=dev), sums[ch[i]:], sums[:ch[i]])
        else:
            grads[(0, i)] = (gw, sums[:ch[i]].clone())
        d_a = ops.convT4x4s2_fprop(d_raw, _dgrad_pack(conv.weight), ch[i - 1])
    # ---- encoder 0: a_in[1] = lrelu(e0) has the sign of e0, so it doubles as the activation mask
    c0 = ch[0]
    d_raw = _bf16(*s.a_in[1].shape, device=dev)
    sums = ops.act_bwd(s.a_in[1], d_a, ACT_LEAKY, dskip[0], ACT_NONE, d_raw, slope=SLOPE)
    if s.xc is not None:
        dw0 = ops.wgrad_finish(ops.conv4x4_wgrad(s.xc, d_raw, stride=2))         # [c0, 64, 4, 4]
        grads[(0, 0)] = (dw0[:, :spec.in_ch].contiguous(), sums[:c0].clone())
    else:
        if THIN_DIRECT and ops.thin_wgrad_ok(d_raw, [s.plane]):
            dw0 = ops.thin_conv_wgrad(d_raw, [s.plane])                          # [c0, 16]
        else:
            xcol = s.xcol if s.xcol is not None else ops.im2col4x4([s.plane], h // 2, w // 2, stride=2)
            dw0 = ops.pointwise_wgrad(d_raw, xcol)                               # [c0, 64]
        grads[(0, 0)] = (dw0[:, :16].reshape(c0, 1, 4, 4), sums[:c0].clone())
    out = []
    for i in range(L):
        out += list(grads[(0, i)])
    for j in range(L):
        out += list(grads[(1, j)])
    dp.finish_async()
    return out


class UnetFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, spec: UnetSpec, training: bool, x: torch.Tensor, *params):
        need = any(ctx.needs_input_grad[3:])
        if ctx.needs_input_grad[2]:
            raise RuntimeError("pai_b200: the fused generator node has no gradient w.r.t. its input image "
                               "(the reference never asks for one, models/wrapper.py:117-162); detach x")
        y, saved = unet_forward(spec, x, training, save=need)
        ctx.spec, ctx.saved, ctx.training = spec, saved, training
        return y

    @staticmethod
    def backward(ctx, grad_y):
        if ctx.saved is None:
            raise RuntimeError("pai_b200: generator backward requested but the forward ran without a graph")
        if not ctx.training and any(b is not None for b in ctx.spec.enc_bns + ctx.spec.dec_bns):
            # the fused backward implements the TRAIN-mode BatchNorm backward (batch-statistic terms); with running
            # statistics the gradient is a different formula -- refuse instead of returning wrong numbers
            raise RuntimeError("pai_b200: gradients through an eval-mode BatchNorm generator are not implemented "
                               "(the reference only differentiates in train mode, models/wrapper.py:117-162)")
        grads = unet_backward(ctx.spec, ctx.saved, grad_y)
        ctx.saved = None
        need = ctx.needs_input_grad[3:]
        return (None, None, None) + tuple(g if nd else None for g, nd in zip(grads, need))


# ------------------------------------------------------------------------------------------ discriminator
class DiscSpec:
    def __init__(self, convs):
        self.convs = convs                       # 4 stride-2 convs (bias) + final stride-1 conv (no bias)
        self.ch = [c.weight.shape[0] for c in convs]
        cin0 = convs[0].weight.shape[1]
        if cin0 % 2 or not (2 <= cin0 <= CARRIER):
            raise RuntimeError("pai_b200: the PatchGAN's first conv reads cat([x, y]) of two images with the same number "
                               f"of channels (at most {CARRIER} together); it has {cin0} inputs")
        self.img_ch = cin0 // 2                  # 1: thin-layer kernels; more: 64-channel carrier (reference default 3)
        if self.ch[-1] != 1 or convs[-1].bias is not None:
            raise RuntimeError("pai_b200: unexpected PatchGAN head")

    def params(self):
        ps = []
        for c in self.convs[:-1]:
            ps += [c.weight, c.bias]
        ps.append(self.convs[-1].weight)
        return ps


def disc_forward(spec: DiscSpec, x: torch.Tensor, y: torch.Tensor, save: bool):
    n, _, h, w = x.shape
    dev = x.device
    if not (x.is_cuda and y.is_cuda and spec.convs[0].weight.is_cuda):
        raise RuntimeError("pai_b200: the PatchGAN runs on the B200 kernels only: inputs and parameters must be CUDA tensors "
                           "(there is no CPU or PyTorch fallback)")
    if x.shape[1] != spec.img_ch or y.shape[1] != spec.img_ch:
        raise RuntimeError(f"pai_b200: this PatchGAN takes two {spec.img_ch}-channel images, got {x.shape[1]} and {y.shape[1]}")
    c0 = spec.convs[0]
    xycol = xyc = px = py = None
    if spec.img_ch == 1:
        px = x.contiguous().float().view(n, h, w)
        py = y.contiguous().float().view(n, h, w)                                # cat([x, y]) is never materialised
    if spec.img_ch != 1:
        xyc = _carrier(x.float(), y.float())
        hcur = ops.conv4x4_fprop(xyc, _carrier_in_pack(c0.weight), spec.ch[0], stride=2, bias=c0.bias.detach(), act=ACT_LEAKY,
                                 slope=SLOPE)
    elif THIN_DIRECT and spec.ch[0] <= 256:
        hcur = _bf16(n, h // 2, w // 2, spec.ch[0], device=dev)
        ops.thin_conv_fprop([px, py], _thin_in_pack(c0.weight), spec.ch[0], c0.bias.detach(), hcur, ACT_LEAKY, slope=SLOPE)
    else:
        xycol = ops.im2col4x4([px, py], h // 2, w // 2, stride=2)
        hcur = ops.pointwise_gemm(xycol, _thin_in_pack(c0.weight), spec.ch[0], bias=c0.bias.detach(), act=ACT_LEAKY,
                                  slope=SLOPE, k_valid=32)
    hs = [hcur]
    for k in range(1, len(spec.convs) - 1):
        c = spec.convs[k]
        hcur = ops.conv4x4_fprop(hcur, _fprop_pack(c.weight), spec.ch[k], stride=2, bias=c.bias.detach(),
                                 act=ACT_LEAKY, slope=SLOPE)
        hs.append(hcur)
    head = spec.convs[-1]
    if THIN_DIRECT:
        # 512 -> 1 channels: ONE GEMM over the input gives the 16 per-tap partial products of every pixel, a small gather
        # sums the 4x4 window (instead of 16 shifted tensor-core passes over the same 16 MB for a 1-column output)
        part = ops.pointwise_gemm(hcur, _head_fprop_pack(head.weight), 16, out_f32=True)
        logits = ops.col2im4x4s1(part)
        nb, lh, lw = logits.shape
    else:
        logits = ops.conv4x4_fprop(hcur, _fprop_pack(head.weight), 1, stride=1, out_f32=True)
        nb, lh, lw, _ = logits.shape
    logits = logits.view(nb, 1, lh, lw)
    if not save:
        return logits, None
    s = _Saved()
    s.px, s.py, s.hs, s.xycol, s.xyc, s.hw = px, py, hs, xycol, xyc, (h, w)
    return logits, s


def disc_backward(spec: DiscSpec, s: _Saved, g_logits: torch.Tensor, need_params: bool, need_y: bool):
    dev = g_logits.device
    n, _, lh, lw = g_logits.shape
    g = g_logits.contiguous().float().view(n, lh, lw)
    K = len(spec.convs)
    head = spec.convs[-1]
    h_last = s.hs[-1]
    c_last = h_last.shape[3]
    grads = [None] * (2 * (K - 1) + 1)
    # head (Conv4x4 s1 p1, 512 -> 1): its backward is 1 channel wide on the gradient side, so -- like dec7 -- the 16
    # shifted copies of the logit gradient become the K = 16 operand of two tensor-core GEMMs
    gcol = ops.im2col4x4([g], h_last.shape[1], h_last.shape[2], stride=1, flip=True)    # [N, 16, 16, 64 (16 used)]
    if need_params:
        dwh = ops.pointwise_wgrad(h_last, gcol)[:, :16]                             # [c, 16]
        grads[-1] = dwh.reshape(1, c_last, 4, 4)
    dh = ops.pointwise_gemm(gcol, _head_dgrad_pack(head.weight), c_last, k_valid=16)
    fused = None                                    # (d_pre, bias-gradient column sums) made by the previous dgrad GEMM
    for k in range(K - 2, -1, -1):
        conv = spec.convs[k]
        hk = s.hs[k]                                # lrelu output: same sign as the pre-activation
        ck = hk.shape[3]
        if fused is not None:
            d_pre, sums = fused
            fused = None
        else:
            d_pre = _bf16(*hk.shape, device=dev)
            sums = ops.act_bwd(hk, dh, ACT_LEAKY, None, ACT_NONE, d_pre, slope=SLOPE)
        if k > 0:
            if need_params:
                grads[2 * k] = ops.wgrad_finish(ops.conv4x4_wgrad(s.hs[k - 1], d_pre, stride=2))
                dp.allreduce_async(grads[2 * k])
                grads[2 * k + 1] = sums[:ck].clone()
            cprev = s.hs[k - 1].shape[3]
            if FUSE_ACT_BWD and ops.bn_fusable(s.hs[k - 1].numel() // cprev, cprev):
                # the LeakyReLU backward of block k-1 (and its bias gradient) rides on this data-gradient GEMM's epilogue
                d_next, part = ops.conv4x4_dgrad_act(d_pre, _dgrad_pack(conv.weight), cprev, s.hs[k - 1], slope=SLOPE,
                                                     want_colsum=need_params)
                fused = (d_next, part.sum(0) if part is not None else None)
            else:
                dh = ops.convT4x4s2_fprop(d_pre, _dgrad_pack(conv.weight), cprev)
        elif s.xyc is not None:
            h, w = s.hw
            if need_params:
                dw0 = ops.wgrad_finish(ops.conv4x4_wgrad(s.xyc, d_pre, stride=2))   # [c, 64, 4, 4]
                grads[0] = dw0[:, :2 * spec.img_ch].contiguous()
                grads[1] = sums[:ck].clone()
            gy = None
            if need_y:
                gyc = ops.convT4x4s2_fprop(d_pre, _carrier_in_dgrad_pack(conv.weight), CARRIER, out_f32=True)
                gy = gyc[..., spec.img_ch:2 * spec.img_ch].permute(0, 3, 1, 2).contiguous()
        else:
            h, w = s.hw
            if need_params:
                if THIN_DIRECT and ops.thin_wgrad_ok(d_pre, [s.px, s.py]):
                    dw0 = ops.thin_conv_wgrad(d_pre, [s.px, s.py])               # [c, 32], column = tap*2 + j
                else:
                    xycol = s.xycol if s.xycol is not None else ops.im2col4x4([s.px, s.py], h // 2, w // 2, stride=2)
                    dw0 = ops.pointwise_wgrad(d_pre, xycol)                      # [c, 64]
                grads[0] = dw0[:, :32].reshape(ck, 4, 4, 2).permute(0, 3, 1, 2)
                grads[1] = sums[:ck].clone()
            gy = None
            if need_y:
                if THIN_DIRECT and ops.thin_plane_ok(d_pre):
                    gy = ops.thin_convT_plane(d_pre, _thin_in_dgrad_pack(conv.weight, 1)).view(n, 1, h, w)
                else:
                    part = ops.pointwise_gemm(d_pre, _thin_in_dgrad_pack(conv.weight, 1), 16, out_f32=True)
                    gy = ops.col2im4x4s2(part).view(n, 1, h, w)
    dp.finish_async()
    return grads, gy


class DiscFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, spec: DiscSpec, x, y, *params):
        need_params = any(ctx.needs_input_grad[3:])
        need_y = ctx.needs_input_grad[2]
        if ctx.needs_input_grad[1]:
            raise RuntimeError("pai_b200: the fused PatchGAN node has no gradient w.r.t. its first (conditioning) input "
                               "x (models/wrapper.py:126-128,147 only differentiate w.r.t. the prediction y); detach x")
        logits, saved = disc_forward(spec, x, y, save=need_params or need_y)
        ctx.spec, ctx.saved, ctx.need_params, ctx.need_y = spec, saved, need_params, need_y
        return logits

    @staticmethod
    def backward(ctx, g_logits):
        grads, gy = disc_backward(ctx.spec, ctx.saved, g_logits, ctx.need_params, ctx.need_y)
        ctx.saved = None
        need = ctx.needs_input_grad[3:]
        return (None, None, gy) + tuple(g if nd else None for g, nd in zip(grads, need))
