"""GPU checks of the Residual / Attention / Trans U-Nets on 1-4 image planes (RGB, RGBA, ...).

1. Kernels and autograd nodes of the first and last layers against fp64 ``F.conv2d`` / ``F.conv_transpose2d`` on the
   same bf16-rounded operands; with one plane, each multi-plane entry point against its 1-plane twin.
2. Lifted reference parity: a C-channel model whose first layer is ``W[:, j] = a_j W1`` (sum a_j = 1), fed
   ``x_j = x + r_j`` (sum a_j r_j = 0), with every output channel a copy of the 1-channel head, IS the 1-channel model of
   ``tests/golden/variants_ref.npz`` (fixtures of the unmodified reference) and is held to that test's bounds.
3. The reference's default constructors (3 channels, GAN loss with the 3-channel PatchGAN, dropout 0.5) train eagerly
   and as a step graph.  ``TransUnetGAN()``'s own default bottleneck (channel_mults (1, 2, 4, 8), patch 16) has a
   131 072-wide token (a 17 G-parameter patch embedding), so the Trans U-Net runs with the small bottleneck of the
   parity fixtures (channel_mults (1, 2, 2), patch 4) and every other default.
4. Channel counts the kernels do not take raise."""
import importlib
import os

import numpy as np
import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

import pix2pix_port as port
from test_variants_gpu import CASES, _build

pytestmark = pytest.mark.gpu
torch.backends.cudnn.allow_tf32 = False
torch.backends.cuda.matmul.allow_tf32 = False


def _bf(t):
    return t.bfloat16().float()


def _gen(seed):
    return torch.Generator(device="cuda").manual_seed(seed)


# ------------------------------------------------------------------------------------------------ 1. kernels / nodes
def _bound_bf16(ref):
    return 1e-2 * max(1.0, ref.abs().max().item())


def _bound_f32(ref):
    return 1e-3 * ref.abs().max().item()


@pytest.mark.parametrize("np_", [1, 2, 3, 4])
@pytest.mark.parametrize("k", [1, 3])
@pytest.mark.parametrize("flip,bias_act", [(False, True), (False, False), (True, False)])
def test_plane_kernels(np_, k, flip, bias_act):
    """pai_conv_planes_to_wide (forward / flipped = summed data gradient), pai_conv_wide_to_planes and
    pai_conv_planes_wide_wgrad on odd-sized images; fp32 arithmetic, bf16 or fp32 outputs."""
    from pai_b200 import ops
    n, h, w, c, pad = 2, 17, 23, 64, k // 2
    g = _gen(10 * np_ + k)
    planes = _bf(torch.randn(n, np_, h, w, generator=g, device="cuda"))
    wt = _bf(torch.randn(c, np_, k, k, generator=g, device="cuda") * 0.3)
    bias = torch.randn(c, generator=g, device="cuda") if bias_act else None
    act = ops.ACT_LEAKY if bias_act else ops.ACT_NONE
    wk = wt.flip(2, 3) if flip else wt                       # flip = correlation with the point-mirrored taps
    ref = F.conv2d(planes.double(), wk.double(), None if bias is None else bias.double(), padding=pad)
    if bias_act:
        ref = F.leaky_relu(ref, 0.2)
    y = ops.conv_planes_to_wide(planes, wt.reshape(c, -1), bias, k, pad, act, flip=flip)
    err = (y.double().permute(0, 3, 1, 2) - ref).abs().max().item()
    assert err < _bound_bf16(ref), err

    x = torch.randn(n, h, w, c, generator=g, device="cuda").bfloat16()
    wo = _bf(torch.randn(np_, c, k, k, generator=g, device="cuda") * 0.05)
    bo = torch.randn(np_, generator=g, device="cuda") if bias_act else None
    ref = F.conv2d(x.double().permute(0, 3, 1, 2), wo.double(), None if bo is None else bo.double(), padding=pad)
    if bias_act:
        ref = torch.tanh(ref)
    yo = ops.conv_wide_to_planes(x, wo.permute(0, 2, 3, 1).reshape(np_, k * k, c).contiguous(), bo, k, pad,
                                 ops.ACT_TANH if bias_act else ops.ACT_NONE)
    assert yo.shape == (n, np_, h, w)
    err = (yo.double() - ref).abs().max().item()
    assert err < _bound_f32(ref), err

    # weight gradient: dw[c][j][t] = sum_p x[p, c] * plane_j[p + off_t]  (off_t negated when flip)
    dw = ops.conv_planes_wide_wgrad(planes, x, k, pad, flip=flip)
    wr = torch.zeros(c, np_, k, k, dtype=torch.float64, device="cuda", requires_grad=True)
    F.conv2d(planes.double(), wr.flip(2, 3) if flip else wr, None, padding=pad).backward(x.double().permute(0, 3, 1, 2))
    ref = wr.grad
    err = (dw.double().view(c, np_, k, k) - ref).abs().max().item()
    assert err < _bound_f32(ref), err

    if np_ == 1:    # the 1-plane twins: same kernels, same FMAs in the same order
        y1 = ops.conv_plane_to_wide(planes[:, 0].contiguous(), wt.reshape(c, -1), bias, k, pad, act, flip=flip)
        assert torch.equal(y1, y)
        yo1 = ops.conv_wide_to_plane(x, wo.permute(0, 2, 3, 1).reshape(k * k, c).contiguous(), bo, k, pad,
                                     ops.ACT_TANH if bias_act else ops.ACT_NONE)
        assert torch.equal(yo1, yo[:, 0])
        # the weight gradients are block partial sums added with float atomics, whose order varies from call to call,
        # for the 1-plane twin as for the new entry point
        dw1 = ops.conv_plane_wide_wgrad(planes[:, 0].contiguous(), x, k, pad, flip=flip)
        assert (dw1 - dw.view(c, k * k)).abs().max().item() <= 1e-5 * dw1.abs().max().item()


@pytest.mark.parametrize("np_", [1, 2, 3, 4])
def test_im2col_col2im_planes(np_):
    """pai_im2col4x4_planes (tap-major) and pai_col2im4x4s2_planes (plane-major, per-plane bias, Tanh)."""
    from pai_b200 import ops
    n, h, w = 2, 18, 26
    g = _gen(100 + np_)
    planes = torch.randn(n, np_, h, w, generator=g, device="cuda")
    for stride, flip, oh, ow in ((2, False, h // 2, w // 2), (1, True, h - 1, w - 1)):
        col = ops.im2col4x4_planes(planes, oh, ow, stride=stride, flip=flip)
        pad = torch.zeros(n, np_, h + 4, w + 4, device="cuda")
        pad[:, :, 2:2 + h, 2:2 + w] = planes
        for t in range(16):
            ky, kx = divmod(t, 4)
            dy, dx = (1 - ky, 1 - kx) if flip else (ky - 1, kx - 1)
            want = pad[:, :, 2 + dy:2 + dy + stride * oh:stride, 2 + dx:2 + dx + stride * ow:stride]
            got = col[..., t * np_:(t + 1) * np_].permute(0, 3, 1, 2).float()
            assert torch.equal(got, _bf(want)), (stride, t)
        if np_ == 1:
            assert torch.equal(col[..., :16], ops.im2col4x4([planes[:, 0].contiguous()], oh, ow, stride, flip)[..., :16])
    hh, ww = 9, 13
    part = torch.randn(n, hh, ww, 16 * np_, generator=g, device="cuda")
    bias = torch.randn(np_, generator=g, device="cuda")
    y = ops.col2im4x4s2_planes(part, np_, bias, ops.ACT_TANH)
    # col2im of plane-major partials == transposed conv of a one-hot "identity" weight on the partial products
    eye = torch.eye(16 * np_, dtype=torch.float64, device="cuda").view(16 * np_, np_, 4, 4)
    ref = torch.tanh(F.conv_transpose2d(part.double().permute(0, 3, 1, 2), eye, bias.double(), stride=2, padding=1))
    assert (y.double() - ref).abs().max().item() < 1e-5
    if np_ == 1:
        assert torch.equal(y[:, 0], ops.col2im4x4s2(part, bias, ops.ACT_TANH))


@pytest.mark.parametrize("np_", [1, 2, 3, 4])
@pytest.mark.parametrize("k", [1, 3])
def test_plane_nodes_forward_backward(np_, k):
    """The Res / Trans U-Net first and last layer nodes (conv_in_planes, conv_out_planes + Tanh): forward, data
    gradient (last layer) and weight / bias gradients, odd image size."""
    from pai_b200 import layers as L
    n, h, w, c = 2, 15, 21, 64
    g = _gen(200 + 10 * np_ + k)
    torch.manual_seed(np_ * 7 + k)
    cin = nn.Conv2d(np_, c, k, padding=k // 2).cuda()
    cout = nn.Conv2d(c, np_, k, padding=k // 2).cuda()
    with torch.no_grad():
        cin.weight.copy_(_bf(cin.weight))
        cout.weight.copy_(_bf(cout.weight))
    planes = _bf(torch.randn(n, np_, h, w, generator=g, device="cuda"))
    y = L.conv_in_planes(planes, cin)
    wi = cin.weight.detach().double().requires_grad_(True)
    bi = cin.bias.detach().double().requires_grad_(True)
    ref = F.conv2d(planes.double(), wi, bi, padding=k // 2)
    assert (y.double().permute(0, 3, 1, 2) - ref).abs().max().item() < _bound_bf16(ref)
    gy = torch.randn(n, h, w, c, generator=g, device="cuda").bfloat16()
    y.backward(gy)
    ref.backward(gy.double().permute(0, 3, 1, 2))
    assert (cin.weight.grad.double() - wi.grad).abs().max().item() < _bound_f32(wi.grad)
    assert (cin.bias.grad.double() - bi.grad).abs().max().item() < _bound_f32(bi.grad)

    x = torch.randn(n, h, w, c, generator=g, device="cuda").bfloat16().requires_grad_(True)
    out = L.conv_out_planes(x, cout, L.ACT_TANH)
    xr = x.detach().double().permute(0, 3, 1, 2).requires_grad_(True)
    wo = cout.weight.detach().double().requires_grad_(True)
    bo = cout.bias.detach().double().requires_grad_(True)
    ref = torch.tanh(F.conv2d(xr, wo, bo, padding=k // 2))
    assert out.shape == (n, np_, h, w)
    assert (out.double() - ref).abs().max().item() < _bound_f32(ref)
    go = torch.randn(n, np_, h, w, generator=g, device="cuda")
    out.backward(go)
    ref.backward(go.double())
    gx_ref = xr.grad.permute(0, 2, 3, 1)
    assert (x.grad.double() - gx_ref).abs().max().item() < _bound_bf16(gx_ref)
    # the node's fp32 gradient of the pre-Tanh value uses the fp32 output, the reference the fp64 one
    assert (cout.weight.grad.double() - wo.grad).abs().max().item() < _bound_f32(wo.grad)
    assert (cout.bias.grad.double() - bo.grad).abs().max().item() < _bound_f32(bo.grad)


@pytest.mark.parametrize("np_", [1, 2, 3, 4])
def test_conv4x4s2_planes_nodes(np_):
    """The Attention U-Net's Conv2d(C, 64, 4, 2, 1) input and ConvTranspose2d(128, C, 4, 2, 1) + Tanh output nodes on
    the im2col / col2im + pointwise GEMM path, with the bounds its 1-plane version meets in test_kernels_gpu."""
    from pai_b200 import layers as L
    n, h, w = 2, 32, 32
    g = _gen(300 + np_)
    torch.manual_seed(np_)
    enc = nn.Conv2d(np_, 64, 4, 2, 1).cuda()
    planes = torch.randn(n, np_, h, w, generator=g, device="cuda")
    y = L.conv4x4s2_in_planes(planes, enc)
    wi = _bf(enc.weight.detach()).double().requires_grad_(True)
    bi = enc.bias.detach().double().requires_grad_(True)
    ref = F.conv2d(_bf(planes).double(), wi, bi, stride=2, padding=1)
    assert (y.double().permute(0, 3, 1, 2) - ref).abs().max().item() < _bound_bf16(ref)
    gy = torch.randn(n, h // 2, w // 2, 64, generator=g, device="cuda").bfloat16()
    y.backward(gy)
    ref.backward(gy.double().permute(0, 3, 1, 2))
    assert (enc.weight.grad.double() - wi.grad).abs().max().item() < 3e-3 * max(1.0, wi.grad.abs().max().item())
    assert (enc.bias.grad.double() - bi.grad).abs().max().item() < 1e-3 * max(1.0, bi.grad.abs().max().item())

    cin, hh, ww = 128, 16, 16
    dec = nn.ConvTranspose2d(cin, np_, 4, 2, 1).cuda()
    with torch.no_grad():
        dec.weight.mul_(0.5)
    x = torch.randn(n, hh, ww, cin, generator=g, device="cuda").bfloat16().requires_grad_(True)
    out = L.convT4x4s2_out_planes_tanh(x, dec)
    xr = x.detach().double().permute(0, 3, 1, 2).requires_grad_(True)
    wq = _bf(dec.weight.detach()).double().requires_grad_(True)
    bq = dec.bias.detach().double().requires_grad_(True)
    ref = torch.tanh(F.conv_transpose2d(xr, wq, bq, stride=2, padding=1))
    assert out.shape == (n, np_, 2 * hh, 2 * ww)
    assert (out.double() - ref).abs().max().item() < 2e-3
    go = torch.randn(n, np_, 2 * hh, 2 * ww, generator=g, device="cuda")
    out.backward(go)
    ref.backward(go.double())
    gx_ref = xr.grad.permute(0, 2, 3, 1)
    assert (x.grad.double() - gx_ref).abs().max().item() < 2e-2 * max(1.0, gx_ref.abs().max().item())
    assert (dec.weight.grad.double() - wq.grad).abs().max().item() < 1e-2 * max(1.0, wq.grad.abs().max().item())
    assert (dec.bias.grad.double() - bq.grad).abs().max().item() < 1e-2 * max(1.0, bq.grad.abs().max().item())


# ------------------------------------------------------------------------------------------------ 2. lifted parity
_FIRST = {"models.res_unet": "unet.in_conv", "models.trans_unet": "unet.in_conv", "models.attention_unet": "unet.encoders.0"}
_LIFTS = [(name, (3, 3)) for name in CASES] + [(name, io) for name in ("res_18_small", "attention", "trans_small")
                                               for io in ((2, 1), (1, 3), (4, 4))]
_A = {1: [1.0], 2: [0.6, 0.4], 3: [0.5, 0.3, 0.2], 4: [0.4, 0.3, 0.2, 0.1]}


def _last_key(module, sd):
    if module == "models.attention_unet":
        return "unet.decoders.%d" % max(int(k.split(".")[2]) for k in sd if k.startswith("unet.decoders."))
    return "unet.out.0"


def _lift(name, cin, cout):
    """-> (1-channel model, C-channel model, x1, xC, t1, tC, a, first, last)."""
    module, cls, kwargs, n, res, loss_type = CASES[name]
    m1, x, t = _build(name)
    torch.manual_seed(0)
    mc = getattr(importlib.import_module(module), cls)(in_channels=cin, out_channels=cout, dropout=0.0,
                                                       loss_type=loss_type, **kwargs)
    sd1, sdc = m1.state_dict(), mc.state_dict()
    first, last = _FIRST[module], _last_key(module, sd1)
    a = torch.tensor(_A[cin], dtype=torch.float64)
    with torch.no_grad():
        for k, v in sd1.items():
            if k == first + ".weight":
                sdc[k].copy_((a.view(1, cin, 1, 1) * v.double()).float())     # W[:, j] = a_j W1
            elif k == last + ".weight":
                dim = 1 if module == "models.attention_unet" else 0            # ConvT [Cin, C, 4, 4] / Conv [C, 64, 3, 3]
                sdc[k].copy_(v.expand_as(sdc[k]) if dim == 1 else v.expand(cout, *v.shape[1:]))
            elif k == last + ".bias":
                sdc[k].copy_(v.expand(cout))
            else:
                sdc[k].copy_(v)
    g = torch.Generator().manual_seed(77)
    r = (torch.rand(cin, *x.shape[-2:], generator=g, dtype=torch.float64) - 0.5) * 0.24
    r = r - (a.view(cin, 1, 1) * r).sum(0, keepdim=True)                       # sum_j a_j r_j = 0 at every pixel
    assert r.abs().max() < 0.25
    xc = (x.double() + r.to(x.device).unsqueeze(0)).float().contiguous()
    return m1, mc.cuda(), x, xc, t, t.expand(-1, cout, -1, -1).contiguous(), a, first, last


@pytest.mark.parametrize("name,io", _LIFTS, ids=[f"{n}-{i}x{o}" for n, (i, o) in _LIFTS])
def test_lifted_reference_parity(name, io, golden_dir):
    gz = np.load(os.path.join(golden_dir, "variants_ref.npz"))
    if f"{name}/state_keys" not in gz:
        pytest.skip("no golden vectors for this case")
    cin, cout = io
    m1, m, x1, x, _, target, a, first, last = _lift(name, cin, cout)
    sd = m1.state_dict()
    keys = sorted(sd.keys())
    assert keys == list(gz[f"{name}/state_keys"]) == sorted(m.state_dict().keys())
    cs = np.array([[float(sd[k].double().sum()), float(sd[k].double().abs().sum())] for k in keys])
    assert np.allclose(cs, gz[f"{name}/state_checksums"], rtol=1e-5, atol=1e-6)
    del m1
    m.eval()
    with torch.no_grad():
        y = m(x)
    assert y.shape == (x.shape[0], cout, *x.shape[2:]) and y.dtype == torch.float32
    for o in range(cout):
        err = np.abs(y.cpu()[:, o:o + 1, ::4, ::4].numpy() - gz[f"{name}/eval_sub"])
        assert err.max() < 2e-2, ("eval", o, err.max(), err.mean())
    m.train()
    y = m(x)
    gap_max, gap_mean = gz[f"{name}/bf16_gap"]
    for o in range(cout):
        err = np.abs(y.detach().cpu()[:, o:o + 1, ::4, ::4].numpy() - gz[f"{name}/train_sub"])
        assert err.max() < max(5e-2, 1.5 * gap_max) and err.mean() < max(1e-2, 1.5 * gap_mean), \
            ("train", o, err.max(), err.mean(), gap_max, gap_mean)
    loss = m.loss(x, y, target)
    loss.backward()
    ref_loss = float(gz[f"{name}/loss"])
    assert abs(float(loss) - ref_loss) <= 0.02 * abs(ref_loss) + 2e-3 + gap_mean, (float(loss), ref_loss)
    named = dict(m.named_parameters())

    def folded(k):      # the gradient of the 1-channel parameter, by the chain rule through the lift
        gr = named[k].grad
        if gr is None:
            return None
        gr = gr.double()
        if k == first + ".weight":
            return (gr * a.to(gr.device).view(1, -1, 1, 1)).sum(1)
        if k == last + ".weight":
            return gr.sum(1) if last.startswith("unet.decoders") else gr.sum(0)
        if k == last + ".bias":
            return gr.sum()
        return gr

    gk = list(gz[f"{name}/grad_keys"])
    ref = gz[f"{name}/grad_norms"]
    got = np.array([float(folded(k).norm()) if folded(k) is not None else 0.0 for k in gk])
    order = np.argsort(-ref)
    energy = np.cumsum(ref[order] ** 2) / np.sum(ref ** 2)
    major = order[: int(np.searchsorted(energy, 0.99)) + 1]
    rel = np.abs(got[major] - ref[major]) / ref[major]
    gtol = 0.2 + 1.5 * float(gap_mean)
    assert rel.max() < gtol, [(gk[i], got[i], ref[i]) for i in major if abs(got[i] - ref[i]) / ref[i] >= gtol]
    assert np.all(np.isfinite(got))
    # every input plane of the first layer gets its share a_j of the 1-channel gradient
    gw = named[first + ".weight"].grad.double()
    for j in range(cin):
        assert gw[:, j].abs().max() > 0


# ------------------------------------------------------------------------------------------------ 3. default constructors
_DEFAULTS = [("models.res_unet", "ResUnetGAN"), ("models.attention_unet", "AttentionUnetGAN"),
             ("models.trans_unet", "TransUnetGAN")]


def _default_model(module, cls, **kw):
    torch.manual_seed(0)
    if cls == "TransUnetGAN":
        kw = dict(channel_mults=(1, 2, 2), patch_size=4, **kw)
    return getattr(importlib.import_module(module), cls)(**kw).cuda().train()


def _rgb_batch(n=2):
    x, t = port.synthetic_pairs(n, seed=4321)
    x, t = x[:, :, :256, :256], t[:, :, :256, :256]
    shift = torch.tensor([0.0, 0.1, -0.1]).view(1, 3, 1, 1)
    return ((x + shift).clamp(-1, 1).contiguous().cuda(), (t * torch.tensor([1.0, 0.9, 0.8]).view(1, 3, 1, 1)).contiguous().cuda())


def _ends(m, module):
    sd_keys = dict(m.named_parameters())
    first = _FIRST[module]
    last = _last_key(module, sd_keys)
    return sd_keys[first + ".weight"], sd_keys[last + ".weight"], module == "models.attention_unet"


@pytest.mark.parametrize("module,cls", _DEFAULTS, ids=[c for _, c in _DEFAULTS])
def test_reference_default_constructor_trains(module, cls):
    """``ResUnetGAN()`` / ``AttentionUnetGAN()`` / ``TransUnetGAN()`` with every default (3 channels, GAN loss with the
    default 3-channel Discriminator(), dropout 0.5): 3 eager steps, then 4 as a step graph."""
    m = _default_model(module, cls)
    assert m.discriminator is not None
    x, t = _rgb_batch()
    w_in, w_out, convt = _ends(m, module)
    w_in0, w_out0 = w_in.detach().clone(), w_out.detach().clone()
    for i in range(3):
        m.training_step((x, t), i)
    torch.cuda.synchronize()
    for gw in (w_in.grad, w_out.grad):
        assert gw is not None and torch.isfinite(gw).all()
    for j in range(3):
        assert w_in.grad[:, j].abs().max() > 0
        assert (w_out.grad[:, j] if convt else w_out.grad[j]).abs().max() > 0
    m.enable_step_graph(warmup=1)
    for i in range(3, 7):
        m.training_step((x, t), i)
    torch.cuda.synchronize()
    assert m.__dict__["_pai_step_graph"].replays == 3
    for k, vals in m.logged.items():
        assert len(vals) == 7 and all(np.isfinite(float(v)) for v in vals), k
    w_in, w_out = w_in.detach(), w_out.detach()
    for j in range(3):
        assert (w_in[:, j] - w_in0[:, j]).abs().max() > 0
        assert ((w_out[:, j] - w_out0[:, j]) if convt else (w_out[j] - w_out0[j])).abs().max() > 0
    m.eval()
    with torch.no_grad():
        pred = m(x)
    assert pred.shape == (2, 3, 256, 256) and torch.isfinite(pred).all()


@pytest.mark.parametrize("module,cls", _DEFAULTS, ids=[c for _, c in _DEFAULTS])
def test_reference_default_constructor_step_graph_matches_eager(module, cls):
    """With dropout 0, 4 steps replayed as a step graph log what 4 eager steps log, within 5x the spread of two eager
    runs, floor 2 % (the criterion of test_variant_step_graph_matches_eager)."""
    x, t = _rgb_batch()
    logs = {}
    for mode in ("eager_a", "eager_b", "graph"):
        m = _default_model(module, cls, dropout=0.0)
        if mode == "graph":
            m.enable_step_graph(warmup=1)
        for i in range(4):
            m.training_step((x, t), i)
        torch.cuda.synchronize()
        if mode == "graph":
            assert m.__dict__["_pai_step_graph"].replays == 3
        logs[mode] = {k: np.array([float(v) for v in vals]) for k, vals in m.logged.items()}
        del m
    for k, a in logs["eager_a"].items():
        g, b = logs["graph"][k], logs["eager_b"][k]
        assert len(a) == len(g) == 4 and np.all(np.isfinite(g))
        scale = np.abs(a) + 1e-3
        dev_graph, dev_eager = float((np.abs(g - a) / scale).max()), float((np.abs(b - a) / scale).max())
        assert dev_graph <= max(5 * dev_eager, 2e-2), (k, dev_graph, dev_eager, a, b, g)


# ------------------------------------------------------------------------------------------------ 4. failures
@pytest.mark.parametrize("module,cls", _DEFAULTS, ids=[c for _, c in _DEFAULTS])
def test_unsupported_channel_counts_raise(module, cls):
    kw = dict(channel_mults=(1, 2, 2), patch_size=2) if cls == "TransUnetGAN" else dict(channel_mults=(1, 2))
    torch.manual_seed(0)
    m5 = getattr(importlib.import_module(module), cls)(in_channels=5, out_channels=3, dropout=0.0, loss_type="ssim", **kw)
    with pytest.raises(RuntimeError, match="in_channels=5.*1 to 4 image channels"):
        m5.cuda()(torch.zeros(1, 5, 256, 256, device="cuda"))
    m3 = getattr(importlib.import_module(module), cls)(dropout=0.0, loss_type="ssim", **kw).cuda()
    with pytest.raises(RuntimeError, match=r"expected a \[N, 3, H, W\] input"):
        m3(torch.zeros(1, 1, 256, 256, device="cuda"))
