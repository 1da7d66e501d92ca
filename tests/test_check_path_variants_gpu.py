"""The fp32 check path (``engine.check_path()``, csrc/check_f32.cu) of the Residual, Attention and Trans U-Nets, forward and
backward, against the UNMODIFIED reference's golden vectors (tests/golden/variants_ref.npz) and against the functional
restatement ``oracle/variants_port.py`` evaluated in fp64 (the exact answer).

Bounds (the methodology of tests/test_check_path_gpu.py): the reference's own fp32 arithmetic is not exact either, so each
case is held to 3x the gap between the port in fp32 (on the CPU, as the fixture was made) and the port in fp64:
* eval outputs: max-abs <= max(1e-5, 3 x gap); train outputs: max-abs <= max(1e-4, 3 x gap) and mean-abs <=
  max(1e-5, 3 x the mean gap) (train-mode BatchNorm over a few values amplifies rounding: on res_next the fixture's own
  mean-abs distance from fp64 is 3.9e-5); running statistics 1e-4 relative + 1e-5 absolute of the fp32 port's; the loss
  1e-4 relative of the fixture's, or 3x the port's fp32 loss error where that is larger (trans_small: an SSIM of -0.004
  whose fp32 evaluation is 6e-4 relative from fp64);
* gradients: per tensor, relative L2 error against fp64 <= 3 x the fp32 port's + 2e-3; conv biases in front of a
  BatchNorm (exactly cancelled) ~0.  A ReLU input within fp32 rounding of zero can land on the other side of the kink
  than in fp64, in the check path as in any fp32 evaluation, and the whole gradient upstream then follows the other
  subgradient (res_v2_small: one upsampled 2x2 block of decoders.3's input, +4.5e-6 in fp64, -1.6e-6 on the check path,
  moves every upstream gradient by 2-7e-3).  So each implementation is compared with the exact gradient of the branches it
  took: the CPU fp32 port with the plain fp64 port, the check path with the fp64 port whose ReLU / LeakyReLU masks are
  pinned to the ones the check path evaluated.  Nothing else of the fp64 evaluation changes.
``res_next_b8`` and ``trans_full`` (the BASELINE configurations) are checked forward only, for the host memory of their
fp64 gradient oracle (``trans_full`` alone has about 8 GB of fp64 parameters, and as much again in gradients)."""
import contextlib
import math

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import pix2pix_port as port
import variants_port
from test_check_variants_cpu import build, family, inputs
from test_variants_gpu import CASES

pytestmark = pytest.mark.gpu

GRAD_CASES = ["res_18_small", "res_v2_small", "res_50_small", "res_next", "attention", "trans_small"]
# each family at the size of its smallest case
FAMILY_CASES = ["res_18_small", "attention", "trans_small"]


@pytest.fixture(scope="module")
def gz(golden_dir):
    import os
    return np.load(os.path.join(golden_dir, "variants_ref.npz"))


def _state(m):
    return {k: v.detach().cpu().clone() for k, v in m.state_dict().items()}


def _cast(sd, dtype, grad=False):
    out = {}
    for k, v in sd.items():
        if v.is_floating_point():
            w = v.detach().clone().to(dtype)
            if grad and port._is_param(k):
                w.requires_grad_(True)
            out[k] = w
        else:
            out[k] = v.clone()
    return out


def _port(sd, dtype, x, training, name):
    """-> (output, state after the forward) of the port in ``dtype`` on the CPU."""
    s = _cast(sd, dtype)
    with torch.no_grad():
        y = variants_port.forward(s, x.to(dtype), training, *family(name))
    return y, s


@contextlib.contextmanager
def _record_branches(masks):
    """Appends (act, input > 0) of every ReLU / LeakyReLU the check path evaluates, in order."""
    from pai_b200 import check
    from pai_b200.ops import ACT_LEAKY, ACT_RELU
    orig = check._act

    def act(x, a):
        if a in (ACT_RELU, ACT_LEAKY):
            masks.append((a, (x.detach() > 0).cpu()))
        return orig(x, a)
    check._act = act
    try:
        yield
    finally:
        check._act = orig


@contextlib.contextmanager
def _pinned_branches(masks):
    """The port's ReLUs / LeakyReLUs take the branches recorded from the check path (same call order, shapes checked)."""
    from pai_b200.ops import ACT_LEAKY, ACT_RELU
    it = iter(masks)

    def take(kind, h):
        a, m = next(it)
        assert a == kind and tuple(m.shape) == tuple(h.shape), (a, kind, tuple(m.shape), tuple(h.shape))
        return m
    orig = variants_port._relu, variants_port._leaky
    variants_port._relu = lambda h: h * take(ACT_RELU, h).to(h.dtype)
    variants_port._leaky = lambda h: torch.where(take(ACT_LEAKY, h), h, 0.2 * h)
    try:
        yield
        assert next(it, None) is None, "the check path evaluated more activations than the port"
    finally:
        variants_port._relu, variants_port._leaky = orig


def _port_grads(sd, dtype, x, target, name, loss_type, masks=None):
    """Gradients of the port in ``dtype``; with ``masks``, on the ReLU branches the check path took."""
    s = _cast(sd, dtype, grad=True)
    with _pinned_branches(masks) if masks is not None else contextlib.nullcontext():
        y = variants_port.forward(s, x.to(dtype), True, *family(name))
    loss = port.generator_loss(s, loss_type, x.to(dtype), y, target.to(dtype))
    loss.backward()
    return {k: v.grad.double() for k, v in s.items() if k.startswith("unet.") and v.grad is not None}, y.detach()


def _gap(a, b):
    return float((a.double() - b.double()).abs().max())


@pytest.mark.parametrize("name", list(CASES))
def test_check_path_forward_matches_reference(name, gz):
    """Eval and train forward inside ``check_path()`` against the fixture, running statistics against the fp32 port."""
    from pai_b200 import engine, lib
    torch.set_num_threads(8)
    m = build(name).cuda()
    sd = _state(m)
    x, target = inputs(name)
    gap_eval = _gap(_port(sd, torch.float32, x, False, name)[0], _port(sd, torch.float64, x, False, name)[0])
    y32, s32 = _port(sd, torch.float32, x, True, name)
    y64, s64 = _port(sd, torch.float64, x, True, name)
    gap_train = _gap(y32, y64)
    mean_train = float((y32.double() - y64)[:, :, ::4, ::4].abs().mean())
    loss_type = CASES[name][5]
    l32 = float(port.generator_loss(s32, loss_type, x, y32, target))
    l64 = float(port.generator_loss(s64, loss_type, x.double(), y64, target.double()))
    m.eval()
    before = lib.launches
    with engine.check_path(), torch.no_grad():
        y = m(x.cuda())
    assert lib.launches > before
    assert y.shape == x.shape and y.dtype == torch.float32
    d = np.abs(y.cpu()[:, :, ::4, ::4].numpy() - gz[f"{name}/eval_sub"])
    assert d.max() <= max(1e-5, 3 * gap_eval), ("eval", d.max(), gap_eval)
    m.train()
    with engine.check_path():
        y = m(x.cuda())
        loss = m.loss(x.cuda(), y, target.cuda())
    d = np.abs(y.detach().cpu()[:, :, ::4, ::4].numpy() - gz[f"{name}/train_sub"])
    assert d.max() <= max(1e-4, 3 * gap_train) and d.mean() <= max(1e-5, 3 * mean_train), \
        ("train", d.max(), d.mean(), gap_train, mean_train)
    ref_loss = float(gz[f"{name}/loss"])
    assert abs(float(loss) - ref_loss) <= max(1e-4 * abs(ref_loss), 3 * abs(l32 - l64)), (float(loss), ref_loss, l32, l64)
    n_bn = 0
    for k, v in m.state_dict().items():
        if k.endswith("running_mean") or k.endswith("running_var"):
            assert torch.allclose(v.cpu(), s32[k], rtol=1e-4, atol=1e-5), k
        if k.endswith("num_batches_tracked"):
            assert int(v) == int(s32[k]) == 1, k
            n_bn += 1
    assert n_bn > 0
    print(f"{name}: eval {gap_eval:.2e} train {gap_train:.2e} / mean {mean_train:.2e} (fp32-fp64 port gaps)")


def _check_grads(m, r32, r64, r64_pinned):
    """Each implementation against the exact gradient of the ReLU branches it took: the CPU fp32 port against the plain
    fp64 port (whose branches it shares), the check path against the fp64 port pinned to the check path's branches."""
    named = dict(m.named_parameters())
    worst = (0.0, 0.0, "")
    assert set(r64) == set(r64_pinned) == {k for k in named if k.startswith("unet.")}
    for k, go in r64_pinned.items():
        assert named[k].grad is not None, k
        g = named[k].grad.cpu().double()
        gn = float(go.norm())
        if gn < 1e-5:            # conv bias in front of a BatchNorm: exactly cancelled (SURVEY Q11), only rounding noise
            assert float(g.norm()) < 1e-4, (k, float(g.norm()))
            continue
        e_check = float((g - go).norm()) / gn
        e_cpu = float((r32[k] - r64[k]).norm()) / float(r64[k].norm())
        worst = max(worst, (e_check, e_cpu, k))
        assert e_check < 3 * e_cpu + 2e-3, (k, e_check, e_cpu)
    return worst


@pytest.mark.parametrize("name", GRAD_CASES)
def test_check_path_backward_every_parameter_gradient(name):
    """One ``loss.backward()`` inside ``check_path()`` with the case's own loss: every generator parameter gradient (the
    grouped 3x3 weights, the attention gates, ``pos_embedding`` and every ViT tensor included) against fp64."""
    from pai_b200 import engine
    torch.set_num_threads(8)
    loss_type = CASES[name][5]
    m = build(name).cuda().train()
    sd = _state(m)
    x, target = inputs(name)
    r32, _ = _port_grads(sd, torch.float32, x, target, name, loss_type)
    r64, _ = _port_grads(sd, torch.float64, x, target, name, loss_type)
    masks = []
    with engine.check_path(), _record_branches(masks):
        y = m(x.cuda())
        loss = m.loss(x.cuda(), y, target.cuda())
        loss.backward()
    r64_pinned, _ = _port_grads(sd, torch.float64, x, target, name, loss_type, masks)
    worst = _check_grads(m, r32, r64, r64_pinned)
    print(f"{name}: worst gradient error vs fp64 {worst[0]:.2e} (CPU fp32: {worst[1]:.2e}) at {worst[2]}")


def _rgb_inputs(name, cin, cout, seed=77):
    _, _, _, n, res, _ = CASES[name]
    g = torch.Generator().manual_seed(seed)
    return torch.rand(n, cin, res, res, generator=g) * 2 - 1, torch.rand(n, cout, res, res, generator=g) * 2 - 1


@pytest.mark.parametrize("name", FAMILY_CASES)
@pytest.mark.parametrize("cin,cout", [(3, 3), (4, 1)])
def test_check_path_multichannel(name, cin, cout):
    """Each family with 3 -> 3 and 4 -> 1 image channels: eval and train outputs and every gradient against the fp64 port;
    the bf16 tensor-core path on the same weights within 2e-2 of the check path in eval mode."""
    from pai_b200 import engine
    torch.set_num_threads(8)
    loss_type = CASES[name][5]
    m = build(name, cin, cout).cuda()
    sd = _state(m)
    x, target = _rgb_inputs(name, cin, cout)
    p32, p64 = _port(sd, torch.float32, x, False, name)[0], _port(sd, torch.float64, x, False, name)[0]
    m.eval()
    with engine.check_path(), torch.no_grad():
        y = m(x.cuda())
    assert y.shape == (x.shape[0], cout) + tuple(x.shape[2:])
    gap = _gap(p32, p64)
    e = _gap(y.cpu(), p64)
    assert e <= max(1e-5, 3 * gap), ("eval", e, gap)
    with torch.no_grad():
        yb = m(x.cuda())
    assert float((yb - y).abs().max()) < 2e-2
    r32, y32 = _port_grads(sd, torch.float32, x, target, name, loss_type)
    r64, y64 = _port_grads(sd, torch.float64, x, target, name, loss_type)
    m.train()
    masks = []
    with engine.check_path(), _record_branches(masks):
        y = m(x.cuda())
        loss = m.loss(x.cuda(), y, target.cuda())
        loss.backward()
    r64_pinned, _ = _port_grads(sd, torch.float64, x, target, name, loss_type, masks)
    d = (y.detach().cpu().double() - y64).abs()
    gap, mean_gap = _gap(y32, y64), float((y32.double() - y64).abs().mean())
    assert float(d.max()) <= max(1e-4, 3 * gap) and float(d.mean()) <= max(1e-5, 3 * mean_gap), \
        ("train", float(d.max()), float(d.mean()), gap, mean_gap)
    _check_grads(m, r32, r64, r64_pinned)


# ------------------------------------------------------------------------------------------ kernels alone
def _close(got, ref, tol=1e-5):
    """max-abs error of ``got`` (CUDA fp32) against the fp64 ``ref``, relative to the largest |ref| (at least 1)."""
    err = float((got.detach().cpu().double() - ref.detach()).abs().max())
    assert err <= tol * max(1.0, float(ref.detach().abs().max())), (err, float(ref.abs().max()))


def _leaf(t):
    return t.detach().cuda().float().requires_grad_(True), t.detach().double().requires_grad_(True)


@pytest.mark.parametrize("stride,bias,hw", [(1, True, (11, 9)), (2, False, (11, 9)), (2, True, (10, 8))])
def test_grouped_conv_kernels(stride, bias, hw):
    """Grouped Conv2d forward, data and weight (+ bias) gradients at odd sizes (and at even sizes with stride 2, whose
    data gradient needs the transposed convolution's output padding), against fp64 ``F.conv2d``."""
    from pai_b200 import engine
    g = torch.Generator().manual_seed(3)
    x = torch.randn(3, 12, *hw, generator=g)
    w = torch.randn(8, 3, 3, 3, generator=g) * 0.3
    b = torch.randn(8, generator=g) if bias else None
    xc, xd = _leaf(x)
    wc, wd = _leaf(w)
    bc, bd = _leaf(b) if bias else (None, None)
    yc = engine._CheckConv2d.apply(xc, wc, bc, stride, 1, 4, False)
    yd = F.conv2d(xd, wd, bd, stride, 1, 1, 4)
    _close(yc, yd)
    gy = torch.randn(yd.shape, generator=g, dtype=torch.float64)
    yc.backward(gy.cuda().float())
    yd.backward(gy)
    assert xc.grad.shape == x.shape
    _close(xc.grad, xd.grad)
    _close(wc.grad, wd.grad, 1e-5 * 10)
    if bias:
        _close(bc.grad, bd.grad)


def test_maxpool_ties_follow_torch_index():
    """MaxPool2d(2) with many ties (and an odd row / column that no window covers): the gradient goes where torch's does."""
    from pai_b200 import engine
    g = torch.Generator().manual_seed(5)
    x = torch.randint(0, 3, (2, 3, 9, 7), generator=g).double()
    xc, xd = _leaf(x)
    yc = engine._CheckMaxPool2.apply(xc)
    yd = F.max_pool2d(xd, 2)
    assert torch.equal(yc.detach().cpu().double(), yd.detach())
    gy = torch.randn(yd.shape, generator=g, dtype=torch.float64)
    yc.backward(gy.cuda().float())
    yd.backward(gy)
    assert torch.equal(xc.grad.cpu().double(), xd.grad.float().double())


def test_upsample_layernorm_linear_gelu_sigmoid():
    from pai_b200 import engine, ops
    g = torch.Generator().manual_seed(7)
    # nearest Upsample(x2)
    x = torch.randn(2, 5, 3, 7, generator=g, dtype=torch.float64)
    xc, xd = _leaf(x)
    yc, yd = engine._CheckUpsample2.apply(xc), F.interpolate(xd, scale_factor=2, mode="nearest")
    _close(yc, yd)
    gy = torch.randn(yd.shape, generator=g, dtype=torch.float64)
    yc.backward(gy.cuda().float())
    yd.backward(gy)
    _close(xc.grad, xd.grad)
    # LayerNorm over the rows of [m, d]
    x = torch.randn(37, 300, generator=g, dtype=torch.float64) * 3 + 1
    gam, bet = torch.randn(300, generator=g, dtype=torch.float64), torch.randn(300, generator=g, dtype=torch.float64)
    (xc, xd), (gc, gd), (bc, bd) = _leaf(x), _leaf(gam), _leaf(bet)
    yc, yd = engine._CheckLayerNorm.apply(xc, gc, bc, 1e-5), F.layer_norm(xd, (300,), gd, bd, 1e-5)
    _close(yc, yd)
    gy = torch.randn(yd.shape, generator=g, dtype=torch.float64)
    yc.backward(gy.cuda().float())
    yd.backward(gy)
    for a, r in ((xc, xd), (gc, gd), (bc, bd)):
        _close(a.grad, r.grad)
    # Linear
    x, w, b = (torch.randn(*s, generator=g, dtype=torch.float64) for s in ((19, 70), (33, 70), (33,)))
    (xc, xd), (wc, wd), (bc, bd) = _leaf(x), _leaf(w), _leaf(b)
    yc, yd = engine._CheckLinear.apply(xc, wc, bc), F.linear(xd, wd, bd)
    _close(yc, yd)
    gy = torch.randn(yd.shape, generator=g, dtype=torch.float64)
    yc.backward(gy.cuda().float())
    yd.backward(gy)
    for a, r in ((xc, xd), (wc, wd), (bc, bd)):
        _close(a.grad, r.grad)
    # exact GELU and sigmoid
    for act, fn in ((ops.ACT_GELU, F.gelu), (ops.ACT_SIGMOID, torch.sigmoid)):
        x = torch.linspace(-8, 8, 4001, dtype=torch.float64)
        xc, xd = _leaf(x)
        yc, yd = engine._CheckAct.apply(xc, act), fn(xd)
        _close(yc, yd)
        gy = torch.randn(yd.shape, generator=g, dtype=torch.float64)
        yc.backward(gy.cuda().float())
        yd.backward(gy)
        _close(xc.grad, xd.grad)


def _attention_ref(qkv, s, b, heads):
    e = qkv.shape[1] // 3
    hd = e // heads
    q, k, v = (u.reshape(s, b, heads, hd).permute(1, 2, 0, 3) for u in qkv.split(e, dim=1))
    p = torch.softmax(q @ k.transpose(-1, -2) / math.sqrt(hd), dim=-1)
    return (p @ v).permute(2, 0, 1, 3).reshape(s * b, e)


@pytest.mark.parametrize("s", [1, 2, 7])
def test_attention_kernels(s):
    """Attention over the sequence axis (the images of a batch) with 8 heads, forward and d(qkv), against fp64."""
    from pai_b200 import engine
    g = torch.Generator().manual_seed(11 + s)
    b, heads, hd = 5, 8, 16
    qkv = torch.randn(s * b, 3 * heads * hd, generator=g, dtype=torch.float64)
    qc, qd = _leaf(qkv)
    yc, yd = engine._CheckAttention.apply(qc, s, b, heads), _attention_ref(qd, s, b, heads)
    _close(yc, yd)
    gy = torch.randn(yd.shape, generator=g, dtype=torch.float64)
    yc.backward(gy.cuda().float())
    yd.backward(gy)
    _close(qc.grad, qd.grad)


# ------------------------------------------------------------------------------------------ refusals
@pytest.mark.parametrize("name", ["res_next", "attention", "trans_small"])      # configurations with Dropout2d / ViT dropout
def test_dropout_refused_in_training_runs_in_eval(name):
    from pai_b200 import engine
    module, cls, kwargs, n, res, loss_type = CASES[name]
    torch.manual_seed(0)
    import importlib
    m = getattr(importlib.import_module(module), cls)(in_channels=1, out_channels=1, dropout=0.5, loss_type=loss_type,
                                                      **kwargs).cuda()
    x, _ = inputs(name)
    m.train()
    with engine.check_path(), torch.no_grad(), pytest.raises(RuntimeError, match="deterministic"):
        m(x.cuda())
    m.eval()
    with engine.check_path(), torch.no_grad():
        y = m(x.cuda())
    assert bool(torch.isfinite(y).all())


@pytest.mark.parametrize("name", FAMILY_CASES)
def test_more_than_four_channels_refused(name):
    from pai_b200 import engine
    m = build(name, 5, 3).cuda().eval()
    x = torch.zeros(2, 5, CASES[name][4], CASES[name][4], device="cuda")
    with engine.check_path(), torch.no_grad(), pytest.raises(RuntimeError, match="1 to 4 image channels"):
        m(x)
