"""GPU checks of the implicit-GEMM fprop epilogue that writes bf16 tiles with TMA stores (and reads the saved
activations of the fused activation backward with TMA loads): every output view is compared with PyTorch's fp32
convolution of the same bf16 operands, and every byte of the allocation OUTSIDE the view must keep the sentinel it was
filled with -- the stores are clipped to the view's channels, pixel grid and (convT) phase."""
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu
torch.backends.cudnn.allow_tf32 = False
torch.backends.cuda.matmul.allow_tf32 = False

SENTINEL = -1234.0          # exactly representable in bf16, never produced by these inputs


def _ops():
    from pai_b200 import ops
    return ops


def _rand(shape, seed, scale=1.0):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return (torch.randn(shape, generator=g, device="cuda") * scale).bfloat16()


def _nchw(t):
    return t.float().permute(0, 3, 1, 2)


def _nhwc(t):
    return t.permute(0, 2, 3, 1).contiguous()


def _slot(shape, ld, off):
    """A sentinel-filled NHWC allocation with `ld` channels per pixel and the view of channels off .. off + c.  (Every
    case has more than ops.SPLITK_MAX_PIXELS output pixels, so no layer is split along K onto the fp32 path.)"""
    n, h, w, c = shape
    big = torch.full((n, h, w, ld), SENTINEL, dtype=torch.bfloat16, device="cuda")
    return big, big[..., off:off + c]


def _outside_untouched(big, off, c):
    keep = torch.ones(big.shape[-1], dtype=torch.bool, device="cuda")
    keep[off:off + c] = False
    rest = big[..., keep]
    assert bool((rest == SENTINEL).all()), f"{int((rest != SENTINEL).sum())} elements outside the view were written"


def _close(y, ref, tol=1e-2):
    scale = max(1.0, ref.abs().max().item())
    err = (y.float() - ref).abs().max().item()
    assert err < tol * scale, (err, scale)


@pytest.mark.parametrize("n,h,w,cin,cout,stride,ld,off", [
    (40, 32, 32, 64, 128, 2, 256, 64),      # concat slot: y_ld > cout with a channel offset
    (12, 32, 32, 64, 64, 1, 64, 0),         # PatchGAN stride 1: 31 x 31 outputs, ragged in w and h
    (12, 32, 32, 64, 128, 1, 192, 64),      # the same into a slot
    (4, 100, 100, 64, 64, 2, 64, 0),        # 50 x 50: gw is not a multiple of the 64-wide pixel box
    (640, 8, 8, 64, 128, 2, 128, 0),        # 4 x 4 images: one 128-pixel box spans 8 images
    (401, 10, 10, 64, 64, 2, 128, 64),      # 5 x 5 images, 2 per box, ragged in w, h and n, into a slot
])
def test_conv_fprop_view(n, h, w, cin, cout, stride, ld, off):
    ops = _ops()
    x = _rand((n, h, w, cin), 1)
    wt = _rand((cout, cin, 4, 4), 2, 0.05)
    bias = torch.randn(cout, device="cuda")
    ho, wo = (h // 2, w // 2) if stride == 2 else (h - 1, w - 1)
    big, y = _slot((n, ho, wo, cout), ld, off)
    ops.conv4x4_fprop(x, ops.pack_conv_weight(wt.float()), cout, stride=stride, bias=bias, act=ops.ACT_LEAKY, slope=0.2,
                      out=y)
    ref = F.leaky_relu(_nhwc(F.conv2d(_nchw(x), wt.float(), bias, stride=stride, padding=1)), 0.2)
    torch.cuda.synchronize()
    _close(y, ref)
    _outside_untouched(big, off, cout)


@pytest.mark.parametrize("n,h,w,cin,cout,ld,off", [
    (4, 32, 32, 128, 128, 256, 128),        # 4 phases by tile, into a slot
    (8, 20, 20, 128, 128, 128, 0),          # 4 phases by tile, ragged grid
    (4, 32, 32, 128, 64, 128, 64),          # phase-fused (cout 64), into a slot
    (8, 20, 20, 128, 64, 64, 0),            # phase-fused, ragged grid
])
def test_convT_fprop_view(n, h, w, cin, cout, ld, off):
    ops = _ops()
    x = _rand((n, h, w, cin), 3)
    wt = _rand((cin, cout, 4, 4), 4, 0.05)
    bias = torch.randn(cout, device="cuda")
    big, y = _slot((n, 2 * h, 2 * w, cout), ld, off)
    ops.convT4x4s2_fprop(x, ops.pack_convT_weight(wt.float()), cout, bias=bias, act=ops.ACT_RELU, out=y)
    ref = F.relu(_nhwc(F.conv_transpose2d(_nchw(x), wt.float(), bias, stride=2, padding=1)))
    torch.cuda.synchronize()
    _close(y, ref)
    _outside_untouched(big, off, cout)


def test_conv_fprop_dual_views():
    ops = _ops()
    n, h, w, cin, cout = 2, 40, 40, 64, 128
    x = _rand((n, h, w, cin), 5)
    wt = _rand((cout, cin, 4, 4), 6, 0.05)
    bias = torch.randn(cout, device="cuda")
    big1, y1 = _slot((n, h // 2, w // 2, cout), 128, 0)
    big2, y2 = _slot((n, h // 2, w // 2, cout), 320, 128)
    ops.conv4x4_fprop_dual(x, ops.pack_conv_weight(wt.float()), cout, bias, y1, ops.ACT_LEAKY, y2, ops.ACT_RELU, slope=0.2)
    ref = _nhwc(F.conv2d(_nchw(x), wt.float(), bias, stride=2, padding=1))
    torch.cuda.synchronize()
    _close(y1, F.leaky_relu(ref, 0.2))
    _close(y2, F.relu(ref))
    _outside_untouched(big2, 128, cout)


@pytest.mark.parametrize("m", [1000, 4099])
def test_pointwise_gemm_ragged(m):
    ops = _ops()
    cin, cout = 128, 128
    x = _rand((m, cin), 7)
    wt = _rand((cout, cin), 8, 0.1)
    bias = torch.randn(cout, device="cuda")
    big1 = torch.full((m + 200, 192), SENTINEL, dtype=torch.bfloat16, device="cuda")
    big2 = torch.full((m + 200, 128), SENTINEL, dtype=torch.bfloat16, device="cuda")
    y1, y2 = big1[:m, 64:], big2[:m]
    ops.pointwise_gemm(x, ops.pack_conv1x1_weight(wt.float()), cout, bias=bias, act=ops.ACT_LEAKY, slope=0.2, out=y1,
                       out2=y2, act2=ops.ACT_NONE)
    ref = x.float() @ wt.float().t() + bias
    torch.cuda.synchronize()
    _close(y1, F.leaky_relu(ref, 0.2))
    _close(y2, ref)
    assert bool((big1[:, :64] == SENTINEL).all()) and bool((big1[m:] == SENTINEL).all())
    assert bool((big2[m:] == SENTINEL).all())


@pytest.mark.parametrize("n,h,w,cgy,cin,want_colsum", [
    (4, 20, 20, 128, 64, True),     # phase-fused, 1-CTA, 40 x 40 output: rows outside the grid in every box row
    (4, 20, 20, 128, 64, False),
    (32, 20, 20, 128, 64, True),    # phase-fused, CTA pairs
    (4, 20, 20, 256, 128, True),    # 4 phases by tile, 1-CTA
    (32, 20, 20, 256, 128, True),   # 4 phases by tile, CTA pairs
    (32, 20, 20, 256, 128, False),
])
def test_dgrad_act_masked(n, h, w, cgy, cin, want_colsum):
    ops = _ops()
    gy = _rand((n, h, w, cgy), 9)
    wt = _rand((cgy, cin, 4, 4), 10, 0.05)       # Conv2d(cin -> cgy) weight; its data gradient is convT(gy, wt)
    saved = _rand((n, 2 * h, 2 * w, cin), 11)
    gx, part = ops.conv4x4_dgrad_act(gy, ops.pack_convT_weight(wt.float()), cin, saved, slope=0.2,
                                     want_colsum=want_colsum)
    ref = _nhwc(F.conv_transpose2d(_nchw(gy), wt.float(), stride=2, padding=1))
    ref = ref * torch.where(saved.float() > 0, 1.0, 0.2)
    torch.cuda.synchronize()
    _close(gx, ref)
    if want_colsum:
        g = gx.float().reshape(-1, cin)
        s = part.sum(0)
        torch.testing.assert_close(s[:cin], g.sum(0), rtol=1e-4, atol=1e-2)
        torch.testing.assert_close(s[cin:], (g * g).sum(0), rtol=1e-4, atol=1e-2)


@pytest.mark.parametrize("kind,n,h,w,cin,cout", [
    ("conv", 8, 26, 26, 64, 128),       # 13 x 13 outputs
    ("conv", 96, 10, 10, 64, 64),       # 5 x 5 outputs, two images per box
    ("convT", 4, 13, 13, 128, 128),     # 26 x 26 outputs
    ("convT", 8, 13, 13, 128, 64),      # phase-fused, 26 x 26 outputs
])
def test_bnstats_ragged(kind, n, h, w, cin, cout):
    """Rows outside the pixel grid are computed but neither stored nor summed: the partial sums equal fp32 sums over
    exactly the stored bf16 output."""
    ops = _ops()
    x = _rand((n, h, w, cin), 12)
    bias = torch.randn(cout, device="cuda")
    if kind == "conv":
        wt = _rand((cout, cin, 4, 4), 13, 0.05)
        y, part = ops.conv4x4_fprop_bnstats(x, ops.pack_conv_weight(wt.float()), cout, bias=bias)
        ref = _nhwc(F.conv2d(_nchw(x), wt.float(), bias, stride=2, padding=1))
    else:
        wt = _rand((cin, cout, 4, 4), 13, 0.05)
        y, part = ops.convT4x4s2_fprop_bnstats(x, ops.pack_convT_weight(wt.float()), cout, bias=bias)
        ref = _nhwc(F.conv_transpose2d(_nchw(x), wt.float(), bias, stride=2, padding=1))
    torch.cuda.synchronize()
    _close(y, ref)
    g = y.float().reshape(-1, cout)
    s = part.sum(0)
    torch.testing.assert_close(s[:cout], g.sum(0), rtol=1e-4, atol=1e-2)
    torch.testing.assert_close(s[cout:], (g * g).sum(0), rtol=1e-4, atol=1e-2)
