"""GPU checks of the Trans U-Net's train-mode ViT dropout (csrc/pai_dropout.cuh, the fused dropout kernels of
csrc/transformer.cu, models/trans_unet.py ``VisionTransformer``).

* the kernels' mask is bit-for-bit the numpy Philox restatement of oracle/vit_dropout_ref.py, and keeps 1 - p;
* one ViT forward / backward with dropout equals the fp32 restatement run with the SAME masks (rebuilt in numpy from
  the key the module drew) as closely as the p = 0 path equals it without masks: a wrong mask, site or index would
  give O(1) errors;
* torch.manual_seed reproduces the key and the output, consecutive forwards draw new keys;
* TransUnetGAN with its default dropout = 0.5 trains eagerly and as a step graph (a new key at every replay);
* with dropout = 0 the ViT issues the launches it always did and none of the new entry points."""
import collections

import numpy as np
import pytest
import torch

import pix2pix_port as port
import vit_dropout_ref as ref

pytestmark = pytest.mark.gpu

DEV = torch.device("cuda")
NEW_ENTRY_POINTS = {"pai_dropout_mask", "pai_attn_fwd_dropout", "pai_attn_bwd_dropout", "pai_add_dropout_layernorm_fwd",
                    "pai_layernorm_bwd_dropout", "pai_gelu_dropout_fwd", "pai_gelu_dropout_bwd"}


def _key_tensor(k):
    return torch.tensor([k], dtype=torch.int64, device=DEV)


@pytest.mark.parametrize("key", [0, 0x0123456789ABCDEF, -2, 2 ** 62 + 12345])
@pytest.mark.parametrize("site", [0, 1, 6, 47])
def test_mask_bits_match_numpy_philox(key, site):
    from pai_b200 import ops
    n = 1 << 20
    for p in (0.5, 0.1):
        got = ops.dropout_mask(_key_tensor(key), site, n, p).cpu().numpy().astype(bool)
        want = ref.dropout_keep(key, site, n, p)
        assert np.array_equal(got, want), (key, site, p, int((got != want).sum()))
    # an odd length ends inside a Philox block
    got = ops.dropout_mask(_key_tensor(key), site, 1001, 0.5).cpu().numpy().astype(bool)
    assert np.array_equal(got, ref.dropout_keep(key, site, 1001, 0.5))


@pytest.mark.parametrize("p", [0.1, 0.5, 0.9])
def test_keep_fraction(p):
    from pai_b200 import ops
    n = 1 << 24
    frac = float(ops.dropout_mask(_key_tensor(0x5EED), 3, n, p).double().mean())
    sigma = (p * (1 - p) / n) ** 0.5
    assert abs(frac - (1 - p)) < 5 * sigma, (frac, 1 - p, sigma)


# ------------------------------------------------------------------------------------------ one ViT, same masks
VIT_CASES = {
    # d = 256, 16 patches, 2 layers, S = 8 images
    "d256": (dict(channels=64, input_size=8, patch_size=2, transformer_layers=2), 8),
    # the trans_full width: d = 4096, 4 patches, one layer, S = 4
    "d4096": (dict(channels=256, input_size=8, patch_size=4, transformer_layers=1), 4),
}


def _vit(case):
    import models.trans_unet as tu
    kw, s = VIT_CASES[case]
    torch.manual_seed(0)
    vit = tu.VisionTransformer(num_heads=8, dropout=0.5, **kw)
    with torch.no_grad():                  # both sides see the same bf16-representable parameters
        for prm in vit.parameters():
            prm.copy_(prm.bfloat16().float())
    side, c = kw["input_size"], kw["channels"]
    x = torch.randn(s, side, side, c, generator=torch.Generator().manual_seed(1)).bfloat16()
    gout = torch.randn(s, side, side, c, generator=torch.Generator().manual_seed(2))
    return vit.to(DEV).train(), x, gout, kw


def _vit_reference(vit, x, masks):
    """fp32 restatement of VisionTransformer.forward (models/trans_unet.py) with explicit per-layer masks."""
    import torch.nn.functional as F
    n, hh, ww, c = x.shape
    p = vit.patch_size
    gh, gw = hh // p, ww // p
    tokens, d = gh * gw, p * p * c
    emb = vit.to_patch_embedding
    t = x.view(n, gh, p, gw, p, c).permute(0, 1, 3, 2, 4, 5).reshape(n * tokens, d)
    t = F.layer_norm(t, (d,), emb[1].weight, emb[1].bias, emb[1].eps)
    t = t @ emb[2].weight.t() + emb[2].bias
    t = F.layer_norm(t, (d,), emb[3].weight, emb[3].bias, emb[3].eps)
    t = (t.view(n, tokens, d) + vit.pos_embedding).reshape(n * tokens, d)
    for i, lyr in enumerate(vit.transformer.layers):
        t = ref.encoder_layer(t, ref.layer_params(lyr), n, tokens, vit.num_heads, None if masks is None else masks[i])
    return t.view(n, gh, gw, p, p, c).permute(0, 1, 3, 2, 4, 5).reshape(n, hh, ww, c)


def _cos(a, b):
    a, b = a.double().flatten(), b.double().flatten()
    return float(a @ b / (a.norm() * b.norm() + 1e-30))


def _vit_errors(vit, kw, x, gout, p):
    """Runs the B200 ViT at dropout p, and the restatement on a CPU fp32 copy with the masks of the key it drew.
    -> (relative output error, min cosine over the input gradient and every parameter gradient, its tensor)."""
    import models.trans_unet as tu
    vit.dropout = p
    vit.zero_grad()
    xg = x.to(DEV).requires_grad_(True)
    torch.manual_seed(123)
    y = vit(xg)
    (y.float() * gout.to(DEV)).sum().backward()
    torch.cuda.synchronize()
    masks = None
    if p > 0:
        key = int(vit._dropout_key.item())
        s, (tokens, d) = x.shape[0], vit.pos_embedding.shape[1:]
        d_ff = vit.transformer.layers[0].linear1.out_features
        masks = [ref.layer_masks(key, i, s, tokens, d, vit.num_heads, d_ff, p) for i in range(len(vit.transformer.layers))]
    cpu = tu.VisionTransformer(num_heads=vit.num_heads, dropout=p, **kw)
    cpu.load_state_dict(vit.state_dict())
    xr = x.float().requires_grad_(True)
    yr = _vit_reference(cpu, xr, masks)
    (yr * gout).sum().backward()
    err = float((y.float().cpu() - yr.detach()).norm() / yr.detach().norm())
    cosines = {"x": _cos(xg.grad.float().cpu(), xr.grad)}
    ref_params = dict(cpu.named_parameters())
    for name, prm in vit.named_parameters():
        cosines[name] = _cos(prm.grad.float().cpu(), ref_params[name].grad)
    worst = min(cosines, key=cosines.get)
    return err, cosines[worst], worst


@pytest.mark.parametrize("case", list(VIT_CASES))
def test_vit_dropout_matches_restatement_with_the_same_masks(case):
    vit, x, gout, kw = _vit(case)
    err0, cos0, worst0 = _vit_errors(vit, kw, x, gout, 0.0)
    err5, cos5, worst5 = _vit_errors(vit, kw, x, gout, 0.5)
    print(f"\n{case}: p=0   output rel err {err0:.3e}, worst grad cosine {cos0:.6f} ({worst0})"
          f"\n{case}: p=0.5 output rel err {err5:.3e}, worst grad cosine {cos5:.6f} ({worst5})")
    # margin: the 1/(1-p) = 2 scaling doubles what bf16 rounds away at the dropout sites; a wrong mask is O(1)
    assert err5 <= 3 * err0 + 1e-2, (err5, err0)
    assert 1 - cos5 <= 4 * (1 - cos0) + 5e-3, (cos5, cos0, worst5)


def test_seed_reproduces_key_and_output_and_keys_are_fresh():
    vit, x, _, _ = _vit("d256")
    x = x.to(DEV)
    with torch.no_grad():
        torch.manual_seed(7)
        y1 = vit(x)
        k1 = int(vit._dropout_key.item())
        torch.manual_seed(7)
        y2 = vit(x)
        k2 = int(vit._dropout_key.item())
        y3 = vit(x)
        k3 = int(vit._dropout_key.item())
    assert k1 == k2 and torch.equal(y1, y2)
    assert k3 != k2 and not torch.equal(y3, y2)
    vit.eval()
    with torch.no_grad():
        assert torch.equal(vit(x), vit(x))            # eval mode: no dropout, no draw


# ------------------------------------------------------------------------------------------ whole model
def _trans_gan(seed):
    import models.trans_unet as tu
    from models.utils import init_weights
    from models.wrapper import Discriminator
    torch.manual_seed(0)
    m = tu.TransUnetGAN(in_channels=1, out_channels=1, channel_mults=(1, 2, 2), patch_size=4)
    assert m.unet.vit_bottleneck.dropout == 0.5            # the constructor's default
    m.discriminator = Discriminator(in_channels=1)         # grayscale pairs need the 1-channel PatchGAN (SURVEY Q1)
    m.discriminator.apply(init_weights)
    x, t = port.synthetic_pairs(2, seed=1234)
    torch.manual_seed(seed)
    return m.to(DEV).train(), x[:, :, :256, :256].contiguous().to(DEV), t[:, :, :256, :256].contiguous().to(DEV)


def test_trans_unet_default_dropout_trains_eager_and_as_step_graph():
    logs, keys = {}, {}
    for mode, seed in (("eager_a", 0), ("eager_b", 1), ("graph", 0)):
        m, x, target = _trans_gan(seed)
        if mode == "graph":
            m.enable_step_graph(warmup=1)
        keys[mode] = []
        for i in range(4):
            m.training_step((x, target), i)
            torch.cuda.synchronize()
            keys[mode].append(int(m.unet.vit_bottleneck._dropout_key.item()))
        if mode == "graph":
            assert m.__dict__["_pai_step_graph"].replays == 3
        logs[mode] = {k: np.array([float(v) for v in vals]) for k, vals in m.logged.items()}
    assert len(set(keys["graph"])) == 4 and len(set(keys["eager_a"])) == 4, keys
    for k, a in logs["eager_a"].items():
        g, b = logs["graph"][k], logs["eager_b"][k]
        assert len(a) == len(g) == 4 and np.all(np.isfinite(a)) and np.all(np.isfinite(b)) and np.all(np.isfinite(g))
        scale = np.abs(a) + 1e-3
        dev_graph, dev_eager = float((np.abs(g - a) / scale).max()), float((np.abs(b - a) / scale).max())
        print(f"{k}: graph vs eager {dev_graph:.4f}, eager seed 0 vs seed 1 {dev_eager:.4f}")
        assert dev_graph <= max(5 * dev_eager, 2e-2), (k, dev_graph, dev_eager, a, b, g)


def test_no_dropout_keeps_the_launches(monkeypatch):
    from pai_b200 import lib
    vit, x, gout, _ = _vit("d256")
    vit.dropout = 0.0
    calls = collections.Counter()
    real = lib.call

    def counting(name, *args, **kw):
        calls[name] += 1
        return real(name, *args, **kw)

    monkeypatch.setattr(lib, "call", counting)
    xg = x.to(DEV).requires_grad_(True)
    n0 = lib.launches
    (vit(xg).float() * gout.to(DEV)).sum().backward()
    torch.cuda.synchronize()
    layers = len(vit.transformer.layers)
    assert not (set(calls) & NEW_ENTRY_POINTS), calls
    want = {"pai_attn_fwd": layers, "pai_attn_bwd": layers, "pai_gelu_fwd": layers, "pai_gelu_bwd": layers,
            "pai_add_act": 2 * layers, "pai_layernorm_fwd": 2 * layers + 2, "pai_layernorm_bwd": 2 * layers + 2}
    assert {k: calls[k] for k in want} == want, calls
    # every launch of the ViT goes through these entry points and the Linear layers' GEMMs
    linears = 4 * layers + 1
    assert calls["pai_pointwise_gemm"] == 2 * linears and calls["pai_pointwise_wgrad"] == linears, calls
    print(f"\nViT (2 layers, d = 256) forward + backward without dropout: {lib.launches - n0} library launches, {dict(calls)}")
