"""Outputs of every layer of bench_igemm.py's list on seeded inputs, for comparing two builds of the library bit for bit.

    PAI_LIB_PATH=<build A> python profiles/scripts/igemm_outputs.py save A.pt
    PAI_LIB_PATH=<build B> python profiles/scripts/igemm_outputs.py save B.pt
    python profiles/scripts/igemm_outputs.py compare A.pt B.pt

bf16 outputs must be bitwise equal; BatchNorm / column partial sums (fp32 atomics, whose order varies from run to run)
are compared as per-channel totals with a relative tolerance."""
import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.join(ROOT, "thesis-pai-reconstruction_b200"))
import torch

# name, kind, hin, cin, cout (bench_igemm.py)
LAYERS = [("enc1", "conv", 128, 64, 128), ("enc2", "conv", 64, 128, 256), ("enc3", "conv", 32, 256, 512),
          ("enc4", "conv", 16, 512, 512), ("dec3", "convT", 8, 1024, 512), ("dec4", "convT", 16, 1024, 256),
          ("dec5", "convT", 32, 512, 128), ("dec6", "convT", 64, 256, 64),
          ("D1dgrad", "dgrad_act", 64, 128, 64), ("D1dgrad-ns", "dgrad_act_nosum", 64, 128, 64),
          ("D2dgrad", "dgrad_act", 32, 256, 128), ("D3dgrad", "dgrad_act", 16, 512, 256),
          ("dec4dgrad", "conv", 32, 256, 1024), ("dec5dgrad", "conv", 64, 128, 512), ("dec6dgrad", "conv", 128, 64, 256)]


def save(path):
    from pai_b200 import ops
    dev = torch.device("cuda")
    n = int(os.environ.get("N", 64))
    out = {}
    for i, (name, kind, hin, cin, cout) in enumerate(LAYERS):
        g = torch.Generator(device=dev).manual_seed(1000 + i)
        rnd = lambda *s, scale=0.5: (torch.randn(*s, generator=g, device=dev) * scale).bfloat16()
        x = rnd(n, hin, hin, cin)
        bias = torch.randn(cout, generator=g, device=dev)
        if kind == "conv":
            wp = ops.pack_conv_weight(rnd(cout, cin, 4, 4, scale=0.05).float())
            y, part = ops.conv4x4_fprop_bnstats(x, wp, cout, bias=bias)
            # the activated form (no statistics) of the same layer, where it is not split along K (fp32 atomics)
            if n * (hin // 2) ** 2 > ops.SPLITK_MAX_PIXELS:
                out[name + "/leaky"] = ops.conv4x4_fprop(x, wp, cout, bias=bias, act=ops.ACT_LEAKY, slope=0.2).cpu()
        elif kind == "convT":
            wp = ops.pack_convT_weight(rnd(cin, cout, 4, 4, scale=0.05).float())
            y, part = ops.convT4x4s2_fprop_bnstats(x, wp, cout, bias=bias)
            if 4 * n * hin * hin > ops.SPLITK_MAX_PIXELS:
                out[name + "/relu"] = ops.convT4x4s2_fprop(x, wp, cout, bias=bias, act=ops.ACT_RELU).cpu()
        else:
            wp = ops.pack_convT_weight(rnd(cin, cout, 4, 4, scale=0.05).float())
            saved = rnd(n, 2 * hin, 2 * hin, cout)
            y, part = ops.conv4x4_dgrad_act(x, wp, cout, saved, want_colsum=kind == "dgrad_act")
        torch.cuda.synchronize()
        out[name] = y.cpu()
        if part is not None:
            out[name + "/part"] = part.double().sum(0).cpu()
        print(f"{name:10s} {tuple(y.shape)}", flush=True)
    torch.save(out, path)


def compare(a_path, b_path):
    a, b = torch.load(a_path), torch.load(b_path)
    assert a.keys() == b.keys(), (sorted(a), sorted(b))
    bad = 0
    for k in a:
        if k.endswith("/part"):
            d = ((a[k] - b[k]).abs() / a[k].abs().clamp_min(1.0)).max().item()
            ok = d < 1e-5
            print(f"{k:18s} partial sums: max rel diff {d:.2e} {'ok' if ok else 'DIFFERENT'}")
        else:
            ne = int((a[k].view(torch.int16) != b[k].view(torch.int16)).sum())
            ok = ne == 0
            print(f"{k:18s} bf16 {tuple(a[k].shape)}: {ne} elements differ {'ok' if ok else 'DIFFERENT'}")
        bad += not ok
    print("bitwise equal" if bad == 0 else f"{bad} outputs differ")
    return bad


if __name__ == "__main__":
    if sys.argv[1] == "save":
        save(sys.argv[2])
    else:
        sys.exit(1 if compare(sys.argv[2], sys.argv[3]) else 0)
