"""Cost of 3-channel (RGB) images in the Residual / Attention / Trans U-Nets.

1. CUDA-event time per launch of each multi-plane kernel at batch 64, 256 x 256 (the Attention U-Net's 4x4 stride-2
   layers: 128 x 128 on the wide side), for P = 1 and P = 3 planes.  Algorithmic bytes and FMAs come from the shapes
   (``counts`` below); each rate is reported against HBM (7.7 TB/s) and the FP32 FMA lanes (148 SMs x 128 x the SM
   clock), and the larger of the two lower bounds names the bound.  Working sets are 0.3-1.1 GB (no L2 residency).
2. Step-graph time (whole training step replayed as one CUDA graph, SSIM loss) of ResUnetGAN(res_type="next") at
   batch 32 and AttentionUnetGAN / TransUnetGAN(channel_mults=(1, 2, 2, 4, 4), patch_size=4) at batch 64, each with
   1 and 3 image channels; both models of a family live at once and their timed windows alternate.

    python profiles/scripts/bench_multichannel.py OUT.txt
"""
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
for p in (os.path.join(ROOT, "thesis-pai-reconstruction_b200"), os.path.join(ROOT, "oracle")):
    sys.path.insert(0, p)
import torch

from pai_b200 import ops
from pix2pix_port import synthetic_pairs

dev = torch.device("cuda")
HBM = 7.7e12
STEPS, ROUNDS = 10, 3


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader,nounits"],
                       capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    name, power, sm, sm_max = [s.strip() for s in q.split(",")]
    return name, float(power), float(sm), float(sm_max)


def timed(fn, reps=50):
    for _ in range(3):
        fn()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps * 1e-3


def counts(kind, n, h, w, p, c=64):
    """-> (bytes, fma) the algorithm needs: each operand read once, each result written once."""
    px = n * h * w
    if kind in ("planes_to_wide", "planes_to_wide_flip"):       # 3x3, fp32 planes in, bf16 [px, 64] out
        return 4 * p * px + 2 * c * px, 9 * c * p * px
    if kind == "wide_to_planes":                                # bf16 [px, 64] in, fp32 planes out
        return 2 * c * px + 4 * p * px, 9 * c * p * px
    if kind == "planes_wide_wgrad":                             # bf16 [px, 64] + fp32 planes in, [64, p, 9] out
        return 2 * c * px + 4 * p * px, 9 * c * p * px
    if kind == "im2col4x4_planes":                              # fine planes in, 16p bf16 columns per coarse pixel out
        return 4 * p * px + 2 * 16 * p * (px // 4), 0
    if kind == "col2im4x4s2_planes":                            # 16p fp32 partials per coarse pixel in, fine planes out
        return 4 * 16 * p * (px // 4) + 4 * p * px, 0
    raise KeyError(kind)


def kernel_table(lines, fma_peak):
    n, h, w, c = 64, 256, 256, 64
    lines.append(f"Kernels at batch {n}, {h} x {w} (4x4 stride-2 layers: {h // 2} x {w // 2} wide side), 64 channels "
                 f"(CUDA events, 50 launches after 3 warm-up)")
    lines.append(f"  {'kernel':<22} {'P':>2} {'time':>10} {'GB':>7} {'GFMA':>7} {'TB/s':>6} {'%HBM':>6} {'%FMA':>6}  bound")
    g = torch.Generator(device="cuda").manual_seed(1)
    wide = torch.randn(n, h, w, c, generator=g, device=dev).bfloat16()
    res = {}
    for p in (1, 3):
        planes = torch.randn(n, p, h, w, generator=g, device=dev)
        w_in = torch.randn(c, p * 9, generator=g, device=dev) * 0.1
        w_out = torch.randn(p, 9, c, generator=g, device=dev) * 0.1
        part = torch.randn(n, h // 2, w // 2, 16 * p, generator=g, device=dev)
        out = torch.empty(n, h, w, c, dtype=torch.bfloat16, device=dev)
        runs = {
            "planes_to_wide": lambda: ops.conv_planes_to_wide(planes, w_in, None, 3, 1, out=out),
            "planes_to_wide_flip": lambda: ops.conv_planes_to_wide(planes, w_in, None, 3, 1, flip=True, out=out),
            "wide_to_planes": lambda: ops.conv_wide_to_planes(wide, w_out, None, 3, 1),
            "planes_wide_wgrad": lambda: ops.conv_planes_wide_wgrad(planes, wide, 3, 1),
            "im2col4x4_planes": lambda: ops.im2col4x4_planes(planes, h // 2, w // 2, stride=2),
            "col2im4x4s2_planes": lambda: ops.col2im4x4s2_planes(part, p),
        }
        for kind, fn in runs.items():
            t = timed(fn)
            b, f = counts(kind, n, h, w, p, c)
            t_hbm, t_fma = b / HBM, f / fma_peak
            bound = "FMA" if t_fma > t_hbm else "HBM"
            res[(kind, p)] = t
            lines.append(f"  {kind:<22} {p:>2} {t * 1e6:>8.1f}us {b / 1e9:>7.3f} {f / 1e9:>7.2f} {b / t / 1e12:>6.2f} "
                         f"{100 * t_hbm / t:>5.1f}% {100 * t_fma / t:>5.1f}%  {bound}")
        del planes, part
    lines.append("  P = 3 vs P = 1: " + ", ".join(f"{k} x{res[(k, 3)] / res[(k, 1)]:.2f}" for k in runs))
    return res


FAMILIES = [
    ("res_unet_next_b32", "models.res_unet", "ResUnetGAN", dict(res_type="next"), 32),
    ("attention_unet_b64", "models.attention_unet", "AttentionUnetGAN", dict(), 64),
    ("trans_unet_b64", "models.trans_unet", "TransUnetGAN", dict(channel_mults=(1, 2, 2, 4, 4), patch_size=4), 64),
]


def step_table(lines):
    import importlib
    lines.append("")
    lines.append(f"Training step replayed as one CUDA graph, SSIM loss: {ROUNDS} alternating windows of {STEPS} steps "
                 "(ms / step)")
    for label, module, cls, kw, batch in FAMILIES:
        x1, t1 = synthetic_pairs(batch, seed=4242)
        x1, t1 = x1[:, :, :256, :256].contiguous().to(dev), t1[:, :, :256, :256].contiguous().to(dev)
        x3 = torch.cat([x1, (x1 + 0.1).clamp(-1, 1), (x1 - 0.1).clamp(-1, 1)], 1).contiguous()
        t3 = torch.cat([t1, t1 * 0.9, t1 * 0.8], 1).contiguous()
        models = {}
        for ch, batch_ in ((1, (x1, t1)), (3, (x3, t3))):
            torch.manual_seed(0)
            m = getattr(importlib.import_module(module), cls)(in_channels=ch, out_channels=ch, dropout=0.0,
                                                              loss_type="ssim", **kw).to(dev).train()
            m.enable_step_graph(warmup=2)
            for i in range(4):
                m.training_step(batch_, i)
            torch.cuda.synchronize()
            m.logged.clear()
            models[ch] = (m, batch_)
        ms = {ch: [] for ch in models}
        for _ in range(ROUNDS):
            for ch, (m, batch_) in models.items():
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for i in range(STEPS):
                    m.training_step(batch_, i)
                e1.record()
                torch.cuda.synchronize()
                m.logged.clear()
                ms[ch].append(e0.elapsed_time(e1) / STEPS)
        for ch in models:
            lines.append(f"  {label} {ch} ch: " + " ".join(f"{v:7.2f}" for v in ms[ch]) + f"   best {min(ms[ch]):.2f} ms")
        lines.append(f"  {label}: 3 ch vs 1 ch {100 * (min(ms[3]) / min(ms[1]) - 1):+.2f} % step time (best windows)")
        del models, m
        torch.cuda.empty_cache()


def main(out_path):
    name, power, sm, sm_max = gpu_info()
    fma_peak = 148 * 128 * sm_max * 1e6
    lines = [f"GPU: {name}, power limit {power:.0f} W, SM clock {sm:.0f} MHz (max {sm_max:.0f} MHz); "
             f"bounds: HBM {HBM / 1e12:.1f} TB/s, FP32 FMA {fma_peak / 1e12:.1f} T FMA/s (148 x 128 x max SM clock)", ""]
    kernel_table(lines, fma_peak)
    print("\n".join(lines), flush=True)
    step_table(lines)
    text = "\n".join(lines) + "\n"
    print("\n".join(lines[-3 * len(FAMILIES) - 2:]))
    with open(out_path, "w") as f:
        f.write(text)


if __name__ == "__main__":
    main(sys.argv[1])
