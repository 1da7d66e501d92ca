"""Cost of the Trans U-Net's train-mode ViT dropout.

1. The ``trans_unet_ssim_b64`` step of bench.py (TransUnetGAN(1, 1, channel_mults=(1, 2, 2, 4, 4), patch_size=4,
   loss "ssim"), batch 64, whole step replayed as one CUDA graph) with dropout = 0.0 and 0.5: both models live at once
   and their timed windows alternate, so drift of the shared host hits both alike.
2. CUDA-event time per launch of each fused dropout kernel next to the kernel(s) it replaces, at that model's ViT
   shapes (S = 64 images, 4 patches, d = 4096, 8 heads, d_ff = 2048).  The operands (< 10 MB) stay in L2.
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
BATCH, STEPS, ROUNDS = 64, 10, 4


def gpu_line():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as ex:  # pragma: no cover
        q = f"{torch.cuda.get_device_name()} (nvidia-smi: {ex})"
    return q


def step_times():
    from models.trans_unet import TransUnetGAN
    x, t = synthetic_pairs(BATCH, seed=4242)
    x, t = x.to(dev), t.to(dev)
    models = {}
    for p in (0.0, 0.5):
        torch.manual_seed(0)
        m = TransUnetGAN(in_channels=1, out_channels=1, channel_mults=(1, 2, 2, 4, 4), patch_size=4, dropout=p,
                         loss_type="ssim").to(dev).train()
        for i in range(3):
            m.training_step((x, t), i)
        m.enable_step_graph(warmup=1)
        for i in range(3):
            m.training_step((x, t), i)
        torch.cuda.synchronize()
        m.logged.clear()
        models[p] = m
    ms = {p: [] for p in models}
    for _ in range(ROUNDS):
        for p, m in models.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for i in range(STEPS):
                m.training_step((x, t), i)
            e1.record()
            torch.cuda.synchronize()
            m.logged.clear()
            ms[p].append(e0.elapsed_time(e1) / STEPS)
    for p, m in models.items():
        assert m.__dict__["_pai_step_graph"].replays == 2 + ROUNDS * STEPS     # 3 calls after enabling: 1 eager
    return ms


def timeit(fn, reps=200):
    for _ in range(10):
        fn()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e3 / reps


def kernel_times():
    s, b, d, heads, dff, p = 64, 4, 4096, 8, 2048, 0.5
    m = s * b
    g = torch.Generator(device="cuda").manual_seed(0)

    def rnd(*shape):
        return torch.randn(*shape, device=dev, generator=g).bfloat16()

    key = torch.randint(-2 ** 63, 2 ** 63 - 1, (1,), dtype=torch.int64, device=dev)
    qkv, dout, x, y, h, gh = rnd(m, 3 * d), rnd(m, d), rnd(m, d), rnd(m, d), rnd(m, dff), rnd(m, dff)
    gamma, beta = torch.ones(d, device=dev), torch.zeros(d, device=dev)
    _, probs = ops.attn_fwd(qkv, s, b, heads)
    z, _, mean, rstd = ops.add_dropout_layernorm_fwd(x, y, gamma, beta, 1e-5, key, 1, p)
    rows = [
        ("attention forward", lambda: ops.attn_fwd(qkv, s, b, heads),
         lambda: ops.attn_fwd_dropout(qkv, s, b, heads, key, 0, p)),
        ("attention backward (2 kernels)", lambda: ops.attn_bwd(qkv, dout, probs, s, b, heads),
         lambda: ops.attn_bwd_dropout(qkv, dout, probs, s, b, heads, key, 0, p)),
        ("residual add + LayerNorm forward", lambda: ops.layernorm_fwd(ops.add_act(x, y), gamma, beta, 1e-5),
         lambda: ops.add_dropout_layernorm_fwd(x, y, gamma, beta, 1e-5, key, 1, p)),
        ("LayerNorm backward (+ dropout branch)", lambda: ops.layernorm_bwd(z, dout, gamma, mean, rstd),
         lambda: ops.layernorm_bwd_dropout(z, dout, gamma, mean, rstd, key, 1, p)),
        ("GELU forward", lambda: ops.gelu_fwd(h), lambda: ops.gelu_dropout_fwd(h, key, 2, p)),
        ("GELU backward", lambda: ops.gelu_bwd(h, gh), lambda: ops.gelu_dropout_bwd(h, gh, key, 2, p)),
    ]
    return [(name, timeit(plain), timeit(drop)) for name, plain, drop in rows]


def main():
    print(f"GPU: {gpu_line()}")
    ms = step_times()
    print(f"\ntrans_unet_ssim_b64 step graph, batch {BATCH}: {ROUNDS} alternating windows of {STEPS} steps (ms / step)")
    for p, v in ms.items():
        best = min(v)
        print(f"  dropout {p:.1f}: " + " ".join(f"{t:7.2f}" for t in v) +
              f"   best {best:.2f} ms = {BATCH / (best * 1e-3):7.1f} images/s")
    a, c = min(ms[0.0]), min(ms[0.5])
    print(f"  dropout 0.5 vs 0.0: {100 * (c / a - 1):+.2f} % step time (best windows)")
    print("\nViT kernels at S = 64, 4 patches, d = 4096, d_ff = 2048, p = 0.5 (CUDA events, 200 launches, L2-resident)")
    print(f"  {'':40s} {'without':>10s} {'with dropout':>14s}")
    for name, t0, t1 in kernel_times():
        print(f"  {name:40s} {t0:8.1f} us {t1:12.1f} us")


if __name__ == "__main__":
    main()
