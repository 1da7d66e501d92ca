"""Dumps the eval-mode output and one train-mode gradient set of the 1-channel res_18_small, attention and trans_small
models (the cases of tests/test_variants_gpu.py, same seeds and inputs) as DIR/<case>.npz, so two builds of the
project can be compared bit for bit.  ``--tree`` runs another checkout (with its library built) instead of this one.

    python profiles/scripts/dump_1ch.py OUT_DIR [--tree CHECKOUT]
    python profiles/scripts/dump_1ch.py --compare DIR_A DIR_B
"""
import argparse
import os
import sys

import numpy as np

CASES = {
    "res_18_small": ("models.res_unet", "ResUnetGAN", dict(res_type="18", channel_mults=(1, 2, 4, 8)), 4, 64, "ssim+psnr"),
    "attention": ("models.attention_unet", "AttentionUnetGAN", dict(), 2, 256, "ssim"),
    "trans_small": ("models.trans_unet", "TransUnetGAN", dict(channel_mults=(1, 2, 2), patch_size=4), 2, 256, "ssim"),
}


def dump(out, tree):
    for p in (os.path.join(tree, "thesis-pai-reconstruction_b200"), os.path.join(tree, "oracle")):
        sys.path.insert(0, p)
    import importlib

    import torch

    import pix2pix_port as port
    os.makedirs(out, exist_ok=True)
    for name, (module, cls, kwargs, n, res, loss_type) in CASES.items():
        torch.manual_seed(0)
        m = getattr(importlib.import_module(module), cls)(in_channels=1, out_channels=1, dropout=0.0, loss_type=loss_type,
                                                          **kwargs).cuda()
        x, t = port.synthetic_pairs(n, seed=1234)
        x, t = x[:, :, :res, :res].contiguous().cuda(), t[:, :, :res, :res].contiguous().cuda()
        m.eval()
        with torch.no_grad():
            y_eval = m(x)
        m.train()
        y = m(x)
        m.loss(x, y, t).backward()
        arrs = {"eval": y_eval.cpu().numpy(), "train": y.detach().cpu().numpy()}
        for k, p in m.named_parameters():
            if p.grad is not None:
                arrs["grad/" + k] = p.grad.cpu().numpy()
        np.savez(os.path.join(out, name + ".npz"), **arrs)
        print(f"{name}: {len(arrs) - 2} gradients")


def compare(a, b):
    for name in CASES:
        za, zb = np.load(os.path.join(a, name + ".npz")), np.load(os.path.join(b, name + ".npz"))
        assert sorted(za.files) == sorted(zb.files), name
        diff = [k for k in za.files if not np.array_equal(za[k], zb[k])]
        worst = max((float(np.abs(za[k] - zb[k]).max() / max(np.abs(za[k]).max(), 1e-30)) for k in diff), default=0.0)
        print(f"{name}: {len(za.files) - len(diff)}/{len(za.files)} arrays bit-identical; eval "
              f"{'identical' if 'eval' not in diff else 'DIFFERENT'}, train output "
              f"{'identical' if 'train' not in diff else 'different'}; largest relative difference {worst:.2e}"
              + (f" in {len(diff)} arrays ({', '.join(diff[:4])}{', ...' if len(diff) > 4 else ''})" if diff else ""))


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("out", nargs="?")
    ap.add_argument("--tree", default=os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
    ap.add_argument("--compare", nargs=2)
    args = ap.parse_args()
    if args.compare:
        compare(*args.compare)
    else:
        dump(args.out, os.path.abspath(args.tree))
