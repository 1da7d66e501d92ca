"""CPU-only checks of the bench.py contract and of the host-side optimizer logic (no GPU needed)."""
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line_with_the_contract_keys(tmp_path):
    """`bench.py --impl reference` times the reference's CPU path (oracle port) and prints exactly one JSON line;
    --dump-outputs writes the values the last step logged."""
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                          "--warmup", "1", "--batch", "8", "--dump-outputs", str(tmp_path)],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, out.stdout
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "pix2pix_gan_train_images_per_sec_256x256"
    assert d["unit"] == "images/s" and d["higher_is_better"] is True and d["value"] > 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and d["n_gpus"] == 1 and d["steps"] == 1 and d["warmup"] == 1
    assert d["config"]["batch_per_gpu"] == 8      # the arm runs the batch it is given (default: 64, the same as our arm)
    check_dumped_outputs(tmp_path)


def check_dumped_outputs(out_dir):
    """What `bench.py --dump-outputs` writes for the GAN step: the five values it logged, float32 scalars."""
    import numpy as np
    arrays = {p.name[:-4]: np.load(p) for p in out_dir.iterdir()}
    assert set(arrays) == {"d_loss", "loss", "train_ssim", "train_psnr", "train_rmse"}
    for name, a in arrays.items():
        assert a.dtype == np.float32 and a.shape == () and np.isfinite(a), name
    assert 0 < arrays["train_ssim"] < 1 and arrays["train_rmse"] > 0


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2",
                          "--steps", "1", "--warmup", "1"], capture_output=True, text=True, timeout=600, cwd=ROOT, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_fused_adam_on_cpu_parameters_is_torch_adam():
    """Non-CUDA parameters take torch.optim.Adam.step unchanged (optimizer plumbing, not the hot path)."""
    from pai_b200.optim import FusedAdam
    torch.manual_seed(0)
    w = torch.nn.Parameter(torch.randn(8, 4, 4, 4))
    r = torch.nn.Parameter(w.detach().clone())
    hyper = dict(lr=2e-4, betas=(0.5, 0.999), eps=1e-7)
    a, b = FusedAdam([w], **hyper), torch.optim.Adam([r], **hyper)
    for _ in range(3):
        g = torch.randn_like(w)
        w.grad, r.grad = g.clone(), g.clone()
        a.step()
        b.step()
    assert torch.equal(w, r)
    sa, sb = a.state_dict(), b.state_dict()
    assert float(sa["state"][0]["step"]) == float(sb["state"][0]["step"]) == 3.0
    assert torch.equal(sa["state"][0]["exp_avg"], sb["state"][0]["exp_avg"])
