"""Pins oracle/pix2pix_port.py (the travelling CPU restatement of the reference's Pix2Pix
training path) against fixtures produced by the real reference (oracle/gen_golden.py) and,
when $PAI_REFERENCE_DIR names a checkout of it, against the reference modules directly."""
import os
import sys

import numpy as np
import pytest
import torch

import pix2pix_port as port


@pytest.fixture(scope="module")
def gz(golden_dir):
    return np.load(os.path.join(golden_dir, "pix2pix_ref.npz"))


@pytest.fixture(scope="module")
def state():
    return port.init_state(0, in_channels=1, out_channels=1, loss_type="gan", disc_in_channels=1)


def test_init_replay_matches_reference_checksums(gz, state):
    keys = list(gz["state_keys"])
    assert sorted(state.keys()) == keys
    cs = np.array([[float(state[k].double().sum()), float(state[k].double().abs().sum())] for k in keys])
    assert np.array_equal(cs, gz["state_checksums"])


def test_parameter_counts(state):
    g = sum(v.numel() for k, v in state.items() if k.startswith("unet.") and port._is_param(k))
    d = sum(v.numel() for k, v in state.items() if k.startswith("discriminator."))
    assert g == 54_413_313 and d == 2_763_712        # SURVEY.md 8(a) A1/A3


def test_eval_forward_and_discriminator(gz, state):
    x, target = port.synthetic_pairs(2, seed=1234)
    sd = {k: v.clone() for k, v in state.items()}
    with torch.no_grad():
        y = port.unet_forward(sd, x, training=False)
        logits = port.disc_forward(sd, x, target)
    assert np.abs(y[:, :, ::4, ::4].numpy() - gz["gen_eval_sub"]).max() < 1e-5
    assert np.abs(logits.numpy() - gz["disc_logits"]).max() < 1e-5


def test_train_forward_and_gradients(gz, state):
    x, target = port.synthetic_pairs(2, seed=1234)
    tr = port.OracleTrainer(state, "gan")
    y = port.unet_forward(tr.sd, x, training=True)
    assert np.abs(y.detach()[:, :, ::4, ::4].numpy() - gz["gen_train_sub"]).max() < 2e-5
    loss = port.generator_loss(tr.sd, "gan", x, y, target)
    assert float(loss) == pytest.approx(float(gz["gan_gloss0"]), rel=1e-5)
    loss.backward()
    norms = {k: float(tr.sd[k].grad.double().norm()) for k in tr.g_keys + tr.d_keys if tr.sd[k].grad is not None}
    for k, want in zip(gz["grad_keys"], gz["grad_norms"]):
        assert norms[str(k)] == pytest.approx(float(want), rel=2e-3, abs=1e-6), k


@pytest.mark.parametrize("loss_type,prefix", [("gan", "gan_log_"), ("ssim+psnr", "sp_log_")])
def test_three_training_steps(gz, loss_type, prefix):
    x, target = port.synthetic_pairs(2, seed=1234)
    sd = port.init_state(0, 1, 1, loss_type=loss_type, disc_in_channels=1)
    tr = port.OracleTrainer(sd, loss_type)
    for _ in range(3):
        tr.training_step(x, target)
    for k, v in tr.logged.items():
        want = gz[prefix + k]
        assert np.allclose(np.array(v), want, rtol=2e-3, atol=1e-5), (k, v, want)
    if loss_type == "gan":
        keys = list(gz["state_keys"])
        cs = np.array([float(tr.sd[k].detach().double().abs().sum()) for k in keys])
        assert np.allclose(cs, gz["state_checksums_after3"][:, 1], rtol=1e-3)


@pytest.mark.reference
def test_against_live_reference(state, reference_dir):
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    import torchvision  # noqa: F401  (its import inspects sys.modules; do it before the namespace swap)
    sys.path.insert(0, os.path.join(root, "oracle", "shim"))
    sys.path.insert(0, reference_dir)
    saved = {k: sys.modules.pop(k) for k in list(sys.modules) if k == "models" or k.startswith("models.")}
    # the reference's ``models`` is a namespace package (no __init__.py): a regular package of the same
    # name anywhere on sys.path would win, so the drop-in package's directory steps aside for this test
    pkg = os.path.join(root, "thesis-pai-reconstruction_b200")
    hidden = [p for p in sys.path if os.path.abspath(p) == pkg]
    sys.path[:] = [p for p in sys.path if os.path.abspath(p) != pkg]
    try:
        from models.pix2pix import Pix2Pix
        from models.wrapper import Discriminator
        from models.utils import init_weights
        torch.manual_seed(0)
        m = Pix2Pix(in_channels=1, out_channels=1, dropout=0.0, loss_type="gan")
        m.discriminator = Discriminator(in_channels=1)
        m.discriminator.apply(init_weights)
        for k, v in m.state_dict().items():
            assert torch.equal(v, state[k]), k
        x, target = port.synthetic_pairs(2, seed=99)
        m.train()
        tr = port.OracleTrainer(state, "gan")
        for _ in range(2):
            m.training_step((x, target), 0)
            tr.training_step(x, target)
        for k in m.logged:
            assert np.allclose(m.logged[k], tr.logged[k], rtol=1e-4, atol=1e-6), k
    finally:
        for k in [k for k in sys.modules if k == "models" or k.startswith("models.")]:
            del sys.modules[k]
        sys.modules.update(saved)
        sys.path[:0] = hidden
        sys.path.remove(reference_dir)
        sys.path.remove(os.path.join(root, "oracle", "shim"))
