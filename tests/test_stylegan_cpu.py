"""CPU: StyleGAN2 generator host logic (weight folds, modulation-as-scaling, up-conv + blur as 4 phase convs, batched
mapping MLP, code mixing) through the torch emulation of the kernels, against the committed fixture produced by the
UNMODIFIED reference Generator (oracle/make_golden.py)."""
import os

import pytest
import torch

from gen_adversarial_b200 import synth, stylegan_engine
from tests import emu_ops

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "stylegan2_gen32.pt")


@pytest.fixture()
def emu(monkeypatch):
    monkeypatch.setattr(stylegan_engine, "ops", emu_ops)
    return emu_ops


@pytest.mark.parametrize("mode,tol", [("fp32", 2e-4), ("bf16", 6e-2)])
def test_generator_matches_reference(emu, mode, tol):
    """full-resolution image and mapping-network output of the reference Generator (generator.py:407-479, models.py:120), as stored
    in the fixture for its seeded weights, latents and z"""
    g = torch.load(GOLDEN, weights_only=True)
    sd = synth.make_stylegan2_state_dict(g["size"], seed=g["seed"])
    latent, z, img_ref, w_ref = g["latent"], g["z"], g["image"], g["w"]
    n_latent = latent.shape[1]
    eng = stylegan_engine.StyleGan2Engine(sd, g["size"], "cpu", mode, _host_logic_test=True)
    img = eng.decode(latent, pool=1)
    w = eng.mapping(z.reshape(-1, 512)).reshape(z.shape)
    scale = img_ref.abs().max().item()
    assert (img - img_ref).abs().max().item() <= tol * scale, ((img - img_ref).abs().max().item(), scale)
    assert (w - w_ref).abs().max().item() <= tol * max(1.0, w_ref.abs().max().item())
    # per-level mixing (models.py:117-127)
    alphas = torch.linspace(0, 1, n_latent)
    mixed_ref = ((1 - alphas.view(-1, 1, 1)) * latent.permute(1, 0, 2) + alphas.view(-1, 1, 1) * w_ref).permute(1, 0, 2)
    mixed = eng.mix_codes(latent, z, alphas)
    assert (mixed - mixed_ref).abs().max().item() <= tol * max(1.0, mixed_ref.abs().max().item())


def test_generator_matches_reference_fixture(emu):
    if not os.path.exists(GOLDEN):
        pytest.skip("fixture not generated")
    g = torch.load(GOLDEN, weights_only=True)
    sd = synth.make_stylegan2_state_dict(32, seed=g["seed"])
    eng = stylegan_engine.StyleGan2Engine(sd, 32, "cpu", "fp32", _host_logic_test=True)
    img = eng.decode(g["latent"], pool=2)
    scale = g["image_pool2"].abs().max().item()
    assert (img - g["image_pool2"]).abs().max().item() <= 2e-4 * scale


def test_superpixel_weights_are_the_same_convolution():
    """stylegan_engine.superpixel_weights: a 3x3 conv on [h][w][c] equals the transformed conv on the [h][w/2][2c] view (exact in fp64)"""
    import torch
    import torch.nn.functional as F
    from gen_adversarial_b200.stylegan_engine import superpixel_weights
    g = torch.Generator().manual_seed(0)
    for cin, cout, h, w in ((4, 6, 5, 8), (32, 32, 6, 12), (3, 2, 4, 2)):
        wt = torch.randn(cout, cin, 3, 3, generator=g, dtype=torch.float64)
        x = torch.randn(2, h, w, cin, generator=g, dtype=torch.float64)                      # NHWC
        ref = F.conv2d(x.permute(0, 3, 1, 2), wt, padding=1).permute(0, 2, 3, 1)              # [n, h, w, cout]
        xs = x.reshape(2, h, w // 2, 2 * cin)
        got = F.conv2d(xs.permute(0, 3, 1, 2), superpixel_weights(wt), padding=1).permute(0, 2, 3, 1).reshape(2, h, w, cout)
        assert (got - ref).abs().max().item() <= 1e-12
