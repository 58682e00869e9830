"""CPU: the oracle restatement (oracle/nvae_ref.py) against fixtures produced by the reference itself."""
import torch

from oracle import nvae_ref
from gen_adversarial_b200 import synth
from gen_adversarial_b200.nvae_spec import NvaeSpec, NVAE_C32_CONFIG, NVAE_C32_RESOLUTION


def test_oracle_matches_reference_fixture_tiny(golden_tiny):
    g = golden_tiny
    spec = NvaeSpec(g["cfg"], g["resolution"])
    for case in g["cases"]:
        alphas = [a * case["attenuation"] for a in case["alphas"]]
        with torch.no_grad():
            _, pur = nvae_ref.defense_call(g["state_dict"], spec, None, g["x"], alphas, g["noises"],
                                           case["eps"], case["blur"])
        err = (pur - case["purified"]).abs().max().item()
        assert err <= 1e-5, (case["name"], err)


def test_oracle_matches_reference_fixture_c32_first_sample(golden_c32):
    """C32 + VGG11 fixture (weights regenerated from seeds): purifier on all 4 samples of one yaml."""
    g = golden_c32
    spec = NvaeSpec(NVAE_C32_CONFIG, NVAE_C32_RESOLUTION)
    sd = synth.make_nvae_state_dict(seed=g["nvae_seed"])
    x, _ = synth.synthetic_batch(g["batch"], seed=g["x_seed"])
    noises = synth.synthetic_noise(spec, g["batch"], seed=g["noise_seed"])
    case = g["cases"][1]
    alphas = [a * case["attenuation"] for a in case["alphas"]]
    with torch.no_grad():
        _, pur = nvae_ref.defense_call(sd, spec, None, x, alphas, noises, case["eps"], case["blur"])
    err = (pur - case["purified"]).abs().max().item()
    assert err <= 1e-4, err


def test_blur_kernel_sizes():
    # src/defenses/ours/abstract_models.py:150-156
    assert nvae_ref.gaussian_blur_ksize(64) == 15
    assert nvae_ref.gaussian_blur_ksize(128) == 31
    assert nvae_ref.gaussian_blur_ksize(256) == 255


def test_noise_is_l2_normalised_and_clamped():
    x = torch.rand(3, 3, 16, 16)
    n = torch.randn(3, 3, 16, 16)
    y = nvae_ref.add_gaussian_noise(x, n, 2.0)
    assert y.min() >= 0 and y.max() <= 1
    d = (x + n * (2.0 / n.flatten(1).norm(dim=1).view(-1, 1, 1, 1))).clamp(0, 1)
    assert torch.equal(y, d)
    # eps = 0 leaves the image unchanged but still clamps
    assert torch.equal(nvae_ref.add_gaussian_noise(x, n, 0.0), x)


def test_pgd_step_projection():
    x = torch.rand(2, 3, 8, 8)
    xa = x.clone()
    g = torch.randn_like(x)
    eps, step = 8 / 255, 2 / 255
    for _ in range(10):
        xa = nvae_ref.pgd_linf_step(xa, g, x, step, eps)
    assert (xa - x).abs().max() <= eps + 1e-7
    assert xa.min() >= 0 and xa.max() <= 1


def test_stylegan_oracle_matches_reference_fixtures():
    """oracle/stylegan_ref.py (configs 3 and 4, full-size architectures, batch 2) against the reference's own outputs"""
    import os
    from oracle import stylegan_ref
    from oracle.make_golden import stored_purified
    golden = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
    for kind, res, n_codes, mk_ae, mk_clf, fn in (
            ("e4e_gender_b2.pt", 256, 18, lambda: synth.make_e4e_checkpoint(1024), synth.make_resnet50_checkpoint, stylegan_ref.e4e_defense_call),
            ("trans_cars_b2.pt", 128, 16, lambda: synth.make_trans_checkpoint(512), synth.make_resnext50_checkpoint, stylegan_ref.trans_defense_call)):
        g = torch.load(os.path.join(golden, kind), weights_only=True)
        x, noises = synth.synthetic_stylegan_inputs(g["batch"], res, n_codes, seed=g["x_seed"])
        alphas = [a * g["attenuation"] for a in g["alphas"]]
        with torch.no_grad():
            logits, pur = fn(mk_ae(), mk_clf()["state_dict"], x, alphas, noises, g["eps"], g["blur"])
        got, ref = stored_purified(g, pur)
        assert (got - ref).abs().max().item() <= 1e-5, kind
        assert ((logits - g["logits"]).abs().max() / g["logits"].abs().max()).item() <= 1e-4, kind
