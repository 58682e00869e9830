"""CPU: the oracle restatement against the UNMODIFIED reference.  The state-dict layout is checked against the committed fixtures;
the other tests import the reference tree through oracle/ref_import.py and skip where it is absent (the repository does not contain
it: oracle/ref_import.py says where it looks, GA_REFERENCE_ROOT among them)."""
import math
import os

import pytest
import torch

from oracle import ref_import, nvae_ref
from oracle.make_golden import sd_digest
from gen_adversarial_b200 import synth
from gen_adversarial_b200.nvae_spec import NvaeSpec, NVAE_C32_CONFIG, NVAE_C32_RESOLUTION, tiny_config

needs_reference = pytest.mark.skipif(not ref_import.reference_available(), reason="reference tree not found (oracle/ref_import.py)")


class _MeanClassifier:
    def set_device(self, d):
        pass

    def __call__(self, x):
        return x.mean(dim=(2, 3))


@pytest.mark.parametrize("cfg,res", [(tiny_config(), (3, 32, 32)), (NVAE_C32_CONFIG, NVAE_C32_RESOLUTION)])
def test_state_dict_layout_matches_reference(cfg, res, golden_tiny, golden_c32):
    """The reference's AutoEncoder loaded the state dicts behind the committed fixtures with strict=True (loading_utils.py:63).  Tiny:
    the fixture stores that state dict's key layout.  C32: oracle/make_golden.py fed exactly make_nvae_state_dict(seed=0) to the
    reference's loader and stored its value digest, so the digest pins the layout (and the values) the reference accepted."""
    if (cfg, tuple(res)) == (NVAE_C32_CONFIG, tuple(NVAE_C32_RESOLUTION)):
        assert sd_digest(synth.make_nvae_state_dict(cfg, res, seed=golden_c32["nvae_seed"])) == golden_c32["nvae_digest"]
        return
    assert (cfg, tuple(res)) == (golden_tiny["cfg"], tuple(golden_tiny["resolution"])), "tiny_config() no longer matches nvae_tiny.pt"
    ref_layout = golden_tiny["state_dict_layout"]
    mine = synth.make_nvae_state_dict(cfg, res, seed=0)
    assert set(ref_layout) == set(mine)
    for k in ref_layout:
        assert tuple(ref_layout[k]) == tuple(mine[k].shape), k


@needs_reference
def test_restatement_matches_reference_call(tmp_path):
    cfg, res = tiny_config(initial_channels=8, groups=3, scales=3, latent=6), (3, 64, 64)
    spec = NvaeSpec(cfg, res)
    ckpt = synth.make_nvae_checkpoint(cfg, res, seed=5)
    path = os.path.join(tmp_path, "nvae.pt")
    torch.save(ckpt, path)
    mm = ref_import.ref_models()
    n = spec.n_latents
    alphas = [0.5 * (1 - math.cos(math.pi * i / n)) for i in range(1, n + 1)]
    dm = mm.NVAEDefenseModel(_MeanClassifier(), path, alphas, 0.7, 2.0, True, "cpu")
    x, _ = synth.synthetic_batch(2, res, seed=1)
    noises = synth.synthetic_noise(spec, 2, seed=2)
    with torch.no_grad(), ref_import.ExplicitNoise(noises):
        _, pur_ref = dm(x, preds_only=False)
    with torch.no_grad():
        _, pur = nvae_ref.defense_call(ckpt["state_dict_temp=0.6"], spec, None, x, [a * 0.7 for a in alphas],
                                       noises, 2.0, True)
    assert (pur - pur_ref).abs().max().item() <= 1e-5


@needs_reference
def test_normalizing_flow_config_matches_reference(tmp_path):
    """A12: a configuration with num_nf_cells = 1 -- state_dict layout (incl. the MaskedConv2d mask buffers, architecture.py:9-34) and
    the whole defense call against the unmodified reference (src/defenses/ours/models.py:209-210,253-254)."""
    cfg, res = tiny_config(initial_channels=8, groups=2, scales=2, latent=4), (3, 32, 32)
    cfg["num_nf_cells"] = 1
    spec = NvaeSpec(cfg, res)
    ae = ref_import.ref_nvae_module().AutoEncoder(cfg, res)
    ref_sd = ae.state_dict()
    mine = synth.make_nvae_state_dict(cfg, res, seed=12)
    assert set(ref_sd) == set(mine)
    for k in ref_sd:
        assert tuple(ref_sd[k].shape) == tuple(mine[k].shape), k
        if k.endswith(".mask"):
            assert torch.equal(ref_sd[k], mine[k]), k              # the masks are fixed by (mirror, zero_diag), not learned
    ckpt = synth.make_nvae_checkpoint(cfg, res, seed=12)
    path = os.path.join(tmp_path, "nvae_nf.pt")
    torch.save(ckpt, path)
    mm = ref_import.ref_models()
    n = spec.n_latents
    alphas = [i / n for i in range(1, n + 1)]
    dm = mm.NVAEDefenseModel(_MeanClassifier(), path, alphas, 0.7, 1.0, True, "cpu")
    x, _ = synth.synthetic_batch(2, res, seed=1)
    noises = synth.synthetic_noise(spec, 2, seed=2)
    with torch.no_grad(), ref_import.ExplicitNoise(noises):
        _, pur_ref = dm(x, preds_only=False)
    with torch.no_grad():
        _, pur = nvae_ref.defense_call(ckpt["state_dict_temp=0.6"], spec, None, x, [a * 0.7 for a in alphas], noises, 1.0, True)
    assert (pur - pur_ref).abs().max().item() <= 1e-5


@needs_reference
def test_restatement_gradient_matches_reference(tmp_path):
    """input-gradient of the oracle == autograd through the reference (attack path, untargeted.py:146)."""
    cfg, res = tiny_config(), (3, 32, 32)
    spec = NvaeSpec(cfg, res)
    ckpt = synth.make_nvae_checkpoint(cfg, res, seed=6)
    path = os.path.join(tmp_path, "nvae.pt")
    torch.save(ckpt, path)
    mm = ref_import.ref_models()
    n = spec.n_latents
    alphas = [i / n for i in range(1, n + 1)]
    dm = mm.NVAEDefenseModel(_MeanClassifier(), path, alphas, 1.0, 1.0, True, "cpu")
    x, _ = synth.synthetic_batch(2, res, seed=3)
    noises = synth.synthetic_noise(spec, 2, seed=4)
    w = torch.randn(2, 3, 32, 32, generator=torch.Generator().manual_seed(7))
    xr = x.clone().requires_grad_(True)
    with ref_import.ExplicitNoise(noises):
        _, pur_ref = dm(xr, preds_only=False)
    g_ref, = torch.autograd.grad((pur_ref * w).sum(), [xr])
    xo = x.clone().requires_grad_(True)
    _, pur = nvae_ref.defense_call(ckpt["state_dict_temp=0.6"], spec, None, xo, alphas, noises, 1.0, True)
    g, = torch.autograd.grad((pur * w).sum(), [xo])
    assert (g - g_ref).abs().max().item() <= 1e-5 * max(1.0, g_ref.abs().max().item())


@needs_reference
@pytest.mark.parametrize("kind", ["e4e", "trans"])
def test_stylegan_restatement_matches_reference_call(tmp_path, kind):
    """configs 3 / 4: oracle/stylegan_ref.py against the reference's own defense classes (different seeds, blur AND noise on,
    other alpha schedule than the committed fixtures); also checks that the synthetic checkpoints load through the
    reference loaders with strict=True (loading_utils.py:10-49,69-81)."""
    from oracle import stylegan_ref
    mm = ref_import.ref_models()
    if kind == "e4e":
        ckpt, clf = synth.make_e4e_checkpoint(1024, seed=14), synth.make_resnet50_checkpoint(seed=16)
        Clf, Def, res, n_codes, fn = mm.CelebaGenderClassifier, mm.E4EStyleGanDefenseModel, 256, 18, stylegan_ref.e4e_defense_call
    else:
        ckpt, clf = synth.make_trans_checkpoint(512, seed=15), synth.make_resnext50_checkpoint(seed=17)
        Clf, Def, res, n_codes, fn = mm.CarsTypeClassifier, mm.TransStyleGanDefenseModel, 128, 16, stylegan_ref.trans_defense_call
    ap, cp = os.path.join(tmp_path, "ae.pt"), os.path.join(tmp_path, "clf.pt")
    torch.save(ckpt, ap)
    torch.save(clf, cp)
    alphas = [0.5 * (1 - math.cos(math.pi * i / n_codes)) for i in range(1, n_codes + 1)]
    dm = Def(Clf(cp, "cpu"), ap, alphas, 0.8, 2.0, True, "cpu")
    x, noises = synth.synthetic_stylegan_inputs(1, res, n_codes, seed=5)
    with torch.no_grad(), ref_import.ExplicitNoise(noises):
        logits_ref, pur_ref = dm(x, preds_only=False)
    with torch.no_grad():
        logits, pur = fn(ckpt, clf["state_dict"], x, [a * 0.8 for a in alphas], noises, 2.0, True)
    assert (pur - pur_ref).abs().max().item() <= 1e-5
    assert ((logits - logits_ref).abs().max() / logits_ref.abs().max()).item() <= 1e-4
