"""CPU: host-side logic of the StyleGAN purification paths (BASELINE configs 3 and 4: IR-SE50 + map2style / transformer
encoders, latent mixing, generator, output pooling, ResNet-50 / ResNeXt-50) driven through the torch emulation of the
kernels (tests/emu_ops.py), against the oracle restatement and against the fixtures produced by the unmodified reference."""
import functools
import os

import pytest
import torch

from gen_adversarial_b200 import synth, stylegan_engine, irse_engine, resnet_engine
from gen_adversarial_b200.defenses.ours import models as ga_models, abstract_models as ga_abstract
from oracle import stylegan_ref
from oracle.make_golden import stored_purified
from tests import emu_ops

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


@pytest.fixture()
def emu(monkeypatch):
    for m in (stylegan_engine, irse_engine, resnet_engine, ga_models, ga_abstract):
        monkeypatch.setattr(m, "ops", emu_ops)
    for name in ("E4EEncoderEngine", "TransEncoderEngine", "StyleGan2Engine", "ResNetEngine"):
        monkeypatch.setattr(ga_models, name, functools.partial(getattr(ga_models, name), _host_logic_test=True))
    return emu_ops


def _alphas_dev_cpu(self):
    return torch.tensor([float(a) for a in self.interpolation_alphas], dtype=torch.float32)


@pytest.fixture()
def cpu_alphas(monkeypatch):
    monkeypatch.setattr(ga_abstract.MLVGMDefenseModel, "_alphas_device", _alphas_dev_cpu)


def test_resnet_engines_match_oracle(emu):
    for groups, mk, res in ((1, synth.make_resnet50_checkpoint, 128), (32, synth.make_resnext50_checkpoint, 64)):
        sd = mk()["state_dict"]
        x = torch.rand(2, 3, res, res, generator=torch.Generator().manual_seed(0))
        with torch.no_grad():
            ref = stylegan_ref.resnet_forward(sd, (x - 0.5) / 0.5, groups)
        eng = resnet_engine.ResNetEngine(sd, "cpu", "fp32", groups=groups, _host_logic_test=True)
        out = eng.forward(emu.nchw_to_nhwc(x, torch.float32, 2.0, -1.0))
        rel = ((out - ref).abs().max() / ref.abs().max()).item()
        assert rel <= 1e-4, (groups, rel)


def _defense(kind, mode):
    if kind == "e4e":
        clf = ga_models.CelebaGenderClassifier(synth.make_resnet50_checkpoint(), "cpu", mode=mode)
        alphas = [round((i + 1) / 18, 2) for i in range(18)]
        return ga_models.E4EStyleGanDefenseModel(clf, synth.make_e4e_checkpoint(1024), alphas, 1.0, 4.0, False, "cpu", mode=mode)
    clf = ga_models.CarsTypeClassifier(synth.make_resnext50_checkpoint(), "cpu", mode=mode)
    alphas = [0.5 * (1 - __import__("math").cos(__import__("math").pi * i / 16)) for i in range(1, 17)]
    return ga_models.TransStyleGanDefenseModel(clf, synth.make_trans_checkpoint(512), alphas, 0.7, 0.0, True, "cpu", mode=mode)


@pytest.mark.parametrize("kind,res,n_codes", [("e4e", 256, 18), ("trans", 128, 16)])
def test_defense_host_logic_matches_reference_fixture(emu, cpu_alphas, kind, res, n_codes):
    """whole `__call__` of the drop-in defense classes (fp32 host logic) against the reference's own outputs"""
    path = os.path.join(GOLDEN, "e4e_gender_b2.pt" if kind == "e4e" else "trans_cars_b2.pt")
    if not os.path.exists(path):
        pytest.skip("fixture not generated")
    g = torch.load(path, weights_only=True)
    x, noises = synth.synthetic_stylegan_inputs(g["batch"], res, n_codes, seed=g["x_seed"])
    dm = _defense(kind, "fp32")
    dm.interpolation_alphas = [a * g["attenuation"] for a in g["alphas"]]
    dm.eps, dm.blur_input = g["eps"], g["blur"]
    dm.set_explicit_noise(noises)
    logits, pur = dm(x, preds_only=False)
    got, ref = stored_purified(g, pur)
    err = (got - ref).abs().max().item()
    rel = ((logits - g["logits"]).abs().max() / g["logits"].abs().max()).item()
    assert err <= 1e-4, (kind, err)
    assert rel <= 1e-3, (kind, rel)
    assert logits.argmax(1).tolist() == g["logits"].argmax(1).tolist()
    # standalone purify(): normalised in, normalised out (abstract_models.py:176-185)
    if kind == "e4e":
        dm.set_explicit_noise([noises[0], noises[1]])
        xn = stylegan_ref._preprocess(x, noises[0], g["eps"], g["blur"])
        p2 = dm.purify(xn)
        got, ref = stored_purified(g, p2 * 0.5 + 0.5)
        assert (got - ref).abs().max().item() <= 1e-4
