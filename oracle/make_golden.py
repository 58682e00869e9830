"""TEST INFRASTRUCTURE ONLY -- generates tests/golden/*.pt by running the UNMODIFIED reference
(located by oracle/ref_import.py) on seeded synthetic checkpoints, inputs and explicit noise.
Run where the reference is available:  python -m oracle.make_golden

No fixture may exceed 1 MB: seeded weights are stored as their seed, layout and digest (load_nvae_tiny),
and a large `purified` tensor as a fixed, seeded sample of its elements (stored_purified).

The reference ships no golden vectors (SURVEY.md section 4), so these fixtures -- outputs of the
reference's own `NVAEDefenseModel.__call__` (src/defenses/ours/abstract_models.py:161-193,
models.py:160-274) and `CelebaIdentityClassifier` (models.py:40-58) -- are what pins the oracle
and the CUDA path on the GPU box, where /root/reference does not exist.
"""
from __future__ import annotations

import hashlib
import math
import os
import shutil
import sys
import tempfile

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)

from oracle import ref_import                                    # noqa: E402
from gen_adversarial_b200 import synth                           # noqa: E402
from gen_adversarial_b200.nvae_spec import (NvaeSpec, NVAE_C32_CONFIG, NVAE_C32_RESOLUTION, tiny_config)  # noqa: E402

GOLDEN = os.path.join(ROOT, "tests", "golden")
SCRATCH = os.path.join(HERE, "_ref", "scratch")


def cosine_alphas(n):   # src/experiments/alpha_learning/common_utils.py:20-22
    return [0.5 * (1 - math.cos(math.pi * (i / n))) for i in range(1, n + 1)]


def linear_alphas(n):   # common_utils.py:15-17
    return [i / n for i in range(1, n + 1)]


def sd_digest(sd) -> str:
    h = hashlib.sha256()
    for k in sorted(sd):
        h.update(k.encode())
        h.update(sd[k].detach().cpu().contiguous().numpy().tobytes())
    return h.hexdigest()


PURIFIED_KEEP = 196608          # elements of a sampled `purified` (half of the 2 x 3 x 256 x 256 E4E output: 786 KB in float32)


def _sample_index(numel: int, keep: int, seed: int) -> torch.Tensor:
    # numpy's legacy RandomState stream is frozen across releases, so the positions never move
    return torch.from_numpy(np.sort(np.random.RandomState(seed).permutation(numel)[:keep]).astype(np.int64))


def sample_purified(out: dict, keep: int = PURIFIED_KEEP, seed: int = 0) -> dict:
    """replace out["purified"] by a seeded sample of `keep` of its elements (full float32 precision)"""
    pur = out.pop("purified")
    idx = _sample_index(pur.numel(), keep, seed)
    out.update(purified_shape=tuple(pur.shape), purified_seed=seed, purified_sample=pur.flatten()[idx].clone())
    return out


def stored_purified(g: dict, pur: torch.Tensor):
    """-> (pur at the positions the fixture stores, the reference's values there): all of `purified`, or its seeded sample"""
    if "purified" in g:
        return pur, g["purified"]
    assert tuple(pur.shape) == tuple(g["purified_shape"]), (tuple(pur.shape), g["purified_shape"])
    idx = _sample_index(pur.numel(), g["purified_sample"].numel(), g["purified_seed"])
    return pur.reshape(-1)[idx.to(pur.device)], g["purified_sample"]


def load_nvae_tiny(path: str) -> dict:
    """tests/golden/nvae_tiny.pt with its "state_dict" regenerated from the stored seed and checked against the stored digest"""
    from gen_adversarial_b200 import synth
    g = torch.load(path, weights_only=True)
    sd = synth.make_nvae_state_dict(g["cfg"], g["resolution"], seed=g["state_dict_seed"])
    assert sd_digest(sd) == g["state_dict_digest"], "synth.make_nvae_state_dict no longer gives the weights the fixture was made with"
    g["state_dict"] = sd
    return g


class _MeanClassifier:
    """stand-in classifier for the purifier-only fixtures (the reference only needs set_device/__call__)."""

    def set_device(self, d):
        pass

    def __call__(self, x):
        return x.mean(dim=(2, 3))


def run_reference_nvae(ckpt, alphas, attenuation, eps, blur, x, noises, classifier=None):
    mm = ref_import.ref_models()
    os.makedirs(SCRATCH, exist_ok=True)
    path = os.path.join(SCRATCH, "nvae_ckpt.pt")
    torch.save(ckpt, path)
    dm = mm.NVAEDefenseModel(classifier or _MeanClassifier(), path, alphas, attenuation, eps, blur, "cpu")
    with torch.no_grad(), ref_import.ExplicitNoise(noises):
        logits, purified = dm(x, preds_only=False)
    return logits, purified


def run_reference_stylegan(kind: str, batch: int = 2):
    """configs 3 / 4 of BASELINE.json through the reference's own `E4EStyleGanDefenseModel` / `TransStyleGanDefenseModel`
    + `CelebaGenderClassifier` / `CarsTypeClassifier` (src/defenses/ours/models.py:17-132,277-353), full-size architectures,
    YAMLs verbatim, seeded synthetic checkpoints in the loaders' formats, explicit noise."""
    import yaml
    mm = ref_import.ref_models()
    os.makedirs(SCRATCH, exist_ok=True)
    if kind == "e4e":
        ckpt, clf, yml, res, n_codes = synth.make_e4e_checkpoint(1024), synth.make_resnet50_checkpoint(), "ours_linear_noise_gender.yaml", 256, 18
        Clf, Def = mm.CelebaGenderClassifier, mm.E4EStyleGanDefenseModel
    else:
        ckpt, clf, yml, res, n_codes = synth.make_trans_checkpoint(512), synth.make_resnext50_checkpoint(), "ours_cosine_blur_cars.yaml", 128, 16
        Clf, Def = mm.CarsTypeClassifier, mm.TransStyleGanDefenseModel
    ap, cp = os.path.join(SCRATCH, f"{kind}_ae.pt"), os.path.join(SCRATCH, f"{kind}_clf.pt")
    torch.save(ckpt, ap)
    torch.save(clf, cp)
    with open(os.path.join(ref_import.REFERENCE_ROOT, "configs", yml)) as f:
        p = yaml.safe_load(f)
    dm = Def(Clf(cp, "cpu"), ap, p["interpolation_alphas"], p["alpha_attenuation"], p["initial_noise_eps"], p["gaussian_blur_input"], "cpu")
    x, noises = synth.synthetic_stylegan_inputs(batch, res, n_codes, seed=42)
    with torch.no_grad(), ref_import.ExplicitNoise(noises):
        logits, purified = dm(x, preds_only=False)
    out = {"yaml": yml, "alphas": p["interpolation_alphas"], "attenuation": p["alpha_attenuation"], "eps": p["initial_noise_eps"],
           "blur": p["gaussian_blur_input"], "batch": batch, "x_seed": 42, "purified": purified, "logits": logits,
           "ae_digest": sd_digest(ckpt["state_dict"]), "clf_digest": sd_digest(clf["state_dict"])}
    print(kind, yml, "purified", purified.min().item(), purified.max().item(), purified.std().item(), "logits", logits.tolist())
    return out


def main_stylegan_paths():
    os.makedirs(GOLDEN, exist_ok=True)
    torch.save(sample_purified(run_reference_stylegan("e4e")), os.path.join(GOLDEN, "e4e_gender_b2.pt"))
    torch.save(run_reference_stylegan("trans"), os.path.join(GOLDEN, "trans_cars_b2.pt"))
    shutil.rmtree(SCRATCH, ignore_errors=True)


def main_stylegan_counts(batch: int = 64, chunk: int = 8):
    """north star: clean-accuracy COUNTS identical on the fp32 path -- logits of the reference's own E4E / Style-Transformer defense calls
    (configs 3 / 4, full-size architectures, YAMLs verbatim) on 64 seeded images, explicit noise; only the logits are stored"""
    import yaml
    mm = ref_import.ref_models()
    os.makedirs(SCRATCH, exist_ok=True)
    for kind in ("e4e", "trans"):
        if kind == "e4e":
            ckpt, clf, yml, res, n_codes = synth.make_e4e_checkpoint(1024), synth.make_resnet50_checkpoint(), "ours_linear_noise_gender.yaml", 256, 18
            Clf, Def = mm.CelebaGenderClassifier, mm.E4EStyleGanDefenseModel
        else:
            ckpt, clf, yml, res, n_codes = synth.make_trans_checkpoint(512), synth.make_resnext50_checkpoint(), "ours_cosine_blur_cars.yaml", 128, 16
            Clf, Def = mm.CarsTypeClassifier, mm.TransStyleGanDefenseModel
        with open(os.path.join(ref_import.REFERENCE_ROOT, "configs", yml)) as f:
            p = yaml.safe_load(f)
        with ref_import.InMemoryCheckpoints({"mem://ae": ckpt, "mem://clf": clf}):
            dm = Def(Clf("mem://clf", "cpu"), "mem://ae", p["interpolation_alphas"], p["alpha_attenuation"], p["initial_noise_eps"],
                     p["gaussian_blur_input"], "cpu")
        x, noises = synth.synthetic_stylegan_inputs(batch, res, n_codes, seed=4242)
        logits = []
        for i in range(0, batch, chunk):
            with torch.no_grad(), ref_import.ExplicitNoise([noises[0][i:i + chunk], noises[1][:, i:i + chunk]]):
                logits.append(dm(x[i:i + chunk]))
            print(kind, "chunk", i, flush=True)
        logits = torch.cat(logits)
        torch.save({"yaml": yml, "alphas": p["interpolation_alphas"], "attenuation": p["alpha_attenuation"], "eps": p["initial_noise_eps"],
                    "blur": p["gaussian_blur_input"], "batch": batch, "x_seed": 4242, "logits": logits,
                    "ae_digest": sd_digest(ckpt["state_dict"]), "clf_digest": sd_digest(clf["state_dict"])},
                   os.path.join(GOLDEN, f"{kind}_counts_b{batch}.pt"))
        print(kind, "argmax histogram", torch.bincount(logits.argmax(1)).tolist())


def main_generator():
    import importlib
    ref_import.install()
    gen = importlib.import_module("src.mlvgms_autoencoders.StyleGan_E4E.stylegan2.generator")
    sd = synth.make_stylegan2_state_dict(32, seed=2)
    G = gen.Generator(32, 512, 8, channel_multiplier=2).eval()
    G.load_state_dict(sd, strict=True)
    g = torch.Generator().manual_seed(0)
    latent = torch.randn(3, G.n_latent, 512, generator=g) * 0.7
    z = torch.randn(G.n_latent, 3, 512, generator=g)
    with torch.no_grad():
        img, _ = G([latent], input_is_latent=True, randomize_noise=False)           # Generator.forward, generator.py:407-479
        w = torch.stack([G.style(n) for n in z], dim=0)                              # models.py:120
    torch.save({"seed": 2, "size": 32, "latent": latent, "z": z, "image": img, "image_pool2": torch.nn.functional.avg_pool2d(img, 2),
                "w": w}, os.path.join(GOLDEN, "stylegan2_gen32.pt"))
    print("stylegan2 gen32", img.abs().max().item(), img.std().item())


def main():
    os.makedirs(GOLDEN, exist_ok=True)
    torch.manual_seed(0)
    # ---------------------------------------------------------------- tiny architecture, weights stored
    cfg, res = tiny_config(), (3, 32, 32)
    spec = NvaeSpec(cfg, res)
    ckpt = synth.make_nvae_checkpoint(cfg, res, seed=3)
    x, _ = synth.synthetic_batch(3, res, seed=11)
    noises = synth.synthetic_noise(spec, 3, seed=12)
    cases = []
    for name, alphas, att, eps, blur in [("cosine_noise", cosine_alphas(spec.n_latents), 0.7, 2.0, False),
                                         ("linear_blur", linear_alphas(spec.n_latents), 1.0, 0.0, True),
                                         ("alpha0_blur_noise", [0.0] * spec.n_latents, 1.0, 1.0, True)]:
        _, pur = run_reference_nvae(ckpt, alphas, att, eps, blur, x, noises)
        cases.append({"name": name, "alphas": alphas, "attenuation": att, "eps": eps, "blur": blur, "purified": pur})
        print("tiny", name, pur.mean().item(), pur.std().item())
    sd = ckpt["state_dict_temp=0.6"]
    torch.save({"cfg": cfg, "resolution": res, "state_dict_seed": 3, "state_dict_digest": sd_digest(sd),
                "state_dict_layout": {k: tuple(v.shape) for k, v in sd.items()}, "x": x,
                "noises": noises, "cases": cases}, os.path.join(GOLDEN, "nvae_tiny.pt"))

    # ---------------------------------------------------------------- C32 + VGG11 (weights regenerated from seeds)
    cfg, res = NVAE_C32_CONFIG, NVAE_C32_RESOLUTION
    spec = NvaeSpec(cfg, res)
    ckpt = synth.make_nvae_checkpoint(cfg, res, seed=0)
    vgg_ckpt = synth.make_vgg11_checkpoint(100, seed=1)
    vpath = os.path.join(SCRATCH, "vgg_ckpt.pt")
    os.makedirs(SCRATCH, exist_ok=True)
    torch.save(vgg_ckpt, vpath)
    mm = ref_import.ref_models()
    clf = mm.CelebaIdentityClassifier(vpath, "cpu")
    import yaml
    out = {"nvae_seed": 0, "vgg_seed": 1, "x_seed": 42, "noise_seed": 7, "batch": 4,
           "nvae_digest": sd_digest(ckpt["state_dict_temp=0.6"]),
           "vgg_small_digest": sd_digest({k: v for k, v in vgg_ckpt["state_dict"].items() if "classifier.0" not in k}),
           "cases": []}
    x, y = synth.synthetic_batch(4, res, seed=42)
    noises = synth.synthetic_noise(spec, 4, seed=7)
    for yml in ("ours_cosine_noise_ids.yaml", "ours_learned_blur_ids.yaml"):
        with open(os.path.join(ref_import.REFERENCE_ROOT, "configs", yml)) as f:
            p = yaml.safe_load(f)
        logits, pur = run_reference_nvae(ckpt, p["interpolation_alphas"], p["alpha_attenuation"],
                                         p["initial_noise_eps"], p["gaussian_blur_input"], x, noises, clf)
        out["cases"].append({"yaml": yml, "alphas": p["interpolation_alphas"], "attenuation": p["alpha_attenuation"],
                             "eps": p["initial_noise_eps"], "blur": p["gaussian_blur_input"],
                             "purified": pur, "logits": logits})
        print("c32", yml, pur.mean().item(), pur.std().item(), logits.abs().mean().item(), logits.argmax(1).tolist())
    torch.save(out, os.path.join(GOLDEN, "nvae_c32_vgg11.pt"))
    main_generator()
    main_stylegan_paths()
    shutil.rmtree(SCRATCH, ignore_errors=True)
    for f in sorted(os.listdir(GOLDEN)):
        print(f, os.path.getsize(os.path.join(GOLDEN, f)))


if __name__ == "__main__":
    which = sys.argv[1] if len(sys.argv) > 1 else "all"
    {"all": main, "generator": main_generator, "stylegan_paths": main_stylegan_paths, "stylegan_counts": main_stylegan_counts}[which]()
