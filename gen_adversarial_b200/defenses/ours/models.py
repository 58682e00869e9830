"""Concrete defense models -- drop-in for /root/reference/src/defenses/ours/models.py on the CUDA path.

Implemented here: the three classifier wrappers (models.py:17-76) and the three MLVGM defense models
(`NVAEDefenseModel` :135-274, `E4EStyleGanDefenseModel` :79-132, `TransStyleGanDefenseModel` :277-353), i.e. all five
BASELINE configs.  Constructor signatures are the reference's (positional use at
src/experiments/load_defense.py:134-140); `mode` is a keyword-only extension selecting the bf16 tensor-core path or
the exact fp32 path.  Checkpoints are read in the reference's on-disk formats (loading_utils.py:20-26,51-66); a
checkpoint dict may be passed in place of a path (used with synthetic weights).
"""
from __future__ import annotations

import torch
from torch import nn

from ... import ops
from ...nvae_engine import NvaeEngine
from ...nvae_spec import NvaeSpec
from ...vgg_engine import Vgg11Engine
from ...resnet_engine import ResNetEngine
from ...stylegan_engine import StyleGan2Engine
from ...irse_engine import E4EEncoderEngine, TransEncoderEngine
from .abstract_models import BaseClassificationModel, MLVGMDefenseModel, default_mode


def _load_ckpt(path_or_dict):
    if isinstance(path_or_dict, dict):
        return path_or_dict
    return torch.load(path_or_dict, map_location="cpu")


class CelebaIdentityClassifier(BaseClassificationModel, torch.nn.Module):

    def __init__(self, model_path: str, device: str, *, mode: str = None, n_classes: int = 100, image_size: int = 64):
        """
        Wrapper for the CelebA-64 Identities VGG-11 custom model.
        """
        mean = (0.5, 0.5, 0.5)
        std = (0.5, 0.5, 0.5)
        self._mode = mode or default_mode()
        self._image_size = image_size
        super().__init__(model_path, device, mean, std)

    def load_classifier(self, model_path: str, device: str):
        ckpt = _load_ckpt(model_path)           # loading_utils.py:20-26: ckpt['state_dict']
        return Vgg11Engine(ckpt["state_dict"], device, self._mode, in_hw=self._image_size)


class NVAEDefenseModel(MLVGMDefenseModel, torch.nn.Module):

    def __init__(self, classifier: BaseClassificationModel, autoencoder_path: str,
                 interpolation_alphas: tuple, alpha_attenuation: float = 1.0, initial_noise_eps: float = 0.0,
                 apply_gaussian_blur: bool = False, device: str = 'cpu', temperature: float = 0.6, *, mode: str = None):
        """
        Defense model using an NVAE.
        :param temperature: temperature for sampling.
        """
        self.temperature = temperature
        self._mode = mode or default_mode()
        # no need for preprocessing, since it is done directly in NVAE forward pass.
        super().__init__(classifier, autoencoder_path, interpolation_alphas, alpha_attenuation, initial_noise_eps,
                         apply_gaussian_blur, device)
        if len(self.interpolation_alphas) != self.autoencoder.spec.n_latents:
            raise ValueError(f"{len(self.interpolation_alphas)} interpolation alphas for "
                             f"{self.autoencoder.spec.n_latents} latent levels")

    def load_autoencoder(self, model_path: str, device: str):
        ckpt = _load_ckpt(model_path)           # loading_utils.py:51-66
        config = ckpt["configuration"]
        spec = NvaeSpec(config["autoencoder"], config["resolution"])
        return NvaeEngine(ckpt[f"state_dict_temp={self.temperature}"], spec, device, self._mode, self.temperature)

    # ------------------------------------------------------------------
    def _noise_args(self):
        if self._explicit_noise is not None:
            return self._explicit_noise[0], list(self._explicit_noise[1:])
        return None, None

    def purify(self, batch: torch.Tensor) -> torch.Tensor:
        """
        MLVGM encoding procedure to extract the codes.
        :param batch: pre-processed images of shape (B, C, H, W) in [0, 1].
        :return: post_precessed purified reconstructions (B, C, H, W)
        """
        eng = self.autoencoder
        x = ops.nchw_to_nhwc(batch.detach().to(torch.float32), eng.adt, 2.0, -1.0)      # (x-0.5)/0.5, models.py:170
        _, eps_levels = self._noise_args()
        purified, _ = eng.purify(x, self._alphas_device(), eps_levels, self._next_seed(), self.sample_offset)
        return purified

    def _forward_cuda(self, batch: torch.Tensor, tape=None):
        """fused `__call__` body (abstract_models.py:161-193): blur -> noise -> normalise -> purify -> classify."""
        eng = self.autoencoder
        noise0, eps_levels = self._noise_args()
        seed = self._next_seed()
        x, pre = ops.preprocess(batch.to(torch.float32), noise0, float(self.eps), bool(self.blur_input), eng.adt,
                                seed=seed, sample0=self.sample_offset, normalize=True, save_pre=tape is not None,
                                taps_cache=self._taps_cache)
        if tape is not None:
            tape.pre = pre
        purified, cls_in = eng.purify(x, self._alphas_device(), eps_levels, seed, self.sample_offset,
                                      cls_dtype=self.classifier.classifier.adt, tape=tape)
        preds = self.classifier.classifier.forward(cls_in, tape=tape) if tape is not None \
            else self.classifier.classifier.forward(cls_in)
        return preds, purified


class CelebaGenderClassifier(BaseClassificationModel, torch.nn.Module):

    def __init__(self, model_path: str, device: str, *, mode: str = None):
        """
        Wrapper for the CelebA-HQ Gender Resnet-50 custom model.
        """
        mean = (0.5, 0.5, 0.5)
        std = (0.5, 0.5, 0.5)
        self._mode = mode or default_mode()
        super().__init__(model_path, device, mean, std)

    def load_classifier(self, model_path: str, device: str):
        ckpt = _load_ckpt(model_path)           # loading_utils.py:10-17
        return ResNetEngine(ckpt["state_dict"], device, self._mode, groups=1)


class CarsTypeClassifier(BaseClassificationModel, torch.nn.Module):

    def __init__(self, model_path: str, device: str, *, mode: str = None):
        """
        Wrapper for the Stanford Cars type ResNeXt-50 custom model.
        """
        mean = (0.5, 0.5, 0.5)
        std = (0.5, 0.5, 0.5)
        self._mode = mode or default_mode()
        super().__init__(model_path, device, mean, std)

    def load_classifier(self, model_path: str, device: str):
        ckpt = _load_ckpt(model_path)           # loading_utils.py:29-36
        return ResNetEngine(ckpt["state_dict"], device, self._mode, groups=32)


class _StyleGanAutoencoder:
    """encoder + generator engines of one checkpoint (what `pSp` / `StyleTransformer` are in the reference)."""

    def __init__(self, encoder, decoder, opts):
        self.encoder, self.decoder, self.opts = encoder, decoder, opts
        self.device = decoder.device
        self.adt = decoder.adt


def _sub_state_dict(sd, prefix):
    n = len(prefix) + 1
    return {k[n:]: v for k, v in sd.items() if k.startswith(prefix + ".")}      # get_keys(), psp.py:8-12


class _StyleGanDefenseBase(MLVGMDefenseModel):
    """shared `__call__` body of the two StyleGAN purifiers: preprocess -> encode -> mix -> synthesise -> pool -> classify."""

    noise_std = 1.0
    max_chunk = None            # generator batch chunk (None: sized from the output resolution)

    def _style_noise(self, n_codes, b, d):
        if self._explicit_noise is not None:
            z = self._explicit_noise[1]
            if tuple(z.shape) != (n_codes, b, d):
                raise ValueError(f"explicit style noise must have shape {(n_codes, b, d)}, got {tuple(z.shape)}")
            return z * self.noise_std if self.noise_std != 1.0 else z
        return ops.philox_codes(self._seed_now, self.sample_offset, self.noise_std, n_codes, b, d, self.autoencoder.device)

    def _mix(self, codes):
        b, n, d = codes.shape
        if len(self.interpolation_alphas) != n:
            raise ValueError(f"{len(self.interpolation_alphas)} interpolation alphas for {n} codes")
        return self.autoencoder.decoder.mix_codes(codes, self._style_noise(n, b, d), self._alphas_device())

    def _preprocessed(self, batch, normalize=True):
        noise0 = self._explicit_noise[0] if self._explicit_noise is not None else None
        self._seed_now = self._next_seed()
        # fp32 image into the encoder stem (a 3-channel SIMT conv either way): a bf16 input would perturb the image by up to 2e-3
        x, _ = ops.preprocess(batch.detach().to(torch.float32), noise0, float(self.eps), bool(self.blur_input), torch.float32,
                              seed=self._seed_now, sample0=self.sample_offset, normalize=normalize, taps_cache=self._taps_cache)
        return x

    def _decode(self, codes, cls_dtype, want_purified=True, denorm=(0.5, 0.5), tape=None):
        """synthesis in batch chunks + the fused output kernel -> (purified NCHW [0,1], classifier input NHWC)"""
        dec = self.autoencoder.decoder
        dec.max_chunk = self.max_chunk
        outs = dec.synthesis(codes, sink=lambda img: self._pool_out(img, cls_dtype, want_purified, denorm), tape=tape)
        cat = lambda ts: None if ts[0] is None else (ts[0] if len(ts) == 1 else torch.cat(ts, dim=0))
        return cat([o[0] for o in outs]), cat([o[1] for o in outs])

    def purify(self, batch: torch.Tensor) -> torch.Tensor:
        """
        MLVGM encoding procedure to extract the codes.
        :param batch: pre-processed (normalised) images of shape (B, C, H, W).
        :return: purified reconstructions (B, C, H, W), still normalised (the caller de-normalises, abstract_models.py:184-185)
        """
        self._seed_now = self._next_seed()
        x = ops.nchw_to_nhwc(batch.detach().to(torch.float32), torch.float32)
        pur, _ = self._decode(self._mix(self._encode(x)), None, denorm=(1.0, 0.0))
        return pur

    def _forward_cuda(self, batch: torch.Tensor, tape=None):
        if tape is not None:
            raise NotImplementedError("input-gradient backward through the StyleGAN purifiers: the encoder half (image -> codes) is not "
                                      "built; the decode half is differentiable through from_codes()")
        x = self._preprocessed(batch)
        codes = self._mix(self._encode(x))
        purified, cls_in = self._decode(codes, self.classifier.classifier.adt)
        return self.classifier.classifier.forward(cls_in), purified

    def from_codes(self, codes: torch.Tensor, preds_only: bool = True):
        """The tail of `__call__` from the encoder's W+ codes (B, n_codes, 512) fp32: mix with the style noise (same seed / explicit-noise /
        `sample_offset` rules as a call) -> synthesis -> pool -> classifier.  -> logits, or (logits, purified) when not preds_only.
        Differentiable w.r.t. `codes` (input gradient only; repeated backward through one forward works)."""
        if codes.requires_grad and torch.is_grad_enabled():
            from ...autograd import codes_apply
            preds, purified = codes_apply(self, codes)
        else:
            preds, purified = self._from_codes_cuda(codes.detach())
        return preds if preds_only else (preds, purified)

    def _from_codes_cuda(self, codes: torch.Tensor, tape=None):
        """-> (logits, purified); tape: an `autograd.CodesTape` to fill for `_from_codes_backward`"""
        self._seed_now = self._next_seed()
        alphas = self._alphas_device()
        latent = self._mix(codes.to(self.autoencoder.device, torch.float32).contiguous())
        cls_eng = self.classifier.classifier
        purified, cls_in = self._decode(latent, cls_eng.adt, tape=tape.syn if tape is not None else None)
        if tape is None:
            return cls_eng.forward(cls_in), purified
        tape.alphas = alphas.clone()                     # the caller may reassign interpolation_alphas before a backward
        return cls_eng.forward(cls_in, tape=tape.cls), purified

    def _from_codes_backward(self, tape, g_preds, g_purified) -> torch.Tensor:
        """(d loss / d logits | None, d loss / d purified | None) -> d loss / d codes (B, n_codes, 512) fp32"""
        g_cls = self.classifier.classifier.backward(tape.cls, g_preds.contiguous().to(torch.float32)) if g_preds is not None else None
        g_pur = g_purified.contiguous().to(torch.float32) if g_purified is not None else None
        dec = self.autoencoder.decoder
        g_img = [self._pool_out_bwd(g_pur[lo:lo + n] if g_pur is not None else None, g_cls[lo:lo + n] if g_cls is not None else None,
                                    dec.size) for lo, n in tape.syn.slices]
        dec.max_chunk = self.max_chunk
        return ops.latent_lerp_bwd(dec.synthesis_backward(tape.syn, g_img), tape.alphas)


class E4EStyleGanDefenseModel(_StyleGanDefenseBase, torch.nn.Module):

    def __init__(self, classifier: BaseClassificationModel, autoencoder_path: str,
                 interpolation_alphas: tuple, alpha_attenuation: float = 1.0,
                 initial_noise_eps: float = 0.0, apply_gaussian_blur: bool = False,
                 device: str = 'cpu', *, mode: str = None):
        """
        Defense model using an StyleGan pretrained on FFHQ.
        """
        mean = (0.5, 0.5, 0.5)
        std = (0.5, 0.5, 0.5)
        self._mode = mode or default_mode()
        super().__init__(classifier, autoencoder_path, interpolation_alphas, alpha_attenuation,
                         initial_noise_eps, apply_gaussian_blur, device, mean, std)

    def load_autoencoder(self, model_path: str, device: str):
        ckpt = _load_ckpt(model_path)           # loading_utils.py:38-49, psp.py:39-45
        opts = dict(ckpt["opts"])
        if opts.get("encoder_type", "Encoder4Editing") != "Encoder4Editing":
            raise NotImplementedError(f"encoder_type {opts['encoder_type']}")            # psp.py:32 asserts the same
        size = int(opts["stylegan_size"])
        lat = ckpt.get("latent_avg") if opts.get("start_from_latent_avg", True) else None
        if lat is None and opts.get("start_from_latent_avg", True):
            raise NotImplementedError("checkpoint without latent_avg (psp.py:121-124 samples 10,000 latents)")
        enc = E4EEncoderEngine(_sub_state_dict(ckpt["state_dict"], "encoder"), size, lat, device, self._mode)
        dec = StyleGan2Engine(_sub_state_dict(ckpt["state_dict"], "decoder"), size, device, self._mode)
        return _StyleGanAutoencoder(enc, dec, opts)

    def _encode(self, x_nhwc):
        return self.autoencoder.encoder.encode(x_nhwc)                                    # psp.py:88-101

    def _pool_out(self, img, cls_dtype, want_purified, denorm):
        k = img.shape[1] // 256                                                           # face_pool -> 256 x 256, psp.py:26,114
        return ops.image_pool_out(img, k, 1, 0, denorm, cls_dtype, want_purified)

    def _pool_out_bwd(self, g_pur, g_cls, size):
        return ops.image_pool_out_bwd(g_pur, g_cls, size, size // 256, 1, 0, 0.5)


class TransStyleGanDefenseModel(_StyleGanDefenseBase, torch.nn.Module):

    noise_std = 0.8                              # torch.normal(0, 0.8, ...), models.py:334

    def __init__(self, classifier: BaseClassificationModel, autoencoder_path: str,
                 interpolation_alphas: tuple, alpha_attenuation: float = 1.0,
                 initial_noise_eps: float = 0.0, apply_gaussian_blur: bool = False,
                 device: str = 'cpu', *, mode: str = None):
        mean = (0.5, 0.5, 0.5)
        std = (0.5, 0.5, 0.5)
        self._mode = mode or default_mode()
        super().__init__(classifier, autoencoder_path, interpolation_alphas, alpha_attenuation,
                         initial_noise_eps, apply_gaussian_blur, device, mean, std)

    def load_autoencoder(self, model_path: str, device: str):
        ckpt = _load_ckpt(model_path)           # loading_utils.py:69-81, style_transformer.py:30-36
        opts = dict(ckpt["opts"])
        if opts.get("learn_in_w", False):
            raise NotImplementedError("learn_in_w checkpoints (single-w codes) are not supported")
        size = int(opts["output_size"])
        lat = ckpt.get("latent_avg") if opts.get("start_from_latent_avg", True) else None
        enc = TransEncoderEngine(_sub_state_dict(ckpt["state_dict"], "encoder.module"), lat, device, self._mode)
        dec = StyleGan2Engine(_sub_state_dict(ckpt["state_dict"], "decoder.module"), size, device, self._mode)
        return _StyleGanAutoencoder(enc, dec, opts)

    def _encode(self, x_nhwc):
        ae = self.autoencoder
        n, h, w, c = x_nhwc.shape
        # resize(x, 256) then rows 32:-32 (models.py:307-308): bilinear to (256 * h / w ...) short side 256, crop fused in the kernel
        # kornia `_side_to_image_size(256, w / h, 'short')` truncates: (256, int(256 * w/h)) if w/h > 1 else (int(256 / (w/h)), 256)
        ar = w / h
        full_h, full_w = (256, int(256 * ar)) if ar > 1 else (int(256 / ar), 256)
        x = ops.resize_bilinear(x_nhwc, full_h, full_w, 32, full_h - 64)
        query = ae.encoder.query(ae.decoder.mapping)                                      # models.py:310-315
        return ae.encoder.encode(x, query)

    def _pool_out(self, img, cls_dtype, want_purified, denorm):
        k = img.shape[1] // 256                                                           # face_pool, models.py:346
        return ops.image_pool_out(img, k, 2, 32, denorm, cls_dtype, want_purified)        # rows := -1, resize 256 -> 128 (:347-351)

    def _pool_out_bwd(self, g_pur, g_cls, size):
        return ops.image_pool_out_bwd(g_pur, g_cls, size, size // 256, 2, 32, 0.5)
