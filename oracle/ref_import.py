"""TEST INFRASTRUCTURE ONLY -- imports the *unmodified* reference from /root/reference.

This module is the "real reference" leg of the oracle (SURVEY.md section 8c / Appendix C).
The tree is /root/reference in the build container, or its byte-identical copy under the git-ignored
oracle/_ref/reference/ (oracle/build_ref.sh) on the GPU box.  It is used by
  * tests/test_oracle_vs_reference.py  (validates oracle/nvae_ref.py against the reference),
  * oracle/make_golden.py              (generates tests/golden/* fixtures), and
  * bench.py: `--impl reference` (the reference's own modules on the host cores, kind "reference") and the
    `incumbent_gpu` block (the same modules on cuda:0 -- `install(cpu_stylegan_ops=False)` lets the reference
    JIT-build and use its own upfirdn2d / fused_bias_act CUDA kernels there).
The product never imports it.

No reference file is copied or modified: three import-time shims make the tree importable
(the committed reference has import-time defects, SURVEY.md section 4.3):

  1. builtins.Union = typing.Union               (src/defenses/ours/abstract_models.py:162)
  2. sys.modules['src.hl_autoencoders'] -> src.mlvgms_autoencoders  (stale package name,
     StyleGan_Trans/models/style_transformer.py:5-6 and friends)
  3. an in-memory `kornia` exposing the seven functions the path calls (kornia is not installed;
     version unpinned in environment.yml:17).  Semantics restated from kornia's documented
     behaviour: normalize=(x-mean)/std, denormalize=x*std+mean, gaussian_blur2d = separable
     reflect-padded 1-D gaussian exp(-t^2/2s^2)/sum with t=arange(k)-k//2, resize(int)=short-side
     bilinear (align_corners=None, antialias=False).
  4. the two JIT-compiled CUDA ops of the StyleGAN2 copies (`fused`, `upfirdn2d`) refuse CPU
     tensors (CHECK_CUDA, fused_bias_act.cpp:7-9); their `op` packages are replaced by a CPU
     restatement: fused_leaky_relu(x,b)=leaky_relu(x+b,0.2)*sqrt(2) (fused_bias_act_kernel.cu:28-47)
     and upfirdn2d = pad/zero-insert/FIR/decimate (upfirdn2d.py:150-184).
"""
from __future__ import annotations

import builtins
import importlib
import math
import os
import sys
import tempfile
import types
import typing

import torch
import torch.nn.functional as F

_HERE = os.path.dirname(os.path.abspath(__file__))


def _find_reference_root() -> str:
    """/root/reference in the build container; on the GPU box the byte-identical copy that oracle/build_ref.sh placed under the
    git-ignored oracle/_ref/reference/ (it travels with the snapshot like a built .so)."""
    env = os.environ.get("GA_REFERENCE_ROOT")
    if env:
        return env
    for cand in ("/root/reference", os.path.join(_HERE, "_ref", "reference")):
        if os.path.isdir(os.path.join(cand, "src", "defenses", "ours")):
            return cand
    return "/root/reference"


REFERENCE_ROOT = _find_reference_root()


def reference_available() -> bool:
    return os.path.isdir(os.path.join(REFERENCE_ROOT, "src", "defenses", "ours"))


# --------------------------------------------------------------------------- kornia restatement
def _bcast(v, ref: torch.Tensor) -> torch.Tensor:
    if not torch.is_tensor(v):
        v = torch.tensor(v, dtype=ref.dtype, device=ref.device)
    v = v.to(device=ref.device, dtype=ref.dtype)
    if v.dim() == 0:
        return v
    return v.view(1, -1, 1, 1)


def k_normalize(data, mean, std):
    return (data - _bcast(mean, data)) / _bcast(std, data)


def k_denormalize(data, mean, std):
    return data * _bcast(std, data) + _bcast(mean, data)


class KNormalize(torch.nn.Module):
    def __init__(self, mean, std):
        super().__init__()
        self.mean, self.std = mean, std

    def forward(self, x):
        return k_normalize(x, self.mean, self.std)


class KDenormalize(torch.nn.Module):
    def __init__(self, mean, std):
        super().__init__()
        self.mean, self.std = mean, std

    def forward(self, x):
        return k_denormalize(x, self.mean, self.std)


def gaussian_kernel1d(k: int, sigma: float, dtype=torch.float32) -> torch.Tensor:
    t = torch.arange(k, dtype=dtype) - k // 2
    if k % 2 == 0:
        t = t + 0.5
    g = torch.exp(-(t ** 2) / (2.0 * sigma ** 2))
    return g / g.sum()


def k_gaussian_blur2d(x, kernel_size, sigma, border_type="reflect", separable=True):
    if isinstance(kernel_size, int):
        kernel_size = (kernel_size, kernel_size)
    ky, kx = kernel_size
    sy, sx = float(sigma[0]), float(sigma[1])
    b, c, h, w = x.shape
    gy = gaussian_kernel1d(ky, sy, x.dtype).to(x.device)
    gx = gaussian_kernel1d(kx, sx, x.dtype).to(x.device)
    py, px = ky // 2, kx // 2
    xp = F.pad(x, (px, px, py, py), mode=border_type)
    xp = F.conv2d(xp, gx.view(1, 1, 1, kx).expand(c, 1, 1, kx), groups=c)
    xp = F.conv2d(xp, gy.view(1, 1, ky, 1).expand(c, 1, ky, 1), groups=c)
    return xp


def k_resize(x, size, interpolation="bilinear", align_corners=None, side="short", antialias=False):
    if isinstance(size, int):
        # kornia.geometry.transform.affwarp._side_to_image_size: truncation, not rounding
        h, w = x.shape[-2:]
        ar = w / h
        if side == "vert":
            size = (size, int(size * ar))
        elif side == "horz":
            size = (int(size / ar), size)
        elif (side == "short") ^ (ar < 1.0):
            size = (size, int(size * ar))
        else:
            size = (int(size / ar), size)
    return F.interpolate(x, size=size, mode=interpolation, align_corners=align_corners, antialias=antialias)


def _install_kornia():
    if "kornia" in sys.modules and not getattr(sys.modules["kornia"], "_ga_shim", False):
        return  # a real kornia is installed; use it
    k = types.ModuleType("kornia"); k._ga_shim = True
    ke = types.ModuleType("kornia.enhance")
    kf = types.ModuleType("kornia.filters")
    kg = types.ModuleType("kornia.geometry")
    ke.normalize, ke.denormalize = k_normalize, k_denormalize
    ke.Normalize, ke.Denormalize = KNormalize, KDenormalize
    kf.gaussian_blur2d = k_gaussian_blur2d
    kg.resize = k_resize
    k.enhance, k.filters, k.geometry = ke, kf, kg
    sys.modules.update({"kornia": k, "kornia.enhance": ke, "kornia.filters": kf, "kornia.geometry": kg})


# --------------------------------------------------------------------------- StyleGAN2 op restatement (CPU)
def fused_leaky_relu_cpu(input, bias=None, negative_slope=0.2, scale=2 ** 0.5):
    if bias is not None:
        rest = [1] * (input.dim() - bias.dim() - 1)
        input = input + bias.view(1, bias.shape[0], *rest)
    return F.leaky_relu(input, negative_slope) * scale


class FusedLeakyReLUCPU(torch.nn.Module):
    def __init__(self, channel, bias=True, negative_slope=0.2, scale=2 ** 0.5):
        super().__init__()
        self.bias = torch.nn.Parameter(torch.zeros(channel)) if bias else None
        self.negative_slope, self.scale = negative_slope, scale

    def forward(self, input):
        return fused_leaky_relu_cpu(input, self.bias, self.negative_slope, self.scale)


def upfirdn2d_cpu(input, kernel, up=1, down=1, pad=(0, 0)):
    """zero-insert up-sample -> pad -> correlate with flipped FIR -> decimate; NCHW."""
    b, c, h, w = input.shape
    kh, kw = kernel.shape
    p0, p1 = pad
    x = input.reshape(b * c, 1, h, 1, w, 1)
    x = F.pad(x, [0, up - 1, 0, 0, 0, up - 1])
    x = x.reshape(b * c, 1, h * up, w * up)
    x = F.pad(x, [max(p0, 0), max(p1, 0), max(p0, 0), max(p1, 0)])
    x = x[:, :, max(-p0, 0): x.shape[2] - max(-p1, 0), max(-p0, 0): x.shape[3] - max(-p1, 0)]
    wk = torch.flip(kernel, [0, 1]).view(1, 1, kh, kw).to(x.dtype)
    x = F.conv2d(x, wk)
    x = x[:, :, ::down, ::down]
    return x.reshape(b, c, x.shape[2], x.shape[3])


def _install_stylegan_ops():
    for pkg in ("src.mlvgms_autoencoders.StyleGan_E4E.stylegan2.op",
                "src.mlvgms_autoencoders.StyleGan_Trans.models.stylegan2.op",
                "src.hl_autoencoders.StyleGan_Trans.models.stylegan2.op"):
        m = types.ModuleType(pkg)
        m.FusedLeakyReLU = FusedLeakyReLUCPU
        m.fused_leaky_relu = fused_leaky_relu_cpu
        m.upfirdn2d = upfirdn2d_cpu
        m.__path__ = []  # behave like a package
        sys.modules[pkg] = m


_INSTALLED = False


def install(cpu_stylegan_ops: bool = True):
    """Make `import src...` resolve to the unmodified reference tree."""
    global _INSTALLED
    if _INSTALLED:
        return
    if not reference_available():
        raise RuntimeError(f"reference tree not found at {REFERENCE_ROOT} (only present in the build container)")
    # keep any torch JIT cache inside the repo (oracle/_ref is git-ignored); a read-only tree gets a per-run temporary directory
    if "TORCH_EXTENSIONS_DIR" not in os.environ:
        ext = os.path.join(_HERE, "_ref", "torch_ext")
        try:
            os.makedirs(ext, exist_ok=True)
            writable = os.access(ext, os.W_OK)
        except OSError:
            writable = False
        os.environ["TORCH_EXTENSIONS_DIR"] = ext if writable else tempfile.mkdtemp(prefix="ga_torch_ext_")
    builtins.Union = typing.Union                                             # shim 1
    _install_kornia()                                                         # shim 3
    if REFERENCE_ROOT not in sys.path:
        sys.path.insert(0, REFERENCE_ROOT)
    if cpu_stylegan_ops:
        _install_stylegan_ops()                                               # shim 4
    sys.modules["src.hl_autoencoders"] = importlib.import_module("src.mlvgms_autoencoders")  # shim 2
    _INSTALLED = True


def ref_models():
    """-> module src.defenses.ours.models of the reference."""
    install()
    return importlib.import_module("src.defenses.ours.models")


def ref_nvae_module():
    install()
    return importlib.import_module("src.mlvgms_autoencoders.NVAE.model")


class ExplicitNoise:
    """Context manager: make the reference consume explicit noise tensors instead of drawing RNG.

    The reference draws (SURVEY 8c "RNG order"): `torch.ones_like(x).normal_(0,1)`
    (abstract_models.py:132) then `torch.zeros_like(mu).normal_()` per latent level
    (distributions.py:43) and `torch.normal(mean, std, size)` for the StyleGAN models
    (models.py:119,334).  While active, every such draw pops the next tensor of `queue`
    (scaled by std and shifted by mean, so queue entries are always N(0,1) draws).
    """

    def __init__(self, queue):
        self.queue = list(queue)
        self._orig_normal_ = None
        self._orig_normal = None

    def _pop(self, shape, dtype, device):
        if not self.queue:
            raise RuntimeError("ExplicitNoise: queue exhausted")
        e = self.queue.pop(0)
        if tuple(e.shape) != tuple(shape):
            raise RuntimeError(f"ExplicitNoise: shape mismatch, wanted {tuple(shape)} got {tuple(e.shape)}")
        return e.to(device=device, dtype=dtype)

    def __enter__(self):
        self._orig_normal_ = torch.Tensor.normal_
        self._orig_normal = torch.normal
        outer = self

        def normal_(t, mean=0.0, std=1.0, *, generator=None):
            e = outer._pop(t.shape, t.dtype, t.device)
            with torch.no_grad():
                t.copy_(e * std + mean)
            return t

        def normal(mean, std=None, size=None, **kw):
            if size is None or torch.is_tensor(mean) or torch.is_tensor(std):
                return outer._orig_normal(mean, std, size, **kw) if size is not None else outer._orig_normal(mean, std, **kw)
            dev = kw.get("device", "cpu")
            e = outer._pop(tuple(size), kw.get("dtype", torch.float32) or torch.float32, dev)
            return e * std + mean

        torch.Tensor.normal_ = normal_
        torch.normal = normal
        return self

    def __exit__(self, *exc):
        torch.Tensor.normal_ = self._orig_normal_
        torch.normal = self._orig_normal
        return False


class InMemoryCheckpoints:
    """Context manager: `torch.load(path)` returns a prepared object for the given pseudo-paths, so the reference's own loaders
    (src/defenses/loading_utils.py:10-81, psp.py:39-45, style_transformer.py:30-36) ingest synthetic checkpoints without a multi-GB
    round trip through the file system (the VGG11 head alone is 2.5 GB).  No reference code is changed."""

    def __init__(self, table):
        self.table = dict(table)
        self._orig = None

    def __enter__(self):
        self._orig = torch.load
        outer = self

        def load(f, *a, **kw):
            if isinstance(f, str) and f in outer.table:
                return outer.table[f]
            return outer._orig(f, *a, **kw)

        torch.load = load
        return self

    def __exit__(self, *exc):
        torch.load = self._orig
        return False


REFERENCE_YAMLS = {"purify": "ours_learned_blur_ids.yaml", "pgd": "ours_cosine_noise_ids.yaml",
                   "gender": "ours_linear_noise_gender.yaml", "cars": "ours_cosine_blur_cars.yaml"}


def build_reference_defense(workload: str, device: str = "cpu"):
    """The reference's OWN defense model for one BASELINE workload -- classes of src/defenses/ours/models.py constructed exactly as
    src/experiments/load_defense.py:134-140 does, from the YAML in the reference's configs/ and the seeded synthetic checkpoints of
    gen_adversarial_b200/synth.py (the same weights the CUDA path loads).  device "cpu": the two StyleGAN CUDA ops are replaced by
    their CPU restatement (they refuse CPU tensors); device "cuda:*": the reference JIT-builds and runs its own kernels.
    -> (defense model, resolution (C,H,W), n_classes, yaml dict)"""
    import yaml
    from gen_adversarial_b200 import synth
    on_gpu = str(device).startswith("cuda")
    install(cpu_stylegan_ops=not on_gpu)
    mm = importlib.import_module("src.defenses.ours.models")
    with open(os.path.join(REFERENCE_ROOT, "configs", REFERENCE_YAMLS[workload])) as f:
        p = yaml.safe_load(f)
    if workload in ("purify", "pgd"):
        from gen_adversarial_b200.nvae_spec import NVAE_C32_RESOLUTION
        table = {"mem://ae": synth.make_nvae_checkpoint(seed=0), "mem://clf": synth.make_vgg11_checkpoint(100, seed=1)}
        Clf, Def, res, n_cls = mm.CelebaIdentityClassifier, mm.NVAEDefenseModel, NVAE_C32_RESOLUTION, 100
    elif workload == "gender":
        table = {"mem://ae": synth.make_e4e_checkpoint(1024), "mem://clf": synth.make_resnet50_checkpoint()}
        Clf, Def, res, n_cls = mm.CelebaGenderClassifier, mm.E4EStyleGanDefenseModel, (3, 256, 256), 2
    elif workload == "cars":
        table = {"mem://ae": synth.make_trans_checkpoint(512), "mem://clf": synth.make_resnext50_checkpoint()}
        table["mem://ae"]["opts"]["device"] = str(device)      # style_transformer.py:30-36 reads the device from the checkpoint's opts
        Clf, Def, res, n_cls = mm.CarsTypeClassifier, mm.TransStyleGanDefenseModel, (3, 128, 128), 4
    else:
        raise ValueError(workload)
    with InMemoryCheckpoints(table):
        clf = Clf("mem://clf", device)
        dm = Def(clf, "mem://ae", p["interpolation_alphas"], p["alpha_attenuation"], p["initial_noise_eps"], p["gaussian_blur_input"],
                 device)
    return dm, res, n_cls, p
