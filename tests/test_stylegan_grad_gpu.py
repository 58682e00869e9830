"""GPU: input gradient of the StyleGAN purifiers' decode half (W+ codes -> generator -> pool -> classifier) against torch.autograd through
the functional oracle (oracle/stylegan_ref.py): the new kernels one by one, the generator's reverse sweep, and `from_codes` of both
defenses."""
import contextlib
import functools
import math
import os

import pytest
import torch
import torch.nn.functional as F

from gen_adversarial_b200 import ops, synth
from gen_adversarial_b200.autograd import CodesTape
from gen_adversarial_b200.stylegan_engine import StyleGan2Engine, SynthesisTape
from gen_adversarial_b200.defenses.ours.models import (E4EStyleGanDefenseModel, TransStyleGanDefenseModel, CelebaGenderClassifier,
                                                       CarsTypeClassifier)
from oracle import stylegan_ref

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "stylegan2_gen32.pt")


def rel_l2(a, b):
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    return ((a - b).norm() / b.norm().clamp_min(1e-300)).item()


def cosine(a, b):
    a, b = a.detach().double().cpu().flatten(), b.detach().double().cpu().flatten()
    return (a @ b / (a.norm() * b.norm())).item()


def _d64(sd):
    return {k: v.double() if v.is_floating_point() else v for k, v in sd.items()}


def _interleave(t4, n, h, w, c):
    """[n, h/2, w/2, 4c] phase-major -> [n, h, w, c]"""
    return t4.view(n, h // 2, w // 2, 2, 2, c).permute(0, 1, 3, 2, 4, 5).reshape(n, h, w, c)


def _deinterleave(t, n, h, w, c):
    """[n, h, w, c] -> [n, h/2, w/2, 4c] phase-major"""
    return t.reshape(n, h // 2, 2, w // 2, 2, c).permute(0, 1, 3, 2, 4, 5).reshape(n, h // 2, w // 2, 4 * c)


# ------------------------------------------------------------------------------------------------ kernels
@pytest.mark.parametrize("dt", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("rgb", [False, True])
@pytest.mark.parametrize("phases", [False, True])
@pytest.mark.parametrize("n,h,w,c", [(1, 6, 10, 32), (3, 10, 14, 64), (3, 5, 7, 16), (2, 4, 4, 512)])
def test_styled_bias_act_bwd(n, h, w, c, phases, rgb, dt):
    """mirror of styled_bias_act + the ToRGB 1x1 adjoint against autograd of the restated forward
    v = lrelu(y * demod + noise_w * noise + bias) * sqrt(2), consumers v * s_next and conv1x1(v * s_rgb, W_rgb)"""
    if phases and (h % 2 or w % 2):
        pytest.skip("an up-sampling layer's output has even sides")
    g = torch.Generator().manual_seed(n * 100 + h + c)
    y = torch.randn(n, h, w, c, generator=g, dtype=torch.float64).requires_grad_()
    demod = (torch.rand(n, c, generator=g, dtype=torch.float64) + 0.5).requires_grad_()
    s_next = (torch.rand(n, c, generator=g, dtype=torch.float64) + 0.5).requires_grad_()
    s_rgb = (torch.rand(n, c, generator=g, dtype=torch.float64) + 0.5).requires_grad_()
    noise, bias = torch.randn(h, w, generator=g, dtype=torch.float64), torch.randn(c, generator=g, dtype=torch.float64)
    w_rgb = torch.randn(c, 4, generator=g, dtype=torch.float64) / math.sqrt(c)
    g_next = torch.randn(n, h, w, c, generator=g, dtype=torch.float64).to(dt).double()
    g_rgb = torch.randn(n, h, w, 4, generator=g, dtype=torch.float64)
    nw = 0.37
    v = F.leaky_relu(y * demod[:, None, None, :] + nw * noise[None, :, :, None] + bias, 0.2) * math.sqrt(2.0)
    loss = (v * s_next[:, None, None, :] * g_next).sum()
    if rgb:
        loss = loss + (((v * s_rgb[:, None, None, :]) @ w_rgb) * g_rgb).sum()
    gy_ref, gd_ref, gsn_ref, gsr_ref = torch.autograd.grad(loss, [y, demod, s_next, s_rgb], allow_unused=True)

    f = lambda t: t.to(DEV, torch.float32).contiguous()
    v_t = v.detach().to(dt).to(DEV)
    parts = ops.styled_bias_act_bwd_parts(h * w, c)
    dot_next, dot_rgb, dot_dem = (torch.full((n, parts, c), float("nan"), device=DEV) for _ in range(3))
    g_y = ops.styled_bias_act_bwd(v_t, g_next.to(DEV, dt), f(s_next.detach()), f(g_rgb) if rgb else None, f(w_rgb) if rgb else None,
                                  f(s_rgb.detach()) if rgb else None, f(demod.detach()), f(noise), nw, f(bias), phases, dt,
                                  dot_next=dot_next, dot_rgb=dot_rgb if rgb else None, dot_demod=dot_dem)
    assert g_y.dtype == dt and g_y.shape == ((n, h // 2, w // 2, 4 * c) if phases else (n, h, w, c))
    got_y = _interleave(g_y.float(), n, h, w, c) if phases else g_y.float()
    tol_y, tol_dot = (1e-5, 1e-5) if dt == torch.float32 else (1e-2, 3e-2)
    assert (got_y.cpu().double() - gy_ref).abs().max().item() <= tol_y * gy_ref.abs().max().item()
    assert rel_l2(dot_next.sum(1), gsn_ref) <= tol_dot
    assert rel_l2(dot_dem.sum(1), demod.detach() * gd_ref) <= tol_dot
    if rgb:
        assert rel_l2(dot_rgb.sum(1), gsr_ref) <= tol_dot


@pytest.mark.parametrize("variant", ["e4e", "trans"])
def test_image_pool_out_bwd(variant):
    """adjoint of image_pool_out: face_pool k x k mean; cars: rows := -1 (no gradient) then the 256 -> 128 2 x 2 mean; denormalise"""
    k1, k2, mask = (2, 1, 0) if variant == "e4e" else (2, 2, 32)
    n, S = 2, 512
    so = S // (k1 * k2)
    g = torch.Generator().manual_seed(7)
    img = torch.randn(n, 3, S, S, generator=g, dtype=torch.float64).requires_grad_()
    gp, gc = torch.randn(n, 3, so, so, generator=g, dtype=torch.float64), torch.randn(n, so, so, 3, generator=g, dtype=torch.float64)
    p = F.avg_pool2d(img, k1)
    if k2 == 2:
        p = p.clone()
        p[:, :, :mask] = -1.0
        p[:, :, -mask:] = -1.0
        p = F.avg_pool2d(p, 2)
    for use_p, use_c in ((True, True), (True, False), (False, True)):
        loss = (p * 0.5 + 0.5).mul(gp).sum() * use_p + (p.permute(0, 2, 3, 1) * gc).sum() * use_c
        ref, = torch.autograd.grad(loss, [img], retain_graph=True)
        got = ops.image_pool_out_bwd(gp.float().to(DEV) if use_p else None, gc.float().to(DEV) if use_c else None, S, k1, k2, mask, 0.5)
        assert got.shape == (n, S, S, 4) and bool((got[..., 3] == 0).all())
        assert (got[..., :3].cpu().double() - ref.permute(0, 2, 3, 1)).abs().max().item() <= 1e-6 * ref.abs().max().item()


def test_phase_conv_dgrad_matches_modconv_upsample():
    """the up-sampling conv's adjoint (ONE 3x3 conv over the de-interleaved gradient) against autograd through the reference modulated
    transposed conv + blur (oracle _modconv(..., upsample=True))"""
    sd = synth.make_stylegan2_state_dict(16, seed=5)
    eng = StyleGan2Engine(sd, 16, DEV, "fp32")
    eng._build_adjoint()
    up = eng.blocks[1][0]                                                  # 8 -> 16
    g = torch.Generator().manual_seed(3)
    n, h = 2, 8
    x = torch.randn(n, up.cin, h, h, generator=g, dtype=torch.float64).requires_grad_()
    lat = torch.randn(n, 512, generator=g)
    out = stylegan_ref._modconv(_d64(sd), "convs.2.conv", x, lat.double(), True, True)
    g_out = torch.randn(out.shape, generator=g, dtype=torch.float64)
    ref, = torch.autograd.grad((out * g_out).sum(), [x])
    s = eng._style(up.mod, lat.to(DEV))
    demod = ops.style_demod(s, up.wsq)
    g_y = _deinterleave(g_out.permute(0, 2, 3, 1).float().to(DEV) * demod[:, None, None, :], n, 2 * h, 2 * h, up.cout).contiguous()
    g_x = ops.conv2d_simt(g_y, up.phase_d, torch.float32) * s[:, None, None, :]
    assert rel_l2(g_x.permute(0, 3, 1, 2), ref) <= 1e-5


# ------------------------------------------------------------------------------------------------ generator
def _engine_branches(eng, tape):
    """the leaky-ReLU branch the engine's forward took in every styled layer (sign of its taped activation), whole batch, NCHW"""
    masks = []
    for kind, layer, _ in eng._plan():
        if kind == "styled":
            v = torch.cat([tape.acts[k] for k in sorted(k for k in tape.acts if k[0] == id(layer))], dim=0)
            masks.append((v > 0).permute(0, 3, 1, 2).cpu())
    return masks


def _classifier_branches(cls_tape):
    """the ReLU branches and the stem max-pool choices the engine's ResNet forward took (from its tape): (ReLU masks in the order
    resnet_forward applies them, NCHW stem ReLU output whose 3x3 / stride-2 window maxima pick the pooled elements)"""
    (_, _, x_stem, recs, h_fc), = [r for r in cls_tape if r[0] == "resnet"]
    nchw = lambda t: t.float().permute(0, 3, 1, 2).cpu()
    masks = [nchw(x_stem) > 0]
    for _, _, h1, h2, out in recs:
        masks += [nchw(h1) > 0, nchw(h2) > 0, nchw(out) > 0]
    masks.append(h_fc.float().reshape(h_fc.shape[0], -1).cpu() > 0)
    return masks, nchw(x_stem)


@contextlib.contextmanager
def _oracle_branches(masks, cls=None):
    """the oracle takes the engine's branches -- leaky ReLUs of the synthesis and, with `cls` (see _classifier_branches), the ReLUs and
    max-pool picks of the classifier -- so autograd differentiates the same piecewise-linear map the engine's backward does.
    Without this an fp32 forward and the fp64 oracle disagree on the slope wherever a pre-activation is within rounding of 0 (about one
    element per sample in the 32^2 generator, dozens in a ResNet-50 at 256^2), and each such element moves the whole gradient by
    ~1/sqrt(elements): 1e-3 in the generator, 2e-3 (random images) to 4e-2 (generator images) in the classifier, as autograd through
    the oracle in fp32 against fp64 shows -- a property of comparing two forwards, not of the backward sweep."""
    it = iter(masks)
    orig = stylegan_ref.fused_leaky_relu

    def fused_leaky_relu(x, bias):
        if x.dim() != 4:                                      # the mapping MLP (no gradient flows through it here)
            return orig(x, bias)
        t = x + bias.view(1, -1, 1, 1)
        return torch.where(next(it), t, 0.2 * t) * math.sqrt(2.0)

    class _Functional:
        """torch.nn.functional with the classifier's ReLUs and stem max-pool following the engine"""

        def __init__(self, relu_masks, stem):
            self.it, self.stem = iter(relu_masks), stem

        def __getattr__(self, name):
            return getattr(F, name)

        def relu(self, x):
            m = next(self.it)
            assert m.shape == x.shape, (m.shape, x.shape)
            return torch.where(m, x, torch.zeros_like(x))

        def max_pool2d(self, x, k, s, p):
            _, idx = F.max_pool2d(self.stem.to(x.dtype), k, s, p, return_indices=True)
            return x.flatten(2).gather(2, idx.flatten(2)).view(idx.shape)

    stylegan_ref.fused_leaky_relu = fused_leaky_relu
    if cls is not None:
        stylegan_ref.F = _Functional(*cls)
    try:
        yield
    finally:
        stylegan_ref.fused_leaky_relu = orig
        stylegan_ref.F = F


@functools.lru_cache(maxsize=None)
def _synthesis_case(which):
    """(state dict, size, latent, image gradient)"""
    if which == "golden32":
        gold = torch.load(GOLDEN, weights_only=True)
        size, sd = gold["size"], synth.make_stylegan2_state_dict(gold["size"], seed=gold["seed"])
    else:
        size, sd = 256, synth.make_stylegan2_state_dict(256, seed=9)
    g = torch.Generator().manual_seed(size)
    batch = 3 if size <= 32 else 2
    lat = torch.randn(batch, 2 * int(math.log2(size)) - 2, 512, generator=g)
    return sd, size, lat, torch.randn(batch, 3, size, size, generator=g)


@pytest.mark.parametrize("mode", ["fp32", "bf16"])
@pytest.mark.parametrize("which", ["golden32", "synthetic256"])
def test_synthesis_backward(which, mode):
    """the reverse sweep on batch slices of one sample (max_chunk = 1) against autograd through generator_synthesis in fp64 (fp32: on the
    engine's leaky-ReLU branches; bf16: on the oracle's own)"""
    sd, size, lat, g_img = _synthesis_case(which)
    eng = StyleGan2Engine(sd, size, DEV, mode)
    eng.max_chunk = 1
    tape = SynthesisTape()
    eng.synthesis(lat.to(DEV), tape=tape)
    assert len(tape.slices) == lat.shape[0]
    g_nhwc = F.pad(g_img.permute(0, 2, 3, 1), (0, 1)).to(DEV)
    got = eng.synthesis_backward(tape, [g_nhwc[lo:lo + n].contiguous() for lo, n in tape.slices])
    latd = lat.double().requires_grad_()
    with _oracle_branches(_engine_branches(eng, tape)) if mode == "fp32" else contextlib.nullcontext():
        img = stylegan_ref.generator_synthesis(_d64(sd), latd, size)
    ref, = torch.autograd.grad((img * g_img.double()).sum(), [latd])
    assert got.shape == ref.shape
    if mode == "fp32":
        assert rel_l2(got, ref) <= 1e-4, rel_l2(got, ref)
    else:
        assert cosine(got, ref) >= 0.99, cosine(got, ref)


# ------------------------------------------------------------------------------------------------ defenses
def _make_defense(kind, size, mode):
    n_codes = 2 * int(math.log2(size)) - 2
    alphas = [0.1 + 0.8 * i / (n_codes - 1) for i in range(n_codes)]
    if kind == "e4e":
        ck, clf_ck = synth.make_e4e_checkpoint(stylegan_size=size), synth.make_resnet50_checkpoint()
        dm = E4EStyleGanDefenseModel(CelebaGenderClassifier(clf_ck, DEV, mode=mode), ck, alphas, 1.0, 0.0, False, DEV, mode=mode)
    else:
        ck, clf_ck = synth.make_trans_checkpoint(output_size=size), synth.make_resnext50_checkpoint()
        dm = TransStyleGanDefenseModel(CarsTypeClassifier(clf_ck, DEV, mode=mode), ck, alphas, 1.0, 0.0, False, DEV, mode=mode)
    return dm, ck, clf_ck, alphas


def _ref_tail(kind, ck, clf_ck, codes, z, alphas, size):
    """the tail of e4e_defense_call / trans_defense_call from the codes: mix -> synthesis -> pool / crop / resize -> classifier, in the
    codes' dtype"""
    cast = _d64 if codes.dtype == torch.float64 else (lambda sd: sd)
    dec = cast(stylegan_ref._sub(ck["state_dict"], "decoder" if kind == "e4e" else "decoder.module"))
    lat = stylegan_ref.mix_codes(dec, codes, z.to(codes.dtype) * (1.0 if kind == "e4e" else 0.8), alphas)
    img = F.adaptive_avg_pool2d(stylegan_ref.generator_synthesis(dec, lat, size), (256, 256))
    if kind != "e4e":
        img = img.clone()
        img[:, :, :32] = -1.0
        img[:, :, -32:] = -1.0
        img = F.interpolate(img, size=(128, 128), mode="bilinear", align_corners=False)
    pur = img * 0.5 + 0.5
    return stylegan_ref.resnet_forward(cast(clf_ck["state_dict"]), (pur - 0.5) / 0.5, 1 if kind == "e4e" else 32), pur


def _check_from_codes(kind, size, batch, tol, ref_dtype=torch.float64):
    dm, ck, clf_ck, alphas = _make_defense(kind, size, "fp32")
    n_codes = len(alphas)
    g = torch.Generator().manual_seed(size + batch)
    codes = torch.randn(batch, n_codes, 512, generator=g)
    z = torch.randn(n_codes, batch, 512, generator=g)
    hw = 256 if kind == "e4e" else 128
    dm.set_explicit_noise([torch.zeros(batch, 3, hw, hw), z])
    tape = CodesTape()
    dm._from_codes_cuda(codes.to(DEV), tape=tape)                             # the forward from_codes runs, for its branches
    masks, cls = _engine_branches(dm.autoencoder.decoder, tape.syn), _classifier_branches(tape.cls)
    branches = lambda: _oracle_branches(masks, cls)
    with branches():
        logits_ref, pur_ref = _ref_tail(kind, ck, clf_ck, codes.to(ref_dtype).requires_grad_(), z, alphas, size)
    g_l, g_p = torch.randn(logits_ref.shape, generator=g), torch.randn(pur_ref.shape, generator=g)
    for preds_only in (True, False):
        cd = codes.to(DEV).requires_grad_()
        if preds_only:
            logits = dm.from_codes(cd)
            loss = (logits * g_l.to(DEV)).sum()
            cr = codes.to(ref_dtype).requires_grad_()
            with branches():
                lr, _ = _ref_tail(kind, ck, clf_ck, cr, z, alphas, size)
            ref, = torch.autograd.grad((lr * g_l.to(ref_dtype)).sum(), [cr])
        else:
            logits, pur = dm.from_codes(cd, preds_only=False)
            assert rel_l2(pur, pur_ref) <= 1e-4
            loss = (logits * g_l.to(DEV)).sum() + (pur * g_p.to(DEV)).sum()
            cr = codes.to(ref_dtype).requires_grad_()
            with branches():
                lr, pr = _ref_tail(kind, ck, clf_ck, cr, z, alphas, size)
            ref, = torch.autograd.grad((lr * g_l.to(ref_dtype)).sum() + (pr * g_p.to(ref_dtype)).sum(), [cr])
        # the fp32 forward (the same kernels as __call__) at the project's fp32 logits criterion (test_stylegan_paths_gpu.py)
        assert (logits.detach().cpu().double() - logits_ref.detach().double()).abs().max() <= 1e-3 * logits_ref.detach().abs().max()
        got, = torch.autograd.grad(loss, [cd])
        assert rel_l2(got, ref) <= tol, (kind, preds_only, rel_l2(got, ref))
    return dm


@pytest.mark.parametrize("kind", ["e4e", "trans"])
def test_from_codes_gradient(kind):
    dm = _check_from_codes(kind, 256, 2, 1e-4)
    # the encoder half is still missing: a differentiable call on the images refuses
    hw = 256 if kind == "e4e" else 128
    dm.set_explicit_noise(None)
    with pytest.raises(NotImplementedError, match="encoder half"):
        dm(torch.rand(1, 3, hw, hw, device=DEV).requires_grad_())


@pytest.mark.parametrize("kind,size", [("e4e", 1024), ("trans", 512)])
def test_from_codes_gradient_full_size(kind, size):
    _check_from_codes(kind, size, 1, 1e-4, ref_dtype=torch.float32)          # fp32 oracle: the fp64 one takes minutes at 1024^2


@pytest.mark.parametrize("kind", ["e4e", "trans"])
def test_from_codes_repeated_backward_and_batch_position(kind):
    dm, _, _, alphas = _make_defense(kind, 256, "fp32")
    dm.max_chunk = 1
    dm.noise_seed = 1234
    g = torch.Generator().manual_seed(11)
    codes = torch.randn(3, len(alphas), 512, generator=g).to(DEV).requires_grad_()
    logits = dm.from_codes(codes)
    g1, g2 = torch.randn(logits.shape, generator=g).to(DEV), torch.randn(logits.shape, generator=g).to(DEV)
    a, = torch.autograd.grad(logits, [codes], g1, retain_graph=True)
    b, = torch.autograd.grad(logits, [codes], g2, retain_graph=True)
    c, = torch.autograd.grad(logits, [codes], g1)
    assert torch.equal(a, c) and not torch.equal(a, b)
    # Philox style noise is keyed by the global sample index: sample 1 alone at sample_offset 1 sees the same noise and gradient
    dm.sample_offset = 1
    one = codes.detach()[1:2].clone().requires_grad_()
    l1 = dm.from_codes(one)
    d, = torch.autograd.grad(l1, [one], g1[1:2])
    assert (l1.detach() - logits.detach()[1:2]).abs().max().item() <= 1e-5 * logits.abs().max().item()
    assert rel_l2(d, a[1:2]) <= 1e-5
