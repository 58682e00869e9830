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


def worst_code_rel_l2(a, b):
    """largest rel-L2 of one code index of a (B, n_codes, 512) gradient: a wrong term in one layer moves its code's gradient by far more
    than the whole gradient"""
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    return ((a - b).norm(dim=(0, 2)) / b.norm(dim=(0, 2)).clamp_min(1e-300)).max().item()


def _d64(sd, device="cpu"):
    return {k: v.to(device, torch.float64) if v.is_floating_point() else v.to(device) for k, v in sd.items()}


def _bf16_ulp(t):
    """spacing of bf16 numbers (8 significant bits) at |t|, elementwise, for float64 t"""
    _, e = torch.frexp(t.abs())                                                # |t| = m 2^e, m in [0.5, 1)
    return torch.ldexp(torch.ones_like(t), e - 8) * (t != 0)


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


@functools.lru_cache(maxsize=None)
def _bf16_generator(size, cm):
    eng = StyleGan2Engine(synth.make_stylegan2_state_dict(size, channel_multiplier=cm, seed=size + cm), size, DEV, "bf16",
                          channel_multiplier=cm)
    eng._build_adjoint()
    return eng


@pytest.mark.parametrize("out", ["bf16", "fp32"])
@pytest.mark.parametrize("size,cm,j,up,n,h,w", [
    (1024, 2, 7, False, 1, 1024, 1024),         # 32 -> 32 at 1024^2: the superpixel adjoint on the [n, H, W/2, 64] pair view
    (512, 1, 6, False, 1, 512, 512),            # the same at 512^2 with channel_multiplier = 1
    (1024, 2, 6, False, 1, 512, 512),           # plain 64 -> 64 dgrad at 512^2
    (1024, 2, 5, False, 1, 256, 256),           # plain 128 -> 128 dgrad at 256^2
    (1024, 2, 7, True, 1, 512, 512),            # up layer 512 -> 1024 (64 -> 32 ch): phase dgrad 128 -> 64 at 512^2
    (1024, 2, 6, True, 1, 256, 256),            # up layer 256 -> 512 (128 -> 64 ch): phase dgrad 256 -> 128 at 256^2
    (1024, 2, 6, False, 2, 136, 384),           # 64 -> 64 on two images of 17 x 12 windows of 8 x 32: window and image seams
], ids=["sp1024", "sp512cm1", "c64at512", "c128at256", "up512to1024", "up256to512", "c64seams"])
def test_adjoint_conv_bf16_shapes(size, cm, j, up, n, h, w, out):
    """the conv adjoints the bf16 engine runs above f32_conv_out_res (tensor cores, wide-window mode of the persistent 3x3 kernel), built by
    _build_adjoint and run through StyleGan2Engine._dgrad on a bf16 conv-output gradient, against autograd of F.conv2d in fp64 on the same
    bf16-rounded operands (the forward layer's weights).  What is left is fp32 accumulation order and the output rounding, so the gate is
    elementwise: one bf16 ulp of the reference (bf16 output) or 1e-5 max|ref| (fp32 output).  Max-abs, not rel-L2: one tap dropped at a
    window seam moves a few border pixels only."""
    eng = _bf16_generator(size, cm)
    s = eng.blocks[j][0 if up else 1]
    L = s.phase_convs if up else s.conv                                     # forward conv: [b, h, w, cin] -> [b, h, w, (4) cout]
    f32 = out == "fp32"
    g = torch.Generator(device=DEV).manual_seed(size + j + n)
    g_y = torch.randn(n, h, w, L.cout, generator=g, device=DEV).to(torch.bfloat16)
    sp = not up and s.conv_sp_d is not None and not f32
    assert sp == (not up and s.cin == 32 and not f32)                       # the superpixel adjoint exists exactly for the 32-channel layers
    D = s.conv_sp_d if sp else (s.phase_d if up else s.conv_d)
    assert ops.conv2d_tc_supported(g_y.view(n, h, w // 2, 2 * L.cout) if sp else g_y, D)   # no silent fall-back to the SIMT kernel
    got = eng._dgrad(s, g_y, f32)
    assert got.dtype == (torch.float32 if f32 else torch.bfloat16) and got.shape == (n, h, w, L.cin)

    wb = L.w_simt.view(3, 3, L.cin, L.cout).permute(3, 2, 0, 1).to(torch.bfloat16).double()
    x = torch.zeros(n, L.cin, h, w, dtype=torch.float64, device=DEV, requires_grad=True)
    ref, = torch.autograd.grad(F.conv2d(x, wb, padding=1), [x], g_y.double().permute(0, 3, 1, 2))
    ref = ref.permute(0, 2, 3, 1)
    err = (got.double() - ref).abs()
    big = ref.abs().max().item()
    if f32:
        assert err.max().item() <= 1e-5 * big, err.max().item() / big
    else:
        # one ulp of the reference, plus 1e-6 max|ref| for the few sums that nearly cancel (there fp32 accumulation error can exceed the
        # ulp); the floor is below one ulp of every element above 2.6e-4 max|ref|
        bad = err > _bf16_ulp(ref) + 1e-6 * big
        assert not bool(bad.any()), (int(bad.sum()), bad.nonzero()[:8].tolist(), (err / _bf16_ulp(ref)).max().item())


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
        return torch.where(next(it).to(t.device), t, 0.2 * t) * math.sqrt(2.0)

    class _Functional:
        """torch.nn.functional with the classifier's ReLUs and stem max-pool following the engine"""

        def __init__(self, relu_masks, stem):
            self.it, self.stem = iter(relu_masks), stem

        def __getattr__(self, name):
            return getattr(F, name)

        def relu(self, x):
            m = next(self.it)
            assert m.shape == x.shape, (m.shape, x.shape)
            return torch.where(m.to(x.device), x, torch.zeros_like(x))

        def max_pool2d(self, x, k, s, p):
            # the element each window picks, from the engine's own stem output: the first maximum in scan order, which is also what
            # maxpool3x3s2_bwd routes the gradient to, so ties (frequent in a bf16 stem) resolve alike
            _, idx = F.max_pool2d(self.stem.contiguous(), k, s, p, return_indices=True)
            idx = idx.to(x.device)
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
    """(state dict, size, channel multiplier, latent, image gradient)"""
    cm = 2
    if which == "golden32":
        gold = torch.load(GOLDEN, weights_only=True)
        size, sd = gold["size"], synth.make_stylegan2_state_dict(gold["size"], seed=gold["seed"])
    elif which == "synthetic256":
        size, sd = 256, synth.make_stylegan2_state_dict(256, seed=9)
    elif which == "synthetic512cm1":
        size, cm = 512, 1
        sd = synth.make_stylegan2_state_dict(512, channel_multiplier=1, seed=10)
    else:
        size, sd = 1024, synth.make_stylegan2_state_dict(1024, seed=11)
    g = torch.Generator().manual_seed(size)
    batch = 2 if size == 256 else 3
    lat = torch.randn(batch, 2 * int(math.log2(size)) - 2, 512, generator=g)
    return sd, size, cm, lat, torch.randn(batch, 3, size, size, generator=g)


def _mixed_slices(eng):
    """blocks at >= 128^2 run on slices of 2 (a batch of 3: 2 + 1) while the lower resolutions run on the whole batch -- the engine's
    recursive split at full size (_cap gives 16 images at 1024^2, 32 at 512^2) on a batch small enough for the fp64 oracle"""
    eng.max_chunk = None
    eng._cap = lambda j: 2 if (8 << j) >= 128 else 1 << 20


# bf16 against the fp64 oracle on the engine's branches, measured on a B200: (rel-L2, worst rel-L2 of one code index); each gate is
# about twice the measurement
BF16_SYNTHESIS_GATES = {"golden32": (7e-3, 8e-3),             # measured 3.5e-3, 3.9e-3
                        "synthetic256": (1e-2, 1.2e-2),         # 5.0e-3, 6.1e-3
                        "synthetic512cm1": (1e-2, 1.7e-2),      # 4.9e-3, 8.6e-3
                        "synthetic1024": (1.2e-2, 1.5e-2)}      # 6.1e-3, 7.4e-3
MIXED = ("synthetic512cm1", "synthetic1024")


@pytest.mark.parametrize("mode", ["fp32", "bf16"])
@pytest.mark.parametrize("which", ["golden32", "synthetic256", "synthetic512cm1", "synthetic1024"])
def test_synthesis_backward(which, mode):
    """the reverse sweep against autograd through generator_synthesis in fp64 on the engine's leaky-ReLU branches: on batch slices of one
    sample (max_chunk = 1), and for 512^2 with channel_multiplier = 1 and for 1024^2 (32-channel superpixel layers) on mixed slices
    (_mixed_slices: a ragged last slice, the low-resolution layers' dots written whole-batch, the high-resolution ones per slice)"""
    sd, size, cm, lat, g_img = _synthesis_case(which)
    eng = StyleGan2Engine(sd, size, DEV, mode, channel_multiplier=cm)
    if which in MIXED:
        _mixed_slices(eng)
    else:
        eng.max_chunk = 1
    tape = SynthesisTape()
    eng.synthesis(lat.to(DEV), tape=tape)
    if which in MIXED:
        assert tape.slices == [(0, 2), (2, 1)]
        assert {k[1] for k in tape.acts if k[0] == id(eng.blocks[3][1])} == {0}          # 64^2: whole batch
        assert {k[1] for k in tape.acts if k[0] == id(eng.blocks[4][0])} == {0, 2}       # 128^2: slices
        assert (eng.blocks[-1][1].conv_sp is not None) == (mode == "bf16")                # 32 channels at the top: superpixel in bf16
    else:
        assert len(tape.slices) == lat.shape[0]
    g_nhwc = F.pad(g_img.permute(0, 2, 3, 1), (0, 1)).to(DEV)
    got = eng.synthesis_backward(tape, [g_nhwc[lo:lo + n].contiguous() for lo, n in tape.slices])
    latd = lat.to(DEV, torch.float64).requires_grad_()
    with _oracle_branches(_engine_branches(eng, tape)):
        img = stylegan_ref.generator_synthesis(_d64(sd, DEV), latd, size)
    ref, = torch.autograd.grad((img * g_img.to(img)).sum(), [latd])
    assert got.shape == ref.shape
    err, worst = rel_l2(got, ref), worst_code_rel_l2(got, ref)
    print(f"synthesis backward {which} {mode}: rel-L2 {err:.3e}, worst code {worst:.3e}")
    if mode == "fp32":
        assert err <= 1e-4, err
    else:
        gate, gate_code = BF16_SYNTHESIS_GATES[which]
        assert err <= gate and worst <= gate_code, (err, worst)


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
    codes' dtype, on the codes' device"""
    cast = lambda sd: {k: v.to(codes.device, codes.dtype) if v.is_floating_point() else v.to(codes.device) for k, v in sd.items()}
    dec = cast(stylegan_ref._sub(ck["state_dict"], "decoder" if kind == "e4e" else "decoder.module"))
    lat = stylegan_ref.mix_codes(dec, codes, z.to(codes) * (1.0 if kind == "e4e" else 0.8), alphas)
    img = F.adaptive_avg_pool2d(stylegan_ref.generator_synthesis(dec, lat, size), (256, 256))
    if kind != "e4e":
        img = img.clone()
        img[:, :, :32] = -1.0
        img[:, :, -32:] = -1.0
        img = F.interpolate(img, size=(128, 128), mode="bilinear", align_corners=False)
    pur = img * 0.5 + 0.5
    return stylegan_ref.resnet_forward(cast(clf_ck["state_dict"]), (pur - 0.5) / 0.5, 1 if kind == "e4e" else 32), pur


def _check_from_codes(kind, size, batch, tol, mode="fp32", mixed_slices=False):
    """from_codes forward and input gradient (preds_only both ways) against the fp64 oracle on the GPU, on the branches the engine's
    generator and classifier took (from their tapes).  tol: rel-L2 gate of the gradient, or {preds_only: (rel-L2 gate, gate of the worst
    code index)}"""
    dm, ck, clf_ck, alphas = _make_defense(kind, size, mode)
    if mixed_slices:
        _mixed_slices(dm.autoencoder.decoder)
    n_codes = len(alphas)
    g = torch.Generator().manual_seed(size + batch)
    codes = torch.randn(batch, n_codes, 512, generator=g)
    z = torch.randn(n_codes, batch, 512, generator=g)
    hw = 256 if kind == "e4e" else 128
    dm.set_explicit_noise([torch.zeros(batch, 3, hw, hw), z])
    tape = CodesTape()
    dm._from_codes_cuda(codes.to(DEV), tape=tape)                             # the forward from_codes runs, for its branches
    if mixed_slices:
        assert tape.syn.slices == [(0, 2), (2, 1)]
    masks, cls = _engine_branches(dm.autoencoder.decoder, tape.syn), _classifier_branches(tape.cls)
    branches = lambda: _oracle_branches(masks, cls)
    with branches(), torch.no_grad():
        logits_ref, pur_ref = _ref_tail(kind, ck, clf_ck, codes.to(DEV, torch.float64), z, alphas, size)
    g_l, g_p = torch.randn(logits_ref.shape, generator=g).to(DEV), torch.randn(pur_ref.shape, generator=g).to(DEV)
    for preds_only in (True, False):
        cd = codes.to(DEV).requires_grad_()
        cr = codes.to(DEV, torch.float64).requires_grad_()
        if preds_only:
            logits = dm.from_codes(cd)
            loss = (logits * g_l).sum()
            with branches():
                lr, _ = _ref_tail(kind, ck, clf_ck, cr, z, alphas, size)
            ref, = torch.autograd.grad((lr * g_l.double()).sum(), [cr])
        else:
            logits, pur = dm.from_codes(cd, preds_only=False)
            if mode == "fp32":
                assert rel_l2(pur, pur_ref) <= 1e-4
            else:                                                           # the project's bf16 criterion on purified images in [0, 1]
                assert (pur.double() - pur_ref).abs().max().item() <= 1e-2
            loss = (logits * g_l).sum() + (pur * g_p).sum()
            with branches():
                lr, pr = _ref_tail(kind, ck, clf_ck, cr, z, alphas, size)
            ref, = torch.autograd.grad((lr * g_l.double()).sum() + (pr * g_p.double()).sum(), [cr])
        lerr = ((logits.detach().double() - logits_ref).abs().max() / logits_ref.abs().max()).item()
        got, = torch.autograd.grad(loss, [cd])
        err, worst = rel_l2(got, ref), worst_code_rel_l2(got, ref)
        print(f"from_codes {kind} {size}^2 {mode} batch {batch} preds_only={preds_only}: logits max-abs / max {lerr:.3e}, "
              f"gradient rel-L2 {err:.3e}, worst code {worst:.3e}")
        if mode == "fp32":
            # the fp32 forward (the same kernels as __call__) at the project's fp32 logits criterion (test_stylegan_paths_gpu.py)
            assert lerr <= 1e-3, lerr
            assert err <= tol, (kind, preds_only, err)
        else:
            # bf16 logits are reported only, as in test_classifier_grad_gpu.py: the random-init ResNets amplify bf16 rounding to about
            # one logit unit (2e-2 of the cars logits, 0.8 of the small gender ones) even on the engine's branches
            gate, gate_code = tol[preds_only]
            assert err <= gate and worst <= gate_code, (kind, preds_only, err, worst)
    return dm


@pytest.mark.parametrize("kind", ["e4e", "trans"])
def test_from_codes_gradient(kind):
    dm = _check_from_codes(kind, 256, 2, 1e-4)
    # the encoder half is still missing: a differentiable call on the images refuses
    hw = 256 if kind == "e4e" else 128
    dm.set_explicit_noise(None)
    with pytest.raises(NotImplementedError, match="encoder half"):
        dm(torch.rand(1, 3, hw, hw, device=DEV).requires_grad_())


# bf16 gradient against the fp64 oracle on the engine's branches, batch 3 on mixed slices, measured on a B200: {preds_only: (rel-L2,
# worst rel-L2 of one code index)}; each gate is about twice the measurement
BF16_FROM_CODES_GATES = {"e4e": {True: (3e-2, 4e-2),           # measured 1.55e-2, 1.94e-2
                                False: (2.5e-2, 3e-2)},         # 1.23e-2, 1.46e-2
                         "trans": {True: (3e-2, 3.3e-2),        # 1.44e-2, 1.64e-2
                                   False: (3e-2, 3.3e-2)}}      # 1.41e-2, 1.64e-2


@pytest.mark.parametrize("kind,size,mode", [("e4e", 1024, "fp32"), ("trans", 512, "fp32"), ("e4e", 1024, "bf16"), ("trans", 512, "bf16")],
                         ids=["e4e-1024", "trans-512", "e4e-1024-bf16", "trans-512-bf16"])
def test_from_codes_gradient_full_size(kind, size, mode):
    """fp32: one sample; bf16 (the timed configuration): 3 samples, the generator's blocks at >= 128^2 on slices of 2 + 1"""
    if mode == "fp32":
        _check_from_codes(kind, size, 1, 1e-4)
    else:
        _check_from_codes(kind, size, 3, BF16_FROM_CODES_GATES[kind], mode="bf16", mixed_slices=True)


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
