"""GPU: input gradient of the E4E encode half -- images -> preprocess -> IR-SE50 -> FPN -> map2style heads -> W+ codes (`to_codes`).

Kernels: the PReLU mask mode of the conv epilogues against fp64 autograd of conv + PReLU, the fused phase interleave, subsample2x_bwd and
codes_assemble_bwd bit-exact against torch emulations, se_residual_bwd without biases against autograd of the SE module.
Engine and defense: against autograd of oracle/stylegan_ref in fp64 on the GPU, on the ENGINE's branches (see _encoder_masks and _branches)."""
import contextlib
import math

import pytest
import torch
import torch.nn.functional as F

from gen_adversarial_b200 import _lib, ops, synth
from gen_adversarial_b200._lib import MUL_RELU_MASK, MUL_PRELU_FROM_Y
from gen_adversarial_b200.autograd import CodesTape, ImagesTape
from gen_adversarial_b200.fold import Folder
from gen_adversarial_b200.irse_engine import E4EEncoderEngine, EncoderTape
from gen_adversarial_b200.defenses.ours.models import (E4EStyleGanDefenseModel, TransStyleGanDefenseModel, CelebaGenderClassifier,
                                                       CarsTypeClassifier)
from oracle import stylegan_ref
from tests.test_stylegan_grad_gpu import _engine_branches, _classifier_branches, _mixed_slices

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def rel_l2(a, b):
    a, b = a.double(), b.double()
    return ((a - b).norm() / b.norm()).item()


def worst_image_rel_l2(a, b):
    a, b = a.double().flatten(1), b.double().flatten(1)
    return ((a - b).norm(dim=1) / b.norm(dim=1)).max().item()


def _bf16_ulp(t):
    """spacing of bf16 numbers (8 significant bits) at |t|, elementwise, for float64 t"""
    _, e = torch.frexp(t.abs())
    return torch.ldexp(torch.ones_like(t), e - 8) * (t != 0)


def _cast(sd, dtype=torch.float64):
    return {k: v.to(DEV, dtype) if v.is_floating_point() else v.to(DEV) for k, v in sd.items()}


def _enc_sd(ck):
    return stylegan_ref._sub(ck["state_dict"], "encoder")


# ------------------------------------------------------------------------------------------------ kernels
@pytest.mark.parametrize("path,n,h,w,cin,cout,k,out", [
    ("tc", 3, 16, 16, 64, 64, 3, "bf16"),          # persistent 3x3, lean add/mul epilogue
    ("tc", 1, 32, 32, 128, 64, 3, "f32"),
    ("tc", 3, 64, 64, 64, 128, 3, "bf16"),
    ("tc", 1, 4, 256, 64, 64, 3, "f32"),            # > 128-wide image
    ("tc", 3, 12, 16, 64, 24, 3, "bf16"),           # partial tiles, Cout not a multiple of 16: general epilogue
    ("tc", 3, 16, 16, 128, 256, 1, "bf16"),         # 1x1: per-tap kernel, generic epilogue
    ("tc", 1, 8, 8, 512, 40, 1, "f32"),
    ("simt", 3, 12, 10, 32, 24, 3, "f32"),
    ("simt", 1, 7, 9, 16, 8, 3, "bf16"),
])
def test_prelu_mask_epilogue(path, n, h, w, cin, cout, k, out):
    """(conv(g) + add) * PReLU'(z) with the derivative from the sign of y = PReLU(z) against fp64 autograd of conv + PReLU"""
    g = torch.Generator().manual_seed(n * 1000 + h * 10 + cout)
    wt = torch.randn(cout, cin, k, k, generator=g, dtype=torch.float64) / math.sqrt(cin * k * k)
    f = Folder({}, DEV, want_tc=path == "tc")
    L = f.conv(wt, None, pad=k // 2)
    slope = torch.rand(cout, generator=g, dtype=torch.float64) * 0.4 + 0.05
    L.act_slope = slope.float().to(DEV)
    x = torch.randn(n, h, w, cin, generator=g)
    z = torch.randn(n, h, w, cout, generator=g, dtype=torch.float64)
    y = torch.where(z > 0, z, z * slope).to(torch.bfloat16)                      # the taped PReLU output
    add = torch.randn(n, h, w, cout, generator=g)
    od = torch.float32 if out == "f32" else torch.bfloat16
    if path == "tc":
        xin = x.to(torch.bfloat16)
        wref = L.w_tc.double().cpu().view(cout, k, k, cin).permute(0, 3, 1, 2)
        assert ops.conv2d_tc_supported(xin.to(DEV), L)
        ob, of = ops.conv2d_tc(xin.to(DEV), L, want_bf16=out == "bf16", want_f32=out == "f32", add=add.to(DEV), mul=y.to(DEV),
                               mul_mode=MUL_PRELU_FROM_Y)
        got = of if out == "f32" else ob
    else:
        xin = x
        wref = L.w_simt.double().cpu().view(k, k, cin, cout).permute(3, 2, 0, 1)
        got = ops.conv2d_simt(xin.to(DEV), L, od, add=add.to(DEV), mul=y.to(DEV), mul_mode=MUL_PRELU_FROM_Y)
    v = F.conv2d(xin.double().permute(0, 3, 1, 2), wref, padding=k // 2) + add.double().permute(0, 3, 1, 2)
    zz = y.double().permute(0, 3, 1, 2).requires_grad_()
    ref, = torch.autograd.grad(F.prelu(zz, slope), [zz], v)
    ref = ref.permute(0, 2, 3, 1)
    d = (got.double().cpu() - ref).abs()
    big = ref.abs().max().item()
    if out == "f32":
        assert d.max().item() <= 1e-5 * big
    else:
        # one ulp of the reference, plus 1e-6 max|ref| for the sums that nearly cancel (there the fp32 accumulation error exceeds the ulp)
        bad = d > _bf16_ulp(ref) + 1e-6 * big
        assert not bool(bad.any()), (int(bad.sum()), (d / _bf16_ulp(ref)).max().item())


def _d2s(x4):
    n, h, w, c4 = x4.shape
    c = c4 // 4
    return x4.view(n, h, w, 2, 2, c).permute(0, 1, 3, 2, 4, 5).reshape(n, 2 * h, 2 * w, c)


@pytest.mark.parametrize("mode", [MUL_RELU_MASK, MUL_PRELU_FROM_Y, None])
@pytest.mark.parametrize("add_dt", [None, torch.float32, torch.bfloat16])
@pytest.mark.parametrize("out_dt", [torch.float32, torch.bfloat16])
def test_phase_interleave(mode, add_dt, out_dt):
    g = torch.Generator().manual_seed(7)
    n, h, w, c = 3, 5, 7, 24
    x4 = torch.randn(n, h, w, 4 * c, generator=g)
    add = torch.randn(n, 2 * h, 2 * w, c, generator=g).to(add_dt) if add_dt is not None else None
    mul = torch.randn(n, 2 * h, 2 * w, c, generator=g).to(torch.bfloat16) if mode is not None else None
    slope = torch.rand(c, generator=g) * 0.3 + 0.05
    got = ops.phase_interleave(x4.to(DEV), add.to(DEV) if add is not None else None, mul.to(DEV) if mul is not None else None,
                               mode if mode is not None else 0, slope.to(DEV), out_dt)
    ref = _d2s(x4)
    assert torch.equal(ops.depth_to_space2(x4.to(DEV)).cpu(), ref)
    if add is not None:
        ref = ref + add.float()
    if mul is not None:
        m = mul.float()
        ref = ref * (torch.where(m > 0, torch.ones_like(m), torch.zeros_like(m)) if mode == MUL_RELU_MASK
                     else torch.where(m > 0, torch.ones_like(m), slope.expand_as(m)))
    assert torch.equal(got.cpu(), ref.to(out_dt))


@pytest.mark.parametrize("h,w", [(8, 12), (7, 9)])
@pytest.mark.parametrize("dt", [torch.float32, torch.bfloat16])
def test_subsample2x_bwd(h, w, dt):
    g = torch.Generator().manual_seed(3)
    x = torch.randn(3, h, w, 16, generator=g)
    gs = torch.randn(3, (h + 1) // 2, (w + 1) // 2, 16, generator=g)
    assert torch.equal(ops.subsample2x(x.to(DEV)).cpu(), x[:, ::2, ::2])
    got = ops.subsample2x_bwd(gs.to(DEV), (h, w), dt).cpu()
    ref = torch.zeros(3, h, w, 16)
    ref[:, ::2, ::2] = gs
    assert torch.equal(got, ref.to(dt))


@pytest.mark.parametrize("b,l", [(1, 14), (5, 18)])
def test_codes_assemble_bwd(b, l):
    g = torch.Generator().manual_seed(b)
    gc = torch.randn(b, l, 512, generator=g)
    got = ops.codes_assemble_bwd(gc.to(DEV)).cpu()
    ref = gc.permute(1, 0, 2).clone()
    s = gc[:, 0].clone()
    for i in range(1, l):
        s = s + gc[:, i]
    ref[0] = s
    assert torch.equal(got, ref)
    # the adjoint of the forward assembly, on the device
    h = torch.randn(l, b, 1, 1, 512, generator=g)
    codes = ops.codes_assemble(h.to(DEV), True, True, None, b, l, 512).cpu().double()
    lhs, rhs = (codes * gc.double()).sum().item(), (h.double().view(l, b, 512) * got.double()).sum().item()
    assert abs(lhs - rhs) <= 1e-5 * abs(lhs)
    if b > 1:                                                                   # batch-independent
        assert torch.equal(ops.codes_assemble_bwd(gc[1:2].to(DEV)).cpu(), got[:, 1:2])


@pytest.mark.parametrize("dt", [torch.float32, torch.bfloat16])
def test_se_residual_bwd_without_biases(dt):
    g = torch.Generator().manual_seed(5)
    n, hh, ww, c, hid = 2, 16, 16, 64, 4
    r = torch.randn(n, hh, ww, c, generator=g)
    skip = torch.randn(n, hh, ww, c, generator=g)
    w1 = torch.randn(hid, c, generator=g) / math.sqrt(c)
    w2 = torch.randn(c, hid, generator=g) / math.sqrt(hid)
    go = torch.randn(n, hh, ww, c, generator=g)
    se = (w1.to(DEV), None, w2.to(DEV), None)
    sums = ops.channel_sum(r.to(DEV))
    out, _, _, _ = ops.se_residual(r.to(DEV), sums, se, 1.0, skip.to(DEV), torch.float32, act_op=0)
    got = ops.se_residual_bwd(go.to(DEV), r.to(DEV), sums, se, 1.0, dt).double().cpu()
    rr = r.double().permute(0, 3, 1, 2).requires_grad_()
    s = torch.sigmoid(F.conv2d(F.relu(F.conv2d(rr.mean(dim=(2, 3), keepdim=True), w1.double().view(hid, c, 1, 1))),
                               w2.double().view(c, hid, 1, 1)))
    o = rr * s + skip.double().permute(0, 3, 1, 2)
    assert rel_l2(out.cpu().permute(0, 3, 1, 2), o.detach()) <= 1e-6
    ref, = torch.autograd.grad(o, [rr], go.double().permute(0, 3, 1, 2))
    assert rel_l2(got.permute(0, 3, 1, 2), ref) <= (1e-6 if dt == torch.float32 else 4e-3)


# ------------------------------------------------------------------------------------------------ oracle on the engine's branches
def _encoder_masks(enc_sd, tape: EncoderTape):
    """the branches the engine's encoder forward took: PReLU (sign of the taped stem output and conv1 outputs), the SE hidden ReLUs
    (recomputed in fp64 from the taped channel sums) and the heads' LeakyReLUs (sign of the taped head activations), all NCHW"""
    nchw = lambda t: (t.float() > 0).permute(0, 3, 1, 2)
    prelu = [nchw(tape.stem)] + [nchw(h) for h, _, _ in tape.units]
    relu = []
    for i, (_, r, sums) in enumerate(tape.units):
        mean = sums.double().sum(dim=1) / (r.shape[1] * r.shape[2])                          # [n][parts][c] -> [n][c]
        w1 = enc_sd[f"body.{i}.res_layer.5.fc1.weight"].to(DEV, torch.float64).flatten(1)
        relu.append((mean @ w1.t() > 0).view(mean.shape[0], -1, 1, 1))
    leaky = [nchw(a) for acts in tape.heads for a in acts]
    return prelu, relu, leaky


@contextlib.contextmanager
def _branches(prelu=(), relu=(), leaky=(), gen=None, cls_stem=None):
    """oracle/stylegan_ref with its PReLUs, ReLUs (SE hidden ReLUs first, then the classifier's), LeakyReLUs, the generator's fused leaky
    ReLUs (gen) and the classifier's stem max-pool picks (cls_stem) following the engine, in the oracle's call order"""
    orig_flr = stylegan_ref.fused_leaky_relu
    it_p, it_r, it_l = iter(prelu), iter(relu), iter(leaky)

    class _Functional:
        def __getattr__(self, name):
            return getattr(F, name)

        def prelu(self, x, a):
            m = next(it_p)
            assert m.shape == x.shape
            return torch.where(m, x, x * a.view(1, -1, 1, 1))

        def relu(self, x):
            m = next(it_r)
            assert m.shape == x.shape, (m.shape, x.shape)
            return torch.where(m.to(x.device), x, torch.zeros_like(x))

        def leaky_relu(self, x, s):
            if s != 0.01:                                     # the generator's mapping MLP (fused_leaky_relu, slope 0.2)
                return F.leaky_relu(x, s)
            m = next(it_l)
            assert m.shape == x.shape
            return torch.where(m, x, s * x)

        def max_pool2d(self, x, k, s, p):
            _, idx = F.max_pool2d(cls_stem.contiguous(), k, s, p, return_indices=True)
            return x.flatten(2).gather(2, idx.to(x.device).flatten(2)).view(idx.shape)

    if gen is not None:
        it_g = iter(gen)

        def fused_leaky_relu(x, bias):
            if x.dim() != 4:
                return orig_flr(x, bias)
            t = x + bias.view(1, -1, 1, 1)
            return torch.where(next(it_g).to(t.device), t, 0.2 * t) * math.sqrt(2.0)
        stylegan_ref.fused_leaky_relu = fused_leaky_relu
    stylegan_ref.F = _Functional()
    try:
        yield
    finally:
        stylegan_ref.F = F
        stylegan_ref.fused_leaky_relu = orig_flr


# bf16 against the fp64 oracle on the engine's branches, measured on a B200: (rel-L2, worst rel-L2 of one image); each gate is about
# twice the measurement
BF16_BACKBONE_GATES = {"tf32": (1e-2, 1e-2),        # measured 5.0e-3, 5.0e-3
                       "bf16": (1e-2, 1e-2)}        # 5.1e-3, 5.1e-3
BF16_ENCODE_GATES = {256: (1.6e-2, 1.6e-2),         # 7.9e-3, 7.9e-3
                     1024: (1.6e-2, 1.6e-2)}        # 7.9e-3, 7.9e-3
BF16_CHAIN_GATES = (3e-2, 3.6e-2)                   # 1.53e-2, 1.83e-2


@pytest.mark.parametrize("mode", ["fp32", "tf32", "bf16"])
def test_backbone_backward(mode, monkeypatch):
    """random gradients on c1 / c2 / c3 at 256^2, batch 2; bf16 with the TF32 backbone (E4E's default) and the bf16 one"""
    monkeypatch.setenv("GA_E4E_TF32_BACKBONE", "0" if mode == "bf16" else "1")
    ck = synth.make_e4e_checkpoint(stylegan_size=256)
    sd = _enc_sd(ck)
    eng = E4EEncoderEngine(sd, 256, None, DEV, "fp32" if mode == "fp32" else "bf16")
    assert eng.backbone.tf32 == (mode == "tf32")
    eng.build_dgrad()
    g = torch.Generator().manual_seed(21)
    x = torch.rand(2, 256, 256, 3, generator=g) * 2 - 1
    tape = EncoderTape()
    c1, c2, c3 = eng.backbone.forward(x.to(DEV), tape)
    gs = [torch.randn(t.shape, generator=g) for t in (c1, c2, c3)]
    got = eng.backbone.backward(tape, *[t.to(DEV) for t in gs])
    got2 = eng.backbone.backward(tape, *[t.to(DEV) for t in gs])
    assert torch.equal(got, got2)                                                           # the tape is left intact
    prelu, relu, _ = _encoder_masks(sd, tape)
    xr = x.to(DEV, torch.float64).permute(0, 3, 1, 2).requires_grad_()
    with _branches(prelu, relu):
        taps = stylegan_ref.irse50_backbone(_cast(sd), xr)
    loss = sum((t * gt.to(DEV, torch.float64).permute(0, 3, 1, 2)).sum() for t, gt in zip(taps, gs))
    ref, = torch.autograd.grad(loss, [xr])
    got = got.permute(0, 3, 1, 2)
    err, worst = rel_l2(got, ref), worst_image_rel_l2(got, ref)
    print(f"backbone backward {mode}: rel-L2 {err:.3e}, worst image {worst:.3e}")
    if mode == "fp32":
        assert err <= 1e-4, err
    else:
        gate, gate_img = BF16_BACKBONE_GATES[mode]
        assert err <= gate and worst <= gate_img, (err, worst)


@pytest.mark.parametrize("mode", ["fp32", "bf16"])
@pytest.mark.parametrize("size", [256, 1024])
def test_encode_backward(size, mode):
    """encode_backward against autograd of e4e_encode (14 heads at 256, 18 at 1024), batch 2"""
    ck = synth.make_e4e_checkpoint(stylegan_size=size)
    sd = _enc_sd(ck)
    eng = E4EEncoderEngine(sd, size, ck["latent_avg"], DEV, mode)
    g = torch.Generator().manual_seed(size)
    x = torch.rand(2, 256, 256, 3, generator=g) * 2 - 1
    tape = EncoderTape()
    codes = eng.encode(x.to(DEV), tape)
    assert torch.equal(codes, eng.encode(x.to(DEV)))                                        # taping does not change the forward
    assert len(tape.heads) == eng.style_count == (14 if size == 256 else 18)
    gc = torch.randn(codes.shape, generator=g)
    got = eng.encode_backward(tape, gc.to(DEV)).permute(0, 3, 1, 2)
    xr = x.to(DEV, torch.float64).permute(0, 3, 1, 2).requires_grad_()
    with _branches(*_encoder_masks(sd, tape)):
        ref_codes = stylegan_ref.e4e_encode(_cast(sd), xr, size, ck["latent_avg"].to(DEV, torch.float64))
    ref, = torch.autograd.grad((ref_codes * gc.to(DEV, torch.float64)).sum(), [xr])
    err, worst = rel_l2(got, ref), worst_image_rel_l2(got, ref)
    cerr = rel_l2(codes, ref_codes.detach())
    print(f"encode backward {size} {mode}: codes rel-L2 {cerr:.3e}, gradient rel-L2 {err:.3e}, worst image {worst:.3e}")
    if mode == "fp32":
        assert cerr <= 1e-4 and err <= 1e-4, (cerr, err)
    else:
        gate, gate_img = BF16_ENCODE_GATES[size]
        assert err <= gate and worst <= gate_img, (err, worst)


# ------------------------------------------------------------------------------------------------ defenses
def _e4e_defense(size, mode, eps=0.0, blur=False, ck=None):
    n_codes = 2 * int(math.log2(size)) - 2
    alphas = [0.1 + 0.8 * i / (n_codes - 1) for i in range(n_codes)]
    ck = ck or synth.make_e4e_checkpoint(stylegan_size=size)
    clf_ck = synth.make_resnet50_checkpoint()
    dm = E4EStyleGanDefenseModel(CelebaGenderClassifier(clf_ck, DEV, mode=mode), ck, alphas, 1.0, eps, blur, DEV, mode=mode)
    return dm, ck, clf_ck, alphas


def test_to_codes_forward_matches_call_head():
    dm, _, _, _ = _e4e_defense(256, "fp32", eps=0.05, blur=True)
    dm.noise_seed = 77
    x = torch.rand(2, 3, 256, 256, generator=torch.Generator().manual_seed(0)).to(DEV)
    plain = dm.to_codes(x)
    taped = dm.to_codes(x.clone().requires_grad_())
    assert taped.requires_grad and torch.equal(plain, taped.detach())                       # bit-identical with and without the tape
    assert torch.equal(plain, dm._encode(dm._preprocessed(x)))


@pytest.mark.parametrize("blur", [False, True])
def test_to_codes_gradient(blur):
    """fp32 against autograd of _preprocess + e4e_encode in fp64, eps > 0 with explicit noise (the clamp mask is exercised)"""
    eps = 8.0
    dm, ck, _, alphas = _e4e_defense(256, "fp32", eps=eps, blur=blur)
    g = torch.Generator().manual_seed(31 + blur)
    x = torch.rand(2, 3, 256, 256, generator=g)
    x[:, :, 100:104], x[:, :, 200:204] = 0.002, 0.998          # flat bands that the noise pushes past 0 and 1 with blur on as well
    noise0 = torch.randn(2, 3, 256, 256, generator=g)
    dm.set_explicit_noise([noise0, torch.randn(len(alphas), 2, 512, generator=g)])
    xd = x.to(DEV).requires_grad_()
    codes = dm.to_codes(xd)
    gc = torch.randn(codes.shape, generator=g).to(DEV)
    got, = torch.autograd.grad(codes, [xd], gc)
    # the taped encoder branches of this forward
    tape = ImagesTape()
    with torch.no_grad():
        assert torch.equal(dm._to_codes_cuda(x.to(DEV), tape), codes.detach())
    pre = tape.pre
    assert bool(((pre < 0) | (pre > 1)).any()), "the clamp is not exercised"
    sd = _enc_sd(ck)
    # the oracle's preprocessing on the host (its blur taps live there), the encoder on the device; autograd spans both
    xr = x.double().requires_grad_()
    with _branches(*_encoder_masks(sd, tape.enc)):
        xn = stylegan_ref._preprocess(xr, noise0.double(), eps, blur).to(DEV)
        ref_codes = stylegan_ref.e4e_encode(_cast(sd), xn, 256, ck["latent_avg"].to(DEV, torch.float64))
    ref, = torch.autograd.grad((ref_codes * gc.double()).sum(), [xr])
    err = rel_l2(got.cpu(), ref)
    print(f"to_codes gradient blur={blur}: codes rel-L2 {rel_l2(codes.detach(), ref_codes.detach()):.3e}, gradient rel-L2 {err:.3e}")
    assert err <= 1e-4, err


def _check_chain(size, batch, mode, mixed_slices=False):
    """from_codes(to_codes(x)) against autograd of e4e_defense_call in fp64 on the engine's branches (encoder, generator, classifier)"""
    dm, ck, clf_ck, alphas = _e4e_defense(size, mode, eps=4.0)
    if mixed_slices:
        _mixed_slices(dm.autoencoder.decoder)
    g = torch.Generator().manual_seed(size + batch)
    x = torch.rand(batch, 3, 256, 256, generator=g)
    noise0 = torch.randn(batch, 3, 256, 256, generator=g)
    z = torch.randn(len(alphas), batch, 512, generator=g)
    dm.set_explicit_noise([noise0, z])
    itape, ctape = ImagesTape(), CodesTape()
    with torch.no_grad():
        codes = dm._to_codes_cuda(x.to(DEV), itape)
        dm._from_codes_cuda(codes, tape=ctape)
        call_logits, _ = dm(x.to(DEV), preds_only=False)
    if mixed_slices:
        assert ctape.syn.slices == [(0, 2), (2, 1)]
    prelu, se_relu, leaky = _encoder_masks(_enc_sd(ck), itape.enc)
    cls_relu, cls_stem = _classifier_branches(ctape.cls)
    branches = lambda: _branches(prelu, se_relu + [m.to(DEV) for m in cls_relu], leaky, gen=_engine_branches(dm.autoencoder.decoder, ctape.syn),
                                 cls_stem=cls_stem)
    xd = x.to(DEV).requires_grad_()
    logits = dm.from_codes(dm.to_codes(xd))
    print(f"chain {size} {mode}: logits bit-identical to __call__: {torch.equal(logits.detach(), call_logits)}")
    assert (logits.detach() - call_logits).abs().max().item() <= 1e-6 * call_logits.abs().max().item()     # = __call__ with explicit noise
    gl = torch.randn(logits.shape, generator=g).to(DEV)
    got, = torch.autograd.grad(logits, [xd], gl)
    xr = x.to(DEV, torch.float64).requires_grad_()
    clf = {k: v for k, v in clf_ck["state_dict"].items()}
    with branches():
        lr, _ = stylegan_ref.e4e_defense_call({**ck, "state_dict": _cast(ck["state_dict"]), "latent_avg": ck["latent_avg"].to(DEV, torch.float64)},
                                              _cast(clf), xr, alphas, [noise0.to(DEV, torch.float64), z.to(DEV, torch.float64)], 4.0, False)
    ref, = torch.autograd.grad((lr * gl.double()).sum(), [xr])
    lerr = ((logits.detach().double() - lr.detach()).abs().max() / lr.detach().abs().max()).item()
    err, worst = rel_l2(got, ref), worst_image_rel_l2(got, ref)
    print(f"chain {size} {mode} batch {batch}: logits max-abs / max {lerr:.3e}, gradient rel-L2 {err:.3e}, worst image {worst:.3e}")
    return lerr, err, worst


def test_chain_gradient_fp32():
    lerr, err, _ = _check_chain(256, 2, "fp32")
    assert lerr <= 1e-3, lerr
    assert err <= 1e-4, err


def test_chain_gradient_bf16_full_size():
    """the timed configuration: 1024^2, batch 3, the generator's blocks at >= 128^2 on slices of 2 + 1"""
    _, err, worst = _check_chain(1024, 3, "bf16", mixed_slices=True)
    gate, gate_img = BF16_CHAIN_GATES
    assert err <= gate and worst <= gate_img, (err, worst)


def test_to_codes_repeated_backward_and_batch_position():
    dm, _, _, _ = _e4e_defense(256, "fp32", eps=0.5)
    dm.noise_seed = 1234
    g = torch.Generator().manual_seed(12)
    x = torch.rand(3, 3, 256, 256, generator=g).to(DEV).requires_grad_()
    codes = dm.to_codes(x)
    g1, g2 = torch.randn(codes.shape, generator=g).to(DEV), torch.randn(codes.shape, generator=g).to(DEV)
    a, = torch.autograd.grad(codes, [x], g1, retain_graph=True)
    b, = torch.autograd.grad(codes, [x], g2, retain_graph=True)
    c, = torch.autograd.grad(codes, [x], g1)
    assert torch.equal(a, c) and not torch.equal(a, b)
    # the preprocessing noise is keyed by the global sample index: sample 1 alone at sample_offset 1 gets the same codes and gradient
    dm.sample_offset = 1
    one = x.detach()[1:2].clone().requires_grad_()
    c1 = dm.to_codes(one)
    d, = torch.autograd.grad(c1, [one], g1[1:2])
    assert rel_l2(c1.detach(), codes.detach()[1:2]) <= 1e-6
    assert rel_l2(d, a[1:2]) <= 1e-5


def test_trans_to_codes_forward_only():
    ck, clf_ck = synth.make_trans_checkpoint(output_size=256), synth.make_resnext50_checkpoint()
    dm = TransStyleGanDefenseModel(CarsTypeClassifier(clf_ck, DEV, mode="fp32"), ck, [0.5] * 14, 1.0, 0.0, False, DEV, mode="fp32")
    dm.noise_seed = 5
    x = torch.rand(2, 3, 128, 128, generator=torch.Generator().manual_seed(1)).to(DEV)
    codes = dm.to_codes(x)
    assert codes.shape == (2, 16, 512) and torch.equal(codes, dm._encode(dm._preprocessed(x)))
    L = _lib.lib()
    torch.cuda.synchronize()
    n0 = L.ga_launch_count(0)
    with pytest.raises(NotImplementedError, match="Style-Transformer"):
        dm.to_codes(x.clone().requires_grad_())
    assert L.ga_launch_count(0) == n0                                                        # refused before any launch


def test_zero_prelu_slope_refuses_taping():
    ck = synth.make_e4e_checkpoint(stylegan_size=256)
    key = "encoder.body.4.res_layer.2.weight"
    ck["state_dict"][key] = ck["state_dict"][key].clone()
    ck["state_dict"][key][0] = 0.0
    dm, _, _, _ = _e4e_defense(256, "fp32", ck=ck)
    x = torch.rand(1, 3, 256, 256, generator=torch.Generator().manual_seed(2)).to(DEV)
    with pytest.raises(NotImplementedError, match="body.4.conv1"):
        dm.to_codes(x.clone().requires_grad_())
    assert dm.to_codes(x).shape == (1, 14, 512)
