"""CPU (fp64): the weights the IR-SE50 / E4E input-gradient backward folds, the codes-assemble adjoint, the PReLU-slope refusal and the new
C-ABI entries.

conv1 of every IR-SE unit runs on BN(x) zero-padded AFTER the BN; its dgrad layer carries the BN scale folded into its weights, so
<conv(pad(a x)), y> = <x, dgrad(y)> exactly and the dgrad equals autograd of conv2d(pad(BN(x))) in fp64."""
import pytest
import torch
import torch.nn.functional as F

from gen_adversarial_b200 import _lib, synth
from gen_adversarial_b200._lib import PRE_AFFINE
from gen_adversarial_b200.fold import Folder
from gen_adversarial_b200.irse_engine import E4EEncoderEngine
from gen_adversarial_b200.nvae_engine import make_dgrad_layer

NEW_ENTRIES = ("ga_phase_interleave", "ga_subsample2x_bwd", "ga_codes_assemble_bwd")


def _w(L):
    """fp32 SIMT weights [kh*kw*cin, cout] of a folded conv -> fp64 [cout, cin, kh, kw]"""
    return L.w_simt.to(torch.float64).view(L.kh, L.kw, L.cin, L.cout).permute(3, 2, 0, 1)


def _encoder_sd(size=256, seed=4):
    return {k[len("encoder."):]: v for k, v in synth.make_e4e_checkpoint(stylegan_size=size, seed=seed)["state_dict"].items()
            if k.startswith("encoder.")}


def test_bn_scale_fold_is_adjoint_of_conv_of_padded_bn():
    g = torch.Generator().manual_seed(0)
    cin, cout = 16, 24
    w = torch.randn(cout, cin, 3, 3, generator=g, dtype=torch.float64).float().double()       # fp32-exact: the layer stores fp32
    a = torch.rand(cin, generator=g, dtype=torch.float64) * 1.5 + 0.25
    b = torch.randn(cin, generator=g, dtype=torch.float64)
    f = Folder({}, "cpu", want_tc=False)
    L = f.conv(w, None, pad=1, pre_op=PRE_AFFINE, pre_affine=(a, b))
    D = make_dgrad_layer(f, L, False, in_scale=a)
    assert D.pad == 1 and D.up == 1 and D.cin == cout and D.cout == cin
    x = torch.randn(2, cin, 7, 9, generator=g, dtype=torch.float64).requires_grad_()
    y = torch.randn(2, cout, 7, 9, generator=g, dtype=torch.float64)
    out = F.conv2d(F.pad(x * a.view(1, -1, 1, 1) + b.view(1, -1, 1, 1), (1, 1, 1, 1)), w)       # zero padding after the BN
    ref, = torch.autograd.grad(out, [x], y)
    got = F.conv2d(y, _w(D), padding=1)
    # the folded weights are rounded to fp32 once: a few fp32 ulps of the weights
    assert ((got - ref).norm() / ref.norm()).item() <= 1e-6
    # without the fold the dgrad is off by the BN scale
    plain = F.conv2d(y, _w(make_dgrad_layer(f, L, False)), padding=1)
    assert ((plain - ref).norm() / ref.norm()).item() > 0.1


def _assemble(h):
    """codes_assemble(heads_lb, use_w0) without latent_avg: h (L, B, D) -> codes (B, L, D), code l = h[l] + h[0] for l > 0"""
    c = h.clone()
    c[1:] = c[1:] + h[0:1]
    return c.permute(1, 0, 2)


def _assemble_bwd(gc):
    """the adjoint the kernel computes: g_heads[l] = g_codes[:, l] (l > 0), g_heads[0] = sum over l, in increasing l"""
    gh = gc.permute(1, 0, 2).clone()
    s = gc[:, 0].clone()
    for l in range(1, gc.shape[1]):
        s = s + gc[:, l]
    gh[0] = s
    return gh


def test_codes_assemble_adjoint():
    g = torch.Generator().manual_seed(1)
    h = torch.randn(18, 3, 512, generator=g, dtype=torch.float64)
    gc = torch.randn(3, 18, 512, generator=g, dtype=torch.float64)
    lhs, rhs = (_assemble(h) * gc).sum().item(), (h * _assemble_bwd(gc)).sum().item()
    assert abs(lhs - rhs) <= 1e-12 * abs(lhs)


def test_engine_dgrad_layers():
    """the engine's conv1 dgrads carry the BN scale, the conv2 / head dgrads the slopes of the activation that produced their mask"""
    eng = E4EEncoderEngine(_encoder_sd(), 256, None, "cpu", "fp32", _host_logic_test=True)
    eng.build_dgrad()
    bb = eng.backbone
    f = Folder({}, "cpu", want_tc=False)
    for i in (0, 3, 11):
        u = bb.units[i]
        ref = make_dgrad_layer(f, u.c1, False, in_scale=u.pre_scale64)
        assert torch.equal(u.c1_d.w_simt, ref.w_simt)
        assert u.c2_d.act_slope is u.c1.act_slope
    assert bb.units[0].c1_d.act_slope is bb.stem.act_slope and bb.units[1].c1_d.act_slope is None
    assert [u.sc_d is not None for u in bb.units] == [u.sc is not None for u in bb.units]
    assert len(eng.heads) == 14
    for hd in eng.heads:
        assert hd.convs_d[0].act_slope is None and all(D.act_slope is eng.slope for D in hd.convs_d[1:] + [hd.linear_d])


@pytest.mark.parametrize("key", ["input_layer.2.weight", "body.9.res_layer.2.weight"])
def test_nonpositive_prelu_slope_refuses_backward(key):
    sd = _encoder_sd()
    sd[key] = sd[key].clone()
    sd[key][5] = 0.0
    eng = E4EEncoderEngine(sd, 256, None, "cpu", "fp32", _host_logic_test=True)
    name = "input_layer" if key.startswith("input") else "body.9.conv1"
    with pytest.raises(NotImplementedError, match=name):
        eng.build_dgrad()
    assert not eng._has_dgrad


def test_new_entries_exported_and_checked():
    L = _lib.lib()
    for name in NEW_ENTRIES:
        assert name in _lib.declared_symbols() and hasattr(L, name), name
    assert L.ga_phase_interleave(None, None, None, 0, None, None, None) != 0
    assert b"ga_phase_interleave" in L.ga_last_error()
    assert L.ga_subsample2x_bwd(None, None, None) != 0
    assert b"ga_subsample2x_bwd" in L.ga_last_error()
    assert L.ga_codes_assemble_bwd(None, 1, 1, 1, None, None) != 0
    assert b"ga_codes_assemble_bwd" in L.ga_last_error()
    assert _lib.MUL_PRELU_FROM_Y == 3
