"""CPU (fp64): the adjoint weights the StyleGAN2 engine folds for its input-gradient backward, and the C-ABI entries of that backward.

<conv(x), y> = <x, conv_adj(y)> for the plain and the up-sampling (phase) convs as the engine folds them, the superpixel pair conv of the
adjoint = the adjoint of the superpixel pair conv, and the ToRGB skip's up-sampling adjoint = the upfirdn2d call the engine makes."""
import ctypes

import pytest
import torch
import torch.nn.functional as F

from gen_adversarial_b200 import _lib, synth
from gen_adversarial_b200.fold import Folder
from gen_adversarial_b200.nvae_engine import make_dgrad_layer
from gen_adversarial_b200.stylegan_engine import StyleGan2Engine, superpixel_weights
from oracle import stylegan_ref

NEW_ENTRIES = ("ga_styled_bias_act_bwd", "ga_styled_bias_act_bwd_parts", "ga_style_bwd", "ga_image_pool_out_bwd", "ga_latent_lerp_bwd")


def _w(L):
    """fp32 SIMT weights [kh*kw*cin, cout] of a folded conv -> fp64 [cout, cin, kh, kw]"""
    return L.w_simt.to(torch.float64).view(L.kh, L.kw, L.cin, L.cout).permute(3, 2, 0, 1)


def _dot(a, b):
    return (a * b).sum().item()


@pytest.fixture(scope="module")
def engine():
    eng = StyleGan2Engine(synth.make_stylegan2_state_dict(16, seed=3), 16, "cpu", "fp32", _host_logic_test=True)
    eng._build_adjoint()
    return eng


def test_plain_and_phase_conv_adjoints(engine):
    g = torch.Generator().manual_seed(0)
    up, conv, _ = engine.blocks[0]
    for layer, fwd, adj, cout in ((engine.conv1, engine.conv1.conv, engine.conv1.conv_d, engine.conv1.cout),
                                  (conv, conv.conv, conv.conv_d, conv.cout),
                                  (up, up.phase_convs, up.phase_d, 4 * up.cout)):      # ONE conv over the de-interleaved [h, w, 4 cout]
        w, wa = _w(fwd), _w(adj)
        assert wa.shape == (layer.cin, cout, 3, 3) and adj.pad == 1 and adj.up == 1
        x = torch.randn(2, layer.cin, 5, 7, generator=g, dtype=torch.float64)
        y = torch.randn(2, cout, 5, 7, generator=g, dtype=torch.float64)
        lhs, rhs = _dot(F.conv2d(x, w, padding=1), y), _dot(x, F.conv2d(y, wa, padding=1))
        assert abs(lhs - rhs) <= 1e-12 * max(1.0, abs(lhs)), (lhs, rhs)


def test_superpixel_of_adjoint_is_adjoint_of_superpixel():
    g = torch.Generator().manual_seed(1)
    w = torch.randn(32, 32, 3, 3, generator=g, dtype=torch.float64)
    f = Folder({}, "cpu", want_tc=False)
    adj_of_sp = make_dgrad_layer(f, f.conv(superpixel_weights(w), None, pad=1), False)
    sp_of_adj = f.conv(superpixel_weights(_w(make_dgrad_layer(f, f.conv(w, None, pad=1), False))), None, pad=1)
    assert torch.equal(adj_of_sp.w_simt, sp_of_adj.w_simt)
    # and as a conv on pixel pairs: <sp(x), y> = <x, sp_adj(y)> in fp64
    x = torch.randn(1, 64, 4, 6, generator=g, dtype=torch.float64)
    y = torch.randn(1, 64, 4, 6, generator=g, dtype=torch.float64)
    lhs = _dot(F.conv2d(x, superpixel_weights(w), padding=1), y)
    rhs = _dot(x, F.conv2d(y, superpixel_weights(w.flip(2, 3).permute(1, 0, 2, 3)), padding=1))
    assert abs(lhs - rhs) <= 1e-12 * max(1.0, abs(lhs))


def test_engine_superpixel_adjoint_weights():
    """bf16 engine with 32-channel layers (512^2, channel multiplier 1): the pair conv of the adjoint is built from the adjoint weights"""
    eng = StyleGan2Engine(synth.make_stylegan2_state_dict(512, channel_multiplier=1, seed=3), 512, "cpu", "bf16", channel_multiplier=1,
                          _host_logic_test=True)
    eng._build_adjoint()
    conv = eng.blocks[-1][1]
    assert conv.cin == 32 and conv.conv_sp is not None and conv.conv_sp_d is not None
    ref = superpixel_weights(_w(conv.conv_d)).permute(0, 2, 3, 1).reshape(64, -1).to(torch.bfloat16)
    assert torch.equal(conv.conv_sp_d.w_tc, ref)


def test_skip_upsample_adjoint(engine):
    g = torch.Generator().manual_seed(2)
    rgb = engine.blocks[0][2]
    k = rgb.up_kernel.to(torch.float64)
    kd = rgb.up_kernel_d.to(torch.float64)
    x = torch.randn(2, 4, 6, 5, generator=g, dtype=torch.float64)
    y = torch.randn(2, 4, 12, 10, generator=g, dtype=torch.float64)
    lhs = _dot(stylegan_ref.upfirdn2d(x, k, up=2, pad=(2, 1)), y)
    rhs = _dot(x, stylegan_ref.upfirdn2d(y, kd, down=2, pad=(1, 1)))
    assert abs(lhs - rhs) <= 1e-12 * max(1.0, abs(lhs)), (lhs, rhs)


def test_new_entries_exported_and_checked():
    L = _lib.lib()
    for name in NEW_ENTRIES:
        assert name in _lib.declared_symbols() and hasattr(L, name), name
    assert L.ga_styled_bias_act_bwd_parts(1024 * 1024, 32) == 1024 * 1024 // 1024
    assert L.ga_styled_bias_act_bwd_parts(16, 512) == 1
    assert L.ga_styled_bias_act_bwd(None, None, None, None, None, None, None, None, 0.0, None, 0, None, None, None, None, None) != 0
    assert b"ga_styled_bias_act_bwd" in L.ga_last_error()
    assert L.ga_style_bwd(None, 0, None, 0, None, None, None, 1, 8, 8, None, None) != 0
    assert b"ga_style_bwd" in L.ga_last_error()
    assert L.ga_image_pool_out_bwd(None, None, 1, 1, 0, 0.5, None, None) != 0
    assert L.ga_latent_lerp_bwd(None, None, 1, 1, 1, None, None) != 0
