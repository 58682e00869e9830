"""GPU: the StyleGAN purification paths (BASELINE configs 3 and 4) through the C-ABI -- the encoder-side kernels against a
torch restatement of the same op (tests/emu_ops.py), the stride-2 / PReLU / act-after-add variants of the conv kernels, and the
whole drop-in defense classes against the fixtures produced by the unmodified reference (full-size architectures, batch 2)."""
import math
import os

import pytest
import torch
import torch.nn.functional as F

from gen_adversarial_b200 import ops, synth
from gen_adversarial_b200._lib import PRE_NONE, PRE_AFFINE, ACT_NONE, ACT_RELU, ACT_PRELU, ACT_SILU
from gen_adversarial_b200.defenses.ours import models as ga_models
from oracle.make_golden import stored_purified
from tests import emu_ops

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def _layer(cin, cout, k, stride, pad, post_act=ACT_NONE, after_add=False, pre_op=PRE_NONE, seed=0):
    g = torch.Generator().manual_seed(seed)
    w = torch.randn(cout, cin, k, k, generator=g) / math.sqrt(cin * k * k)
    L = ops.ConvLayer(k, k, stride, pad, cin, cout, post_act=post_act, pre_op=pre_op, name=f"t{cin}x{cout}k{k}s{stride}")
    L.w_simt = w.permute(2, 3, 1, 0).reshape(k * k * cin, cout).contiguous()
    L.w_tc = w.permute(0, 2, 3, 1).reshape(cout, k * k * cin).to(torch.bfloat16).contiguous()
    L.bias = torch.randn(cout, generator=g) * 0.1
    L.act_after_add = after_add
    if post_act == ACT_PRELU:
        L.act_slope = torch.rand(cout, generator=g) * 0.3 + 0.05
    if pre_op == PRE_AFFINE:
        L.pre_scale = torch.rand(cin, generator=g) + 0.5
        L.pre_shift = torch.randn(cin, generator=g) * 0.2
    return L


def _dev(L):
    import copy
    D = copy.copy(L)
    for f in ("w_simt", "w_tc", "bias", "pre_scale", "pre_shift", "act_slope"):
        v = getattr(L, f)
        setattr(D, f, None if v is None else v.to(DEV))
    return D


TC_CASES = [
    # n, h, w, cin, cout, k, stride, act, after_add, add
    (2, 32, 32, 64, 64, 3, 2, ACT_PRELU, False, False),       # IR-SE50 conv2 of a down unit
    (3, 16, 16, 128, 256, 1, 2, ACT_NONE, False, False),      # IR-SE50 / ResNet shortcut
    (4, 64, 64, 64, 128, 3, 2, ACT_RELU, False, False),       # ResNet stride-on-3x3
    (5, 16, 16, 512, 512, 3, 2, ACT_PRELU, False, False),     # map2style head
    (130, 2, 2, 512, 512, 3, 2, ACT_PRELU, False, False),     # map2style tail: 2x2 -> 1x1, images span tiles
    (2, 256, 256, 64, 64, 3, 2, ACT_NONE, False, False),      # W_out = 128
    (2, 16, 16, 256, 1024, 1, 1, ACT_RELU, True, True),       # bottleneck conv3: relu(conv + identity)
    (2, 8, 8, 64, 64, 3, 1, ACT_PRELU, False, True),
    (3, 12, 16, 64, 128, 3, 1, ACT_PRELU, False, False),      # Style-Transformer 192x256 input: 12x16 maps (partial tiles)
    (3, 24, 32, 64, 64, 3, 2, ACT_NONE, False, True),         # ... stride 2 onto a 12x16 map
    (2, 20, 32, 32, 96, 1, 1, ACT_RELU, True, True),
]


@pytest.mark.parametrize("case", TC_CASES)
def test_conv_tc_stride_prelu_after_add(case):
    n, h, w, cin, cout, k, stride, act, after_add, use_add = case
    L = _layer(cin, cout, k, stride, k // 2, act, after_add, seed=cin + cout + stride)
    x = torch.randn(n, h, w, cin).to(torch.bfloat16)
    ho, wo = ops.conv_out_hw(L, h, w)
    add = torch.randn(n, ho, wo, cout) if use_add else None
    _, ref = emu_ops.conv2d_tc(x, L, want_bf16=False, want_f32=True, add=add)
    D = _dev(L)
    assert ops.conv2d_tc_supported(x.to(DEV), D)
    ob, of = ops.conv2d_tc(x.to(DEV), D, want_bf16=True, want_f32=True, add=add.to(DEV) if use_add else None)
    assert of.shape == ref.shape
    scale = max(1.0, ref.abs().max().item())
    assert (of.cpu() - ref).abs().max().item() <= 2e-3 * scale
    assert (ob.float().cpu() - ref).abs().max().item() <= 1e-2 * scale


@pytest.mark.parametrize("case", [(2, 16, 16, 32, 48, 3, 2, ACT_PRELU, False, False, PRE_AFFINE),
                                  (2, 8, 8, 24, 40, 1, 1, ACT_RELU, True, True, PRE_NONE),
                                  (2, 33, 33, 3, 64, 7, 2, ACT_RELU, False, False, PRE_NONE),      # ResNet stem (persistent stem kernel)
                                  (2, 20, 24, 3, 64, 3, 1, ACT_PRELU, False, False, PRE_NONE),     # IR-SE50 stem
                                  (3, 17, 19, 3, 32, 3, 1, ACT_NONE, False, False, PRE_NONE),      # NVAE stem, odd sizes
                                  (40, 64, 64, 3, 64, 3, 1, ACT_RELU, False, False, PRE_NONE)])    # more pixels than one grid pass
def test_conv_simt_prelu_after_add(case):
    n, h, w, cin, cout, k, stride, act, after_add, use_add, pre = case
    L = _layer(cin, cout, k, stride, k // 2, act, after_add, pre, seed=cin)
    x = torch.randn(n, h, w, cin)
    ho, wo = ops.conv_out_hw(L, h, w)
    add = torch.randn(n, ho, wo, cout) if use_add else None
    ref = emu_ops.conv2d_simt(x, L, torch.float32, add=add)
    got = ops.conv2d_simt(x.to(DEV), _dev(L), torch.float32, add=add.to(DEV) if use_add else None)
    assert (got.cpu() - ref).abs().max().item() <= 3e-5 * max(1.0, ref.abs().max().item())


def test_pools_and_subsample():
    x = torch.randn(3, 17, 12, 8)
    for name in ("subsample2x", "maxpool3x3s2", "global_avgpool"):
        ref = getattr(emu_ops, name)(x)
        got = getattr(ops, name)(x.to(DEV))
        assert got.shape == ref.shape, name
        assert (got.cpu() - ref).abs().max().item() <= 1e-5, name


def test_se_residual_no_bias_affine_output():
    r, skip = torch.randn(2, 8, 8, 64), torch.randn(2, 8, 8, 64)
    w1, w2 = torch.randn(4, 64) * 0.2, torch.randn(64, 4) * 0.5
    aff = (torch.rand(64) + 0.5, torch.randn(64) * 0.1)
    sums_ref = r.reshape(2, 1, 64, 64).sum(dim=2)
    ref = emu_ops.se_residual(r, sums_ref, (w1, None, w2, None), 1.0, skip, act_affine=aff, act_dtype=torch.float32, act_op=ACT_NONE)
    rd = r.to(DEV)
    sums = ops.channel_sum(rd)
    got = ops.se_residual(rd, sums, (w1.to(DEV), None, w2.to(DEV), None), 1.0, skip.to(DEV), act_affine=(aff[0].to(DEV), aff[1].to(DEV)),
                          act_dtype=torch.float32, act_op=ACT_NONE)
    assert (got[0].cpu() - ref[0]).abs().max().item() <= 1e-5
    assert (got[2].cpu() - ref[2]).abs().max().item() <= 1e-5


def test_add_layernorm_and_attention():
    g = torch.Generator().manual_seed(0)
    x, y = torch.randn(3, 16, 1, 512, generator=g), torch.randn(3, 16, 1, 512, generator=g)
    gamma, beta = torch.rand(512, generator=g) + 0.5, torch.randn(512, generator=g) * 0.1
    ref = emu_ops.add_layernorm(x, y, gamma, beta, torch.float32)
    got, got2 = ops.add_layernorm(x.to(DEV), y.to(DEV), gamma.to(DEV), beta.to(DEV), torch.float32, out2_dtype=torch.bfloat16)
    assert (got.cpu() - ref).abs().max().item() <= 1e-5
    assert (got2.float().cpu() - ref).abs().max().item() <= 2e-2
    for s_hw in ((12, 16), (4, 4), (1, 16), (48, 64)):
        q = torch.randn(3, 16, 1, 512, generator=g)
        kv = torch.randn(3, s_hw[0], s_hw[1], 1024, generator=g)
        ref = emu_ops.attention(q, 0, kv, 0, kv, 512, 4, 128, torch.float32)
        got = ops.attention(q.to(DEV), 0, kv.to(DEV), 0, kv.to(DEV), 512, 4, 128, torch.float32)
        assert (got.cpu() - ref).abs().max().item() <= 2e-5, s_hw
    qkv = torch.randn(2, 16, 1, 1536, generator=g)                     # fused self-attention projection
    ref = emu_ops.attention(qkv, 0, qkv, 512, qkv, 1024, 4, 128, torch.float32)
    got = ops.attention(qkv.to(DEV), 0, qkv.to(DEV), 512, qkv.to(DEV), 1024, 4, 128, torch.float32)
    assert (got.cpu() - ref).abs().max().item() <= 2e-5


def test_codes_resize_image_out_philox():
    g = torch.Generator().manual_seed(1)
    heads = torch.randn(18, 3, 512, generator=g)
    avg = torch.randn(18, 512, generator=g)
    ref = emu_ops.codes_assemble(heads, True, True, avg, 3, 18, 512)
    got = ops.codes_assemble(heads.to(DEV), True, True, avg.to(DEV), 3, 18, 512)
    assert torch.equal(got.cpu(), ref)
    codes = torch.randn(3, 16, 512, generator=g)
    ref = emu_ops.codes_assemble(codes, False, False, avg[:16], 3, 16, 512)
    got = ops.codes_assemble(codes.to(DEV), False, False, avg[:16].to(DEV), 3, 16, 512)
    assert torch.equal(got.cpu(), ref)
    x = torch.rand(2, 128, 128, 3, generator=g)
    ref = emu_ops.resize_bilinear(x, 256, 256, 32, 192)
    got = ops.resize_bilinear(x.to(DEV), 256, 256, 32, 192)
    assert got.shape == (2, 192, 256, 3) and (got.cpu() - ref).abs().max().item() <= 1e-6
    ref = emu_ops.resize_bilinear(x, 100, 77, 3, 90)                   # generic scale factors
    got = ops.resize_bilinear(x.to(DEV), 100, 77, 3, 90)
    assert (got.cpu() - ref).abs().max().item() <= 1e-5
    img = torch.randn(2, 64, 64, 4, generator=g)
    for k1, k2, mask in ((4, 1, 0), (2, 2, 2), (1, 1, 0)):
        rp, rc = emu_ops.image_pool_out(img, k1, k2, mask, (0.5, 0.5), torch.float32)
        gp, gc = ops.image_pool_out(img.to(DEV), k1, k2, mask, (0.5, 0.5), torch.float32)
        assert (gp.cpu() - rp).abs().max().item() <= 1e-6 and (gc.cpu() - rc).abs().max().item() <= 1e-6
    # Philox style noise: N(0, std^2) moments; independent of how the batch is sharded (keyed by the global sample index)
    z = ops.philox_codes(123, 0, 0.8, 16, 64, 512, DEV)
    assert abs(z.mean().item()) < 5e-3 and abs(z.std().item() - 0.8) < 5e-3
    z2 = ops.philox_codes(123, 32, 0.8, 16, 32, 512, DEV)
    assert torch.equal(z[:, 32:], z2)


def _defense(kind, mode):
    if kind == "e4e":
        clf = ga_models.CelebaGenderClassifier(synth.make_resnet50_checkpoint(), DEV, mode=mode)
        return ga_models.E4EStyleGanDefenseModel(clf, synth.make_e4e_checkpoint(1024), [0.0] * 18, 1.0, 0.0, False, DEV, mode=mode)
    clf = ga_models.CarsTypeClassifier(synth.make_resnext50_checkpoint(), DEV, mode=mode)
    return ga_models.TransStyleGanDefenseModel(clf, synth.make_trans_checkpoint(512), [0.0] * 16, 1.0, 0.0, False, DEV, mode=mode)


@pytest.mark.parametrize("kind,res,n_codes", [("e4e", 256, 18), ("trans", 128, 16)])
@pytest.mark.parametrize("mode", ["fp32", "bf16"])
def test_defense_matches_reference_fixture(kind, res, n_codes, mode):
    """BASELINE configs 3 / 4, full-size architectures: purified images within 1e-4 (fp32) / 1e-2 (bf16) max-abs of the reference's
    own output, logits within 1e-3 relative (fp32), arg-max identical (fp32)."""
    g = torch.load(os.path.join(GOLDEN, "e4e_gender_b2.pt" if kind == "e4e" else "trans_cars_b2.pt"), weights_only=True)
    x, noises = synth.synthetic_stylegan_inputs(g["batch"], res, n_codes, seed=g["x_seed"])
    dm = _defense(kind, mode)
    dm.interpolation_alphas = [a * g["attenuation"] for a in g["alphas"]]
    dm.eps, dm.blur_input = g["eps"], g["blur"]
    dm.set_explicit_noise(noises)
    ops.launch_count(True)
    logits, pur = dm(x.to(DEV), preds_only=False)
    torch.cuda.synchronize()
    launches = ops.launch_count(True)
    got, ref = stored_purified(g, pur.cpu())
    err = (got - ref).abs().max().item()
    rel = ((logits.cpu() - g["logits"]).abs().max() / g["logits"].abs().max()).item()
    print(f"[{mode}] {kind}: purified max-abs err {err:.3e}; logits rel err {rel:.3e}; kernels {launches}")
    assert launches > 100
    if mode == "fp32":
        assert err <= 1e-4, err
        assert rel <= 1e-3, rel
        assert logits.argmax(1).tolist() == g["logits"].argmax(1).tolist()
    else:
        # bf16 gate of the north star: 1e-2 max-abs on images in [0, 1].  Style-Transformer @512 sits at 7-8e-3.  E4E @1024 measured
        # 0.98-1.1e-2 with a bf16 IR-SE50 backbone; its backbone now multiplies fp32 operands as TF32 (irse_engine.IrSe50Backbone.tf32).
        assert err <= 1e-2, err


def test_defense_philox_mode_is_shard_independent():
    """product mode (in-kernel Philox noise): a sample's result does not depend on where it sits in the batch / which GPU owns it"""
    dm = _defense("trans", "fp32")
    dm.interpolation_alphas = [0.3] * 16
    dm.eps, dm.blur_input, dm.noise_seed = 1.0, True, 77
    x = torch.rand(4, 3, 128, 128, generator=torch.Generator().manual_seed(3)).to(DEV)
    _, full = dm(x, preds_only=False)
    dm.sample_offset = 2
    _, tail = dm(x[2:], preds_only=False)
    assert (full[2:] - tail).abs().max().item() <= 1e-5


@pytest.mark.parametrize("kind,res,n_codes", [("e4e", 256, 18), ("trans", 128, 16)])
def test_clean_counts_identical_on_64_images(kind, res, n_codes):
    """north star: clean accuracy COUNTS identical on the fp32 path -- 64 seeded images per StyleGAN config, explicit noise, against the
    logits of the reference's own defense call (tests/golden/*_counts_b64.pt, oracle/make_golden.py stylegan_counts); bf16 reported."""
    path = os.path.join(GOLDEN, f"{kind}_counts_b64.pt")
    if not os.path.exists(path):
        pytest.skip("fixture not generated")
    g = torch.load(path, weights_only=True)
    x, noises = synth.synthetic_stylegan_inputs(g["batch"], res, n_codes, seed=g["x_seed"])
    ref = g["logits"]
    for mode in ("fp32", "bf16"):
        dm = _defense(kind, mode)
        dm.interpolation_alphas = [a * g["attenuation"] for a in g["alphas"]]
        dm.eps, dm.blur_input = g["eps"], g["blur"]
        got = []
        for i in range(0, g["batch"], 16):
            dm.set_explicit_noise([noises[0][i:i + 16], noises[1][:, i:i + 16]])
            with torch.no_grad():
                got.append(dm(x[i:i + 16].to(DEV)).cpu())
        got = torch.cat(got)
        diff = int((got.argmax(1) != ref.argmax(1)).sum())
        rel = ((got - ref).abs().max() / ref.abs().max()).item()
        print(f"[{mode}] {kind}: 64 images, {diff} arg-max differences, logits rel err {rel:.2e}, class histogram {torch.bincount(ref.argmax(1)).tolist()}")
        if mode == "fp32":
            assert diff == 0 and rel <= 1e-3
        else:
            assert diff <= 6
        del dm
        torch.cuda.empty_cache()
