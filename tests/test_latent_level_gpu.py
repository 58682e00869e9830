"""GPU: the fused tail of a decoder latent level (`ops.latent_level`: prior sampler -> latent mix -> combiner in one tensor-core kernel)
against the three launches it replaces (`conv2d_tc` -> `latent_mix` -> `conv2d_tc` with a second source).  The fused kernel runs the same
MMA shapes in the same K order and the same latent-mix device code, so the new stream (fp32 and bf16) and the taped `pp` are compared for
bit equality."""
import math

import pytest
import torch

from gen_adversarial_b200 import _lib, graphs, ops, synth
from gen_adversarial_b200.defenses.ours.models import CelebaIdentityClassifier, NVAEDefenseModel
from gen_adversarial_b200.nvae_spec import NVAE_C32_CONFIG, NVAE_C32_RESOLUTION, NvaeSpec
from gen_adversarial_b200.ops import gt, ptr, stream

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
ZDIM, TEMP = 20, 0.6
BAND = 4096


def _level_layers(c, zc, seed, zdim=ZDIM):
    g = torch.Generator(device=DEV).manual_seed(seed)
    smp = ops.ConvLayer(1, 1, 1, 0, c, 2 * zdim, name="dec_sampler")
    smp.w_tc = (torch.randn(2 * zdim, c, device=DEV, generator=g) * (0.7 / math.sqrt(c))).bfloat16().contiguous()
    smp.bias = torch.randn(2 * zdim, device=DEV, generator=g) * 0.2
    comb = ops.ConvLayer(1, 1, 1, 0, c, c, cin2=zc, name="dec_comb")
    w = torch.randn(c, c + zc, device=DEV, generator=g) / math.sqrt(c + zdim)
    w[:, c + zdim:] = 0.0                                    # z channels above zdim carry no weight (the engine's zero padding)
    comb.w_tc = w.bfloat16().contiguous()
    comb.bias = torch.randn(c, device=DEV, generator=g) * 0.2
    return smp, comb


def _inputs(n, hw, c, seed, zdim=ZDIM):
    g = torch.Generator(device=DEV).manual_seed(seed)
    x_elu = torch.nn.functional.elu(torch.randn(n, hw, hw, c, device=DEV, generator=g)).bfloat16()
    xa = torch.randn(n, hw, hw, c, device=DEV, generator=g).bfloat16()
    muq = torch.randn(n, hw, hw, zdim, device=DEV, generator=g)
    eps = torch.randn(n, zdim, hw, hw, device=DEV, generator=g)
    return x_elu, xa, muq, eps


def _three_launches(x_elu, xa, muq, eps, smp, comb, seed, level, sample0, alpha, zc, zdim=ZDIM):
    pp = ops.conv2d_tc(x_elu, smp, want_bf16=False, want_f32=True)[1]
    z = ops.latent_mix(muq, pp, eps, seed, level, sample0, alpha, TEMP, zdim, zc, torch.bfloat16)
    ob, of = ops.conv2d_tc(xa, comb, want_bf16=True, want_f32=True, x2=z)
    return ob, of, pp


@pytest.mark.parametrize("hw,c", [(32, 64), (16, 128), (8, 256)])
@pytest.mark.parametrize("n", [1, 3, 5, 512])
def test_latent_level_matches_three_launches(hw, c, n):
    zcs = (24, 32) if n == 5 else (24,)
    for zc in zcs:
        smp, comb = _level_layers(c, zc, seed=c + zc)
        x_elu, xa, muq, eps = _inputs(n, hw, c, seed=n)
        for a in (0.0, 0.37, 1.0):
            alpha = torch.full((1,), a, device=DEV)
            for e in (eps, None):
                for tape in (False, True):
                    ob, of, pp = ops.latent_level(x_elu, xa, muq, e, smp, comb, 77, 5, 3, alpha, TEMP, ZDIM, want_pp=tape)
                    rb, rf, rpp = _three_launches(x_elu, xa, muq, e, smp, comb, 77, 5, 3, alpha, zc)
                    what = (hw, c, n, zc, a, e is None, tape)
                    assert torch.equal(of, rf), (what, (of - rf).abs().max().item())
                    assert torch.equal(ob, rb), what
                    if tape:
                        assert torch.equal(pp, rpp), what
                    else:
                        assert pp is None
                    assert torch.isfinite(of).all()


@pytest.mark.parametrize("zdim,zc", [(4, 8), (12, 16), (24, 24), (32, 32)])
@pytest.mark.parametrize("hw,c", [(32, 64), (8, 256)])
def test_latent_level_other_latent_widths(zdim, zc, hw, c):
    """the kernel is instantiated per zdim / 4 (the NVAE configurations use 20): other widths against the three launches"""
    smp, comb = _level_layers(c, zc, seed=zdim, zdim=zdim)
    x_elu, xa, muq, eps = _inputs(3, hw, c, seed=zdim + 1, zdim=zdim)
    alpha = torch.full((1,), 0.37, device=DEV)
    for e in (eps, None):
        ob, of, pp = ops.latent_level(x_elu, xa, muq, e, smp, comb, 11, 4, 2, alpha, TEMP, zdim, want_pp=True)
        rb, rf, rpp = _three_launches(x_elu, xa, muq, e, smp, comb, 11, 4, 2, alpha, zc, zdim=zdim)
        assert torch.equal(of, rf) and torch.equal(ob, rb) and torch.equal(pp, rpp), (zdim, hw, c, e is None)


def test_latent_level_philox_shard_independence():
    """Philox eps is keyed by the global sample index: a batch split at sample0 gives the rows of the whole batch"""
    c, hw, n = 128, 16, 6
    smp, comb = _level_layers(c, 24, seed=1)
    x_elu, xa, muq, _ = _inputs(n, hw, c, seed=2)
    alpha = torch.full((1,), 0.8, device=DEV)
    full_b, full_f, _ = ops.latent_level(x_elu, xa, muq, None, smp, comb, 1234, 3, 0, alpha, TEMP, ZDIM)
    for lo, hi in ((0, 4), (4, 6)):
        pb, pf, _ = ops.latent_level(x_elu[lo:hi].contiguous(), xa[lo:hi].contiguous(), muq[lo:hi].contiguous(), None, smp, comb, 1234,
                                     3, lo, alpha, TEMP, ZDIM)
        assert torch.equal(pf, full_f[lo:hi]) and torch.equal(pb, full_b[lo:hi])
    # and the noise does reach the output
    other, _, _ = ops.latent_level(x_elu, xa, muq, None, smp, comb, 1235, 3, 0, alpha, TEMP, ZDIM)
    assert not torch.equal(other, full_b)


class _Guarded:
    def __init__(self, shape, dtype):
        n = 1
        for d in shape:
            n *= d
        self.sentinel = 12345.0 if dtype == torch.float32 else 12352.0          # exactly representable in bf16
        self.big = torch.full((n + 2 * BAND,), self.sentinel, device=DEV, dtype=dtype)
        self.view = self.big[BAND:BAND + n].view(shape)

    def check(self):
        torch.cuda.synchronize()
        assert bool((self.big[:BAND] == self.sentinel).all()) and bool((self.big[-BAND:] == self.sentinel).all()), "guard band overwritten"
        return self.view


@pytest.mark.parametrize("n,hw,c", [(1, 32, 64), (3, 8, 256), (5, 16, 128)])
def test_latent_level_stays_inside_its_outputs(n, hw, c):
    """partial last tiles (3 x 8x8 = 192 pixels: the second tile is half empty) must not write past the outputs"""
    smp, comb = _level_layers(c, 24, seed=4)
    x_elu, xa, muq, eps = _inputs(n, hw, c, seed=5)
    alpha = torch.full((1,), 0.5, device=DEV)
    ob, of, pp = _Guarded((n, hw, hw, c), torch.bfloat16), _Guarded((n, hw, hw, c), torch.float32), _Guarded((n, hw, hw, 2 * ZDIM), torch.float32)
    _lib.check(_lib.lib().ga_latent_level(gt(x_elu), gt(xa), gt(muq), ptr(eps), smp.w_tc.data_ptr(), ptr(smp.bias), comb.w_tc.data_ptr(),
                                          ptr(comb.bias), 24, 9, 2, 0, ptr(alpha), TEMP, ZDIM, gt(ob.view), gt(of.view), gt(pp.view), stream()),
               "latent_level")
    rb, rf, rpp = _three_launches(x_elu, xa, muq, eps, smp, comb, 9, 2, 0, alpha, 24)
    assert torch.equal(ob.check(), rb) and torch.equal(of.check(), rf) and torch.equal(pp.check(), rpp)


@pytest.fixture(scope="module")
def c32_models():
    return synth.make_nvae_checkpoint(seed=0), synth.make_vgg11_checkpoint(100, seed=1)


def test_engine_fuse_level_changes_nothing(c32_models):
    """the whole purification with the fused level tail on and off: identical purified images and logits, eagerly, under CUDA-graph replay
    with two part-batches on two streams, and for a taped forward and its input gradient"""
    nv, vg = c32_models
    clf = CelebaIdentityClassifier(vg, DEV, mode="bf16")
    dm = NVAEDefenseModel(clf, nv, [0.5] * 24, 1.0, 2.0, True, DEV, mode="bf16")
    eng = dm.autoencoder
    assert eng.fuse_level
    dm.noise_seed = 23
    x, _ = synth.synthetic_batch(8, seed=5)
    xd = x.to(DEV)
    launches = {}
    outs = {}
    for fuse in (True, False):
        eng.fuse_level = fuse
        with torch.no_grad():
            n0 = ops.launch_count()
            outs[("eager", fuse)] = [t.clone() for t in dm(xd, preds_only=False)]
            launches[fuse] = ops.launch_count() - n0
            dm.set_streams(2).enable_cuda_graph(True)
            for rep in range(2):
                graphs.enable_seed_salt(DEV).zero_()               # the same salt for both builds of the graph
                outs[("graph", fuse, rep)] = [t.clone() for t in dm(xd, preds_only=False)]
            dm.enable_cuda_graph(False).set_streams(1)
    torch.cuda.synchronize()
    assert launches[False] - launches[True] == 2 * (eng.spec.n_latents - 1)      # three launches become one on every level but level 0
    for key in (("eager",), ("graph", 0), ("graph", 1)):
        (l1, p1), (l0, p0) = outs[key[:1] + (True,) + key[1:]], outs[key[:1] + (False,) + key[1:]]
        assert torch.equal(l1, l0) and torch.equal(p1, p0), key
    assert not torch.equal(outs[("eager", True)][1], outs[("graph", True, 0)][1])   # the graph drew its own (salted) noise

    # taped forward + input gradient (the attack path): the fused kernel also writes pp for the tape
    spec = NvaeSpec(NVAE_C32_CONFIG, NVAE_C32_RESOLUTION)
    a_dev = torch.full((spec.n_latents,), 0.5, device=DEV)
    xin, _ = ops.preprocess(xd[:4], None, 0.0, False, torch.bfloat16)
    res = {}
    for fuse in (True, False):
        eng.fuse_level = fuse
        tape = []
        pur, _ = eng.purify(xin, a_dev, None, seed=41, sample0=0, tape=tape)
        g_pur = torch.linspace(-1.0, 1.0, pur.numel(), device=DEV).view(pur.shape)
        res[fuse] = (pur.clone(), eng.backward(tape, g_purified_nchw=g_pur).clone())
    eng.fuse_level = True
    torch.cuda.synchronize()
    assert torch.equal(res[True][0], res[False][0]) and torch.equal(res[True][1], res[False][1])
