"""Thin Python wrappers over the C-ABI (include/ga_b200.h): torch owns memory and streams, the kernels are ours.

Tensors handled here are dense NHWC `torch.Tensor`s of shape (N, H, W, C), dtype float32 or bfloat16, on a
CUDA device.  Every wrapper launches on `torch.cuda.current_stream()` and raises RuntimeError on failure;
nothing here ever falls back to a torch/CPU implementation.
"""
from __future__ import annotations

import ctypes
from dataclasses import dataclass
from typing import Optional

import torch

from . import _lib
from ._lib import GaTensor, GaConvDesc, GA_F32, GA_BF16, PRE_NONE, PRE_ELU, PRE_SILU, PRE_AFFINE_SILU, \
    ACT_NONE, ACT_SILU, ACT_ELU, ACT_RELU, ACT_LRELU_SQRT2, MUL_VALUE, MUL_RELU_MASK, MUL_ELU_FROM_Y, MUL_PRELU_FROM_Y


def _dt(t: torch.Tensor) -> int:
    if t.dtype == torch.float32:
        return GA_F32
    if t.dtype == torch.bfloat16:
        return GA_BF16
    raise TypeError(f"unsupported dtype {t.dtype}")


def gt(t: Optional[torch.Tensor]):
    """torch NHWC tensor -> POINTER(GaTensor) (or None)."""
    if t is None:
        return None
    if not t.is_cuda:
        raise RuntimeError("libga_b200 ops need CUDA tensors (no CPU fallback exists)")
    if t.dim() != 4 or not t.is_contiguous():
        raise RuntimeError(f"expected a contiguous NHWC tensor, got shape {tuple(t.shape)} strides {t.stride()}")
    n, h, w, c = t.shape
    return ctypes.pointer(GaTensor(t.data_ptr(), _dt(t), n, h, w, c))


def ptr(t: Optional[torch.Tensor]):
    if t is None:
        return None
    if not t.is_cuda:
        raise RuntimeError("libga_b200 ops need CUDA tensors (no CPU fallback exists)")
    return t.data_ptr()


def stream():
    return torch.cuda.current_stream().cuda_stream


def torch_dtype(name: str):
    return {"fp32": torch.float32, "bf16": torch.bfloat16}[name]


class KernelTimer:
    """CUDA-event timing of individual launches on the launching stream (bench.py roofline): when installed as
    `ops.TIMER`, every tensor-core conv launch is bracketed by two events and its algorithmic FLOPs / bytes are
    recorded; `summary()` synchronises once and aggregates per problem shape."""

    def __init__(self):
        self.records = []

    def start(self):
        e = torch.cuda.Event(enable_timing=True)
        e.record(torch.cuda.current_stream())
        return e

    def stop(self, e0, key, flops, bytes_):
        e1 = torch.cuda.Event(enable_timing=True)
        e1.record(torch.cuda.current_stream())
        self.records.append((key, flops, bytes_, e0, e1))

    def summary(self):
        torch.cuda.synchronize()
        agg = {}
        for key, flops, bytes_, e0, e1 in self.records:
            a = agg.setdefault(key, {"launches": 0, "ms": 0.0, "flops": 0.0, "bytes": 0.0})
            a["launches"] += 1
            a["ms"] += e0.elapsed_time(e1)
            a["flops"] += flops
            a["bytes"] += bytes_
        return agg


TIMER: Optional[KernelTimer] = None
TIME_ALL = False      # bench.py --breakdown: also bracket every non-conv_tc op (keyed "op:<name> <shape>")


def _tensor_bytes(objs) -> float:
    by = 0.0
    for o in objs:
        if torch.is_tensor(o):
            by += o.numel() * o.element_size()
        elif isinstance(o, (tuple, list)):
            by += _tensor_bytes(o)
    return by


def _timed(name, hbm: bool = False):
    """bench.py instrumented pass: bracket the op with CUDA events.  hbm=True marks a bandwidth-bound kernel: its algorithmic bytes are
    every tensor operand and result counted exactly once (SURVEY 8d: compulsory traffic), keyed "hbm:<name> <shape>"."""
    def deco(fn):
        def wrapper(*a, **k):
            if TIMER is None or not TIME_ALL:
                return fn(*a, **k)
            e0 = TIMER.start()
            out = fn(*a, **k)
            shp = tuple(a[0].shape) if len(a) and torch.is_tensor(a[0]) else ()
            if hbm:
                TIMER.stop(e0, f"hbm:{name} {shp}", 0.0, _tensor_bytes(a) + _tensor_bytes(list(k.values())) + _tensor_bytes([out]))
            else:
                TIMER.stop(e0, f"op:{name} {shp}", 0.0, 0.0)
            return out
        wrapper.__name__ = fn.__name__
        wrapper.__doc__ = fn.__doc__
        return wrapper
    return deco


@dataclass
class ConvLayer:
    """A folded convolution living on the device."""
    kh: int
    kw: int
    stride: int
    pad: int
    cin: int
    cout: int
    w_simt: Optional[torch.Tensor] = None      # fp32 [kh*kw*cin, cout]
    w_tc: Optional[torch.Tensor] = None        # bf16 [cout, ktot]  (ktot = kh*kw*cin + cin2)
    w_tf32: Optional[torch.Tensor] = None      # fp32 [cout, ktot]: tensor-core path with fp32 activations, multiplied as TF32
    bias: Optional[torch.Tensor] = None        # fp32 [cout]
    pre_op: int = PRE_NONE
    pre_scale: Optional[torch.Tensor] = None   # fp32 [cin]
    pre_shift: Optional[torch.Tensor] = None
    post_act: int = ACT_NONE
    up: int = 1
    cin2: int = 0                              # channels of the second (1x1) K source folded into w_tc
    act_slope: Optional[torch.Tensor] = None   # fp32 [cout] negative slopes (ACT_PRELU)
    act_after_add: bool = False                # out = act(conv + bias + add)
    phase: Optional["ConvLayer"] = None        # dgrad of a stride-2 conv as ONE stride-1 conv emitting the 4 output phases (4*cout channels)
    name: str = ""

    def desc(self, tc: bool, mul=None, mul_mode: int = 0, dact=None, tf32: bool = False, csum=None) -> GaConvDesc:
        w = (self.w_tf32 if tf32 else self.w_tc) if tc else self.w_simt
        if w is None:
            raise RuntimeError(f"conv layer {self.name}: no {'tensor-core' if tc else 'SIMT'} weights prepared")
        return GaConvDesc(self.kh, self.kw, self.stride, self.pad, self.up, PRE_NONE if tc else self.pre_op, self.post_act,
                          ptr(self.pre_scale), ptr(self.pre_shift), w.data_ptr(), ptr(self.bias), int(bool(tf32 and tc)),
                          w.shape[1] if tc else 0,
                          ptr(mul), _dt(mul) if mul is not None else 0, mul_mode,
                          ptr(dact), _dt(dact) if dact is not None else 0, int(self.act_after_add), ptr(self.act_slope), ptr(csum))


def conv_out_hw(L: ConvLayer, h: int, w: int):
    hu, wu = (h - 1) * L.up + 1, (w - 1) * L.up + 1
    return (hu + 2 * L.pad - L.kh) // L.stride + 1, (wu + 2 * L.pad - L.kw) // L.stride + 1


@_timed("conv2d_simt")
def conv2d_simt(x: torch.Tensor, L: ConvLayer, out_dtype: torch.dtype, add: Optional[torch.Tensor] = None,
                out_hw=None, mul: Optional[torch.Tensor] = None, mul_mode: int = 0, want_dact: bool = False,
                out: Optional[torch.Tensor] = None):
    """out = (act(conv(pre(x)) + bias) + add) * f(mul).  With want_dact -> (out, act'(pre-activation))."""
    n, h, w, c = x.shape
    assert c == L.cin, (L.name, c, L.cin)
    ho, wo = out_hw if out_hw is not None else conv_out_hw(L, h, w)
    if out is None:
        out = torch.empty((n, ho, wo, L.cout), device=x.device, dtype=out_dtype)
    dact = torch.empty_like(out) if want_dact else None
    d = L.desc(False, mul, mul_mode, dact)
    _lib.check(_lib.lib().ga_conv2d_simt(gt(x), ctypes.byref(d), gt(add), gt(out), stream()), f"conv2d_simt[{L.name}]")
    return (out, dact) if want_dact else out


def conv2d_tc_supported(x: torch.Tensor, L: ConvLayer, x2: Optional[torch.Tensor] = None, tf32: bool = False) -> bool:
    if tf32:
        if L.w_tf32 is None or x.dtype != torch.float32:
            return False
    elif L.w_tc is None or x.dtype != torch.bfloat16:
        return False
    d = L.desc(True, tf32=tf32)
    return bool(_lib.lib().ga_conv2d_tc_supported(gt(x), gt(x2), ctypes.byref(d), L.cout))


def conv2d_tc_csum_supported(x: torch.Tensor, L: ConvLayer) -> bool:
    """can conv2d_tc(x, L) (bf16 output only, no add / mul / tape) also emit the SE channel sums of its output (`want_csum`)?"""
    if L.w_tc is None or x.dtype != torch.bfloat16:
        return False
    d = L.desc(True)
    return bool(_lib.lib().ga_conv2d_tc_csum_supported(gt(x), ctypes.byref(d), L.cout))


def conv2d_tc(x: torch.Tensor, L: ConvLayer, want_bf16: bool = True, want_f32: bool = False,
              add: Optional[torch.Tensor] = None, x2: Optional[torch.Tensor] = None,
              mul: Optional[torch.Tensor] = None, mul_mode: int = 0, dact_out: Optional[torch.Tensor] = None,
              out_bf16: Optional[torch.Tensor] = None, out_f32: Optional[torch.Tensor] = None, tf32: bool = False,
              csum_out: Optional[torch.Tensor] = None):
    """-> (out_bf16 or None, out_f32 or None);  out = (act(conv + bias) + add) * f(mul); dact_out <- act'(conv + bias).
    tf32: x is fp32 and the layer's fp32 weights are used (kind::tf32 MMA: 10-bit mantissas, half the bf16 rate)"""
    n, h, w, c = x.shape
    assert c == L.cin, (L.name, c, L.cin)
    ho, wo = conv_out_hw(L, h, w)
    ob = (out_bf16 if out_bf16 is not None else torch.empty((n, ho, wo, L.cout), device=x.device, dtype=torch.bfloat16)) if want_bf16 else None
    of = (out_f32 if out_f32 is not None else torch.empty((n, ho, wo, L.cout), device=x.device, dtype=torch.float32)) if want_f32 else None
    d = L.desc(True, mul, mul_mode, dact_out, tf32=tf32, csum=csum_out)
    e0 = TIMER.start() if TIMER is not None else None
    _lib.check(_lib.lib().ga_conv2d_tc(gt(x), gt(x2), ctypes.byref(d), gt(add), gt(ob), gt(of), stream()),
               f"conv2d_tc[{L.name}]")
    if e0 is not None:
        m = n * ho * wo
        ktot = (L.w_tf32 if tf32 else L.w_tc).shape[1]
        flops = 2.0 * m * L.cout * ktot
        # compulsory traffic: A once (not per tap), weights once, outputs (+ add) once
        bytes_ = 2.0 * n * h * w * c + 2.0 * m * (x2.shape[3] if x2 is not None else 0) + 2.0 * L.cout * ktot \
            + m * L.cout * ((2 if want_bf16 else 0) + (4 if want_f32 else 0) + (add.element_size() if add is not None else 0))
        TIMER.stop(e0, f"k{L.kh}{'s2' if L.stride == 2 else ''}{' tf32' if tf32 else ''} hw{h} cin{c} cout{L.cout}", flops, bytes_)
    return ob, of


@_timed("dwconv5x5")
def dwconv5x5(x: torch.Tensor, weight: torch.Tensor, bias: Optional[torch.Tensor], act: int, up: bool,
              out_dtype: torch.dtype, mul: Optional[torch.Tensor] = None, want_dact: bool = False):
    """out = act(dwconv5x5(x) + bias) * mul.  With want_dact -> (out, act'(pre-activation))."""
    n, h, w, c = x.shape
    s = 2 if up else 1
    out = torch.empty((n, h * s, w * s, c), device=x.device, dtype=out_dtype)
    if mul is None and not want_dact:
        _lib.check(_lib.lib().ga_dwconv5x5_fwd(gt(x), ptr(weight), ptr(bias), act, int(up), gt(out), stream()), "dwconv5x5")
        return out
    dact = torch.empty_like(out) if want_dact else None
    _lib.check(_lib.lib().ga_dwconv5x5_ex(gt(x), gt(mul), ptr(weight), ptr(bias), act, int(up), gt(out), gt(dact), stream()),
               "dwconv5x5_ex")
    return (out, dact) if want_dact else out


def mbconv_fused_supported(x: torch.Tensor, e: ConvLayer, p: ConvLayer) -> bool:
    if x.dtype != torch.bfloat16 or e.w_tc is None or p.w_tc is None or e.bias is None or p.bias is None:
        return False
    return bool(_lib.lib().ga_mbconv_fused_supported(gt(x), e.cout))


def dw_weights_chunked(dw_w: torch.Tensor) -> torch.Tensor:
    """[25][hidden] depthwise taps -> chunk-major [hidden/64][25][64] (one contiguous 6400-byte block per 64-channel chunk)"""
    t, hidden = dw_w.shape
    return dw_w.reshape(t, hidden // 64, 64).permute(1, 0, 2).contiguous()


def mbconv_fused(x: torch.Tensor, e: ConvLayer, dw_w_chunked: torch.Tensor, dw_b: torch.Tensor, p: ConvLayer, want_sums: bool = False,
                 want_tape: bool = False):
    """decoder-cell body in ONE kernel: project(SiLU(dw5x5(SiLU(expand(x)))))  -> r (bf16); dw_w_chunked = dw_weights_chunked(dw_w).
    want_sums: also the SE channel sums of r ([n][parts][c] fp32, what `channel_sum(r)` returns) from the cell's epilogue;
    want_tape: also SiLU'(expand pre-activation) and SiLU'(depthwise pre-activation), bf16 [n][h][w][hidden] (attack path).
    -> r | (r, sums) | (r, sums | None, dact_e, dact_dw)"""
    n, h, w, c = x.shape
    out = torch.empty(x.shape, device=x.device, dtype=torch.bfloat16)
    sums = torch.empty((n, channel_sum_parts(n, h * w), c), device=x.device, dtype=torch.float32) if want_sums else None
    dact_e = torch.empty((n, h, w, e.cout), device=x.device, dtype=torch.bfloat16) if want_tape else None
    dact_dw = torch.empty((n, h, w, e.cout), device=x.device, dtype=torch.bfloat16) if want_tape else None
    e0 = TIMER.start() if TIMER is not None else None
    _lib.check(_lib.lib().ga_mbconv_fused_ex(gt(x), e.w_tc.data_ptr(), ptr(e.bias), ptr(dw_w_chunked), ptr(dw_b), p.w_tc.data_ptr(), ptr(p.bias),
                                             e.cout, gt(out), ptr(sums), gt(dact_e), gt(dact_dw), stream()), "mbconv_fused")
    if e0 is not None:
        m, hid = n * h * w, e.cout
        # algorithmic work: two 1x1 GEMMs on the tensor cores + 25 MAC per hidden element on the fp32 pipe; compulsory HBM traffic: x in, r out
        # (+ the two hidden-sized tapes when taping)
        TIMER.stop(e0, f"fused:mbconv{'_tape' if want_tape else ''} hw{h} c{c} hidden{hid}", 2.0 * m * hid * c * 2 + 2.0 * m * hid * 25,
                   2.0 * m * c * 2 + 2.0 * hid * c * 2 + (4.0 * m * hid if want_tape else 0.0))
    if want_tape:
        return out, sums, dact_e, dact_dw
    return (out, sums) if want_sums else out


def mbconv_fused_bwd(g: torch.Tensor, p_d: ConvLayer, dw_wT_chunked: torch.Tensor, dact_dw: torch.Tensor, dact_e: torch.Tensor, e_d: ConvLayer,
                     add: Optional[torch.Tensor] = None) -> torch.Tensor:
    """input gradient of the decoder-cell body in ONE kernel: add + e_d(dact_e * dw5x5^T(dact_dw * p_d(g)))  -> fp32 NHWC.
    p_d / e_d: the dgrad layers of project / expand (transposed bf16 weights), dw_wT_chunked = dw_weights_chunked(flipped taps)"""
    out = torch.empty(g.shape, device=g.device, dtype=torch.float32)
    e0 = TIMER.start() if TIMER is not None else None
    _lib.check(_lib.lib().ga_mbconv_fused_bwd(gt(g), p_d.w_tc.data_ptr(), ptr(dw_wT_chunked), gt(dact_dw), gt(dact_e), e_d.w_tc.data_ptr(),
                                              gt(add), p_d.cout, gt(out), stream()), "mbconv_fused_bwd")
    if e0 is not None:
        n, h, w, c = g.shape
        m, hid = n * h * w, p_d.cout
        TIMER.stop(e0, f"fused:mbconv_bwd hw{h} c{c} hidden{hid}", 2.0 * m * hid * c * 2 + 2.0 * m * hid * 25,
                   2.0 * m * c + 4.0 * m * c * (2 if add is not None else 1) + 4.0 * m * hid)
    return out


def channel_sum_parts(n: int, hw: int) -> int:
    return int(_lib.lib().ga_channel_sum_parts(n, hw))


@_timed("channel_sum", hbm=True)
def channel_sum(r: torch.Tensor) -> torch.Tensor:
    parts = _lib.lib().ga_channel_sum_parts(r.shape[0], r.shape[1] * r.shape[2])
    sums = torch.empty((r.shape[0], parts, r.shape[3]), device=r.device, dtype=torch.float32)
    _lib.check(_lib.lib().ga_channel_sum(gt(r), ptr(sums), stream()), "channel_sum")
    return sums


def se_residual(r, sums, se, res_scale: float, skip, out_dtype=torch.float32, want_out2=False, out2_dtype=torch.bfloat16,
                act_affine=None, act_dtype=torch.bfloat16, want_gate=False, act_op: int = ACT_SILU, act_plain: bool = False):
    """se = (w1, b1, w2, b2) fp32 device tensors (biases may be None).  -> (out, out2|None, act|None, gate|None);
    act = act_op(act_scale * out + act_shift), act_op SiLU (NVAE cells) or none (IR-SE50 BatchNorm); act_plain: act = act_op(out)
    without an affine (ELU copy for the decoder sampler / logits head)"""
    w1, b1, w2, b2 = se
    out = torch.empty(r.shape, device=r.device, dtype=out_dtype)
    out2 = torch.empty(r.shape, device=r.device, dtype=out2_dtype) if want_out2 else None
    act = torch.empty(r.shape, device=r.device, dtype=act_dtype) if (act_affine is not None or act_plain) else None
    gate = torch.empty((r.shape[0], r.shape[3]), device=r.device, dtype=torch.float32) if want_gate else None
    a_s, a_b = act_affine if act_affine is not None else (None, None)
    e0 = TIMER.start() if TIMER is not None else None
    _lib.check(_lib.lib().ga_se_residual_fwd(gt(r), ptr(sums), ptr(w1), ptr(b1), ptr(w2), ptr(b2), w1.shape[0], res_scale,
                                             gt(skip), gt(out), gt(out2), gt(act), ptr(a_s), ptr(a_b), act_op, ptr(gate), stream()),
               "se_residual")
    if e0 is not None:     # HBM-bound: every operand is read or written exactly once
        by = sum(t.numel() * t.element_size() for t in (r, skip, out, out2, act) if t is not None)
        TIMER.stop(e0, f"hbm:se_residual {tuple(r.shape)}", 0.0, float(by))
    return out, out2, act, gate


@_timed("latent_mix", hbm=True)
def latent_mix(q, p, eps_nchw, seed: int, level: int, sample0: int, alpha_dev, temperature: float, zdim: int,
               zc: int, out_dtype) -> torch.Tensor:
    n, h, w, _ = q.shape
    z = torch.empty((n, h, w, zc), device=q.device, dtype=out_dtype)
    _lib.check(_lib.lib().ga_latent_mix_fwd(gt(q), gt(p), ptr(eps_nchw), seed, level, sample0, ptr(alpha_dev), temperature,
                                            zdim, gt(z), stream()), "latent_mix")
    return z


def latent_level_supported(x_elu: torch.Tensor, xa: torch.Tensor, sampler: ConvLayer, comb: ConvLayer, zdim: int) -> bool:
    """can `latent_level` run this level (bf16 tensors, C in {64, 128, 256}, zdim a multiple of 4 up to 32)?"""
    c = xa.shape[3]
    return (x_elu is not None and x_elu.dtype == torch.bfloat16 and xa.dtype == torch.bfloat16 and x_elu.shape == xa.shape
            and c in (64, 128, 256) and zdim % 4 == 0 and 4 <= zdim <= 32 and sampler.w_tc is not None and sampler.cout == 2 * zdim
            and sampler.kh == 1 and comb.w_tc is not None and comb.kh == 1 and comb.cin == c and comb.cout == c
            and zdim <= comb.cin2 <= 32 and sampler.bias is not None and comb.bias is not None)


@_timed("latent_level", hbm=True)
def latent_level(x_elu, xa, muq, eps_nchw, sampler: ConvLayer, comb: ConvLayer, seed: int, level: int, sample0: int, alpha_dev,
                 temperature: float, zdim: int, want_pp: bool = False):
    """tail of a decoder latent level in one kernel: pp = sampler(x_elu), z = latent_mix(muq, pp, eps), comb([xa | z]).
    x_elu: ELU(x) in bf16 (the sampler's pre-activated input); comb: the combiner layer with its z weights folded in (cin2 = zc).
    -> (out bf16, out fp32, pp fp32 | None);  pp only with want_pp (taping forward)"""
    n, h, w, c = xa.shape
    ob = torch.empty((n, h, w, c), device=xa.device, dtype=torch.bfloat16)
    of = torch.empty((n, h, w, c), device=xa.device, dtype=torch.float32)
    pp = torch.empty((n, h, w, 2 * zdim), device=xa.device, dtype=torch.float32) if want_pp else None
    _lib.check(_lib.lib().ga_latent_level(gt(x_elu), gt(xa), gt(muq), ptr(eps_nchw), sampler.w_tc.data_ptr(), ptr(sampler.bias),
                                          comb.w_tc.data_ptr(), ptr(comb.bias), comb.cin2, seed, level, sample0, ptr(alpha_dev),
                                          temperature, zdim, gt(ob), gt(of), gt(pp), stream()), "latent_level")
    return ob, of, pp


@_timed("discmix_mean", hbm=True)
def discmix_mean(logits, n_mix: int, cls_dtype=None):
    n, h, w, _ = logits.shape
    purified = torch.empty((n, 3, h, w), device=logits.device, dtype=torch.float32)
    cls = torch.empty((n, h, w, 3), device=logits.device, dtype=cls_dtype) if cls_dtype is not None else None
    _lib.check(_lib.lib().ga_discmix_mean_fwd(gt(logits), n_mix, ptr(purified), gt(cls), stream()), "discmix_mean")
    return purified, cls


@_timed("upsample_nearest2x")
def upsample_nearest2x(x, out_dtype=None):
    n, h, w, c = x.shape
    out = torch.empty((n, 2 * h, 2 * w, c), device=x.device, dtype=out_dtype or x.dtype)
    _lib.check(_lib.lib().ga_upsample_nearest2x(gt(x), gt(out), stream()), "upsample_nearest2x")
    return out


@_timed("upsample_bilinear2x", hbm=True)
def upsample_bilinear2x(x, out_dtype=None):
    n, h, w, c = x.shape
    out = torch.empty((n, 2 * h, 2 * w, c), device=x.device, dtype=out_dtype or x.dtype)
    _lib.check(_lib.lib().ga_upsample_bilinear2x(gt(x), gt(out), stream()), "upsample_bilinear2x")
    return out


@_timed("maxpool2x2", hbm=True)
def maxpool2x2(x, out_dtype=None):
    n, h, w, c = x.shape
    out = torch.empty((n, h // 2, w // 2, c), device=x.device, dtype=out_dtype or x.dtype)
    _lib.check(_lib.lib().ga_maxpool2x2(gt(x), gt(out), stream()), "maxpool2x2")
    return out


@_timed("subsample2x")
def subsample2x(x, out_dtype=None):
    n, h, w, c = x.shape
    out = torch.empty((n, (h + 1) // 2, (w + 1) // 2, c), device=x.device, dtype=out_dtype or x.dtype)
    _lib.check(_lib.lib().ga_subsample2x(gt(x), gt(out), stream()), "subsample2x")
    return out


@_timed("maxpool3x3s2")
def maxpool3x3s2(x, out_dtype=None):
    n, h, w, c = x.shape
    out = torch.empty((n, (h - 1) // 2 + 1, (w - 1) // 2 + 1, c), device=x.device, dtype=out_dtype or x.dtype)
    _lib.check(_lib.lib().ga_maxpool3x3s2(gt(x), gt(out), stream()), "maxpool3x3s2")
    return out


@_timed("global_avgpool")
def global_avgpool(x, out_dtype=None):
    n, h, w, c = x.shape
    out = torch.empty((n, 1, 1, c), device=x.device, dtype=out_dtype or x.dtype)
    _lib.check(_lib.lib().ga_global_avgpool(gt(x), gt(out), stream()), "global_avgpool")
    return out


@_timed("affine_act", hbm=True)
def affine_act(x, scale, shift, act: int, out_dtype):
    out = torch.empty(x.shape, device=x.device, dtype=out_dtype)
    _lib.check(_lib.lib().ga_affine_act(gt(x), ptr(scale), ptr(shift), act, gt(out), stream()), "affine_act")
    return out


def cast(x, out_dtype):
    return affine_act(x, None, None, ACT_NONE, out_dtype)


def f32_round_tf32(on: bool):
    """while on, kernels writing fp32 activations round them to nearest TF32 (operands of the kind::tf32 convs, which truncate)"""
    _lib.check(_lib.lib().ga_f32_round_tf32(int(bool(on))), "f32_round_tf32")


@_timed("nchw_to_nhwc")
def nchw_to_nhwc(x_nchw, out_dtype, scale=1.0, shift=0.0):
    n, c, h, w = x_nchw.shape
    out = torch.empty((n, h, w, c), device=x_nchw.device, dtype=out_dtype)
    _lib.check(_lib.lib().ga_nchw_to_nhwc(ptr(x_nchw.contiguous()), gt(out), scale, shift, stream()), "nchw_to_nhwc")
    return out


def gaussian_taps(h: int, max_radius: int = 12):
    """Blur taps of abstract_models.py:145-159 (k = int(2**(sqrt(h)//2)-1), sigma=1, kornia kernel
    exp(-t^2/2)/sum).  k = 255 at 256x256: taps beyond |t| = 12 are < 6e-32 of the peak and are dropped."""
    import math
    k = int(2 ** (math.sqrt(h) // 2) - 1)
    t = torch.arange(k, dtype=torch.float64) - k // 2
    g = torch.exp(-(t ** 2) / 2.0)
    g = g / g.sum()
    r = k // 2
    if r > max_radius:
        g = g[r - max_radius: r + max_radius + 1]
        r = max_radius
    return g.to(torch.float32), r


@_timed("preprocess", hbm=True)
def preprocess(x_nchw, noise_nchw, eps: float, blur: bool, out_dtype, seed: int = 0, sample0: int = 0,
               normalize: bool = True, save_pre: bool = False, taps_cache=None):
    """blur -> noise -> clamp -> (x-.5)/.5 in one kernel (+ the L2-norm pre-pass).  -> (out NHWC, pre NCHW|None)"""
    L = _lib.lib()
    n, c, h, w = x_nchw.shape
    x_nchw = x_nchw.contiguous()
    out = torch.empty((n, h, w, c), device=x_nchw.device, dtype=out_dtype)
    pre = torch.empty_like(x_nchw) if save_pre else None
    taps, radius = None, 0
    if blur:
        if taps_cache is not None and taps_cache.get("h") == h and taps_cache["taps"].device == x_nchw.device:
            taps, radius = taps_cache["taps"], taps_cache["radius"]
        else:
            t, radius = gaussian_taps(h)
            taps = t.to(x_nchw.device)
            if taps_cache is not None:
                taps_cache.update({"h": h, "taps": taps, "radius": radius})
    if L.ga_preprocess_image_supported(c, h, w, radius, int(blur)):
        # 3 x 64 x 64: one launch, image resident in shared memory, noise norm reduced in the kernel
        if eps != 0.0 and noise_nchw is not None:
            noise_nchw = noise_nchw.contiguous()
        _lib.check(L.ga_preprocess_image_fwd(ptr(x_nchw), ptr(noise_nchw) if eps != 0.0 else None, seed, sample0, eps, ptr(taps), radius,
                                             int(normalize), gt(out), ptr(pre), stream()), "preprocess_image_fwd")
        return out, pre
    sumsq = None
    if eps != 0.0:
        sumsq = torch.empty((n, L.ga_noise_sumsq_parts(c * h * w)), device=x_nchw.device, dtype=torch.float32)
        if noise_nchw is not None:
            noise_nchw = noise_nchw.contiguous()
            _lib.check(L.ga_noise_sumsq(ptr(noise_nchw), n, c * h * w, ptr(sumsq), stream()), "noise_sumsq")
        else:
            _lib.check(L.ga_noise_sumsq_philox(seed, sample0, n, c * h * w, ptr(sumsq), stream()), "noise_sumsq_philox")
    _lib.check(L.ga_preprocess_fwd(ptr(x_nchw), ptr(noise_nchw) if eps != 0.0 else None, ptr(sumsq), seed, sample0, eps,
                                   ptr(taps), radius, int(normalize), gt(out), ptr(pre), stream()), "preprocess_fwd")
    return out, pre


@_timed("pgd_linf_step", hbm=True)
def pgd_linf_step_(x_adv, grad, x_nat, step: float, eps: float):
    assert x_adv.is_contiguous() and grad.is_contiguous() and x_nat.is_contiguous()
    _lib.check(_lib.lib().ga_pgd_linf_step(ptr(x_adv), ptr(grad), ptr(x_nat), step, eps, x_adv.numel(), stream()), "pgd_linf_step")
    return x_adv


def apgd_l2_step_(x_adv, x_adv_old, grad, x_nat, step_size, a: float, bound: float):
    """in place: the APGD update (untargeted.py:176-193) for a batch, per-image norms; step_size: device float32 [n]"""
    n = x_adv.shape[0]
    chw = x_adv.numel() // max(n, 1)
    for t in (x_adv, x_adv_old, grad, x_nat, step_size):
        assert t.is_contiguous() and t.dtype == torch.float32
    _lib.check(_lib.lib().ga_apgd_l2_step(ptr(x_adv), ptr(x_adv_old), ptr(grad), ptr(x_nat), ptr(step_size), float(a), float(bound), n, chw,
                                          stream()), "apgd_l2_step")
    return x_adv


def fgsm_l2_step(x_nat, grad, l2: float):
    """x + l2 * sign(g) / ||sign(g)||, clamped (untargeted.py:736-745; g = gradient of +CE)"""
    n = x_nat.shape[0]
    out = torch.empty_like(x_nat)
    _lib.check(_lib.lib().ga_fgsm_l2_step(ptr(x_nat.contiguous()), ptr(grad.contiguous()), float(l2), ptr(out), n, x_nat.numel() // max(n, 1),
                                          stream()), "fgsm_l2_step")
    return out


def l2_ball_start(x_nat, noise, bound: float):
    """clamp(x + bound * noise / ||noise||, 0, 1) per image (untargeted.py:129-131)"""
    n = x_nat.shape[0]
    out = torch.empty_like(x_nat)
    _lib.check(_lib.lib().ga_l2_ball_start(ptr(x_nat.contiguous()), ptr(noise.contiguous()), float(bound), ptr(out), n,
                                           x_nat.numel() // max(n, 1), stream()), "l2_ball_start")
    return out


@_timed("softmax_xent")
def softmax_xent(logits, labels, want_grad=True, counter=None):
    """-> (loss[n], dlogits|None, pred[n] int32); `counter` (uint64 device scalar) accumulates argmax==label."""
    n, k = logits.shape
    logits = logits.contiguous()
    if not labels.is_cuda or labels.dim() != 1 or labels.shape[0] != n:
        raise RuntimeError(f"softmax_xent: labels must be a CUDA tensor of shape ({n},), got {tuple(labels.shape)} on {labels.device}")
    if labels.dtype != torch.int64:          # the kernel reads const int64_t*: any other integer width would be misread
        if labels.dtype.is_floating_point or labels.dtype == torch.bool:
            raise TypeError(f"softmax_xent: labels must be an integer tensor, got {labels.dtype}")
        labels = labels.to(torch.int64)
    labels = labels.contiguous()
    loss = torch.empty((n,), device=logits.device, dtype=torch.float32)
    dl = torch.empty_like(logits) if want_grad else None
    pred = torch.empty((n,), device=logits.device, dtype=torch.int32)
    _lib.check(_lib.lib().ga_softmax_xent(ptr(logits), ptr(labels), n, k, ptr(loss), ptr(dl), ptr(pred), ptr(counter), stream()),
               "softmax_xent")
    return loss, dl, pred


# ------------------------------------------------------------------------------------------------ StyleGAN2 generator ops
@_timed("pixelnorm")
def pixelnorm(x: torch.Tensor, out_dtype) -> torch.Tensor:
    """x: (rows, d) fp32 -> (rows, 1, 1, d) NHWC view"""
    rows, d = x.shape
    out = torch.empty((rows, 1, 1, d), device=x.device, dtype=out_dtype)
    _lib.check(_lib.lib().ga_pixelnorm(ptr(x.contiguous()), rows, d, gt(out), stream()), "pixelnorm")
    return out


@_timed("style_demod")
def style_demod(s: torch.Tensor, wsq: torch.Tensor) -> torch.Tensor:
    n, cin = s.shape
    cout = wsq.shape[0]
    demod = torch.empty((n, cout), device=s.device, dtype=torch.float32)
    _lib.check(_lib.lib().ga_style_demod(ptr(s), ptr(wsq), n, cin, cout, ptr(demod), stream()), "style_demod")
    return demod


@_timed("channel_scale")
def channel_scale(x, s, out_dtype):
    out = torch.empty(x.shape, device=x.device, dtype=out_dtype)
    _lib.check(_lib.lib().ga_channel_scale(gt(x), ptr(s), gt(out), stream()), "channel_scale")
    return out


@_timed("styled_bias_act", hbm=True)
def styled_bias_act(y, phases: bool, demod, noise_hw, noise_w: float, bias, act: int, skip, out_dtype, scale_a=None, scale_b=None,
                    want_out: bool = True, skip_up_kernel=None):
    """v = act(y * demod + noise + bias) (+ skip, up-sampled x2 on the fly through the 4x4 FIR `skip_up_kernel` when given);
    -> out = v * scale_a (or v), and with scale_b -> (out | None, v * scale_b)"""
    n = y.shape[0]
    h, w, c = (y.shape[1] * 2, y.shape[2] * 2, y.shape[3] // 4) if phases else (y.shape[1], y.shape[2], y.shape[3])
    out = torch.empty((n, h, w, c), device=y.device, dtype=out_dtype) if want_out else None
    out_b = torch.empty((n, h, w, c), device=y.device, dtype=out_dtype) if scale_b is not None else None
    _lib.check(_lib.lib().ga_styled_bias_act(gt(y), int(phases), ptr(demod), ptr(noise_hw), float(noise_w), ptr(bias), act, gt(skip),
                                             ptr(skip_up_kernel), ptr(scale_a), gt(out), ptr(scale_b), gt(out_b), stream()), "styled_bias_act")
    return (out, out_b) if scale_b is not None else out


@_timed("torgb_fused", hbm=True)
def torgb_fused(x: torch.Tensor, L: ConvLayer, bias, skip=None, skip_up_kernel=None) -> torch.Tensor:
    """ToRGB in one pass: conv1x1(x, L.w_tc [4][cin]) + bias + Upsample(skip)  -> fp32 (n, h, w, 4)"""
    n, h, w, _ = x.shape
    out = torch.empty((n, h, w, 4), device=x.device, dtype=torch.float32)
    _lib.check(_lib.lib().ga_torgb_fused(gt(x), L.w_tc.data_ptr(), ptr(bias), gt(skip), ptr(skip_up_kernel), gt(out), stream()), "torgb_fused")
    return out


@_timed("upfirdn2d", hbm=True)
def upfirdn2d(x, kernel, up: int = 1, down: int = 1, pad=(0, 0), out_dtype=None):
    """same semantics as the reference op (stylegan2/op/upfirdn2d.py:141-147) on NHWC tensors"""
    n, h, w, c = x.shape
    kh, kw = kernel.shape
    ho = (h * up + pad[0] + pad[1] - kh) // down + 1
    wo = (w * up + pad[0] + pad[1] - kw) // down + 1
    out = torch.empty((n, ho, wo, c), device=x.device, dtype=out_dtype or x.dtype)
    _lib.check(_lib.lib().ga_upfirdn2d(gt(x), ptr(kernel), kh, kw, up, down, pad[0], pad[1], gt(out), stream()), "upfirdn2d")
    return out


@_timed("avgpool_to_nchw")
def avgpool_to_nchw(x, k: int, out_c: int):
    n, h, w, c = x.shape
    out = torch.empty((n, out_c, h // k, w // k), device=x.device, dtype=torch.float32)
    _lib.check(_lib.lib().ga_avgpool_to_nchw(gt(x), k, out_c, ptr(out), stream()), "avgpool_to_nchw")
    return out


@_timed("latent_lerp")
def latent_lerp(codes, styles, alphas_dev):
    b, l, d = codes.shape
    out = torch.empty_like(codes)
    _lib.check(_lib.lib().ga_latent_lerp(ptr(codes.contiguous()), ptr(styles.contiguous()), ptr(alphas_dev), b, l, d, ptr(out), stream()),
               "latent_lerp")
    return out


# ------------------------------------------------------------------------------------------------ encoder-side ops (encoders.cu)
@_timed("add_layernorm")
def add_layernorm(x, y, gamma, beta, out_dtype, eps: float = 1e-5, out2_dtype=None):
    """LayerNorm(x + y) over channels -> out (and a second copy in out2_dtype)"""
    out = torch.empty(x.shape, device=x.device, dtype=out_dtype)
    out2 = torch.empty(x.shape, device=x.device, dtype=out2_dtype) if out2_dtype is not None else None
    _lib.check(_lib.lib().ga_add_layernorm(gt(x), gt(y), ptr(gamma), ptr(beta), eps, gt(out), gt(out2), stream()), "add_layernorm")
    return (out, out2) if out2_dtype is not None else out


@_timed("attention")
def attention(q, q_off: int, k, k_off: int, v, v_off: int, heads: int, dh: int, out_dtype):
    """q (B,Q,1,Cq), k / v (B,*,*,C): head h = columns [off + h*dh, off + (h+1)*dh).  -> (B,Q,1,heads*dh)"""
    b, nq = q.shape[0], q.shape[1] * q.shape[2]
    s = k.shape[1] * k.shape[2]
    ws = torch.empty((int(_lib.lib().ga_attention_ws_floats(b, heads, nq, s)),), device=q.device, dtype=torch.float32)
    out = torch.empty((b, nq, 1, heads * dh), device=q.device, dtype=out_dtype)
    _lib.check(_lib.lib().ga_attention(gt(q), q_off, gt(k), k_off, gt(v), v_off, heads, dh, ptr(ws), gt(out), stream()), "attention")
    return out


@_timed("codes_assemble")
def codes_assemble(heads, heads_lb: bool, use_w0: bool, latent_avg, b: int, l: int, d: int):
    out = torch.empty((b, l, d), device=heads.device, dtype=torch.float32)
    _lib.check(_lib.lib().ga_codes_assemble(ptr(heads), int(heads_lb), int(use_w0), ptr(latent_avg), b, l, d, ptr(out), stream()),
               "codes_assemble")
    return out


@_timed("resize_bilinear")
def resize_bilinear(x, full_h: int, out_w: int, crop_y0: int, crop_h: int, out_dtype=None):
    n, h, w, c = x.shape
    out = torch.empty((n, crop_h, out_w, c), device=x.device, dtype=out_dtype or x.dtype)
    _lib.check(_lib.lib().ga_resize_bilinear(gt(x), full_h, crop_y0, gt(out), stream()), "resize_bilinear")
    return out


@_timed("image_pool_out", hbm=True)
def image_pool_out(img, k1: int, k2: int = 1, mask_rows: int = 0, denorm=(0.5, 0.5), cls_dtype=None, want_purified: bool = True):
    """generator image NHWC fp32 -> (purified NCHW fp32 denormalised | None, classifier input NHWC | None)"""
    n, s = img.shape[0], img.shape[1]
    so = s // (k1 * k2)
    pur = torch.empty((n, 3, so, so), device=img.device, dtype=torch.float32) if want_purified else None
    cls = torch.empty((n, so, so, 3), device=img.device, dtype=cls_dtype) if cls_dtype is not None else None
    _lib.check(_lib.lib().ga_image_pool_out(gt(img), k1, k2, mask_rows, float(denorm[0]), float(denorm[1]), ptr(pur), gt(cls), stream()),
               "image_pool_out")
    return pur, cls


@_timed("philox_codes")
def philox_codes(seed: int, sample0: int, std: float, l: int, b: int, d: int, device):
    out = torch.empty((l, b, d), device=device, dtype=torch.float32)
    _lib.check(_lib.lib().ga_philox_codes(seed, sample0, float(std), l, b, d, ptr(out), stream()), "philox_codes")
    return out


# ------------------------------------------------------------------------------------------------ backward ops
@_timed("affine_act_bwd", hbm=True)
def affine_act_bwd(g, x, scale, shift, act: int, out_dtype, add=None):
    out = torch.empty(g.shape, device=g.device, dtype=out_dtype)
    _lib.check(_lib.lib().ga_affine_act_bwd(gt(g), gt(x), ptr(scale), ptr(shift), act, gt(add), gt(out), stream()), "affine_act_bwd")
    return out


@_timed("add", hbm=True)
def add(a, b, out_dtype):
    out = torch.empty(a.shape, device=a.device, dtype=out_dtype)
    _lib.check(_lib.lib().ga_add(gt(a), gt(b), gt(out), stream()), "add")
    return out


@_timed("se_residual_bwd", hbm=True)
def se_residual_bwd(g_out, r, sums, se, res_scale: float, out_dtype):
    w1, b1, w2, b2 = se
    g_r = torch.empty(r.shape, device=r.device, dtype=out_dtype)
    dots = torch.empty_like(sums)
    _lib.check(_lib.lib().ga_se_residual_bwd(gt(g_out), gt(r), ptr(sums), ptr(dots), ptr(w1), ptr(b1), ptr(w2), ptr(b2),
                                             w1.shape[0], res_scale, gt(g_r), stream()), "se_residual_bwd")
    return g_r


@_timed("sumpool2x2", hbm=True)
def sumpool2x2(x, out_dtype, mul=None):
    n, h, w, c = x.shape
    out = torch.empty((n, h // 2, w // 2, c), device=x.device, dtype=out_dtype)
    _lib.check(_lib.lib().ga_sumpool2x2(gt(x), gt(mul), gt(out), stream()), "sumpool2x2")
    return out


@_timed("upsample_bilinear2x_bwd")
def upsample_bilinear2x_bwd(g_out, out_dtype):
    n, h, w, c = g_out.shape
    out = torch.empty((n, h // 2, w // 2, c), device=g_out.device, dtype=out_dtype)
    _lib.check(_lib.lib().ga_upsample_bilinear2x_bwd(gt(g_out), gt(out), stream()), "upsample_bilinear2x_bwd")
    return out


@_timed("depth_to_space2", hbm=True)
def depth_to_space2(x: torch.Tensor) -> torch.Tensor:
    """[n,h,w,4c] fp32 (phase-major channels) -> [n,2h,2w,c]"""
    n, h, w, c4 = x.shape
    out = torch.empty((n, 2 * h, 2 * w, c4 // 4), device=x.device, dtype=torch.float32)
    _lib.check(_lib.lib().ga_depth_to_space2(gt(x), gt(out), stream()), "depth_to_space2")
    return out


@_timed("phase_interleave", hbm=True)
def phase_interleave(x: torch.Tensor, add=None, mul=None, mul_mode: int = MUL_VALUE, slope=None, out_dtype=torch.float32) -> torch.Tensor:
    """[n,h,w,4c] fp32 (phase-major channels) -> (depth_to_space2(x) + add) * f(mul) [n,2h,2w,c] in out_dtype, one pass; f is the
    ga_mul_mode factor (MUL_PRELU_FROM_Y: `slope` [c] fp32, the slopes of the layer that produced `mul`)"""
    n, h, w, c4 = x.shape
    out = torch.empty((n, 2 * h, 2 * w, c4 // 4), device=x.device, dtype=out_dtype)
    _lib.check(_lib.lib().ga_phase_interleave(gt(x), gt(add), gt(mul), int(mul_mode), ptr(slope), gt(out), stream()), "phase_interleave")
    return out


@_timed("subsample2x_bwd", hbm=True)
def subsample2x_bwd(g: torch.Tensor, out_hw, out_dtype=torch.float32) -> torch.Tensor:
    """adjoint of subsample2x: g [n,h,w,c] -> [n,H,W,c] with g at the even pixels, zeros elsewhere"""
    out = torch.empty((g.shape[0], out_hw[0], out_hw[1], g.shape[3]), device=g.device, dtype=out_dtype)
    _lib.check(_lib.lib().ga_subsample2x_bwd(gt(g), gt(out), stream()), "subsample2x_bwd")
    return out


@_timed("codes_assemble_bwd")
def codes_assemble_bwd(g_codes: torch.Tensor) -> torch.Tensor:
    """adjoint of codes_assemble(heads_lb=True, use_w0=True): g_codes (b, l, d) fp32 -> g_heads (l, b, d) fp32"""
    b, l, d = g_codes.shape
    g_codes = g_codes.contiguous()
    out = torch.empty((l, b, d), device=g_codes.device, dtype=torch.float32)
    _lib.check(_lib.lib().ga_codes_assemble_bwd(ptr(g_codes), b, l, d, ptr(out), stream()), "codes_assemble_bwd")
    return out


@_timed("maxpool2x2_bwd", hbm=True)
def maxpool2x2_bwd(x_in, g_out, relu: bool, out_dtype):
    out = torch.empty(x_in.shape, device=x_in.device, dtype=out_dtype)
    _lib.check(_lib.lib().ga_maxpool2x2_bwd(gt(x_in), gt(g_out), int(relu), gt(out), stream()), "maxpool2x2_bwd")
    return out


@_timed("maxpool3x3s2_bwd", hbm=True)
def maxpool3x3s2_bwd(x_in, g_out, relu: bool, out_dtype):
    out = torch.empty(x_in.shape, device=x_in.device, dtype=out_dtype)
    _lib.check(_lib.lib().ga_maxpool3x3s2_bwd(gt(x_in), gt(g_out), int(relu), gt(out), stream()), "maxpool3x3s2_bwd")
    return out


@_timed("avgpool_bwd_relu", hbm=True)
def avgpool_bwd_relu(g_feat, y, out_dtype):
    """global-average-pool backward times the ReLU mask of the pooled map y: g_feat (N,1,1,C) -> (N,H,W,C)"""
    out = torch.empty(y.shape, device=y.device, dtype=out_dtype)
    _lib.check(_lib.lib().ga_avgpool_bwd_relu(gt(g_feat), gt(y), gt(out), stream()), "avgpool_bwd_relu")
    return out


@_timed("latent_mix_bwd", hbm=True)
def latent_mix_bwd(g_z, q, p, eps_nchw, seed: int, level: int, sample0: int, alpha_dev, temperature: float, zdim: int, zc: int):
    """-> (g_q fp32 [n,h,w,zc] zero-padded beyond zdim, g_p fp32 [n,h,w,2*zdim] | None)"""
    n, h, w, _ = q.shape
    g_q = torch.empty((n, h, w, zc), device=q.device, dtype=torch.float32)
    g_p = torch.empty((n, h, w, 2 * zdim), device=q.device, dtype=torch.float32) if p is not None else None
    _lib.check(_lib.lib().ga_latent_mix_bwd(gt(g_z), gt(q), gt(p), ptr(eps_nchw), seed, level, sample0, ptr(alpha_dev), temperature,
                                            zdim, gt(g_q), gt(g_p), stream()), "latent_mix_bwd")
    return g_q, g_p


@_timed("discmix_mean_bwd", hbm=True)
def discmix_mean_bwd(logits, n_mix: int, g_purified_nchw, g_cls, pad_to: int = 0):
    """-> d loss / d logits, fp32, channel-padded with zeros to `pad_to` channels (tensor-core alignment of the dgrad conv)"""
    n, h, w, c = logits.shape
    g_logits = torch.empty((n, h, w, max(c, pad_to)), device=logits.device, dtype=torch.float32)
    _lib.check(_lib.lib().ga_discmix_mean_bwd(gt(logits), n_mix, ptr(g_purified_nchw), gt(g_cls), gt(g_logits), stream()),
               "discmix_mean_bwd")
    return g_logits


@_timed("preprocess_bwd", hbm=True)
def preprocess_bwd(g_nhwc, pre_nchw, blur: bool, normalize: bool = True, taps_cache=None):
    """-> gradient w.r.t. the input batch (NCHW fp32)."""
    n, h, w, c = g_nhwc.shape
    gx = torch.empty((n, c, h, w), device=g_nhwc.device, dtype=torch.float32)
    taps, radius, tmp = None, 0, None
    if blur:
        if taps_cache is not None and taps_cache.get("h") == h:
            taps, radius = taps_cache["taps"], taps_cache["radius"]
        else:
            t, radius = gaussian_taps(h)
            taps = t.to(g_nhwc.device)
        tmp = torch.empty_like(gx)
    _lib.check(_lib.lib().ga_preprocess_bwd(gt(g_nhwc), ptr(pre_nchw), ptr(taps), radius, int(normalize), ptr(tmp), ptr(gx), stream()),
               "preprocess_bwd")
    return gx


def styled_bias_act_bwd_parts(hw: int, c: int) -> int:
    """number of fixed pixel slices of the per-(sample, channel) partial sums of `styled_bias_act_bwd`"""
    return int(_lib.lib().ga_styled_bias_act_bwd_parts(hw, c))


@_timed("styled_bias_act_bwd", hbm=True)
def styled_bias_act_bwd(v, g_next, s_next, g_rgb, w_rgb, s_rgb, demod, noise_hw, noise_w: float, bias, phases: bool, gy_dtype,
                        dot_next=None, dot_rgb=None, dot_demod=None, want_gy: bool = True):
    """backward of one styled layer's epilogue (styled_bias_act + the ToRGB 1x1 conv fed by it), v = the taped activation.
    -> g_y (conv-output gradient; phase-major [n,h/2,w/2,4c] when `phases`) or None; the dots land in the caller's
    [n, styled_bias_act_bwd_parts(h*w, c), c] fp32 buffers"""
    n, h, w, c = v.shape
    g_y = None
    if want_gy:
        g_y = torch.empty((n, h // 2, w // 2, 4 * c) if phases else (n, h, w, c), device=v.device, dtype=gy_dtype)
    _lib.check(_lib.lib().ga_styled_bias_act_bwd(gt(v), gt(g_next), ptr(s_next), ptr(g_rgb), ptr(w_rgb), ptr(s_rgb), ptr(demod),
                                                 ptr(noise_hw), float(noise_w), ptr(bias), int(phases), gt(g_y), ptr(dot_next), ptr(dot_rgb),
                                                 ptr(dot_demod), stream()), "styled_bias_act_bwd")
    return g_y


@_timed("style_bwd")
def style_bwd(dot_mod, dot_demod, s, demod, wsq) -> torch.Tensor:
    """d loss / d s (n, cin) of a modulated layer from its partial dots (see `styled_bias_act_bwd`); dot_demod / demod / wsq are None for
    ToRGB layers (no demodulation)"""
    n, cin = s.shape
    cout = wsq.shape[0] if wsq is not None else 0
    ds = torch.empty((n, cin), device=s.device, dtype=torch.float32)
    _lib.check(_lib.lib().ga_style_bwd(ptr(dot_mod), dot_mod.shape[1] if dot_mod is not None else 0, ptr(dot_demod),
                                       dot_demod.shape[1] if dot_demod is not None else 0, ptr(s), ptr(demod), ptr(wsq), n, cin, cout,
                                       ptr(ds), stream()), "style_bwd")
    return ds


@_timed("image_pool_out_bwd", hbm=True)
def image_pool_out_bwd(g_purified, g_cls, size: int, k1: int, k2: int = 1, mask_rows: int = 0, out_scale: float = 0.5):
    """adjoint of `image_pool_out`: (g_purified NCHW fp32 | None, g_cls NHWC | None) -> generator image gradient (n, size, size, 4) fp32"""
    n = (g_purified if g_purified is not None else g_cls).shape[0]
    g_img = torch.empty((n, size, size, 4), device=(g_purified if g_purified is not None else g_cls).device, dtype=torch.float32)
    _lib.check(_lib.lib().ga_image_pool_out_bwd(ptr(g_purified.contiguous()) if g_purified is not None else None,
                                                gt(g_cls.contiguous()) if g_cls is not None else None, k1, k2, mask_rows, float(out_scale),
                                                gt(g_img), stream()), "image_pool_out_bwd")
    return g_img


@_timed("latent_lerp_bwd")
def latent_lerp_bwd(g_out, alphas_dev):
    """adjoint of `latent_lerp` w.r.t. the codes: (1 - alpha_l) * g_out[:, l]"""
    b, l, d = g_out.shape
    g_out = g_out.contiguous()
    out = torch.empty_like(g_out)
    _lib.check(_lib.lib().ga_latent_lerp_bwd(ptr(g_out), ptr(alphas_dev), b, l, d, ptr(out), stream()), "latent_lerp_bwd")
    return out


def launch_count(reset: bool = False) -> int:
    return int(_lib.lib().ga_launch_count(int(reset)))
