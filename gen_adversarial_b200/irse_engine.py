"""IR-SE50 backbone and the two W+ inversion encoders built on it, on the hand-written CUDA kernels.

Replaces (paths under /root/reference/src/mlvgms_autoencoders/):
  * `Encoder4Editing.forward`          StyleGan_E4E/encoding/encoder.py:57-140  (+ `bottleneck_IR_SE`, `SEModule`,
    `_upsample_add`, helpers.py:57-139; `GradualStyleBlock` :33-54; `pSp.encode` psp.py:88-101)        -- SURVEY row A13
  * `GradualStyleEncoder.forward`      StyleGan_Trans/models/encoders/style_transformer_encoders.py:10-84 and the DETR
    `TransformerDecoderLayer.forward_post` StyleGan_Trans/models/transformer.py:40-66                   -- SURVEY row A18

Exact load-time rewrites (fp64): eval BN after a conv folded into the conv; the BN *before* the first 3x3 conv of every unit
stays an affine pre-op because the reference zero-pads after it (bf16 mode: the previous unit's SE/residual kernel
emits BN(x) as a second bf16 output, so no extra pass exists); `MaxPool2d(1, stride)` shortcuts are a strided
sub-sample; the 1x1 stride-2 shortcut convs and the 3x3 stride-2 convs run on the tensor-core kernel with TMA element
strides; `EqualLinear` scales folded; the learned query `z` of the Style-Transformer goes through the mapping MLP once
for its 16 rows (the reference expands it to B x 16 rows first, style_transformer.py:57-61 / models.py:311-315).

Input gradient (E4E; attacks): `IrSe50Backbone.backward` and `E4EEncoderEngine.encode_backward` run the dgrad-only reverse sweep over what a
taped forward (`EncoderTape`) kept: per unit the PReLU output h of conv1, the conv2 output r and its SE channel sums, plus the stem output
and every map2style activation.  The PReLU / LeakyReLU derivatives are recovered from the SIGN of those outputs (exact while every slope is
> 0, checked when the dgrad layers are built); the BN in front of each unit's conv1 is folded into conv1's dgrad weights.
"""
from __future__ import annotations

import math
from typing import Dict, List, Optional

import torch

from . import ops
from ._lib import PRE_NONE, PRE_AFFINE, ACT_NONE, ACT_RELU, ACT_PRELU, MUL_PRELU_FROM_Y
from .fold import Folder
from .resnet_engine import conv_dgrad

IRSE50_BLOCKS = [(64, 64, 3), (64, 128, 4), (128, 256, 14), (256, 512, 3)]      # helpers.py:30-37 (in, depth, units)


def irse50_units():
    """-> [(in_channel, depth, stride)] for the 24 bottleneck units (helpers.py:26-37)."""
    units = []
    for cin, depth, n in IRSE50_BLOCKS:
        units.append((cin, depth, 2))
        units += [(depth, depth, 1)] * (n - 1)
    return units


class _Unit:
    __slots__ = ("cin", "depth", "stride", "pre", "pre_scale64", "c1", "c2", "sc", "se", "c1_d", "c2_d", "sc_d")


class EncoderTape:
    """what a taped `E4EEncoderEngine.encode` keeps for `encode_backward` (tensors the forward produces anyway; nothing is recomputed)"""

    def __init__(self):
        self.stem = None          # stem output (PReLU output: unit 0's input and the stem's mask)
        self.units = []           # per unit (h, r, sums): conv1's PReLU output, conv2's output, r's SE channel sums
        self.heads = []           # per map2style head: the output of each conv (LeakyReLU outputs)
        self.tap_shapes = None    # shapes of c1 / c2 / c3


def conv1x1_any(engine, x, L, want_f32=False, add=None, out=None):
    """1x1 convolution / linear layer on any (N,H,W,C) tensor: every pixel is an independent GEMM row, so the tensor is
    viewed as (M,1,1,C), which the tensor-core kernel always tiles (128 rows per tile)."""
    n, h, w, c = x.shape
    xv = x.reshape(n * h * w, 1, 1, c)
    addv = add.reshape(n * h * w, 1, 1, -1) if add is not None else None
    outv = out.reshape(n * h * w, 1, 1, -1) if out is not None else None
    y = engine._conv(xv, L, want_f32=want_f32, add=addv, out=outv)
    return y.reshape(n, h, w, L.cout)


class IrSe50Backbone:
    """input_layer + 24 `bottleneck_IR_SE` units; returns the taps c1 / c2 / c3 (after units 6, 20, 23)."""

    def __init__(self, f: Folder, bf16: bool, in_channels: int = 3, tf32: bool = False):
        self.bf16 = bf16
        # tf32: in bf16 mode the 48 convs of the backbone keep fp32 activations / weights and multiply them as TF32 (kind::tf32: 10-bit
        # mantissas, half the bf16 MMA rate).  The E4E path needs it: with a bf16 backbone its W+ codes are off by 0.35% of their range and
        # the purified image lands AT the 1e-2 bf16 gate (DESIGN.md section 2); the taps handed to the heads stay bf16.
        self.tf32 = bool(tf32 and bf16)
        self.f32_taps = False                 # tf32 mode: hand the fp32 residual stream (not its bf16 copy) to the heads
        self.adt = torch.bfloat16 if bf16 else torch.float32
        w = f.f64("input_layer.0.weight")
        a, b = f.bn("input_layer.1")
        self.stem = f.conv(w * a.view(-1, 1, 1, 1), b, pad=1, post_act=ACT_PRELU, name="input_layer")
        self.stem.act_slope = f.dev32(f.f64("input_layer.2.weight"))
        self.units: List[_Unit] = []
        for i, (cin, depth, stride) in enumerate(irse50_units()):
            u = _Unit()
            u.cin, u.depth, u.stride = cin, depth, stride
            p = f"body.{i}"
            a0, b0 = f.bn(f"{p}.res_layer.0")
            u.pre = (f.dev32(a0), f.dev32(b0))
            u.pre_scale64 = a0
            u.c1 = f.conv(f.f64(f"{p}.res_layer.1.weight"), None, pad=1, pre_op=PRE_AFFINE, pre_affine=(a0, b0),
                          post_act=ACT_PRELU, name=f"{p}.conv1", tf32=self.tf32)
            u.c1.act_slope = f.dev32(f.f64(f"{p}.res_layer.2.weight"))
            a4, b4 = f.bn(f"{p}.res_layer.4")
            u.c2 = f.conv(f.f64(f"{p}.res_layer.3.weight") * a4.view(-1, 1, 1, 1), b4, stride=stride, pad=1, name=f"{p}.conv2",
                          tf32=self.tf32)
            if cin != depth:
                asc, bsc = f.bn(f"{p}.shortcut_layer.1")
                u.sc = f.conv(f.f64(f"{p}.shortcut_layer.0.weight") * asc.view(-1, 1, 1, 1), bsc, stride=stride, pad=0,
                              name=f"{p}.shortcut", tf32=self.tf32)
            else:
                u.sc = None
            w1 = f.f64(f"{p}.res_layer.5.fc1.weight").flatten(1)
            w2 = f.f64(f"{p}.res_layer.5.fc2.weight").flatten(1)
            u.se = (f.dev32(w1), None, f.dev32(w2), None)
            self.units.append(u)
        self._has_dgrad = False

    def _conv(self, x, L, want_f32=False, add=None, out=None):
        if self.bf16 and x.dtype == torch.float32 and L.w_tf32 is not None and ops.conv2d_tc_supported(x, L, tf32=True):
            ob, of = ops.conv2d_tc(x, L, want_bf16=not want_f32, want_f32=want_f32, add=add, tf32=True,
                                   out_bf16=None if want_f32 else out, out_f32=out if want_f32 else None)
            return of if want_f32 else ob
        if self.bf16 and L.w_tc is not None and x.dtype == torch.bfloat16 and ops.conv2d_tc_supported(x, L):
            ob, of = ops.conv2d_tc(x, L, want_bf16=not want_f32, want_f32=want_f32, add=add,
                                   out_bf16=None if want_f32 else out, out_f32=out if want_f32 else None)
            return of if want_f32 else ob
        return ops.conv2d_simt(x, L, torch.float32 if (want_f32 or not self.bf16) else torch.bfloat16, add=add, out=out)

    def forward(self, x_nhwc: torch.Tensor, tape: Optional[EncoderTape] = None):
        """x_nhwc (N,H,W,3) normalised input in the activation dtype -> (c1, c2, c3) in the activation dtype.
        tape: an EncoderTape receiving what `backward` needs (build_dgrad() first); the values computed do not depend on it."""
        units = self.units
        x32 = ops.conv2d_simt(x_nhwc, self.stem, torch.float32)
        if tape is not None:
            tape.stem = x32
        if self.tf32:
            return self._forward_tf32(x32, tape)
        xa = ops.affine_act(x32, units[0].pre[0], units[0].pre[1], ACT_NONE, torch.bfloat16) if self.bf16 else None
        xb = ops.cast(x32, torch.bfloat16) if (self.bf16 and units[0].sc is not None) else None
        taps = {}
        for i, u in enumerate(units):
            if self.bf16:
                if ops.conv2d_tc_supported(xa, u.c1):
                    h, _ = ops.conv2d_tc(xa, u.c1)
                else:
                    h = ops.conv2d_simt(x32, u.c1, torch.bfloat16)            # SIMT applies the BN pre-op itself
            else:
                h = ops.conv2d_simt(x32, u.c1, torch.float32)
            r = self._conv(h, u.c2, want_f32=True)     # fp32: r only feeds the SE mean and the fp32 residual stream (one bf16 rounding less per unit)
            if u.sc is not None:
                skip = self._conv(xb if self.bf16 else x32, u.sc, want_f32=True)
            else:
                skip = x32 if u.stride == 1 else ops.subsample2x(x32)
            sums = ops.channel_sum(r)
            if tape is not None:
                tape.units.append((h, r, sums))
            nxt = units[i + 1] if i + 1 < len(units) else None
            is_tap = i in (6, 20, 23)
            want_b = self.bf16 and (is_tap or (nxt is not None and nxt.sc is not None))
            x32, xb, xa, _ = ops.se_residual(r, sums, u.se, 1.0, skip, torch.float32, want_out2=want_b,
                                             act_affine=nxt.pre if (self.bf16 and nxt is not None) else None, act_op=ACT_NONE)
            if is_tap:
                taps[i] = xb if self.bf16 else x32
        self.c3_f32 = x32                                  # fp32 copy of the last tap (E4E head 0 reads it)
        return taps[6], taps[20], taps[23]


    def _conv_tf32(self, x32, L, round_out: bool):
        """fp32 activations x fp32 weights on the tensor cores as TF32 -> fp32 (rounded to TF32 when it feeds another TF32 conv);
        shapes the TC kernel cannot tile return None (the caller falls back to the SIMT conv)"""
        if L.w_tf32 is not None and ops.conv2d_tc_supported(x32, L, tf32=True):
            ops.f32_round_tf32(round_out)
            try:
                return ops.conv2d_tc(x32, L, want_bf16=False, want_f32=True, tf32=True)[1]
            finally:
                ops.f32_round_tf32(False)
        return None

    @staticmethod
    def _rounded(fn):
        """run `fn` with fp32 activation outputs rounded to nearest TF32 (operands of kind::tf32 convs, which truncate)"""
        ops.f32_round_tf32(True)
        try:
            return fn()
        finally:
            ops.f32_round_tf32(False)

    def _forward_tf32(self, x32, tape=None):
        units = self.units
        # BN of the first unit (the conv pads AFTER it), rounded to TF32
        xa = self._rounded(lambda: ops.affine_act(x32, units[0].pre[0], units[0].pre[1], ACT_NONE, torch.float32))
        taps = {}
        for i, u in enumerate(units):
            h = self._conv_tf32(xa, u.c1, True)
            if h is None:
                h = ops.conv2d_simt(x32, u.c1, torch.float32)                                   # SIMT applies the BN pre-op itself
            r = self._conv_tf32(h, u.c2, False)                                                 # r feeds the SE mean and the fp32 stream: unrounded
            if r is None:
                r = ops.conv2d_simt(h, u.c2, torch.float32)
            if u.sc is not None:
                xs = self._rounded(lambda: ops.cast(x32, torch.float32))                        # TF32-rounded copy of the stream for the shortcut conv
                skip = self._conv_tf32(xs, u.sc, False)
                if skip is None:
                    skip = ops.conv2d_simt(x32, u.sc, torch.float32)
            else:
                skip = x32 if u.stride == 1 else ops.subsample2x(x32)
            sums = ops.channel_sum(r)
            if tape is not None:
                tape.units.append((h, r, sums))
            nxt = units[i + 1] if i + 1 < len(units) else None
            is_tap = i in (6, 20, 23)
            x32, xb, xa, _ = self._rounded(lambda: ops.se_residual(
                r, sums, u.se, 1.0, skip, torch.float32, want_out2=is_tap, act_affine=nxt.pre if nxt is not None else None,
                act_dtype=torch.float32, act_op=ACT_NONE))                                      # only the fp32 `act` copy is rounded
            if is_tap:
                # bf16 copies for the FPN / heads, or TF32-rounded copies of the fp32 stream
                taps[i] = self._rounded(lambda: ops.cast(x32, torch.float32)) if self.f32_taps else xb
        self.c3_f32 = x32
        return taps[6], taps[20], taps[23]

    # ------------------------------------------------------------------ input gradient
    def build_dgrad(self, device):
        """dgrad layers of the stem and the 24 units (built on the first taped forward: forward-only use pays nothing).  The PReLU masks are
        recovered from the sign of the PReLU outputs, which is exact only for slopes > 0: any other slope refuses the backward."""
        if self._has_dgrad:
            return
        from .nvae_engine import make_dgrad_layer
        for L in [self.stem] + [u.c1 for u in self.units]:
            if bool((L.act_slope <= 0).any()):
                raise NotImplementedError(f"input gradient through the IR-SE50 backbone: PReLU of {L.name} has a slope <= 0, so its derivative "
                                          f"cannot be recovered from the sign of its taped output")
        f = Folder({}, device, want_tc=self.bf16)
        for i, u in enumerate(self.units):
            u.c1_d = make_dgrad_layer(f, u.c1, self.bf16, in_scale=u.pre_scale64)      # BN pre-affine (zero padding after it): scale folded
            u.c1_d.act_slope = self.stem.act_slope if i == 0 else None                 # unit 0's input is the stem's PReLU output
            u.c2_d = make_dgrad_layer(f, u.c2, self.bf16)
            u.c2_d.act_slope = u.c1.act_slope                                          # mask of h = PReLU(conv1)
            u.sc_d = make_dgrad_layer(f, u.sc, self.bf16) if u.sc is not None else None
        self.stem_d = make_dgrad_layer(f, self.stem, self.bf16)
        self._has_dgrad = True

    def backward(self, tape: EncoderTape, g_c1: torch.Tensor, g_c2: torch.Tensor, g_c3: torch.Tensor) -> torch.Tensor:
        """d loss / d (c1, c2, c3) fp32 NHWC -> d loss / d x_nhwc (N,H,W,3) fp32 (w.r.t. the normalised image); the residual-stream gradient
        stays fp32, the gradients that only feed a dgrad conv are bf16 in bf16 mode.  The tape is left intact."""
        dg = lambda g, D, **kw: conv_dgrad(g, D, self.bf16, mul_mode=MUL_PRELU_FROM_Y, **kw)
        tap_grads = {6: g_c1, 20: g_c2, 23: g_c3}
        g = None
        for i in range(len(self.units) - 1, -1, -1):
            u = self.units[i]
            h, r, sums = tape.units[i]
            t = tap_grads.get(i)
            if t is not None:
                g = t.contiguous() if g is None else ops.add(g, t.contiguous(), torch.float32)
            g_r = ops.se_residual_bwd(g, r, sums, u.se, 1.0, self.adt)                 # the skip gradient is g itself
            g_h = dg(g_r, u.c2_d, mul=h)                                                # times PReLU'(conv1) from the sign of h
            if u.sc is not None:
                g_skip = dg(g, u.sc_d, f32=True)                                        # 1x1 stride-2 shortcut
            elif u.stride == 2:
                g_skip = ops.subsample2x_bwd(g, (h.shape[1], h.shape[2]))               # MaxPool2d(1, 2)
            else:
                g_skip = g
            # unit 0: times the stem's PReLU' (its output is unit 0's input), after the shortcut gradient has joined
            g = dg(g_h, u.c1_d, add=g_skip, mul=tape.stem if i == 0 else None, f32=True)
        return ops.conv2d_simt(g, self.stem_d, torch.float32)


class _Head:
    __slots__ = ("convs", "linear", "convs_d", "linear_d")


class E4EEncoderEngine:
    """`Encoder4Editing` at ProgressiveStage.Inference + `pSp.encode`'s latent_avg offset -> codes (B, n_styles, 512)."""

    def __init__(self, state_dict: Dict[str, torch.Tensor], stylegan_size: int, latent_avg: Optional[torch.Tensor], device,
                 mode: str = "fp32", _host_logic_test: bool = False):
        self.device = torch.device(device)
        if self.device.type != "cuda" and not _host_logic_test:
            raise RuntimeError("E4EEncoderEngine runs only on CUDA devices: there is no CPU fallback")
        self.bf16 = mode == "bf16"
        self.adt = torch.bfloat16 if self.bf16 else torch.float32
        f = Folder(state_dict, self.device, want_tc=self.bf16)
        env = __import__("os").environ
        self.backbone = IrSe50Backbone(f, self.bf16, tf32=env.get("GA_E4E_TF32_BACKBONE", "1") != "0")
        self.tf32_heads = self.bf16 and env.get("GA_E4E_TF32_HEADS", "0") != "0"      # FPN + map2style convs on fp32 operands (TF32 MMA)
        self.backbone.f32_taps = self.tf32_heads and self.backbone.tf32
        self.style_count = 2 * int(math.log2(stylegan_size)) - 2
        self.coarse_ind, self.middle_ind = 3, 7
        self.slope = torch.full((512,), 0.01, dtype=torch.float32, device=self.device)        # nn.LeakyReLU() default
        # (measured: fp32 tails / more fp32 heads do not move the end-to-end bf16 error, which is dominated by the 48 bf16 convs of the
        # backbone -- DESIGN.md section 2; the knobs stay for experiments)
        self.fp32_tail_hw = int(__import__("os").environ.get("GA_E4E_FP32_TAIL_HW", "0"))
        self.fp32_heads = int(__import__("os").environ.get("GA_E4E_FP32_HEADS", "1"))      # heads fed by c3 that run fully in fp32
        self.heads: List[_Head] = []
        for i in range(self.style_count):
            spatial = 16 if i < self.coarse_ind else (32 if i < self.middle_ind else 64)
            hd = _Head()
            hd.convs = []
            for j in range(int(math.log2(spatial))):
                L = f.conv(f.f64(f"styles.{i}.convs.{2 * j}.weight"), f.f64(f"styles.{i}.convs.{2 * j}.bias"), stride=2, pad=1,
                           post_act=ACT_PRELU, name=f"styles.{i}.convs.{2 * j}", tf32=self.tf32_heads)
                L.act_slope = self.slope
                hd.convs.append(L)
            wl = f.f64(f"styles.{i}.linear.weight") * (1.0 / math.sqrt(512))                   # EqualLinear, lr_mul = 1
            hd.linear = f.conv(wl.view(512, 512, 1, 1), f.f64(f"styles.{i}.linear.bias"), name=f"styles.{i}.linear")
            self.heads.append(hd)
        self.lat1 = f.conv(f.f64("latlayer1.weight"), f.f64("latlayer1.bias"), name="latlayer1", tf32=self.tf32_heads)
        self.lat2 = f.conv(f.f64("latlayer2.weight"), f.f64("latlayer2.bias"), name="latlayer2", tf32=self.tf32_heads)
        self.latent_avg = None if latent_avg is None else latent_avg.to(torch.float32).reshape(-1, 512)[: self.style_count].contiguous().to(self.device)
        self._has_dgrad = False

    _conv = IrSe50Backbone._conv

    def build_dgrad(self):
        """dgrad layers of the backbone, the FPN laterals and the heads (raises NotImplementedError for a PReLU slope <= 0, see
        IrSe50Backbone.build_dgrad); called by the first taped `encode`"""
        if self._has_dgrad:
            return
        from .nvae_engine import make_dgrad_layer
        self.backbone.build_dgrad(self.device)
        f = Folder({}, self.device, want_tc=self.bf16)
        for hd in self.heads:
            hd.convs_d = [make_dgrad_layer(f, L, self.bf16) for L in hd.convs]
            for D in hd.convs_d[1:]:
                D.act_slope = self.slope                          # its input is the previous conv's LeakyReLU output
            hd.linear_d = make_dgrad_layer(f, hd.linear, self.bf16)
            hd.linear_d.act_slope = self.slope
        self.lat1_d = make_dgrad_layer(f, self.lat1, self.bf16)
        self.lat2_d = make_dgrad_layer(f, self.lat2, self.bf16)
        self._has_dgrad = True

    def _head(self, feat, hd: _Head, out, acts=None):
        """map2style head.  bf16 mode: the final EqualLinear (and, optionally, the convs on maps <= fp32_tail_hw) run in fp32"""
        x = feat
        for L in hd.convs:
            if self.tf32_heads and x.dtype == torch.float32 and L.w_tf32 is not None and ops.conv2d_tc_supported(x, L, tf32=True):
                x = IrSe50Backbone._rounded(lambda: self._conv(x, L, want_f32=True))     # fp32 operands as TF32 on the tensor cores
            elif self.bf16 and (x.shape[1] <= self.fp32_tail_hw or x.dtype == torch.float32):
                x = ops.conv2d_simt(x, L, torch.float32)
            else:
                x = self._conv(x, L)
            if acts is not None:
                acts.append(x)
        ops.conv2d_simt(x.reshape(x.shape[0], 1, 1, -1), hd.linear, torch.float32, out=out)

    def encode(self, x_nhwc: torch.Tensor, tape: Optional[EncoderTape] = None) -> torch.Tensor:
        """x_nhwc (B,256,256,3) normalised -> codes (B, n_styles, 512) fp32 (latent_avg already added, psp.py:92-99).
        tape: an EncoderTape to fill for encode_backward (the codes are the same with and without it)."""
        b = x_nhwc.shape[0]
        if tape is not None:
            self.build_dgrad()
        c1, c2, c3 = self.backbone.forward(x_nhwc, tape)
        if tape is not None:
            tape.tap_shapes = (c1.shape, c2.shape, c3.shape)
        rnd = IrSe50Backbone._rounded if self.tf32_heads else (lambda fn: fn())
        if self.tf32_heads and c3.dtype != torch.float32:
            c1, c2, c3 = (ops.cast(t, torch.float32) for t in (c1, c2, c3))          # bf16 values are exact in TF32
        heads = torch.empty((self.style_count, b, 1, 1, 512), device=x_nhwc.device, dtype=torch.float32)
        feat = c3
        p2 = None
        for i, hd in enumerate(self.heads):
            if i == self.coarse_ind:
                p2 = rnd(lambda: conv1x1_any(self, c2, self.lat1, add=ops.upsample_bilinear2x(c3), want_f32=self.tf32_heads))   # _upsample_add (helpers.py:122-139)
                feat = p2
            elif i == self.middle_ind:
                feat = rnd(lambda: conv1x1_any(self, c1, self.lat2, add=ops.upsample_bilinear2x(p2), want_f32=self.tf32_heads))
            # head 0 (w0, added to all 18 codes) runs in fp32 from the fp32 residual stream in both modes: 1% of the encoder's FLOPs
            acts = [] if tape is not None else None
            self._head(self.backbone.c3_f32 if (i < self.fp32_heads and self.bf16) else feat, hd, heads[i], acts)
            if tape is not None:
                tape.heads.append(acts)
        return ops.codes_assemble(heads, True, True, self.latent_avg, b, self.style_count, 512)

    def encode_backward(self, tape: EncoderTape, g_codes: torch.Tensor) -> torch.Tensor:
        """g_codes (B, n_styles, 512) fp32 -> d loss / d x_nhwc (B,256,256,3) fp32 (w.r.t. the normalised image).  The heads' gradients are
        summed per feature map (c3 / p2 / p1) in head order, each added in the epilogue of the head's last dgrad."""
        dg = lambda g, D, **kw: conv_dgrad(g, D, self.bf16, mul_mode=MUL_PRELU_FROM_Y, **kw)
        b = g_codes.shape[0]
        g_heads = ops.codes_assemble_bwd(g_codes.to(torch.float32))                    # (n_styles, B, 512): w0 collects every code's gradient
        g_feat = [None, None, None]                                                    # c3, p2, p1
        for i, hd in enumerate(self.heads):
            k = 0 if i < self.coarse_ind else (1 if i < self.middle_ind else 2)
            acts = tape.heads[i]
            g = dg(g_heads[i].reshape(b, 1, 1, 512), hd.linear_d, mul=acts[-1])        # EqualLinear transpose x LeakyReLU'
            for j in range(len(hd.convs_d) - 1, 0, -1):
                g = dg(g, hd.convs_d[j], mul=acts[j - 1])
            g_feat[k] = dg(g, hd.convs_d[0], add=g_feat[k], f32=True)
        g_c3, g_p2, g_p1 = g_feat
        # _upsample_add: p2 = lat1(c2) + up(c3), p1 = lat2(c1) + up(p2)   (align_corners=True bilinear x2)
        s1, s2, _ = tape.tap_shapes
        if g_p1 is not None:
            g_c1 = dg(g_p1, self.lat2_d, f32=True)
            up = ops.upsample_bilinear2x_bwd(g_p1, torch.float32)
            g_p2 = up if g_p2 is None else ops.add(g_p2, up, torch.float32)
        else:
            g_c1 = torch.zeros(s1, device=g_codes.device, dtype=torch.float32)
        if g_p2 is not None:
            g_c2 = dg(g_p2, self.lat1_d, f32=True)
            g_c3 = ops.add(g_c3, ops.upsample_bilinear2x_bwd(g_p2, torch.float32), torch.float32)
        else:
            g_c2 = torch.zeros(s2, device=g_codes.device, dtype=torch.float32)
        return self.backbone.backward(tape, g_c1, g_c2, g_c3)


class _TLayer:
    __slots__ = ("sa_in", "sa_out", "ca_q", "ca_kv", "ca_out", "ff1", "ff2", "n1", "n2", "n3")


class TransEncoderEngine:
    """`GradualStyleEncoder` + the query through the generator's mapping MLP -> codes (B, 16, 512)."""

    def __init__(self, state_dict: Dict[str, torch.Tensor], latent_avg: Optional[torch.Tensor], device, mode: str = "fp32",
                 _host_logic_test: bool = False):
        self.device = torch.device(device)
        if self.device.type != "cuda" and not _host_logic_test:
            raise RuntimeError("TransEncoderEngine runs only on CUDA devices: there is no CPU fallback")
        self.bf16 = mode == "bf16"
        self.adt = torch.bfloat16 if self.bf16 else torch.float32
        f = Folder(state_dict, self.device, want_tc=self.bf16)
        self.backbone = IrSe50Backbone(f, self.bf16)
        self.lat1 = f.conv(f.f64("latlayer1.weight"), f.f64("latlayer1.bias"), name="latlayer1")
        self.lat2 = f.conv(f.f64("latlayer2.weight"), f.f64("latlayer2.bias"), name="latlayer2")
        self.z = f.dev32(f.f64("z")[0])                                                       # (16, 512)
        self.n_query = self.z.shape[0]
        self.layers = [self._fold_layer(f, f"transformerlayer_{n}") for n in ("coarse", "medium", "fine")]
        self.latent_avg = None if latent_avg is None else latent_avg.to(torch.float32).reshape(-1, 512).contiguous().to(self.device)
        self._query_cache = None

    _conv = IrSe50Backbone._conv

    @staticmethod
    def _fold_layer(f: Folder, p: str) -> _TLayer:
        def lin(w, b, act=ACT_NONE, name=""):
            return f.conv(w.view(w.shape[0], w.shape[1], 1, 1), b, post_act=act, name=name)
        t = _TLayer()
        wi, bi = f.f64(f"{p}.self_attn.in_proj_weight"), f.f64(f"{p}.self_attn.in_proj_bias")
        t.sa_in = lin(wi, bi, name=p + ".self_attn.in_proj")                                   # q | k | v fused (1536 outputs)
        t.sa_out = lin(f.f64(f"{p}.self_attn.out_proj.weight"), f.f64(f"{p}.self_attn.out_proj.bias"), name=p + ".self_attn.out_proj")
        wi, bi = f.f64(f"{p}.multihead_attn.in_proj_weight"), f.f64(f"{p}.multihead_attn.in_proj_bias")
        d = wi.shape[1]
        t.ca_q = lin(wi[:d], bi[:d], name=p + ".multihead_attn.q")
        t.ca_kv = lin(wi[d:], bi[d:], name=p + ".multihead_attn.kv")                           # k | v fused (1024 outputs)
        t.ca_out = lin(f.f64(f"{p}.multihead_attn.out_proj.weight"), f.f64(f"{p}.multihead_attn.out_proj.bias"),
                       name=p + ".multihead_attn.out_proj")
        t.ff1 = lin(f.f64(f"{p}.linear1.weight"), f.f64(f"{p}.linear1.bias"), ACT_RELU, name=p + ".linear1")
        t.ff2 = lin(f.f64(f"{p}.linear2.weight"), f.f64(f"{p}.linear2.bias"), name=p + ".linear2")
        for k in ("1", "2", "3"):
            setattr(t, "n" + k, (f.dev32(f.f64(f"{p}.norm{k}.weight")), f.dev32(f.f64(f"{p}.norm{k}.bias"))))
        return t

    def _layer(self, tgt32, tgt_a, memory, t: _TLayer):
        """post-norm decoder layer (transformer.py:40-66, dropout inactive in eval).  tgt32 fp32 (B,Q,1,512), tgt_a same in adt."""
        heads, dh = 4, 128
        d = heads * dh
        qkv = conv1x1_any(self, tgt_a, t.sa_in)
        a = ops.attention(qkv, 0, qkv, d, qkv, 2 * d, heads, dh, self.adt)
        o = conv1x1_any(self, a, t.sa_out, want_f32=True)
        tgt32, tgt_a = ops.add_layernorm(tgt32, o, t.n1[0], t.n1[1], torch.float32, out2_dtype=self.adt)
        q = conv1x1_any(self, tgt_a, t.ca_q)
        kv = conv1x1_any(self, memory, t.ca_kv)
        a = ops.attention(q, 0, kv, 0, kv, d, heads, dh, self.adt)
        o = conv1x1_any(self, a, t.ca_out, want_f32=True)
        tgt32, tgt_a = ops.add_layernorm(tgt32, o, t.n2[0], t.n2[1], torch.float32, out2_dtype=self.adt)
        hdn = conv1x1_any(self, tgt_a, t.ff1)
        o = conv1x1_any(self, hdn, t.ff2, want_f32=True)
        return ops.add_layernorm(tgt32, o, t.n3[0], t.n3[1], torch.float32, out2_dtype=self.adt)

    def query(self, mapping_fn) -> torch.Tensor:
        """decoder.style(z) for the 16 learned query rows (weights are frozen: computed once)"""
        if self._query_cache is None:
            self._query_cache = mapping_fn(self.z).reshape(self.n_query, 512).contiguous()
        return self._query_cache

    def encode(self, x_nhwc: torch.Tensor, query: torch.Tensor) -> torch.Tensor:
        """x_nhwc (B,192,256,3) normalised, query (16,512) fp32 -> codes (B,16,512) fp32 (+ latent_avg, models.py:318-325)"""
        b = x_nhwc.shape[0]
        c1, c2, c3 = self.backbone.forward(x_nhwc)
        p2 = conv1x1_any(self, c2, self.lat1, add=ops.upsample_bilinear2x(c3))
        p1 = conv1x1_any(self, c1, self.lat2, add=ops.upsample_bilinear2x(p2))
        tgt32 = query.reshape(1, self.n_query, 1, 512).expand(b, -1, -1, -1).contiguous()
        tgt_a = ops.cast(tgt32, self.adt) if self.bf16 else tgt32
        for t, mem in zip(self.layers, (c3, p2, p1)):
            tgt32, tgt_a = self._layer(tgt32, tgt_a, mem, t)
        return ops.codes_assemble(tgt32, False, False, self.latent_avg, b, self.n_query, 512)
