"""ResNet-50 / ResNeXt-50 (32x4d) + 4-layer head (the `gender` and `cars` classifiers) on the hand-written CUDA kernels.

Replaces `ResNet.forward` / `ResNext.forward` (/root/reference/src/classifier/model.py:10-28,53-70; bodies = torchvision
`resnet50` / `resnext50_32x4d`, head `Linear(2048,2048,bias=False)-BatchNorm1d-ReLU-Linear(2048,n_classes)`), SURVEY row A19.

Exact load-time rewrites (fp64): every eval BatchNorm folded into the conv / linear before it; the residual add and the
ReLU after it are the epilogue of the third 1x1 conv (`act_after_add`); the grouped 3x3 convs of ResNeXt (32 groups) are
expanded to block-diagonal dense weights so they run on the same implicit-GEMM kernels (zeros cost < 3% of the cars path's
FLOPs, SURVEY 8d) -- torchvision's stride-on-3x3 (v1.5) placement is kept.
"""
from __future__ import annotations

from typing import Dict

import torch

from . import ops
from ._lib import ACT_NONE, ACT_RELU, MUL_RELU_MASK
from .fold import Folder

LAYERS = (3, 4, 6, 3)


class _Block:
    __slots__ = ("c1", "c2", "c3", "down", "c1_d", "c2_d", "c3_d", "down_d")


def densify_grouped(w: torch.Tensor, groups: int) -> torch.Tensor:
    """[cout, cin/groups, kh, kw] grouped weights -> block-diagonal [cout, cin, kh, kw]"""
    if groups == 1:
        return w
    cout, cpg, kh, kw = w.shape
    opg = cout // groups
    dense = torch.zeros((cout, cpg * groups, kh, kw), dtype=w.dtype)
    for g in range(groups):
        dense[g * opg:(g + 1) * opg, g * cpg:(g + 1) * cpg] = w[g * opg:(g + 1) * opg]
    return dense


def conv_dgrad(g, D: ops.ConvLayer, bf16: bool, add=None, mul=None, f32: bool = False, mul_mode: int = MUL_RELU_MASK):
    """input gradient through one conv (D from make_dgrad_layer): (dgrad(g) + add) * f(mul), f the mul_mode derivative of the activation whose
    output `mul` is (MUL_PRELU_FROM_Y: D.act_slope holds that activation's slopes).  fp32 mode: SIMT fp32.  bf16 mode: tensor cores on a bf16
    copy of g where the shape tiles, SIMT elsewhere; the output is bf16, or fp32 with f32 (gradients that join the residual stream)."""
    if not bf16:
        out_hw = (g.shape[1] * D.up, g.shape[2] * D.up) if D.up > 1 else None
        return ops.conv2d_simt(g, D, torch.float32, add=add, out_hw=out_hw, mul=mul, mul_mode=mul_mode)
    if g.dtype != torch.bfloat16:
        g = ops.cast(g, torch.bfloat16)
    if D.phase is not None and ops.conv2d_tc_supported(g, D.phase):
        # stride-2 forward conv: the four output phases as one stride-1 tensor-core conv over g, interleaved, then add / mask
        _, o4 = ops.conv2d_tc(g, D.phase, want_bf16=False, want_f32=True)
        if mul_mode != MUL_RELU_MASK:                  # one fused pass (the ReLU-masked classifier path keeps its measured three passes)
            return ops.phase_interleave(o4, add, mul, mul_mode, D.act_slope, torch.float32 if f32 else torch.bfloat16)
        o = ops.depth_to_space2(o4)
        if add is not None:
            o = ops.add(o, add, torch.float32)
        if mul is not None:
            o = ops.affine_act_bwd(o, mul, None, None, ACT_RELU, torch.float32 if f32 else torch.bfloat16)
        return o
    if D.w_tc is not None and ops.conv2d_tc_supported(g, D):
        ob, of = ops.conv2d_tc(g, D, want_bf16=not f32, want_f32=f32, add=add, mul=mul, mul_mode=mul_mode)
        return of if f32 else ob
    out_hw = (g.shape[1] * D.up, g.shape[2] * D.up) if D.up > 1 else None
    return ops.conv2d_simt(g, D, torch.float32 if f32 else torch.bfloat16, add=add, out_hw=out_hw, mul=mul, mul_mode=mul_mode)


class ResNetEngine:
    def __init__(self, state_dict: Dict[str, torch.Tensor], device, mode: str = "fp32", groups: int = 1,
                 _host_logic_test: bool = False):
        self.device = torch.device(device)
        if self.device.type != "cuda" and not _host_logic_test:
            raise RuntimeError("ResNetEngine runs only on CUDA devices: there is no CPU fallback")
        self.mode, self.bf16 = mode, mode == "bf16"
        self.adt = torch.bfloat16 if self.bf16 else torch.float32
        sd = {(k[len("model."):] if k.startswith("model.") else k): v for k, v in state_dict.items()}
        f = Folder(sd, self.device, want_tc=self.bf16)

        def conv_bn(cw, bn, stride=1, pad=0, act=ACT_RELU, g=1, after_add=False):
            a, b = f.bn(bn)
            L = f.conv(densify_grouped(f.f64(cw + ".weight"), g) * a.view(-1, 1, 1, 1), b, stride=stride, pad=pad, post_act=act, name=cw)
            L.act_after_add = after_add
            return L

        self.stem = conv_bn("conv1", "bn1", stride=2, pad=3)
        self.blocks = []
        for li, n in enumerate(LAYERS, start=1):
            for bi in range(n):
                p = f"layer{li}.{bi}"
                stride = 2 if (li > 1 and bi == 0) else 1
                blk = _Block()
                blk.c1 = conv_bn(f"{p}.conv1", f"{p}.bn1")
                blk.c2 = conv_bn(f"{p}.conv2", f"{p}.bn2", stride=stride, pad=1, g=groups)
                blk.c3 = conv_bn(f"{p}.conv3", f"{p}.bn3", act=ACT_RELU, after_add=True)
                blk.down = conv_bn(f"{p}.downsample.0", f"{p}.downsample.1", stride=stride, act=ACT_NONE) \
                    if f"{p}.downsample.0.weight" in sd else None
                self.blocks.append(blk)
        a1, b1 = f.bn("fc.1")
        w0 = f.f64("fc.0.weight") * a1.view(-1, 1)
        self.fc0 = f.conv(w0.view(w0.shape[0], w0.shape[1], 1, 1), b1, post_act=ACT_RELU, name="fc.0")
        w3 = f.f64("fc.3.weight")
        self.fc1 = f.conv(w3.view(w3.shape[0], w3.shape[1], 1, 1), f.f64("fc.3.bias"), name="fc.3")
        self.n_classes = w3.shape[0]
        self._has_dgrad = False

    def _conv(self, x, L, want_f32=False, add=None):
        if self.bf16 and L.w_tc is not None and x.dtype == torch.bfloat16 and ops.conv2d_tc_supported(x, L):
            ob, of = ops.conv2d_tc(x, L, want_bf16=not want_f32, want_f32=want_f32, add=add)
            return of if want_f32 else ob
        return ops.conv2d_simt(x, L, torch.float32 if (want_f32 or not self.bf16) else torch.bfloat16, add=add)

    def forward(self, x_nhwc: torch.Tensor, tape=None) -> torch.Tensor:
        """x_nhwc (N,H,W,3) normalised with mean=std=0.5 (abstract_models.py:59-60) -> logits fp32 (N, classes).
        tape: None or a list receiving the activations the input-gradient needs (every ReLU output is also the next op's input: nothing is
        saved that the forward did not produce anyway)."""
        if tape is not None and not self._has_dgrad:
            self._build_dgrad()
        x_stem = ops.conv2d_simt(x_nhwc, self.stem, self.adt)
        x = ops.maxpool3x3s2(x_stem)
        recs = []
        for blk in self.blocks:
            idt = x if blk.down is None else self._conv(x, blk.down)
            h1 = self._conv(x, blk.c1)
            h2 = self._conv(h1, blk.c2)
            out = self._conv(h2, blk.c3, add=idt)
            if tape is not None:
                recs.append((blk, x, h1, h2, out))
            x = out
        n = x.shape[0]
        feat = ops.global_avgpool(x)
        h = self._conv(feat, self.fc0)
        logits = self._conv(h, self.fc1, want_f32=True)
        if tape is not None:
            tape.append(("resnet", x_nhwc.shape, x_stem, recs, h))
        return logits.reshape(n, self.n_classes)

    # ------------------------------------------------------------------ backward (input gradient only; SURVEY 8f rank 3)
    def _build_dgrad(self):
        """flipped / transposed weights of every conv (built on first use: attacks only)"""
        from .nvae_engine import make_dgrad_layer
        f = Folder({}, self.device, want_tc=self.bf16)
        dg = lambda L: make_dgrad_layer(f, L, self.bf16)
        for blk in self.blocks:
            blk.c1_d, blk.c2_d, blk.c3_d = dg(blk.c1), dg(blk.c2), dg(blk.c3)
            blk.down_d = dg(blk.down) if blk.down is not None else None
        self.stem_d = dg(self.stem)
        self.fc0_d, self.fc1_d = dg(self.fc0), dg(self.fc1)
        self._has_dgrad = True

    def _dg(self, g, D, add=None, mul=None, f32=False):
        """input gradient through one conv: (dgrad(g) + add) * [mul > 0]  (mul = the ReLU output that fed the forward conv)"""
        return conv_dgrad(g, D, self.bf16, add=add, mul=mul, f32=f32)

    def backward(self, tape, g_logits: torch.Tensor) -> torch.Tensor:
        """g_logits (N, classes) fp32 -> d loss / d x_nhwc (N,H,W,3) fp32.  `tape` = the list filled by forward(tape=...)."""
        (_, in_shape, x_stem, recs, h_fc), = [r for r in tape if r[0] == "resnet"]
        n = g_logits.shape[0]
        g = g_logits.contiguous().to(torch.float32).reshape(n, 1, 1, -1)
        g = self._dg(g, self.fc1_d, mul=h_fc)                       # times the ReLU mask of the hidden layer
        g = self._dg(g, self.fc0_d)                                  # w.r.t. the pooled features
        last = recs[-1][4]
        g = ops.avgpool_bwd_relu(g, last, self.adt)                  # average-pool backward x ReLU mask of the last block's output
        for i in range(len(recs) - 1, -1, -1):
            blk, x_in, h1, h2, _ = recs[i]
            # g: gradient at the block's pre-ReLU sum (the output's ReLU mask is already applied)
            g_h2 = self._dg(g, blk.c3_d, mul=h2)
            g_h1 = self._dg(g_h2, blk.c2_d, mul=h1)
            g_idt = g if blk.down is None else self._dg(g, blk.down_d, f32=True)
            # the block input is the previous block's ReLU output (mask applied here) or, for the first block, the pooled stem
            g = self._dg(g_h1, blk.c1_d, add=g_idt, mul=x_in if i > 0 else None)
        g = ops.maxpool3x3s2_bwd(x_stem, g, True, torch.float32)     # first maximum of every 3x3 window, times the stem's ReLU mask
        return ops.conv2d_simt(g, self.stem_d, torch.float32, out_hw=(in_shape[1], in_shape[2]))
