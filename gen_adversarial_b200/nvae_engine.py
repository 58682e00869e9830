"""Host-side driver of the NVAE purification path on the hand-written CUDA kernels.

Mirrors `NVAEDefenseModel.purify` (/root/reference/src/defenses/ours/models.py:160-274) op for op, but on
folded weights (fold.py) and NHWC tensors, calling only entry points of libga_b200.so.

Two product modes:
  * "fp32": every tensor fp32, every convolution through the SIMT implicit-GEMM kernel (exact-arithmetic path,
            tolerance 1e-4 on purified images, identical accuracy counts);
  * "bf16": GEMM operands bf16, accumulation fp32, residual stream kept in fp32; convolutions through the
            tcgen05/TMEM/TMA kernel wherever the problem fits it (everything except the 3-channel stem and the
            stride-2 cells), tolerance 1e-2 on purified images.
"""
from __future__ import annotations

from typing import Dict, List, Optional, Sequence

import torch

from . import ops
from ._lib import PRE_NONE, PRE_ELU, PRE_SILU, PRE_AFFINE_SILU, ACT_NONE, ACT_SILU, ACT_ELU, ACT_RELU
from .fold import Folder, round_up
from .nvae_spec import NvaeSpec, EncCell, DecCell

_PRE_TO_ACT = {PRE_ELU: ACT_ELU, PRE_SILU: ACT_SILU, PRE_AFFINE_SILU: ACT_SILU}


def stride2_dgrad_phase_weights(w: torch.Tensor, pad: int) -> torch.Tensor:
    """w [cout, cin, k, k] of a stride-2 conv (3x3 pad 1, or 1x1 pad 0) -> weights [4*cin, cout, k, k] of the stride-1 conv over grad_out
    (same k and 'same' padding) whose output channels (2*pi + pj)*cin + c are the input gradient at pixels (2a + pi, 2b + pj).
    Forward: out[y] = sum_ky W[ky] in[2y + ky - pad]  =>  gin[2a + pi] = sum over (y, ky) with 2y + ky - pad = 2a + pi:
      3x3 pad 1: pi = 0 -> (y = a, ky = 1);  pi = 1 -> (y = a, ky = 2), (y = a + 1, ky = 0)        1x1 pad 0: pi = 0 -> (y = a, ky = 0)"""
    cout, cin, k, _ = w.shape
    if k == 3 and pad == 1:
        taps = {0: [(0, 1)], 1: [(0, 2), (1, 0)]}          # phase -> [(dy, ky)]
    elif k == 1 and pad == 0:
        taps = {0: [(0, 0)], 1: []}
    else:
        raise NotImplementedError(f"stride-2 dgrad phases for k={k} pad={pad}")
    wd = torch.zeros(4, cin, cout, k, k, dtype=w.dtype)
    c = k // 2
    for pi in (0, 1):
        for pj in (0, 1):
            for dy, ky in taps[pi]:
                for dx, kx in taps[pj]:
                    wd[2 * pi + pj, :, :, c + dy, c + dx] = w[:, :, ky, kx].t()
    return wd.reshape(4 * cin, cout, k, k)


def make_dgrad_layer(f: Folder, L: ops.ConvLayer, bf16: bool, pad_cin_to: Optional[int] = None,
                     in_scale: Optional[torch.Tensor] = None) -> ops.ConvLayer:
    """Input-gradient layer of the forward conv L (weights frozen: dgrad only): flipped taps, transposed channels; a stride-2 forward conv
    becomes an input-dilated (`up`) conv for the SIMT kernel and, in bf16 mode, ONE stride-1 tensor-core conv emitting the four output
    phases (`.phase`, see stride2_dgrad_phase_weights).  pad_cin_to: zero-pad the dgrad's input channels (= forward cout) to this many.
    in_scale: fp64 [cin], the scale of a per-channel affine applied to L's input BEFORE its zero padding (L's PRE_AFFINE); its adjoint
    scales the dgrad's output channels, folded into the weights here (exact: the padding follows the affine, so no border term exists)."""
    w = L.w_simt.detach().to("cpu", torch.float64).view(L.kh, L.kw, L.cin, L.cout).permute(3, 2, 0, 1)   # [cout,cin,kh,kw]
    if in_scale is not None:
        w = w * in_scale.to(torch.float64).view(1, -1, 1, 1)
    if pad_cin_to is not None and pad_cin_to > w.shape[0]:
        w = torch.cat([w, torch.zeros((pad_cin_to - w.shape[0],) + tuple(w.shape[1:]), dtype=w.dtype)], dim=0)
    wt = w.flip(2, 3).permute(1, 0, 2, 3).contiguous()           # [cin, cout(_pad), kh, kw]
    D = f.conv(wt, None, stride=1, pad=L.kh - 1 - L.pad, name=L.name + ".dgrad", up=L.stride)
    if bf16 and L.stride == 2 and w.shape[0] % 8 == 0 and L.cin % 4 == 0 and ((L.kh == 3 and L.pad == 1) or (L.kh == 1 and L.pad == 0)):
        P = f.conv(stride2_dgrad_phase_weights(w, L.pad), None, stride=1, pad=L.kh // 2, name=L.name + ".dgrad4", simt=False)
        D.phase = P if P.w_tc is not None else None
    return D


class _Enc:
    __slots__ = ("c1", "c2", "se", "skip", "down", "pre_affine", "c1_d", "c2_d", "skip_d")


class _Dec:
    __slots__ = ("e", "dw_w", "dw_wc", "dw_b", "p", "se", "skip", "up", "e_d", "p_d", "skip_d", "dw_wT", "dw_wTc")


class NvaeEngine:
    def __init__(self, state_dict: Dict[str, torch.Tensor], spec: NvaeSpec, device, mode: str = "fp32",
                 temperature: float = 0.6, _host_logic_test: bool = False):
        if mode not in ("fp32", "bf16"):
            raise ValueError(f"unknown mode {mode}")
        self.spec = spec
        self.device = torch.device(device)
        if self.device.type != "cuda" and not _host_logic_test:   # (tests/emu_ops.py drives the host logic on CPU)
            raise RuntimeError("NvaeEngine runs only on CUDA devices: there is no CPU fallback")
        self.mode = mode
        self.bf16 = mode == "bf16"
        self.adt = torch.bfloat16 if self.bf16 else torch.float32      # activation dtype
        self.temperature = float(temperature)
        self.zc = round_up(spec.z, 8)
        self.taps: Optional[dict] = None
        # fused decoder-cell kernel (expand -> dw5x5 -> project, hidden tensor on chip); GA_MBCONV_FUSED=0 selects the three-kernel path
        self.fuse_cells = __import__("os").environ.get("GA_MBCONV_FUSED", "1") != "0"
        self.fuse_csum = __import__("os").environ.get("GA_FUSE_CSUM", "1") != "0"     # SE channel sums from the encoder conv2 epilogue
        self.fuse_tape = __import__("os").environ.get("GA_FUSE_TAPE", "1") != "0"     # attack path: taping forward of the decoder cells in the fused kernel
        self.fuse_bwd = int(__import__("os").environ.get("GA_FUSE_BWD", "2"))         # attack path: backward of the decoder cells in the fused kernel
        # level tail (sampler -> latent mix -> combiner) in one kernel; tests/emu_ops.py emulates the unfused ops only
        self.fuse_level = __import__("os").environ.get("GA_FUSE_LEVEL", "1") != "0" and not _host_logic_test
        f = Folder(state_dict, self.device, want_tc=self.bf16)
        self._fold(f)
        self._prior_cache = {}
        self._has_dgrad = False

    # ------------------------------------------------------------------ weight preparation
    def _fold_enc(self, f: Folder, cell: EncCell) -> _Enc:
        p = cell.prefix
        e = _Enc()
        e.down = cell.down
        a1, b1 = f.bn(f"{p}.residual.0")
        w1, bias1 = f.wn(f"{p}.residual.2")
        a2, b2 = f.bn(f"{p}.residual.3")
        w1 = w1 * a2.view(-1, 1, 1, 1)
        bias1 = bias1 * a2 + b2
        e.pre_affine = (f.dev32(a1), f.dev32(b1))
        e.c1 = f.conv(w1, bias1, stride=2 if cell.down else 1, pad=1, pre_op=PRE_AFFINE_SILU, pre_affine=(a1, b1),
                      post_act=ACT_SILU, name=p + ".conv1")
        w2, bias2 = f.wn(f"{p}.residual.5")
        e.c2 = f.conv(w2, bias2, stride=1, pad=1, name=p + ".conv2")
        e.se = f.se(f"{p}.residual.6")
        e.skip = None
        if cell.down:
            ws, bs = f.wn(f"{p}.skip_connection.conv")
            e.skip = f.conv(ws, bs, stride=2, pad=0, pre_op=PRE_SILU, name=p + ".skip")
        return e

    def _fold_dec(self, f: Folder, cell: DecCell) -> _Dec:
        p, o = cell.prefix, cell.off
        d = _Dec()
        d.up = cell.up
        a0, b0 = f.bn(f"{p}.residual.{0 + o}")
        we = f.f64(f"{p}.residual.{1 + o}.weight")                   # [H, C, 1, 1]
        a1, b1 = f.bn(f"{p}.residual.{2 + o}")
        be = a1 * (we[:, :, 0, 0] @ b0) + b1
        we = we * a1.view(-1, 1, 1, 1) * a0.view(1, -1, 1, 1)
        d.e = f.conv(we, be, post_act=ACT_SILU, name=p + ".expand")
        wd = f.f64(f"{p}.residual.{4 + o}.weight")                   # [H, 1, 5, 5]
        a2, b2 = f.bn(f"{p}.residual.{5 + o}")
        wd = wd[:, 0] * a2.view(-1, 1, 1)
        d.dw_w = f.dev32(wd.permute(1, 2, 0).reshape(25, -1))        # [25][H]
        d.dw_wc = ops.dw_weights_chunked(d.dw_w) if d.dw_w.shape[1] % 64 == 0 else None     # chunk-major copy for the fused cell kernel
        d.dw_b = f.dev32(b2)
        wp = f.f64(f"{p}.residual.{7 + o}.weight")                   # [Cout, H, 1, 1]
        a3, b3 = f.bn(f"{p}.residual.{8 + o}")
        d.p = f.conv(wp * a3.view(-1, 1, 1, 1), b3, name=p + ".project")
        d.se = f.se(f"{p}.residual.{9 + o}")
        d.skip = None
        if cell.up:
            ws, bs = f.wn(f"{p}.skip_connection.conv")
            d.skip = f.conv(ws, bs, name=p + ".skip")
        return d

    @staticmethod
    def _nf_shift(f: Folder, cells, z: int) -> torch.Tensor:
        shift = torch.zeros(z, dtype=torch.float64)
        for q, _ in cells:
            w_last = f.f64(f"{q}.4.weight") * f.f64(f"{q}.4.mask")
            if float(w_last.abs().max()) != 0.0:
                raise NotImplementedError(f"NF cell {q}: the 1x1 conv has surviving taps (a mask the reference's MaskedConv2d cannot produce)")
            shift += f.f64(f"{q}.4.bias")
        return shift

    def _fold(self, f: Folder):
        spec = self.spec
        w, b = f.wn("preprocessing_block.init_conv")
        self.init_conv = f.conv(w, b, pad=1, name="init_conv")
        self.pre_cells = [self._fold_enc(f, c) for c in spec.pre_cells]
        self.enc_scales = []
        for sc in spec.enc_scales:
            groups = [[self._fold_enc(f, c) for c in grp] for grp in sc["groups"]]
            down = self._fold_enc(f, sc["down"]) if sc["down"] is not None else None
            self.enc_scales.append({"s": sc["s"], "groups": groups, "down": down})
        w, b = f.wn("encoder_0.1")
        self.enc0 = f.conv(w, b, pre_op=PRE_ELU, post_act=ACT_ELU, name="encoder_0")
        self.levels = []
        z = spec.z
        for lvl in spec.levels:
            L = {"s": lvl.s, "g": lvl.g, "res": lvl.res, "channels": lvl.channels}
            w, b = f.wn(f"enc_sampler.sampler_{lvl.s}:{lvl.g}")
            L["enc_sampler"] = f.conv(w[:z], b[:z], pad=1, name=f"enc_sampler_{lvl.s}:{lvl.g}")     # mu half only
            w, b = f.wn(f"decoder_combiners.combiner_{lvl.s}:{lvl.g}.conv")
            c = lvl.channels
            wx = w[:, :c]
            wz = torch.zeros((c, self.zc), dtype=torch.float64)
            wz[:, :z] = w[:, c:, 0, 0]
            if spec.use_nf:
                # normalizing-flow cells (architecture.py:221-253, applied at models.py:209-210,253-254): NFCell(z) = z - layers(z), and the
                # LAST layer of every cell is a MaskedConv2d 1x1 whose mask keeps (1*1)//2 = 0 taps (architecture.py:17-24): its weight is
                # all zero, layers(z) is that conv's bias, and a chain of cells subtracts a per-channel constant from z.  z only feeds
                # the decoder combiner's 1x1 conv, so the shift folds exactly into that conv's bias: b' = b - Wz . sum(bias_last).
                b = b - wz[:, :z] @ self._nf_shift(f, spec.nf_cells_of(lvl.s, lvl.g), z)
            L["dec_comb"] = f.conv(wx, b, name=f"dec_comb_{lvl.s}:{lvl.g}", w2=wz)
            L["dec_comb_z"] = f.conv(wz.view(c, self.zc, 1, 1), None, name=f"dec_comb_z_{lvl.s}:{lvl.g}")
            if not (lvl.s == 0 and lvl.g == 0):
                w, b = f.wn(f"encoder_combiners.combiner_{lvl.s}:{lvl.g}.conv")
                L["enc_comb"] = f.conv(w, b, name=f"enc_comb_{lvl.s}:{lvl.g}")
                w, b = f.wn(f"dec_sampler.sampler_{lvl.s}:{lvl.g}.1")
                L["dec_sampler"] = f.conv(w, b, pre_op=PRE_ELU, name=f"dec_sampler_{lvl.s}:{lvl.g}")
                L["cells"] = [self._fold_dec(f, c) for c in lvl.cells]
            else:
                # the constant prior goes through the x-half of combiner_0:0 once, at load (models.py:215-218)
                prior = f.f64("const_prior")                                        # [1, C, r, r]
                px = torch.einsum("oc,chw->hwo", wx[:, :, 0, 0], prior[0]) + b      # [r, r, C]
                L["prior_x"] = f.dev32(px.unsqueeze(0))
            self.levels.append(L)
        self.up_cells = {s: self._fold_dec(f, c) for s, c in spec.up_cells.items()}
        self.post_cells = [self._fold_dec(f, c) for c in spec.post_cells]
        w, b = f.wn("to_logits.1")
        self.to_logits = f.conv(w, b, pad=1, pre_op=PRE_ELU, name="to_logits")

    # ------------------------------------------------------------------ op dispatch
    def _tap(self, name, t):
        if self.taps is not None:
            self.taps[name] = t.detach().float().permute(0, 3, 1, 2).contiguous()

    def _conv(self, x, L: ops.ConvLayer, add=None, want_act=True, want_f32=False, x2=None, aux: ops.ConvLayer = None,
              mul=None, mul_mode=0, want_dact=False):
        """-> (out in activation dtype | None, out fp32 | None[, dact]).  fp32 mode: both outputs are the same tensor.
        out = (act(conv(pre(x)) + bias) + add) * f(mul);  dact = act'(pre-activation) (saved for the backward pass)."""
        dact = None
        if not self.bf16:
            if x2 is not None:
                add = ops.conv2d_simt(x2, aux, torch.float32, add=add)
            o = ops.conv2d_simt(x, L, torch.float32, add=add, mul=mul, mul_mode=mul_mode, want_dact=want_dact)
            if want_dact:
                o, dact = o
            return (o, o, dact) if want_dact else (o, o)
        xin = x
        if L.w_tc is not None:
            if L.pre_op != PRE_NONE:
                xin = ops.affine_act(x, L.pre_scale, L.pre_shift, _PRE_TO_ACT[L.pre_op], torch.bfloat16)
            elif x.dtype != torch.bfloat16:
                xin = ops.cast(x, torch.bfloat16)
            if ops.conv2d_tc_supported(xin, L, x2):
                if want_dact:
                    ho, wo = ops.conv_out_hw(L, xin.shape[1], xin.shape[2])
                    dact = torch.empty((xin.shape[0], ho, wo, L.cout), device=xin.device, dtype=torch.bfloat16)
                ob, of = ops.conv2d_tc(xin, L, want_bf16=want_act, want_f32=want_f32, add=add, x2=x2, mul=mul, mul_mode=mul_mode,
                                       dact_out=dact)
                return (ob, of, dact) if want_dact else (ob, of)
        # SIMT (3-channel stem, stride-2 cells, transposed convs, odd shapes): applies the pre-op itself
        if x2 is not None:
            add = ops.conv2d_simt(x2, aux, torch.float32, add=add)
        ob = of = None
        out_hw = None
        if L.up > 1:
            out_hw = (x.shape[1] * L.up, x.shape[2] * L.up)        # transposed conv: full-size output (output_padding)
        if want_act:
            ob = ops.conv2d_simt(x, L, torch.bfloat16, add=add, out_hw=out_hw, mul=mul, mul_mode=mul_mode, want_dact=want_dact)
            if want_dact:
                ob, dact = ob
        if want_f32:
            of = ops.conv2d_simt(x, L, torch.float32, add=add, out_hw=out_hw, mul=mul, mul_mode=mul_mode,
                                 want_dact=want_dact and dact is None)
            if want_dact and dact is None:
                of, dact = of
        return (ob, of, dact) if want_dact else (ob, of)

    def _conv_preact(self, x32, x_pre, L: ops.ConvLayer):
        """fp32 output of a layer with an ELU pre-op: from the pre-activated bf16 copy `x_pre` when one exists and the tensor-core kernel
        takes the shape, else the generic path (which materialises ELU(x32) itself)"""
        if x_pre is not None and L.w_tc is not None and L.pre_op == PRE_ELU and ops.conv2d_tc_supported(x_pre, L):
            return ops.conv2d_tc(x_pre, L, want_bf16=False, want_f32=True)[1]
        return self._conv(x32, L, want_act=False, want_f32=True)[1]

    def _dgrad(self, g, L: ops.ConvLayer, add=None, mul=None, mul_mode=0, f32=True):
        """input-gradient of the forward conv whose dgrad layer is L: -> fp32 (stream gradients) or activation dtype."""
        if not self.bf16:
            out_hw = (g.shape[1] * L.up, g.shape[2] * L.up) if L.up > 1 else None
            return ops.conv2d_simt(g, L, torch.float32, add=add, out_hw=out_hw, mul=mul, mul_mode=mul_mode)
        if L.phase is not None and f32 and mul is None:
            # stride-2 conv: the four output phases as one stride-1 tensor-core conv over g, then interleaved (the zero-stuffed
            # transposed conv ran on the SIMT kernel: 0.35-0.67 ms per launch at batch 128)
            _, o4 = self._conv(g, L.phase, want_act=False, want_f32=True)
            o = ops.depth_to_space2(o4)
            return o if add is None else ops.add(o, add, torch.float32)
        ob, of = self._conv(g, L, add=add, want_act=not f32, want_f32=f32, mul=mul, mul_mode=mul_mode)
        return of if f32 else ob

    # ------------------------------------------------------------------ forward pieces (each returns what backward needs)
    def _enc_cell(self, x32, act, e: _Enc, next_affine, rec):
        """x32: fp32 residual stream.  act: SiLU(BN1(x)) already materialised (bf16 mode) or None."""
        taping = rec is not None
        if self.bf16 and e.c1.w_tc is not None and act is not None and ops.conv2d_tc_supported(act, e.c1):
            dact1 = torch.empty(act.shape[:3] + (e.c1.cout,), device=act.device, dtype=torch.bfloat16) if taping else None
            h, _ = ops.conv2d_tc(act, e.c1, dact_out=dact1)
        elif taping:
            h, _, dact1 = self._conv(x32, e.c1, want_dact=True)
        else:
            h, _ = self._conv(x32, e.c1)
            dact1 = None
        sums = None
        if self.bf16 and self.fuse_csum and ops.conv2d_tc_csum_supported(h, e.c2):
            # SE squeeze fused into conv2's epilogue (persistent 3x3 kernel): per-image channel sums in the 128-pixel slices ga_channel_sum uses
            sums = torch.empty((h.shape[0], ops.channel_sum_parts(h.shape[0], h.shape[1] * h.shape[2]), e.c2.cout), device=h.device,
                               dtype=torch.float32)
            r, _ = ops.conv2d_tc(h, e.c2, csum_out=sums)
        else:
            r, _ = self._conv(h, e.c2)
        if e.down:
            _, skip = self._conv(x32, e.skip, want_act=False, want_f32=True)
        else:
            skip = x32
        if sums is None:
            sums = ops.channel_sum(r)
        out, _, act_next, _ = ops.se_residual(r, sums, e.se, 0.1, skip, torch.float32,
                                              act_affine=next_affine if self.bf16 else None)
        if taping:
            rec.append(("enc", e, x32, dact1, r, sums))
        return out, act_next

    def _enc_cell_bwd(self, g_out, rec):
        _, e, x32, dact1, r, sums = rec
        g_r = ops.se_residual_bwd(g_out, r, sums, e.se, 0.1, self.adt)
        g_v1 = self._dgrad(g_r, e.c2_d, mul=dact1, f32=False)                       # through conv2, times SiLU'(v1)
        g_a = self._dgrad(g_v1, e.c1_d, f32=True)                                   # w.r.t. SiLU(BN1(x))
        if e.down:
            g_s = self._dgrad(g_out, e.skip_d, f32=True)                            # w.r.t. SiLU(x)
            t = ops.affine_act_bwd(g_s, x32, None, None, ACT_SILU, torch.float32)
        else:
            t = g_out
        return ops.affine_act_bwd(g_a, x32, e.pre_affine[0], e.pre_affine[1], ACT_SILU, torch.float32, add=t)

    def _dec_cell(self, x32, xa, d: _Dec, rec, want_elu: bool = False):
        """x32: fp32 residual stream; xa: same values in the activation dtype (GEMM operand).
        want_elu (bf16 mode): the SE kernel also writes ELU(out) in bf16 -- the pre-activated input of the decoder sampler / logits head that
        follows this cell (NVAE/model.py:226-231,310-313) -- and it is left in `self._elu_copy` (saves a pass over the fp32 stream)."""
        taping = rec is not None
        elu = bool(want_elu and self.bf16)
        self._elu_copy = None
        fused_ok = self.fuse_cells and self.bf16 and not d.up and d.dw_wc is not None and ops.mbconv_fused_supported(xa, d.e, d.p)
        if taping and fused_ok and self.fuse_tape:
            # attack path: the same fused kernel also writes the two SiLU' tapes (hidden-sized, write-only) that `_dec_cell_bwd` multiplies by
            r, sums, dact_e, dact_dw = ops.mbconv_fused(xa, d.e, d.dw_wc, d.dw_b, d.p, want_sums=True, want_tape=True)
            out, out2, self._elu_copy, _ = ops.se_residual(r, sums, d.se, 0.1, x32, torch.float32, want_out2=True, act_plain=elu,
                                                           act_op=ACT_ELU if elu else ACT_SILU)
            rec.append(("dec", d, dact_e, dact_dw, r, sums))
            return out, out2
        if not taping and fused_ok:
            # expand -> dw5x5 -> project in one kernel, hidden tensor on chip; the SE squeeze comes out of its epilogue (GA_FUSE_CSUM)
            if self.fuse_csum:
                r, sums = ops.mbconv_fused(xa, d.e, d.dw_wc, d.dw_b, d.p, want_sums=True)
            else:
                r = ops.mbconv_fused(xa, d.e, d.dw_wc, d.dw_b, d.p)
                sums = ops.channel_sum(r)
            out, out2, self._elu_copy, _ = ops.se_residual(r, sums, d.se, 0.1, x32, torch.float32, want_out2=True, act_plain=elu,
                                                           act_op=ACT_ELU if elu else ACT_SILU)
            return out, out2
        if taping:
            h1, _, dact_e = self._conv(xa, d.e, want_dact=True)
            h2, dact_dw = ops.dwconv5x5(h1, d.dw_w, d.dw_b, ACT_SILU, d.up, self.adt, want_dact=True)
        else:
            h1, _ = self._conv(xa, d.e)                               # low resolution for up cells (exact commute)
            h2 = ops.dwconv5x5(h1, d.dw_w, d.dw_b, ACT_SILU, d.up, self.adt)
        r, _ = self._conv(h2, d.p)
        if d.up:
            _, s = self._conv(xa, d.skip, want_act=False, want_f32=True)
            skip = ops.upsample_bilinear2x(s)
        else:
            skip = x32
        sums = ops.channel_sum(r)
        out, out2, self._elu_copy, _ = ops.se_residual(r, sums, d.se, 0.1, skip, torch.float32, want_out2=self.bf16, act_plain=elu,
                                                       act_op=ACT_ELU if elu else ACT_SILU)
        if taping:
            rec.append(("dec", d, dact_e, dact_dw, r, sums))
        return out, (out2 if self.bf16 else out)

    def _dec_cell_bwd(self, g_out, rec):
        _, d, dact_e, dact_dw, r, sums = rec
        g_r = ops.se_residual_bwd(g_out, r, sums, d.se, 0.1, self.adt)
        # (isolated: 332 vs 431 us at 16x16, 197 vs 249 us at 8x8, but 779 vs 707 us at 32x32 -- the 4 halo rows make the first stage read 1.5x the
        #  tape, one 128-byte row load per thread; inside the attack iteration the fused kernel is no slower there either (118.2 vs 117.9 img/s) and
        #  saves two hidden-sized intermediates.  GA_FUSE_BWD=1 keeps the 32x32 cells on the three kernels, 0 all cells.)
        if (self.fuse_bwd and self.bf16 and not d.up and d.dw_wTc is not None and g_r.dtype == torch.bfloat16
                and (g_r.shape[2] <= 16 or self.fuse_bwd >= 2) and ops.mbconv_fused_supported(g_r, d.e, d.p)):
            # project^T -> x SiLU'(dw out) -> transposed depthwise -> x SiLU'(expand out) -> expand^T (+ skip gradient) in one kernel
            return ops.mbconv_fused_bwd(g_r, d.p_d, d.dw_wTc, dact_dw, dact_e, d.e_d, add=g_out)
        g_v2 = self._dgrad(g_r, d.p_d, mul=dact_dw, f32=False)                      # through project, times SiLU'(dw out)
        if d.up:
            g_h1 = ops.dwconv5x5(g_v2, d.dw_wT, None, ACT_NONE, False, self.adt)    # transposed depthwise (flipped taps)
            g_v1 = ops.sumpool2x2(g_h1, self.adt, mul=dact_e)                       # nearest-x2 backward, times SiLU'(expand out)
            g_s = ops.upsample_bilinear2x_bwd(g_out, torch.float32)
            t = self._dgrad(g_s, d.skip_d, f32=True)
        else:
            g_v1 = ops.dwconv5x5(g_v2, d.dw_wT, None, ACT_NONE, False, self.adt, mul=dact_e)
            t = g_out
        return self._dgrad(g_v1, d.e_d, add=t, f32=True)

    def _enc_sequence(self):
        """encoder cells in execution order with the stash / scale boundaries (models.py:176-192)."""
        seq = [("cell", e, None) for e in self.pre_cells]
        for sc in self.enc_scales:
            for g, grp in enumerate(sc["groups"]):
                for i, e in enumerate(grp):
                    stash = (sc["s"], g) if (i == len(grp) - 1 and not (sc["s"] == 0 and g == 0)) else None
                    seq.append(("cell", e, stash))
            if sc["down"] is not None:
                seq.append(("cell", sc["down"], None))
        return seq

    # ------------------------------------------------------------------ forward
    def purify(self, x_nhwc: torch.Tensor, alphas_dev: torch.Tensor, eps_levels: Optional[Sequence[torch.Tensor]] = None,
               seed: int = 0, sample0: int = 0, cls_dtype=None, tape=None):
        """x_nhwc: pre-processed, normalised input (N,H,W,3) in the activation dtype.
        alphas_dev: fp32 device tensor [n_latents] (already attenuated) -- read by the kernels at run time, so it
        can be changed between calls without re-capturing anything (alpha_learning/common_utils.py:88).
        eps_levels: explicit N(0,1) draws per level in NCHW (parity mode) or None (Philox in-kernel).
        tape: None, or a list that receives what `backward` needs (saved activations stay alive with it).
        -> (purified NCHW fp32 in [0,1], classifier input NHWC or None)"""
        spec = self.spec
        n = x_nhwc.shape[0]
        rec = tape
        if rec is not None and not self._has_dgrad:
            self._build_dgrad()
        x32 = ops.conv2d_simt(x_nhwc, self.init_conv, torch.float32)
        self._tap("init_conv", x32)
        seq = self._enc_sequence()
        stash = {}
        act = None
        for i, (_, e, st) in enumerate(seq):
            nxt = seq[i + 1][1].pre_affine if (i + 1 < len(seq) and not seq[i + 1][1].down) else None
            x32, act = self._enc_cell(x32, act, e, nxt, rec)
            if st is not None:
                stash[st] = x32
                if rec is not None:
                    rec.append(("stash", st))
            if i == len(self.pre_cells) - 1:
                self._tap("pre", x32)
        # encoder_0 (models.py:195)
        x32_top = x32
        xa, _ = self._conv(x32, self.enc0)
        self._tap("enc0", xa)
        lv0 = self.levels[0]
        _, muq = self._conv(xa, lv0["enc_sampler"], want_act=False, want_f32=True)
        eps0 = eps_levels[0] if eps_levels is not None else None
        z = ops.latent_mix(muq, None, eps0, seed, 0, sample0, alphas_dev[0:1], self.temperature, spec.z, self.zc, self.adt)
        self._tap("z0", z[..., :spec.z])
        key = (n,)
        if key not in self._prior_cache:
            self._prior_cache = {key: lv0["prior_x"].expand(n, -1, -1, -1).contiguous()}
        prior_x = self._prior_cache[key]
        if self.bf16:
            xa2, x32 = self._conv(z, lv0["dec_comb_z"], add=prior_x, want_act=True, want_f32=True)
        else:
            x32 = ops.conv2d_simt(z, lv0["dec_comb_z"], torch.float32, add=prior_x)
            xa2 = x32
        if rec is not None:
            rec.append(("level0", lv0, x32_top, xa, muq, alphas_dev[0:1]))
        xa = xa2
        idx = 1
        for s in range(spec.num_scales):
            for L in self.levels:
                if L["s"] != s or (L["s"] == 0 and L["g"] == 0):
                    continue
                x_elu = None
                for ci, d in enumerate(L["cells"]):
                    x32, xa = self._dec_cell(x32, xa, d, rec, want_elu=ci == len(L["cells"]) - 1)
                    x_elu = self._elu_copy
                comb, _ = self._conv(xa, L["enc_comb"], add=stash[(L["s"], L["g"])])
                _, muq = self._conv(comb, L["enc_sampler"], want_act=False, want_f32=True)
                eps = eps_levels[idx] if eps_levels is not None else None
                if (self.fuse_level and self.bf16 and self.taps is None
                        and ops.latent_level_supported(x_elu, xa, L["dec_sampler"], L["dec_comb"], spec.z)):
                    # prior sampler -> latent mix -> combiner in one kernel: pp and z stay on chip (pp is written only for the tape)
                    xa2, x32_2, pp = ops.latent_level(x_elu, xa, muq, eps, L["dec_sampler"], L["dec_comb"], seed, idx, sample0,
                                                      alphas_dev[idx:idx + 1], self.temperature, spec.z, want_pp=rec is not None)
                else:
                    pp = self._conv_preact(x32, x_elu, L["dec_sampler"])
                    z = ops.latent_mix(muq, pp, eps, seed, idx, sample0, alphas_dev[idx:idx + 1], self.temperature, spec.z, self.zc,
                                       self.adt)
                    self._tap(f"z{idx}", z[..., :spec.z])
                    xa2, x32_2 = self._conv(xa, L["dec_comb"], want_act=True, want_f32=True, x2=z, aux=L["dec_comb_z"])
                if rec is not None:
                    rec.append(("level", L, x32, muq, pp, eps, seed, idx, sample0, alphas_dev[idx:idx + 1]))
                xa, x32 = xa2, x32_2
                idx += 1
            if s in self.up_cells:
                x32, xa = self._dec_cell(x32, xa, self.up_cells[s], rec)
        self._tap("dec_out", x32)
        x_elu = None
        for ci, d in enumerate(self.post_cells):
            x32, xa = self._dec_cell(x32, xa, d, rec, want_elu=ci == len(self.post_cells) - 1)
            x_elu = self._elu_copy
        self._tap("post", x32)
        logits = self._conv_preact(x32, x_elu, self.to_logits)
        self._tap("logits", logits)
        if rec is not None:
            rec.append(("head", x32, logits))
        return ops.discmix_mean(logits, spec.num_mixtures, cls_dtype)

    # ------------------------------------------------------------------ backward (input gradient only)
    def _build_dgrad(self):
        """flipped / transposed weights of every conv on the path (built on first use: attacks only)."""
        from .fold import Folder
        f = Folder({}, self.device, want_tc=self.bf16)

        def dg(L: ops.ConvLayer, pad_cin_to=None):
            return make_dgrad_layer(f, L, self.bf16, pad_cin_to)

        for _, e, _ in self._enc_sequence():
            e.c1_d, e.c2_d = dg(e.c1), dg(e.c2)
            e.skip_d = dg(e.skip) if e.skip is not None else None
        decs = [d for L in self.levels for d in L.get("cells", [])] + list(self.up_cells.values()) + list(self.post_cells)
        for d in decs:
            d.e_d, d.p_d = dg(d.e), dg(d.p)
            d.skip_d = dg(d.skip) if d.skip is not None else None
            d.dw_wT = d.dw_w.flip(0).contiguous()                        # 5x5 taps reversed = spatial flip
            d.dw_wTc = ops.dw_weights_chunked(d.dw_wT) if (self.bf16 and d.dw_wc is not None) else None
        self.init_conv_d = dg(self.init_conv)
        self.enc0_d = dg(self.enc0)
        self.to_logits_d = dg(self.to_logits, pad_cin_to=round_up(self.to_logits.cout, 8))
        for L in self.levels:
            L["enc_sampler_d"] = dg(L["enc_sampler"], pad_cin_to=self.zc)
            L["dec_comb_x_d"] = dg(L["dec_comb"]) if "prior_x" not in L else None
            L["dec_comb_z_d"] = dg(L["dec_comb_z"])
            if "enc_comb" in L:
                L["enc_comb_d"] = dg(L["enc_comb"])
                L["dec_sampler_d"] = dg(L["dec_sampler"])
        self._has_dgrad = True

    def backward(self, tape, g_purified_nchw=None, g_cls=None):
        """Reverse sweep over `tape` (filled by `purify`).  g_purified_nchw: d loss / d purified (N,3,H,W) fp32 or None;
        g_cls: d loss / d classifier-input (N,H,W,3) or None.  -> d loss / d x_nhwc (N,H,W,3) fp32 (w.r.t. the
        normalised pre-processed input).  The tape is not consumed: backward may be called repeatedly with different
        output gradients (DeepFool / FAB, untargeted.py:529-535,622-627)."""
        spec = self.spec
        g = None                   # gradient w.r.t. the current stream tensor x32
        g_stash = {}
        for rec in reversed(tape):
            kind = rec[0]
            if kind == "head":
                _, x32, logits = rec
                g_logits = ops.discmix_mean_bwd(logits, spec.num_mixtures, g_purified_nchw, g_cls, pad_to=self.to_logits_d.cin)
                t = self._dgrad(g_logits, self.to_logits_d, f32=True)                 # w.r.t. ELU(x)
                g = ops.affine_act_bwd(t, x32, None, None, ACT_ELU, torch.float32)
            elif kind == "dec":
                g = self._dec_cell_bwd(g, rec)
            elif kind == "level":
                _, L, x32, muq, pp, eps, seed, idx, sample0, a_dev = rec
                g1 = self._dgrad(g, L["dec_comb_x_d"], f32=True)
                g_z = self._dgrad(g, L["dec_comb_z_d"], f32=True)
                g_q, g_p = ops.latent_mix_bwd(g_z, muq, pp, eps, seed, idx, sample0, a_dev, self.temperature, spec.z, self.zc)
                g_comb = self._dgrad(g_q, L["enc_sampler_d"], f32=True)
                g_stash[(L["s"], L["g"])] = g_comb                                    # encoder-side stash gets it as is
                g2 = self._dgrad(g_comb, L["enc_comb_d"], add=g1, f32=True)
                t = self._dgrad(g_p, L["dec_sampler_d"], f32=True)                    # w.r.t. ELU(x)
                g = ops.affine_act_bwd(t, x32, None, None, ACT_ELU, torch.float32, add=g2)
            elif kind == "level0":
                _, lv0, x32_top, xa, muq, a_dev = rec
                g_z = self._dgrad(g, lv0["dec_comb_z_d"], f32=True)
                g_q, _ = ops.latent_mix_bwd(g_z, muq, None, None, 0, 0, 0, a_dev, self.temperature, spec.z, self.zc)
                g_v = self._dgrad(g_q, lv0["enc_sampler_d"], mul=xa, mul_mode=2, f32=True)   # times ELU'(v) from y = ELU(v)
                t = self._dgrad(g_v, self.enc0_d, f32=True)                            # w.r.t. ELU(x_top)
                g = ops.affine_act_bwd(t, x32_top, None, None, ACT_ELU, torch.float32)
            elif kind == "stash":
                gs = g_stash.pop(rec[1], None)
                if gs is not None:
                    g = ops.add(g, gs, torch.float32)
            elif kind == "enc":
                g = self._enc_cell_bwd(g, rec)
            else:
                raise RuntimeError(f"unknown tape record {kind}")
        # 32 -> 3 channels at full resolution: tensor cores in bf16 mode (the SIMT conv took 2 ms per iteration at batch 512), SIMT in fp32 mode
        return self._dgrad(g, self.init_conv_d, f32=True)
