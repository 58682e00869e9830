"""StyleGAN2 generator (decoder of the E4E / Style-Transformer purifiers) on the hand-written CUDA kernels.

Replaces `Generator.forward(..., input_is_latent=True, randomize_noise=False)` and `Generator.style`
(/root/reference/src/mlvgms_autoencoders/StyleGan_E4E/stylegan2/generator.py:294-479; SURVEY rows A14-A17).

Exact rewrites done at load (fp64):
  * equalised-lr scales folded into the weights (`EqualLinear`, generator.py:69-100; conv scale :154-155);
  * modulated conv = scale the input channels by the style s[b,ci]  ->  ONE shared-weight dense conv (tcgen05 kernel)
    ->  scale the output channels by demod[b,co] = rsqrt(sum_ci s^2 * sum_k W^2 + 1e-8)   (SURVEY App. D, 6e-15);
    the reference builds B x Cout x Cin x k x k weights and a grouped conv with groups = B (generator.py:163-207);
  * up-sampling StyledConv = conv_transpose2d(stride 2) followed by the 4x4 FIR blur (generator.py:180-191): both are
    linear with zero boundaries, so their composition is a stride-2 transposed conv with a 6x6 kernel, i.e. FOUR
    ordinary 3x3 convolutions (one per output sub-pixel phase) at the INPUT resolution on composed weights
    K_{py,px}[a,b] = G[py+2-2a, px+2-2b], G = W (*) blur.  They share their input, so they run as ONE tensor-core conv with 4 x Cout
    output channels (phase-major) and are interleaved by the fused epilogue kernel -- no zero-insertion, no (2H+1)^2 intermediate,
    no separate blur pass;
  * `noise + bias + leaky_relu * sqrt(2)` (NoiseInjection + FusedLeakyReLU, generator.py:210-268) and the demodulation
    scale are one kernel (`ga_styled_bias_act`, the `fused_bias_act` equivalent);
  * the mapping MLP runs ONCE on all n_codes x B rows (the reference loops over codes in Python, models.py:120,335).
"""
from __future__ import annotations

import math
from typing import Dict, Optional

import torch

from . import ops
from ._lib import ACT_NONE, ACT_LRELU_SQRT2
from .fold import Folder
from .synth import STYLEGAN_CHANNELS


def superpixel_weights(w: torch.Tensor) -> torch.Tensor:
    """3x3 / pad 1 conv weights [cout, cin, 3, 3] -> the weights [2 cout, 2 cin, 3, 3] of the SAME conv evaluated on pairs of horizontally
    adjacent pixels: an NHWC tensor [h][w][cin] is [h][w/2][2 cin] in memory (channel index = parity * cin + ci), output likewise.
    W'[(q,co)][ky][dX + 1][(p,ci)] = W[co][ky][2 dX + p - q + 1][ci], zero where the tap index leaves 0..2."""
    cout, cin = w.shape[0], w.shape[1]
    w2 = torch.zeros((2 * cout, 2 * cin, 3, 3), dtype=w.dtype)
    for q in range(2):
        for p_ in range(2):
            for dX in (-1, 0, 1):
                kx = 2 * dX + p_ - q + 1
                if 0 <= kx < 3:
                    w2[q * cout:(q + 1) * cout, p_ * cin:(p_ + 1) * cin, :, dX + 1] = w[:, :, :, kx]
    return w2


class _Styled:
    __slots__ = ("mod", "conv", "conv_sp", "phase_convs", "wsq", "noise", "noise_w", "bias", "up", "cin", "cout",
                 "mod_d", "conv_d", "conv_sp_d", "phase_d")


class _ToRGB:
    __slots__ = ("mod", "conv", "bias", "up_kernel", "mod_d", "up_kernel_d")


class SynthesisTape:
    """what `StyleGan2Engine.synthesis(..., tape=...)` leaves for `synthesis_backward`: the styles / demodulation factors of the whole
    batch, every styled layer's activation act(pre) per batch slice (as the forward produced it: fp32 up to `f32_conv_out_res`, the
    mode's activation dtype above) and the output slices in forward order"""

    def __init__(self):
        self.batch = 0
        self.n_codes = 0
        self.st = None
        self.acts = {}          # (id(layer), first sample of the slice) -> activation
        self.slices = []        # (first sample, size) of each output slice


class StyleGan2Engine:
    def __init__(self, state_dict: Dict[str, torch.Tensor], size: int, device, mode: str = "fp32", style_dim: int = 512,
                 n_mlp: int = 8, channel_multiplier: int = 2, lr_mlp: float = 0.01, _host_logic_test: bool = False):
        self.device = torch.device(device)
        if self.device.type != "cuda" and not _host_logic_test:
            raise RuntimeError("StyleGan2Engine runs only on CUDA devices: there is no CPU fallback")
        self.mode, self.bf16 = mode, mode == "bf16"
        self.adt = torch.bfloat16 if self.bf16 else torch.float32
        self.size, self.style_dim = size, style_dim
        self.log_size = int(math.log2(size))
        self.n_latent = self.log_size * 2 - 2
        ch = STYLEGAN_CHANNELS(channel_multiplier)
        f = Folder(state_dict, self.device, want_tc=self.bf16)
        sd = state_dict
        # ---- mapping network (generator.py:311-320)
        self.mapping_layers = []
        sc = (1.0 / math.sqrt(style_dim)) * lr_mlp
        for i in range(1, n_mlp + 1):
            w = f.f64(f"style.{i}.weight") * sc
            b = f.f64(f"style.{i}.bias") * lr_mlp
            L = f.conv(w.view(style_dim, style_dim, 1, 1), b, post_act=ACT_LRELU_SQRT2, name=f"style.{i}")
            L.w_tc = None          # the W+ codes steer every modulated conv: the 8-layer MLP stays fp32 in both modes (0.1% of the FLOPs)
            self.mapping_layers.append(L)
        # ---- synthesis
        self.const_input = f.dev32(f.f64("input.input")[0].permute(1, 2, 0).unsqueeze(0))          # [1,4,4,C]
        self.conv1 = self._fold_styled(f, "conv1", up=False)
        self.to_rgb1 = self._fold_rgb(f, "to_rgb1", up=False)
        self.blocks = []
        for j in range(self.log_size - 2):
            self.blocks.append((self._fold_styled(f, f"convs.{2 * j}", up=True), self._fold_styled(f, f"convs.{2 * j + 1}", up=False),
                                self._fold_rgb(f, f"to_rgbs.{j}", up=True)))
        num_layers = (self.log_size - 2) * 2 + 1
        self.noises = [f.dev32(f.f64(f"noises.noise_{i}")[0, 0]) for i in range(num_layers)]
        self._has_adjoint = False

    # ------------------------------------------------------------------ load-time folds
    def _fold_mod(self, f: Folder, prefix: str):
        w = f.f64(f"{prefix}.conv.modulation.weight") * (1.0 / math.sqrt(self.style_dim))           # lr_mul = 1
        b = f.f64(f"{prefix}.conv.modulation.bias")
        L = f.conv(w.view(w.shape[0], w.shape[1], 1, 1), b, name=prefix + ".modulation")
        L.w_tc = None                      # tiny GEMM; keep the style in fp32 (SIMT kernel) in both modes
        return L

    def _fold_styled(self, f: Folder, prefix: str, up: bool) -> _Styled:
        s = _Styled()
        w = f.f64(f"{prefix}.conv.weight")[0]                                                       # [cout, cin, 3, 3]
        cout, cin, k, _ = w.shape
        w = w * (1.0 / math.sqrt(cin * k * k))
        s.cin, s.cout, s.up = cin, cout, up
        s.mod = self._fold_mod(f, prefix)
        s.wsq = f.dev32((w ** 2).sum(dim=(2, 3)))                                                   # [cout, cin]
        s.conv, s.phase_convs = None, None
        s.conv_sp = None
        if not up:
            s.conv = f.conv(w, None, pad=1, name=prefix + ".conv")
            if self.bf16 and cin == 32 and cout % 4 == 0 and self.superpixel:
                # 32-channel layers (1024^2): the same conv on PAIRS of horizontally adjacent pixels -- [h][w][32] is [h][w/2][64] in memory --
                # with 64 -> 2*cout channels and block-sparse weights W'[(q,co)][ky][dX][(p,ci)] = W[co][ky][2 dX + p - q + 1][ci]
                # (zero outside 0..2).  Twice the multiply-adds, but 64-channel K blocks take the layer from the per-tap kernel
                # (1.3 TB/s, 186 TFLOP/s: bound by neither) to the persistent halo kernel.
                s.conv_sp = f.conv(superpixel_weights(w), None, pad=1, name=prefix + ".conv.superpixel", simt=False)
        else:
            kb = f.f64(f"{prefix}.conv.blur.kernel")                                                # 4x4, already x4
            G = torch.zeros((cout, cin, 6, 6), dtype=torch.float64)                                 # index d+2, d in [-2, 3]
            for dy in range(-2, 4):
                for dx in range(-2, 4):
                    for ty in range(4):
                        for tx in range(4):
                            ky, kx = dy + ty - 1, dx + tx - 1
                            if 0 <= ky < 3 and 0 <= kx < 3:
                                G[:, :, dy + 2, dx + 2] += kb[ty, tx] * w[:, :, ky, kx]
            Ks = []
            for py in range(2):
                for px in range(2):
                    K = torch.zeros((cout, cin, 3, 3), dtype=torch.float64)
                    for a in range(3):
                        for b in range(3):
                            K[:, :, a, b] = G[:, :, (py + 2 - 2 * a) + 2, (px + 2 - 2 * b) + 2]
                    Ks.append(K)
            # the four phase convs share their input: ONE conv with 4 * cout output channels (phase-major) reads it once
            s.phase_convs = f.conv(torch.cat(Ks, dim=0), None, pad=1, name=f"{prefix}.conv.phases")
        s.noise_w = float(f.f64(f"{prefix}.noise.weight")[0])
        s.bias = f.dev32(f.f64(f"{prefix}.activate.bias"))
        return s

    def _fold_rgb(self, f: Folder, prefix: str, up: bool) -> _ToRGB:
        r = _ToRGB()
        w = f.f64(f"{prefix}.conv.weight")[0]                                                       # [3, cin, 1, 1]
        cin = w.shape[1]
        w4 = torch.zeros((4, cin, 1, 1), dtype=torch.float64)                                       # RGB padded to 4 channels
        w4[:3] = w * (1.0 / math.sqrt(cin))
        r.mod = self._fold_mod(f, prefix)
        r.conv = f.conv(w4, None, name=prefix + ".conv")
        b4 = torch.zeros(4, dtype=torch.float64)
        b4[:3] = f.f64(f"{prefix}.bias").view(3)
        r.bias = f.dev32(b4)
        r.up_kernel = f.dev32(f.f64(f"{prefix}.upsample.kernel")) if up else None
        return r

    # ------------------------------------------------------------------ ops
    def _conv(self, x, L, want_f32=False, out=None):
        if self.bf16 and ops.conv2d_tc_supported(x, L):
            ob, of = ops.conv2d_tc(x, L, want_bf16=not want_f32, want_f32=want_f32, out_bf16=None if want_f32 else out,
                                   out_f32=out if want_f32 else None)
            return of if want_f32 else ob
        return ops.conv2d_simt(x, L, torch.float32 if (want_f32 or not self.bf16) else torch.bfloat16, out=out)

    def mapping(self, z: torch.Tensor) -> torch.Tensor:
        """z: (rows, style_dim) fp32 -> w: (rows, style_dim) fp32   [`Generator.style`, all codes in one batch]"""
        x = ops.pixelnorm(z.to(torch.float32), torch.float32)
        for L in self.mapping_layers:
            x = ops.conv2d_simt(x, L, torch.float32)
        return x.reshape(z.shape[0], self.style_dim)

    def _style(self, L, latent_i):
        """modulation EqualLinear (generator.py:164): (B, style_dim) -> (B, Cin) fp32"""
        b = latent_i.shape[0]
        return ops.conv2d_simt(latent_i.reshape(b, 1, 1, -1).contiguous(), L, torch.float32).reshape(b, -1)

    def _plan(self):
        """execution order: [(kind, layer, latent index)] -- conv1, to_rgb1, then (up conv, conv, to_rgb) per resolution"""
        plan = [("styled", self.conv1, 0), ("rgb", self.to_rgb1, 1)]
        i = 1
        for up, conv, rgb in self.blocks:
            plan += [("styled", up, i), ("styled", conv, i + 1), ("rgb", rgb, i + 2)]
            i += 2
        return plan

    def _styles(self, latent):
        """all modulation vectors s[b, cin] and demodulation factors of one call, for the WHOLE batch (one small GEMM per layer
        instead of one per layer per generator chunk)"""
        out = {}
        for kind, layer, idx in self._plan():
            st = self._style(layer.mod, latent[:, idx])
            out[id(layer)] = (st, ops.style_demod(st, layer.wsq) if kind == "styled" else None)
        return out

    def _styled(self, xs, s: _Styled, demod, noise, scale_next, scale_rgb, tape=None, key=None):
        """xs: input already scaled by this layer's style.  -> (act * scale_next | None, act * scale_rgb | None): the output is
        handed to its consumers pre-modulated (the fused epilogue kernel applies their style vectors on the fp32 value)"""
        # conv outputs at <= 128^2 stay fp32 until the fused epilogue (one bf16 rounding less per layer where it is almost free:
        # errors made in the early layers pass through every later one)
        b, h, w, _ = xs.shape
        f32 = self.bf16 and h * (2 if s.up else 1) <= self.f32_conv_out_res
        if not s.up:
            if s.conv_sp is not None and not f32 and xs.dtype == torch.bfloat16 and w % 2 == 0 and xs.is_contiguous():
                y = self._conv(xs.view(b, h, w // 2, 2 * s.cin), s.conv_sp).view(b, h, w, s.cout)
            else:
                y = self._conv(xs, s.conv, want_f32=f32)
            phases = False
        else:
            y = self._conv(xs, s.phase_convs, want_f32=f32)              # [b, h, w, 4 * cout]
            phases = True
        r = ops.styled_bias_act(y, phases, demod, noise, s.noise_w, s.bias, ACT_LRELU_SQRT2, None, self.adt, scale_a=scale_next,
                                scale_b=scale_rgb, want_out=scale_next is not None)
        if tape is not None:
            # the unmodulated activation for the backward: a second pass of the same epilogue, so the values handed to the consumers are
            # exactly those of an untaped forward
            tape.acts[(id(s), key)] = ops.styled_bias_act(y, phases, demod, noise, s.noise_w, s.bias, ACT_LRELU_SQRT2, None,
                                                          self._tape_dtype(h * (2 if s.up else 1)))
        return r if scale_rgb is not None else (r, None)

    def _tape_dtype(self, res: int):
        return torch.float32 if (not self.bf16 or res <= self.f32_conv_out_res) else self.adt

    fuse_rgb = __import__("os").environ.get("GA_SG_FUSE_RGB", "1") != "0"

    def _rgb(self, xs, r: _ToRGB, skip):
        if (self.fuse_rgb and self.bf16 and xs.dtype == torch.bfloat16 and r.conv.w_tc is not None and r.conv.w_tc.shape[0] == 4
                and xs.shape[3] % 8 == 0 and r.conv.w_tc.shape[1] == xs.shape[3]):
            # 1x1 conv to RGB + bias + up-sampled skip in one memory-bound pass (the tensor-core kernel ran this 4-column GEMM at 1.25 TB/s)
            return ops.torgb_fused(xs, r.conv, r.bias, skip, r.up_kernel if skip is not None else None)
        y = self._conv(xs, r.conv, want_f32=True)                                                   # [B,H,W,4] fp32
        # the half-resolution skip is up-sampled (Upsample, generator.py:30-47) inside the epilogue kernel
        return ops.styled_bias_act(y, False, None, None, 0.0, r.bias, ACT_NONE, skip, torch.float32,
                                   skip_up_kernel=r.up_kernel if skip is not None else None)

    def _cap(self, j: int) -> int:
        """largest batch slice block j (output resolution 8 * 2^j) runs on: keeps one activation tensor <= 2^29 elements (1 GB bf16)"""
        res = 8 << j
        cout = self.blocks[j][0].cout
        return max(1, (1 << 29) // (res * res * cout))

    def _run_blocks(self, j, x, skip, st, lo, sink, outs, tape=None):
        """blocks j.. on samples [lo, lo + n): low resolutions run on the whole batch, high resolutions on slices (recursive split)"""
        n = skip.shape[0]
        if j == len(self.blocks):
            if tape is not None:
                tape.slices.append((lo, n))
            outs.append(sink(skip) if sink is not None else skip)
            return
        cap = self.max_chunk or self._cap(j)
        if n > cap:
            for o in range(0, n, cap):
                self._run_blocks(j, x[o:o + cap], skip[o:o + cap], st, lo + o, sink, outs, tape)
            return
        up, conv, rgb = self.blocks[j]
        sl = slice(lo, lo + n)
        s_conv, d_conv = st[id(conv)]
        s_rgb, _ = st[id(rgb)]
        s_next = st[id(self.blocks[j + 1][0])][0][sl] if j + 1 < len(self.blocks) else None
        x, _ = self._styled(x, up, st[id(up)][1][sl], self.noises[2 * j + 1], s_conv[sl], None, tape, lo)
        x, xr = self._styled(x, conv, d_conv[sl], self.noises[2 * j + 2], s_next, s_rgb[sl], tape, lo)
        skip = self._rgb(xr, rgb, skip)
        self._run_blocks(j + 1, x, skip, st, lo, sink, outs, tape)

    max_chunk = None
    superpixel = __import__("os").environ.get("GA_SG_SUPERPIXEL", "1") != "0"
    f32_conv_out_res = int(__import__("os").environ.get("GA_SG_F32_RES", "128"))

    def synthesis(self, latent: torch.Tensor, sink=None, tape: Optional[SynthesisTape] = None):
        """latent: (B, >= n_latent, style_dim) fp32 -> list of RGB image slices NHWC (n_i, size, size, 4) fp32 in batch order (4th
        channel is padding), or of `sink(slice)` results when a sink is given (the caller pools each slice as soon as it exists).
        tape: a fresh `SynthesisTape` that records what `synthesis_backward` needs (the outputs do not change)."""
        b = latent.shape[0]
        assert latent.shape[1] >= self.n_latent, (latent.shape, self.n_latent)
        latent = latent.to(torch.float32)
        st = self._styles(latent)
        if tape is not None:
            tape.batch, tape.n_codes, tape.st = b, latent.shape[1], st
        s1, d1 = st[id(self.conv1)]
        x0 = ops.channel_scale(self.const_input.expand(b, -1, -1, -1).contiguous(), s1, self.adt)
        s_next = st[id(self.blocks[0][0])][0] if self.blocks else None
        x, xr = self._styled(x0, self.conv1, d1, self.noises[0], s_next, st[id(self.to_rgb1)][0], tape, 0)
        skip = self._rgb(xr, self.to_rgb1, None)
        outs = []
        self._run_blocks(0, x, skip, st, 0, sink, outs, tape)
        return outs

    # ------------------------------------------------------------------ input-gradient backward (W+ codes; weights frozen)
    def _build_adjoint(self):
        """flipped / transposed weights of every conv, folded in fp64 on the first backward (forward-only use pays nothing):
        3x3 convs -> their dgrad conv (the superpixel pair conv of the 32-channel layers -> superpixel_weights of the adjoint, which IS the
        adjoint of the pair conv), the up-sampling phase conv -> ONE 3x3 conv over the de-interleaved [h, w, 4 cout] gradient, modulation
        EqualLinears -> their transposes (fp32 SIMT), ToRGB skip up-sampling -> the flipped FIR (down 2)"""
        from .nvae_engine import make_dgrad_layer
        f = Folder({}, self.device, want_tc=self.bf16)
        f32 = Folder({}, self.device, want_tc=False)
        for kind, layer, _ in self._plan():
            layer.mod_d = make_dgrad_layer(f32, layer.mod, False)
            if kind == "rgb":
                layer.up_kernel_d = layer.up_kernel.flip(0, 1).contiguous() if layer.up_kernel is not None else None
                continue
            if layer.up:
                layer.phase_d = make_dgrad_layer(f, layer.phase_convs, self.bf16)
                layer.conv_d = layer.conv_sp_d = None
            else:
                layer.phase_d = None
                layer.conv_d = make_dgrad_layer(f, layer.conv, self.bf16)
                layer.conv_sp_d = None
                if layer.conv_sp is not None:
                    wt = layer.conv_d.w_simt.detach().to("cpu", torch.float64).view(3, 3, layer.cout, layer.cin).permute(3, 2, 0, 1)
                    layer.conv_sp_d = f.conv(superpixel_weights(wt), None, pad=1, name=layer.conv.name + ".dgrad.superpixel", simt=False)
        self._has_adjoint = True

    def _dgrad(self, s: _Styled, g, f32: bool):
        """gradient w.r.t. the layer's modulated input from the conv-output gradient g (de-interleaved phases for up-sampling layers)"""
        if s.up:
            return self._conv(g, s.phase_d, want_f32=f32)
        b, h, w, _ = g.shape
        if s.conv_sp_d is not None and not f32 and g.dtype == torch.bfloat16 and w % 2 == 0 and g.is_contiguous():
            return self._conv(g.view(b, h, w // 2, 2 * s.cout), s.conv_sp_d).view(b, h, w, s.cin)
        return self._conv(g, s.conv_d, want_f32=f32)

    def _layer_bwd(self, s: _Styled, tape, lo, n, g_next, nxt, rgb, g_rgb, noise, dots):
        """one styled layer on samples [lo, lo + n): epilogue adjoint (+ partial dots) then the conv's dgrad -> gradient w.r.t. its
        modulated input"""
        st, sl = tape.st, slice(lo, lo + n)
        v = tape.acts[(id(s), lo)]
        hw, c = v.shape[1] * v.shape[2], v.shape[3]
        f32 = not self.bf16 or v.shape[1] // (2 if s.up else 1) <= self.f32_conv_out_res
        g_y = ops.styled_bias_act_bwd(
            v, g_next, st[id(nxt)][0][sl] if nxt is not None else None, g_rgb, rgb.conv.w_simt if rgb is not None else None,
            st[id(rgb)][0][sl] if rgb is not None else None, st[id(s)][1][sl], noise, s.noise_w, s.bias, s.up,
            torch.bfloat16 if self.bf16 else torch.float32,
            dot_next=dots(nxt, "mod", hw, c)[sl] if nxt is not None else None,
            dot_rgb=dots(rgb, "mod", hw, c)[sl] if rgb is not None else None,
            dot_demod=dots(s, "demod", hw, c)[sl])
        return self._dgrad(s, g_y, f32)

    def _bwd_blocks(self, j, lo, n, tape, g_it, dots):
        """reverse of `_run_blocks` on samples [lo, lo + n) -> (gradient w.r.t. the modulated input of block j's up-sampling conv,
        gradient w.r.t. the RGB skip entering block j)"""
        if j == len(self.blocks):
            g = next(g_it)
            if tuple(g.shape) != (n, self.size, self.size, 4):
                raise ValueError(f"image gradient slice must have shape {(n, self.size, self.size, 4)}, got {tuple(g.shape)}")
            return None, g.to(torch.float32).contiguous()
        cap = self.max_chunk or self._cap(j)
        if n > cap:
            parts = [self._bwd_blocks(j, lo + o, min(cap, n - o), tape, g_it, dots) for o in range(0, n, cap)]
            return torch.cat([p[0] for p in parts], dim=0), torch.cat([p[1] for p in parts], dim=0)
        up, conv, rgb = self.blocks[j]
        nxt = self.blocks[j + 1][0] if j + 1 < len(self.blocks) else None
        g_next, g_skip = self._bwd_blocks(j + 1, lo, n, tape, g_it, dots)
        g_x = self._layer_bwd(conv, tape, lo, n, g_next, nxt, rgb, g_skip, self.noises[2 * j + 2], dots)
        g_x = self._layer_bwd(up, tape, lo, n, g_x, conv, None, None, self.noises[2 * j + 1], dots)
        # adjoint of the skip's Upsample (upfirdn2d up 2, pad (2, 1)): the flipped FIR, down 2, pad (1, 1)
        return g_x, ops.upfirdn2d(g_skip, rgb.up_kernel_d, up=1, down=2, pad=(1, 1))

    def synthesis_backward(self, tape: SynthesisTape, g_slices) -> torch.Tensor:
        """input gradient of `synthesis`: g_slices = gradients of the output image slices (n_i, size, size, 4) fp32 in the forward's slice
        order -> gradient w.r.t. the latent (B, n_codes, style_dim) fp32.  The tape is only read: any number of backward passes work."""
        if not self._has_adjoint:
            self._build_adjoint()
        b, st = tape.batch, tape.st
        bufs = {}

        def dots(layer, kind, hw, c):
            key = (id(layer), kind)
            if key not in bufs:
                bufs[key] = torch.empty((b, ops.styled_bias_act_bwd_parts(hw, c), c), device=self.device, dtype=torch.float32)
            return bufs[key]

        g_it = iter(g_slices)
        nxt = self.blocks[0][0] if self.blocks else None
        g_x, g_skip = self._bwd_blocks(0, 0, b, tape, g_it, dots)
        g_x = self._layer_bwd(self.conv1, tape, 0, b, g_x, nxt, self.to_rgb1, g_skip, self.noises[0], dots)
        # conv1's modulation acts on the constant input: its dot is the only thing left to form there
        const = self.const_input.expand(b, -1, -1, -1).contiguous()
        ops.styled_bias_act_bwd(const, g_x, None, None, None, None, None, None, 0.0, None, False, None, want_gy=False,
                                dot_next=dots(self.conv1, "mod", 16, const.shape[3]))
        g_lat = [None] * self.n_latent
        for kind, layer, idx in self._plan():
            s, demod = st[id(layer)]
            ds = ops.style_bwd(bufs[(id(layer), "mod")], bufs.get((id(layer), "demod")), s, demod, layer.wsq if kind == "styled" else None)
            # several layers share a latent index: the modulation EqualLinear's adjoint accumulates through the SIMT conv's add epilogue
            g_lat[idx] = ops.conv2d_simt(ds.view(b, 1, 1, -1), layer.mod_d, torch.float32, add=g_lat[idx])
        g = torch.cat([t.view(b, 1, self.style_dim) for t in g_lat], dim=1)
        if tape.n_codes > self.n_latent:
            g = torch.cat([g, g.new_zeros((b, tape.n_codes - self.n_latent, self.style_dim))], dim=1)
        return g

    def decode(self, latent: torch.Tensor, pool: int = 1, chunk: Optional[int] = None) -> torch.Tensor:
        """`pSp.decode` (psp.py:109-115): synthesis + face_pool (k x k mean) -> NCHW fp32 (B,3,size/pool,size/pool)."""
        if chunk is not None:
            self.max_chunk = chunk
        outs = self.synthesis(latent, sink=lambda img: ops.avgpool_to_nchw(img, pool, 3))
        return outs[0] if len(outs) == 1 else torch.cat(outs, dim=0)

    def mix_codes(self, codes: torch.Tensor, z_noise: torch.Tensor, alphas_dev: torch.Tensor) -> torch.Tensor:
        """per-level latent interpolation (models.py:117-127): styles = mapping(noise) for all n_codes x B rows at once;
        codes (B, n, d), z_noise (n, B, d) in the reference's draw layout (torch.normal(0,1,(n_codes,b,d)), models.py:119)"""
        b, n, d = codes.shape
        styles = self.mapping(z_noise.reshape(n * b, d)).reshape(n, b, d).permute(1, 0, 2).contiguous()
        return ops.latent_lerp(codes.to(torch.float32), styles, alphas_dev)
