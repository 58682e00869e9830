"""torch.autograd bridge for the attack path.

The reference's attacks call `torch.autograd.grad(loss, [x])` / `loss.backward()` on `net(x)`
(/root/reference/src/attacks/untargeted.py:146,201,420,529,625,734); DeepFool and FAB back-propagate through the SAME
graph repeatedly with different output gradients (`retain_graph=True`, :529-535,622-627).  The whole defense call
is therefore ONE autograd node: forward runs the CUDA path while taping the few activations the input-gradient
needs, backward runs the dgrad-only reverse sweep.  The tape lives on the node's ctx and is never consumed, so
any number of backward calls work.  No parameter gradients exist (weights are frozen, callers never step them);
double backward is not supported (no caller needs it, SURVEY 8b).
"""
from __future__ import annotations

import torch

from . import ops


class _DefenseFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, batch, model):
        tape = Tape()
        with torch.no_grad():
            preds, purified = model._forward_cuda(batch.detach(), tape=tape)
        ctx.tape = tape
        ctx.model = model
        ctx.set_materialize_grads(False)
        return preds, purified

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, g_preds, g_purified):
        model, tape = ctx.model, ctx.tape
        eng = model.autoencoder
        g_cls = None
        if g_preds is not None:
            g_cls = model.classifier.classifier.backward(tape.vgg, g_preds.contiguous().to(torch.float32))
        g_pur = g_purified.contiguous().to(torch.float32) if g_purified is not None else None
        if g_cls is None and g_pur is None:
            return None, None
        g_x = eng.backward(tape.nvae, g_pur, g_cls)
        gx = ops.preprocess_bwd(g_x, tape.pre, bool(model.blur_input), normalize=True, taps_cache=model._taps_cache)
        return gx, None


class Tape:
    """what one forward call leaves behind for its backward passes"""

    def __init__(self):
        self.pre = None      # pre-clamp pre-processed image (NCHW fp32) for the clamp mask
        self.nvae = []       # records of NvaeEngine.purify
        self.vgg = []        # records of the classifier engine

    # the engines only `append` -- route by record kind
    def append(self, rec):
        (self.vgg if rec[0].startswith(("vgg_", "resnet")) else self.nvae).append(rec)


class CodesTape:
    """what `_StyleGanDefenseBase._from_codes_cuda` leaves behind: the generator's tape, the classifier's records, the mixing alphas"""

    def __init__(self):
        from .stylegan_engine import SynthesisTape
        self.syn = SynthesisTape()
        self.cls = []
        self.alphas = None


class _CodesFn(torch.autograd.Function):
    """`from_codes` of a StyleGAN defense as ONE node: W+ codes -> mix -> generator -> pool -> classifier.  Same contract as _DefenseFn:
    the forward tapes, the backward runs the dgrad-only reverse sweep and leaves the tape intact (repeated backward works)."""

    @staticmethod
    def forward(ctx, codes, model):
        tape = CodesTape()
        with torch.no_grad():
            preds, purified = model._from_codes_cuda(codes.detach(), tape=tape)
        ctx.tape, ctx.model = tape, model
        ctx.set_materialize_grads(False)
        return preds, purified

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, g_preds, g_purified):
        if g_preds is None and g_purified is None:
            return None, None
        return ctx.model._from_codes_backward(ctx.tape, g_preds, g_purified), None


def codes_apply(model, codes: torch.Tensor):
    """differentiable `_StyleGanDefenseBase.from_codes` body -> (preds, purified)"""
    return _CodesFn.apply(codes, model)


def defense_apply(model, batch: torch.Tensor):
    """differentiable `MLVGMDefenseModel.__call__` body -> (preds, purified)"""
    return _DefenseFn.apply(batch, model)


class _ClassifierFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, batch, wrapper):
        eng = wrapper.classifier
        tape = []
        with torch.no_grad():
            x = ops.nchw_to_nhwc(batch.detach().to(torch.float32), eng.adt, wrapper._norm_scale, wrapper._norm_shift)
            preds = eng.forward(x, tape=tape)
        ctx.tape, ctx.wrapper = tape, wrapper
        return preds

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, g_preds):
        eng = ctx.wrapper.classifier
        g = eng.backward(ctx.tape, g_preds.contiguous().to(torch.float32))           # (N,H,W,3) fp32, w.r.t. normalised input
        return g.permute(0, 3, 1, 2).contiguous() * ctx.wrapper._norm_scale, None


def classifier_apply(wrapper, batch: torch.Tensor):
    """differentiable `BaseClassificationModel.__call__`"""
    return _ClassifierFn.apply(batch, wrapper)


class _PreprocessFn(torch.autograd.Function):
    """blur / L2-normalised noise / clamp used ALONE (ablation defenses, `add_gaussian_noise`, `apply_gaussian_blur`), differentiable
    w.r.t. the batch like the reference's torch/kornia code (src/defenses/ablations/models.py:21-60, abstract_models.py:129-159):
    the noise is a constant, so the input gradient is the clamp mask followed by the transposed (= same symmetric, reflect-scatter) blur."""

    @staticmethod
    def forward(ctx, x, noise, eps, blur, seed, sample0, taps_cache):
        out, pre = ops.preprocess(x.detach().to(torch.float32), noise, float(eps), bool(blur), torch.float32, seed=seed, sample0=sample0,
                                  normalize=False, save_pre=True, taps_cache=taps_cache)
        ctx.pre, ctx.blur, ctx.taps_cache = pre, bool(blur), taps_cache
        return out.permute(0, 3, 1, 2).contiguous()

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, g):
        g_nhwc = g.to(torch.float32).permute(0, 2, 3, 1).contiguous()
        gx = ops.preprocess_bwd(g_nhwc, ctx.pre, ctx.blur, normalize=False, taps_cache=ctx.taps_cache)
        return gx, None, None, None, None, None, None


def preprocess_apply(x: torch.Tensor, noise, eps: float, blur: bool, seed: int, sample0: int, taps_cache=None) -> torch.Tensor:
    """(B,C,H,W) in [0,1] -> blurred / noised / clamped (B,C,H,W) fp32; differentiable w.r.t. x when x requires grad"""
    if x.requires_grad and torch.is_grad_enabled():
        return _PreprocessFn.apply(x, noise, eps, blur, seed, sample0, taps_cache)
    out, _ = ops.preprocess(x.detach().to(torch.float32), noise, float(eps), bool(blur), torch.float32, seed=seed, sample0=sample0,
                            normalize=False, taps_cache=taps_cache)
    return out.permute(0, 3, 1, 2).contiguous()
