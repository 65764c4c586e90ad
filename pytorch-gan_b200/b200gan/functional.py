"""Autograd nodes of the b200gan hot path.  Every forward/backward here is one or more calls into
libb200gan.so; torch only provides the tensors and the autograd tape.

Reference behaviour mirrored (file:line under implementations/):
  conv blocks        dcgan/dcgan.py:52-64, 77-88   pix2pix/models.py:20-52   cyclegan/models.py:22-87
  training-mode BN   dcgan/dcgan.py:53,56,60,80 (eps = 0.8)    InstanceNorm  pix2pix/models.py:25,40
"""
import weakref
from dataclasses import dataclass
from typing import Optional, Tuple

import torch

from . import ops
from ._lib import ConvGeom
from ._lib import (ACT_LRELU, ACT_NONE, ACT_RELU, ACT_SIGMOID, ACT_TANH, ALGO_AUTO, ALGO_SIMT, ALGO_TC, PACK_SIMT_DGRAD,
                   PACK_SIMT_FPROP, PACK_TC_DGRAD, PACK_TC_DGRAD_UP2, PACK_TC_FPROP, PACK_TC_FPROP_UP2, PAD_ZERO)


@dataclass(frozen=True)
class ConvSpec:
    stride: int = 1
    pads: Tuple[int, int, int, int] = (0, 0, 0, 0)  # top, left, bottom, right of the virtual input
    pad_mode: int = PAD_ZERO
    up: int = 1
    transposed: bool = False
    act: int = ACT_NONE
    slope: float = 0.0
    stats: Optional[bool] = None  # None: no fused statistics; False: per channel (BN); True: per sample (IN)
    rtf_out: bool = False         # round the output to TF32 (it feeds a tcgen05 conv)
    rtf_dz: bool = False          # round the epilogue-backward output (feeds tcgen05 dgrad/wgrad)


@dataclass(frozen=True)
class NormSpec:
    per_sample: bool = False
    eps: float = 1e-5
    momentum: float = 0.1
    act: int = ACT_NONE
    slope: float = 0.0
    rtf_out: bool = False
    rtf_dx: bool = False


class PackCache:
    """Derived packed copies of one weight Parameter, invalidated by the tensor version counter.  Caches register
    themselves per parameter so that an optimizer can refresh every packed copy of its weights in ONE launch right
    after the update (refresh_packs) instead of one pack launch per copy at the next forward."""

    registry = weakref.WeakValueDictionary()  # id(parameter storage) -> PackCache

    def __init__(self):
        self._d = {}

    def get(self, g, w, kind):
        key = (kind, g.C, g.K, g.R, g.S, g.transposed)
        ver = (w._version, w.data_ptr())
        hit = self._d.get(key)
        if ops.Config.weight_cache and hit is not None and hit[0] == ver:
            return hit[1]
        if hit is not None and hit[1].device == w.device:
            packed = hit[1]          # same buffer: a CUDA graph that captured it stays valid
            ops.pack_weights(g, w, kind, out=packed)
        else:
            packed = ops.pack_weights(g, w, kind)
        g_copy = ConvGeom.from_buffer_copy(g)
        self._d[key] = (ver, packed, g_copy)
        PackCache.registry[w.data_ptr()] = self
        return packed

    def jobs(self, w):
        """(geometry, kind, packed buffer) of every live copy, for ops.pack_weights_multi."""
        return [(e[2], key[0], e[1]) for key, e in self._d.items() if e[1].device == w.device]

    def mark_fresh(self, w):
        ver = (w._version, w.data_ptr())
        for key, e in list(self._d.items()):
            self._d[key] = (ver, e[1], e[2])


def refresh_packs(params):
    """Re-pack, in one launch, every cached packed copy of the given (just updated) weight tensors."""
    jobs, touched = [], []
    for w in params:
        cache = PackCache.registry.get(w.data_ptr())
        if cache is None:
            continue
        js = cache.jobs(w)
        if js:
            jobs.extend((g, kind, w, packed) for g, kind, packed in js)
            touched.append((cache, w))
    if jobs:
        ops.pack_weights_multi(jobs)
        for cache, w in touched:
            cache.mark_fresh(w)


def _pow2ceil(v):
    p = 1
    while p < v:
        p *= 2
    return p


def _tc_tile_is_one_image(g, spec):
    """True when a 128-pixel tile of the tcgen05 fprop never spans two images, the condition for fusing
    per-sample (InstanceNorm) sums into its epilogue (mirrors the tile choice in conv_tc.cu:run_tc)."""
    if spec.up == 2:
        ho, wo = g.H, g.W                 # per-phase grid of the upsample fold
    elif spec.transposed and spec.stride == 2:
        ho, wo = g.P // 2, g.Q // 2       # per-phase grid of the scatter form
    else:
        ho, wo = g.P, g.Q
    return min(_pow2ceil(wo), 128) * _pow2ceil(ho) >= 128


def _as_cl(t):
    return t if ops.is_cl(t) else ops.to_cl(t)


class ConvFn(torch.autograd.Function):
    """[Upsample x2] [pad] Conv2d/ConvTranspose2d [+bias] [act] [* Dropout2d scale] (+ BN/IN partial sums)."""

    @staticmethod
    def forward(ctx, x, weight, bias, chan_scale, spec: ConvSpec, cache: PackCache):
        ops._require_cuda(x, "conv input")
        ops._require_cuda(weight, "conv weight")
        ctx.in_nchw = not ops.is_cl(x)
        x = _as_cl(x)
        g, _ = ops.make_geom(tuple(x.shape), tuple(weight.shape), spec.stride, spec.pads, spec.pad_mode, spec.up,
                             spec.transposed)
        w = weight.detach()
        if ops.tc_supported(g, 0) and not (g.K < 32 and chan_scale is not None):
            algo = ALGO_TC
            packed = cache.get(g, w, PACK_TC_FPROP_UP2 if spec.up == 2 else PACK_TC_FPROP)
        else:
            algo = ALGO_SIMT
            packed = cache.get(g, w, PACK_SIMT_FPROP)
        stats = None
        if spec.stats is not None:
            stats = ops.zero_scratch(x.device, 2 * (g.N * g.K if spec.stats else g.K))
        fuse_stats = stats is not None and not (algo == ALGO_TC and spec.stats and not _tc_tile_is_one_image(g, spec))
        y = ops.conv_fprop(g, x, packed, algo, bias=None if bias is None else bias.detach(), act=spec.act,
                           slope=spec.slope, chan_scale=chan_scale, stats=stats if fuse_stats else None,
                           stats_per_sample=bool(spec.stats), round_tf32=spec.rtf_out)
        if stats is not None and not fuse_stats:
            stats = None  # caller computes them with a separate pass
        ctx.spec, ctx.cache, ctx.g = spec, cache, g
        ctx.has_bias = bias is not None
        need_y = spec.act != ACT_NONE
        ctx.save_for_backward(x, weight, y if need_y else None, chan_scale)
        if spec.stats is not None:
            if stats is None:
                stats = torch.empty(0, device=x.device, dtype=torch.float64)
            ctx.mark_non_differentiable(stats)
            return y, stats
        return y

    @staticmethod
    def backward(ctx, dy, *unused):
        if torch.is_grad_enabled():
            # autograd.grad(..., create_graph=True): the gradient penalty of a conv critic (stargan.py:142-161,
            # dragan.py:144-167) differentiates THROUGH this backward -- build it from differentiable nodes
            return _conv_backward_differentiable(ctx, dy)
        x, weight, y, chan_scale = ctx.saved_tensors
        spec, g = ctx.spec, ctx.g
        dy = _as_cl(dy)
        if spec.act != ACT_NONE or chan_scale is not None:
            dz = ops.epilogue_bwd(dy, y, chan_scale, spec.act, spec.slope, spec.rtf_dz)
        else:
            dz = dy
        dx = dw = db = None
        w = weight.detach()
        if ctx.needs_input_grad[0]:
            if ops.tc_supported(g, 1):
                packed = ctx.cache.get(g, w, PACK_TC_DGRAD_UP2 if spec.up == 2 else PACK_TC_DGRAD)
                dx = ops.conv_dgrad(g, dz, packed, ALGO_TC)
            else:
                packed = ctx.cache.get(g, w, PACK_SIMT_DGRAD)
                dx = ops.conv_dgrad(g, dz, packed, ALGO_SIMT)
        want_db = ctx.has_bias and ctx.needs_input_grad[2]
        if want_db and dz is not dy and spec.rtf_dz:
            # dz was rounded to TF32 for the tensor-core passes; a bias gradient is a sum with heavy cancellation
            # and must come from the unrounded values
            db = ops.bias_grad(dy, y, chan_scale, spec.act, spec.slope)
            want_db = False
        if ctx.needs_input_grad[1] or want_db:
            algo = ALGO_SIMT if ops.Config.algo == "simt" else ALGO_AUTO
            dw, db2 = ops.conv_wgrad(g, x, dz, tuple(weight.shape), want_db, algo)
            db = db2 if want_db else db
            if not ctx.needs_input_grad[1]:
                dw = None
        return dx, dw, db, None, None, None


# ---- double backward through convolutions (SURVEY.md 8f N2: conv-critic gradient penalties) ---------------------------
# conv is bilinear in (x, w): the backward of its backward needs no new kernels.  With F = fprop(x, w):
#   D = dgrad(dz, w)  (= dF/dx applied to dz):   dD/d(dz) applied to u = fprop(u, w),   dD/dw applied to u = wgrad(u, dz)
#   W = wgrad(x, dz)  (= dF/dw applied to dz):   dW/dx applied to v  = dgrad(dz, v),    dW/d(dz) applied to v = fprop(x, v)
def _plain_fprop(g, x, w):
    tc = ops.tc_supported(g, 0)
    kind = (PACK_TC_FPROP_UP2 if g.up == 2 else PACK_TC_FPROP) if tc else PACK_SIMT_FPROP
    if g.transposed and not tc:
        kind = PACK_SIMT_DGRAD
    return ops.conv_fprop(g, x, ops.pack_weights(g, w, kind), ALGO_TC if tc else ALGO_SIMT)


def _plain_dgrad(g, dz, w):
    tc = ops.tc_supported(g, 1)
    kind = (PACK_TC_DGRAD_UP2 if g.up == 2 else PACK_TC_DGRAD) if tc else PACK_SIMT_DGRAD
    if g.transposed and not tc:
        kind = PACK_SIMT_FPROP
    return ops.conv_dgrad(g, dz, ops.pack_weights(g, w, kind), ALGO_TC if tc else ALGO_SIMT)


def _plain_wgrad(g, x, dz, wshape):
    return ops.conv_wgrad(g, x, dz, wshape, False, ALGO_SIMT if ops.Config.algo == "simt" else ALGO_AUTO)[0]


class ConvDgradFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, dz, weight, g):
        ctx.g = g
        ctx.save_for_backward(dz, weight)
        return _plain_dgrad(g, _as_cl(dz.detach()), weight.detach())

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, u):
        dz, weight = ctx.saved_tensors
        g, u = ctx.g, _as_cl(u)
        ddz = _plain_fprop(g, u, weight.detach()) if ctx.needs_input_grad[0] else None
        dw = _plain_wgrad(g, u, _as_cl(dz.detach()), tuple(weight.shape)) if ctx.needs_input_grad[1] else None
        return ddz, dw, None


class ConvWgradFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, dz, g, wshape):
        ctx.g = g
        ctx.save_for_backward(x, dz)
        return _plain_wgrad(g, _as_cl(x.detach()), _as_cl(dz.detach()), wshape)

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, v):
        x, dz = ctx.saved_tensors
        g, v = ctx.g, v.contiguous()
        dx = _plain_dgrad(g, _as_cl(dz.detach()), v) if ctx.needs_input_grad[0] else None
        ddz = _plain_fprop(g, _as_cl(x.detach()), v) if ctx.needs_input_grad[1] else None
        return dx, ddz, None, None


def _conv_backward_differentiable(ctx, dy):
    x, weight, y, chan_scale = ctx.saved_tensors
    spec, g = ctx.spec, ctx.g
    if spec.up != 1 or spec.pad_mode != PAD_ZERO:
        raise NotImplementedError("b200gan: double backward through a conv with a folded upsample / reflection padding")
    dz = dy
    if spec.act == ACT_LRELU:
        dz = dz * torch.where(y > 0, 1.0, spec.slope)      # piecewise constant mask: no second-order term
    elif spec.act == ACT_RELU:
        dz = dz * (y > 0).to(dy.dtype)
    elif spec.act == ACT_TANH:
        dz = dz * (1 - y * y)                              # y is this node's (differentiable) output
    elif spec.act == ACT_SIGMOID:
        dz = dz * (y * (1 - y))
    if chan_scale is not None:
        dz = dz * chan_scale.view(chan_scale.shape[0], chan_scale.shape[1], 1, 1)
        if spec.act in (ACT_TANH, ACT_SIGMOID):
            raise NotImplementedError("b200gan: double backward through Dropout2d fused with tanh / sigmoid")
    dx = ConvDgradFn.apply(dz, weight, g) if ctx.needs_input_grad[0] else None
    if dx is not None and ctx.in_nchw:
        dx = ToContiguousFn.apply(dx)   # the layout of the input: a script may .view() its gradient (dualgan.py:130)
    dw = ConvWgradFn.apply(x, dz, g, tuple(weight.shape)) if ctx.needs_input_grad[1] else None
    db = dz.sum((0, 2, 3)) if (ctx.has_bias and ctx.needs_input_grad[2]) else None
    return dx, dw, db, None, None, None



class NormFn(torch.autograd.Function):
    """Training-mode BatchNorm2d / InstanceNorm2d with an optional fused activation."""

    @staticmethod
    def forward(ctx, x, gamma, beta, stats, running_mean, running_var, nbt, spec: NormSpec):
        ops._require_cuda(x, "norm input")
        x_in = x
        x = _as_cl(x)
        if stats is not None and stats.numel() == 0:
            stats = None
        y, mean_rstd, scale_shift = ops.norm_forward(
            x, None if gamma is None else gamma.detach(), None if beta is None else beta.detach(), running_mean,
            running_var, nbt, spec.per_sample, spec.eps, spec.momentum, spec.act, spec.slope, stats, spec.rtf_out,
            return_scale_shift=True)
        ctx.spec = spec
        # LeakyReLU / ReLU masks are recomputed from x in backward (sign of x * scale + shift): y need not be kept
        c_ = x.shape[1]
        mask_from_x = (ops.Config.norm_fast and spec.act in (ACT_LRELU, ACT_RELU) and c_ % 4 == 0 and c_ // 4 <= 256
                       and 256 % (c_ // 4) == 0)
        need_y = spec.act != ACT_NONE and not mask_from_x
        ctx.mask_from_x = mask_from_x
        ctx.x_is_input = x is x_in  # else the saved x has no autograd history (create_graph needs it)
        # scale_shift is always kept: the double backward recomputes the activation mask from it
        ctx.save_for_backward(x, y if need_y else None, mean_rstd, gamma, scale_shift)
        return y

    @staticmethod
    def backward(ctx, dy):
        x, y, mean_rstd, gamma, scale_shift = ctx.saved_tensors
        spec = ctx.spec
        if torch.is_grad_enabled():
            # autograd.grad(..., create_graph=True): the gradient penalty of a BatchNorm critic (dragan.py:144-167,
            # dualgan.py:116-135) differentiates THROUGH this backward
            if spec.per_sample:
                raise NotImplementedError("b200gan: double backward through InstanceNorm2d")
            if spec.act not in (ACT_NONE, ACT_LRELU, ACT_RELU):
                raise NotImplementedError("b200gan: double backward through a norm with a fused tanh / sigmoid")
            if not ctx.x_is_input:
                raise NotImplementedError("b200gan: double backward through a norm whose input was not channels_last")
            dx, dgamma, dbeta = NormBwdFn.apply(dy, x, gamma, y, mean_rstd, scale_shift, spec, ctx.mask_from_x)
            want_params = gamma is not None
            return (dx, dgamma if want_params and ctx.needs_input_grad[1] else None,
                    dbeta if want_params and ctx.needs_input_grad[2] else None, None, None, None, None, None)
        scale_shift = scale_shift if ctx.mask_from_x else None
        dy = _as_cl(dy)
        need_params = gamma is not None and (ctx.needs_input_grad[1] or ctx.needs_input_grad[2])
        dx, dgb = ops.norm_backward(dy, x, y, mean_rstd, None if gamma is None else gamma.detach(), spec.per_sample,
                                    spec.eps, spec.act, spec.slope, need_params, spec.rtf_dx, scale_shift)
        dgamma = dbeta = None
        if need_params:
            n, c = x.shape[0], x.shape[1]
            groups = dgb.numel() // 2
            dgamma, dbeta = dgb[:groups], dgb[groups:]
            if spec.per_sample:  # affine InstanceNorm2d: parameters are shared across samples
                dgamma, dbeta = dgamma.view(n, c).sum(0), dbeta.view(n, c).sum(0)
        return dx, dgamma, dbeta, None, None, None, None, None


class NormBwdFn(torch.autograd.Function):
    """The first-order backward of a training-mode BatchNorm2d [+ LeakyReLU / ReLU] as a differentiable node:
    (dy, x, gamma) -> (dx, dgamma, dbeta), with y / mean_rstd / scale_shift / spec as constants.  Forward is the same
    kernel as NormFn.backward (b200gan_norm_bwd); backward is b200gan_norm_bwd_bwd.  mask_from_x: the first-order kernel
    takes the activation mask from scale_shift (else from the saved output y), exactly as NormFn.backward chose."""

    @staticmethod
    def forward(ctx, dy, x, gamma, y, mean_rstd, scale_shift, spec: NormSpec, mask_from_x):
        x = _as_cl(x.detach())
        g = None if gamma is None else gamma.detach()
        dx, dgb = ops.norm_backward(_as_cl(dy.detach()), x, None if y is None else y.detach(), mean_rstd, g, False,
                                    spec.eps, spec.act, spec.slope, True, spec.rtf_dx,
                                    scale_shift if mask_from_x else None)
        c = x.shape[1]
        ctx.spec = spec
        ctx.set_materialize_grads(False)
        ctx.save_for_backward(dy, x, gamma, mean_rstd, scale_shift)
        return dx, dgb[:c].clone(), dgb[c:].clone()  # two outputs, not two views of one buffer

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, u, gg_gamma, gg_beta):
        dy, x, gamma, mean_rstd, scale_shift = ctx.saved_tensors
        spec = ctx.spec
        dy = _as_cl(dy)
        u = torch.zeros_like(dy, memory_format=ops.CL) if u is None else _as_cl(u)
        need_dgamma = gamma is not None and ctx.needs_input_grad[2]
        gx, gdy, dgamma = ops.norm_backward_backward(
            dy, x, u, mean_rstd, scale_shift, None if gamma is None else gamma.detach(),
            None if gg_gamma is None or gamma is None else gg_gamma.contiguous(),
            None if gg_beta is None or gamma is None else gg_beta.contiguous(), spec.eps, spec.act, spec.slope, need_dgamma)
        return gdy, gx, dgamma, None, None, None, None, None


@dataclass(frozen=True)
class TailSpec:
    eps: float = 1e-5
    momentum: float = 0.0
    act_mid: int = ACT_NONE
    slope: float = 0.0
    act_out: int = ACT_NONE
    rtf_dx: bool = False


class TailFn(torch.autograd.Function):
    """Training-mode BatchNorm2d -> LeakyReLU/ReLU -> Conv2d(C, K<=3, 3, 1, 1) [-> Tanh] on the raw output `a` of
    the preceding conv (dcgan.py:60-63), without materialising the normalised tensor or any gradient of it."""

    @staticmethod
    def forward(ctx, a, stats, gamma, beta, running_mean, running_var, nbt, weight, bias, spec: TailSpec):
        ops._require_cuda(a, "tail input")
        a = _as_cl(a)
        if stats is None or stats.numel() == 0:
            stats = ops.norm_stats(a, False)
        mean_rstd, scale_shift = ops.norm_finalize(
            tuple(a.shape), stats, None if gamma is None else gamma.detach(), None if beta is None else beta.detach(),
            running_mean, running_var, nbt, False, spec.eps, spec.momentum, a.device)
        d = ops.tail_desc(tuple(a.shape), weight.shape[0], spec.act_mid, spec.slope, spec.act_out)
        w = weight.detach().contiguous()
        out = ops.tail_fprop(d, a, scale_shift, w, None if bias is None else bias.detach())
        ctx.spec, ctx.d = spec, d
        ctx.has_affine, ctx.has_bias = gamma is not None, bias is not None
        ctx.save_for_backward(a, mean_rstd, scale_shift, weight, out if spec.act_out != ACT_NONE else None)
        return out

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, dout):
        a, mean_rstd, scale_shift, weight, out = ctx.saved_tensors
        spec = ctx.spec
        dout = _as_cl(dout)
        g = ops.epilogue_bwd(dout, out, None, spec.act_out, 0.0) if spec.act_out != ACT_NONE else dout
        need_affine = ctx.has_affine and (ctx.needs_input_grad[2] or ctx.needs_input_grad[3])
        need_bias = ctx.has_bias and ctx.needs_input_grad[8]
        da, dgb, dw, db = ops.tail_bwd(ctx.d, a, mean_rstd, scale_shift, weight.detach().contiguous(), g, need_affine,
                                       need_bias, spec.rtf_dx)
        c = a.shape[1]
        dgamma = dgb[:c] if need_affine else None
        dbeta = dgb[c:] if need_affine else None
        return da, None, dgamma, dbeta, None, None, None, dw, db, None


class AffineActFn(torch.autograd.Function):
    """y = act(x * scale[c] + shift[c]) with constant scale/shift: eval-mode BatchNorm2d."""

    @staticmethod
    def forward(ctx, x, scale_shift, act, slope):
        x = _as_cl(x)
        y = ops.norm_apply_affine(x, scale_shift, False, act, slope)
        ctx.act, ctx.slope = act, slope
        ctx.save_for_backward(y, scale_shift)
        return y

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, dy):
        y, scale_shift = ctx.saved_tensors
        dy = _as_cl(dy)
        dz = ops.epilogue_bwd(dy, y, None, ctx.act, ctx.slope) if ctx.act != ACT_NONE else dy
        c = y.shape[1]
        zero = torch.zeros_like(scale_shift)
        zero[:c] = scale_shift[:c]
        # dx = dz * scale: an affine apply with shift = 0
        return ops.norm_apply_affine(dz, zero, False), None, None, None


class ToChannelsLastFn(torch.autograd.Function):
    """Layout change NCHW -> NHWC.  Linear, so under create_graph=True (gradient penalties, SURVEY.md 8f N2) the
    backward is the opposite layout node rather than a detached copy."""

    @staticmethod
    def forward(ctx, x):
        return ops.to_cl(x)

    @staticmethod
    def backward(ctx, dy):
        if torch.is_grad_enabled() and dy.requires_grad:
            return ToContiguousFn.apply(dy)
        return ops.to_nchw(dy.detach())


class ToContiguousFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x):
        return ops.to_nchw(x)

    @staticmethod
    def backward(ctx, dy):
        if torch.is_grad_enabled() and dy.requires_grad:
            return dy if ops.is_cl(dy) else ToChannelsLastFn.apply(dy)
        return _as_cl(dy.detach())


class UpsampleFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x):
        return ops.upsample2x(_as_cl(x))

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, dy):
        return ops.upsample2x_bwd(_as_cl(dy))


class PadFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, pads, mode, round_tf32=False):
        ctx.pads, ctx.mode = pads, mode
        return ops.pad2d(_as_cl(x), pads, mode, round_tf32)

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, dy):
        return ops.pad2d_bwd(_as_cl(dy), ctx.pads, ctx.mode), None, None, None


class ActFn(torch.autograd.Function):
    """y = mask * act(x).  mask: None, per-(n,c) [N,C] (Dropout2d) or element-wise (Dropout)."""

    @staticmethod
    def forward(ctx, x, act, slope, mask, mask_per_channel):
        x = _as_cl(x)
        y = ops.act_forward(x, act, slope, mask, mask_per_channel)
        ctx.act, ctx.slope, ctx.mpc = act, slope, mask_per_channel
        ctx.save_for_backward(y if act != ACT_NONE else None, mask)
        return y

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, dy):
        y, mask = ctx.saved_tensors
        dy = _as_cl(dy)
        if mask is not None and not ctx.mpc:
            if ctx.act in (ACT_TANH, ACT_SIGMOID):
                raise NotImplementedError("b200gan: element-wise mask fused with tanh/sigmoid")
            dy = ops.act_forward(dy, ACT_NONE, 0.0, mask, False)
            mask = None
        if ctx.act == ACT_NONE and mask is None:
            return dy, None, None, None, None
        return ops.epilogue_bwd(dy, y, mask, ctx.act, ctx.slope), None, None, None, None


@dataclass(frozen=True)
class NbSpec:
    stride: int = 1
    pad: int = 0
    act: int = ACT_NONE
    slope: float = 0.0
    momentum: float = 0.0     # of the BatchNorm on the INPUT edge (its running statistics are updated by this conv)
    want_stats: bool = False  # a training-mode BatchNorm follows: produce the batch sums of the output
    groups: int = 1           # statistics groups of the batch (ops.bn_groups)


def _bn_edge_differentiable(a, gamma, beta, edge, want_xhat=True):
    """The BatchNorm of a chain edge as differentiable nodes, for a create_graph backward: the normalised tensor
    BN(a) (a NormFn of (a, gamma, beta); None unless want_xhat) and a function mapping a gradient w.r.t. BN(a) to
    (gradient w.r.t. the stored a, dgamma, dbeta) through NormBwdFn.  Both use the batch sums the forward kept in edge.stats; norm_finalize consumes
    (zeroes) the sums it is given, so each call gets a copy.  The running statistics are not touched (the forward
    already updated them once)."""
    if edge.groups > 1:
        raise NotImplementedError("b200gan: double backward through a grouped pass (ops.bn_groups)")
    spec = NormSpec(eps=edge.eps)
    xhat = NormFn.apply(a, gamma, beta, edge.stats.clone(), None, None, None, spec) if want_xhat else None
    mean_rstd, scale_shift = ops.norm_finalize(tuple(a.shape), edge.stats.clone(), edge.gamma, edge.beta, None, None,
                                               None, False, edge.eps, 0.0, a.device)

    def backward(g_xhat):
        return NormBwdFn.apply(g_xhat, a, gamma, None, mean_rstd, scale_shift, spec, True)

    return xhat, backward


class NbConvFn(torch.autograd.Function):
    """One layer of a fused narrow chain (csrc/narrow_block.cu): conv over the (virtually normalised) stored output of
    the previous layer, + bias, activation, Dropout2d scale, + the batch sums for the following BatchNorm.

    Chain protocol.  `in_edge` / `out_edge` are ops.BnEdge objects shared with the neighbouring layers.  In backward the
    incoming gradient is w.r.t. the VIRTUAL normalised output (the consumer could not finish the BatchNorm backward
    without the batch sums); by then the consumer has stored those sums in out_edge.sums.  This node finishes the norm
    backward (nb_dz), computes its parameter gradients, and hands ITS producer a virtual gradient plus in_edge.sums.
    Only valid when the stored output has exactly one consumer: the next node of the same chain."""

    @staticmethod
    def forward(ctx, x, weight, bias, chan_scale, in_gamma, in_beta, in_rm, in_rv, in_nbt, in_edge, out_box, spec, cache):
        ops._require_cuda(x, "conv input")
        ctx.in_nchw = not ops.is_cl(x)
        x = _as_cl(x)
        g, _ = ops.make_geom(tuple(x.shape), tuple(weight.shape), spec.stride, (spec.pad,) * 4)
        w = weight.detach()
        packed = cache.get(g, w, PACK_SIMT_FPROP)
        y, stats = ops.nb_fprop(g, x, packed, None if bias is None else bias.detach(), spec.act, spec.slope, chan_scale,
                                in_edge, in_rm, in_rv, in_nbt, spec.momentum, spec.want_stats, spec.groups)
        ctx.g, ctx.spec, ctx.cache, ctx.in_edge, ctx.out_box = g, spec, cache, in_edge, out_box
        ctx.has_bias = bias is not None
        ctx.save_for_backward(x, weight, y, chan_scale, in_gamma, in_beta)
        if spec.want_stats:
            ctx.mark_non_differentiable(stats)
            return y, stats
        return y

    @staticmethod
    def backward(ctx, gy, *unused):
        x, weight, y, chan_scale, in_gamma, in_beta = ctx.saved_tensors
        g, spec, in_edge = ctx.g, ctx.spec, ctx.in_edge
        out_edge = ctx.out_box[0] if ctx.out_box else None
        create_graph = torch.is_grad_enabled()
        # A chain that has been through a create_graph backward stays in the stored protocol for every later backward
        # (the penalty's .backward() reaches these forward nodes with gradients w.r.t. the stored tensors)
        stored = create_graph or any(e is not None and e.grad_of_stored for e in (in_edge, out_edge))
        if stored:
            # autograd.grad(..., create_graph=True) through a chain: the gradient penalty of a conv critic (SURVEY.md 8f
            # N2: stargan/models.py:87-115, and with BatchNorm dragan.py:144-167).  Same differentiable nodes as ConvFn;
            # across a BatchNorm edge every gradient is w.r.t. the STORED tensor (BnEdge.grad_of_stored).
            if spec.groups > 1:
                raise NotImplementedError("b200gan: double backward through a grouped pass (ops.bn_groups)")
            if out_edge is not None and not out_edge.grad_of_stored:
                raise RuntimeError("b200gan: fused conv chain: the consumer of this layer did not run its create_graph "
                                   "backward first")
            dz = gy
            if spec.act == ACT_LRELU:
                dz = dz * torch.where(y > 0, 1.0, spec.slope)
            elif spec.act == ACT_RELU:
                dz = dz * (y > 0).to(gy.dtype)
            if chan_scale is not None:
                dz = dz * chan_scale.view(chan_scale.shape[0], chan_scale.shape[1], 1, 1)
            xin = x
            if in_edge is not None:
                in_edge.grad_of_stored = True
                xin, norm_bwd = _bn_edge_differentiable(x, in_gamma, in_beta, in_edge, ctx.needs_input_grad[1])
            need_params = in_edge is not None and (ctx.needs_input_grad[4] or ctx.needs_input_grad[5])
            gx = dgamma = dbeta = None
            if ctx.needs_input_grad[0] or need_params:
                gx = ConvDgradFn.apply(dz, weight, g)
                if in_edge is not None:
                    gx, dgamma, dbeta = norm_bwd(gx)
                elif ctx.in_nchw:
                    gx = ToContiguousFn.apply(gx)
            dw = ConvWgradFn.apply(xin, dz, g, tuple(weight.shape)) if ctx.needs_input_grad[1] else None
            db = dz.sum((0, 2, 3)) if (ctx.has_bias and ctx.needs_input_grad[2]) else None
            return (gx, dw, db, None, dgamma if ctx.needs_input_grad[4] else None,
                    dbeta if ctx.needs_input_grad[5] else None) + (None,) * 7
        gy, y, x = gy.detach(), y.detach(), x.detach()
        if out_edge is not None and out_edge.sums is None:
            raise RuntimeError("b200gan: fused conv chain: the consumer of this layer did not run its backward first")
        gy = _as_cl(gy)
        want_db = ctx.has_bias and ctx.needs_input_grad[2]
        dz, db = ops.nb_dz(gy, y, chan_scale, spec.act, spec.slope, out_edge, want_db)
        dw = None
        if ctx.needs_input_grad[1]:
            dw = ops.nb_wgrad(g, x, dz, in_edge, tuple(weight.shape))
        gx = dgamma = dbeta = None
        need_in = ctx.needs_input_grad[0] or (in_edge is not None and (ctx.needs_input_grad[4] or ctx.needs_input_grad[5]))
        if need_in:
            packed = ctx.cache.get(g, weight.detach(), PACK_SIMT_DGRAD)
            gx, sums = ops.nb_dgrad(g, dz, packed, in_edge, x)
            if in_edge is not None:
                in_edge.sums = sums
                c = g.C
                if ctx.needs_input_grad[4] or ctx.needs_input_grad[5]:
                    # one conversion kernel for both parameter gradients (summed over the statistics groups)
                    dgb = sums.float() if in_edge.groups == 1 else sums.view(in_edge.groups, 2 * c).sum(0).float()
                    dgamma = dgb[c:] if ctx.needs_input_grad[4] else None
                    dbeta = dgb[:c] if ctx.needs_input_grad[5] else None
        return gx, dw, db, None, dgamma, dbeta, None, None, None, None, None, None, None


class NbTailFn(torch.autograd.Function):
    """End of a fused narrow chain: the last BatchNorm's output as a real tensor (optionally NCHW-contiguous: the layout
    the script's `.view(N, -1)` needs, dcgan.py:96)."""

    @staticmethod
    def forward(ctx, a, gamma, beta, rm, rv, nbt, edge, momentum, nchw):
        a = _as_cl(a)
        out = ops.nb_tail_fwd(a, edge, rm, rv, nbt, momentum, nchw)
        ctx.edge, ctx.nchw = edge, nchw
        ctx.save_for_backward(a, gamma, beta)
        return out

    @staticmethod
    def backward(ctx, dout):
        a, gamma, beta = ctx.saved_tensors
        if torch.is_grad_enabled() or ctx.edge.grad_of_stored:
            # create_graph=True (dragan.py:144-167), and every later backward of the same forward: the gradient handed
            # to the producer is w.r.t. the stored a
            ctx.edge.grad_of_stored = True
            if not ops.is_cl(dout):
                dout = ToChannelsLastFn.apply(dout.contiguous())
            _, norm_bwd = _bn_edge_differentiable(a, gamma, beta, ctx.edge, want_xhat=False)
            g, dgamma, dbeta = norm_bwd(dout)
            return (g, dgamma if ctx.needs_input_grad[1] else None, dbeta if ctx.needs_input_grad[2] else None,
                    None, None, None, None, None, None)
        dout = dout.contiguous() if ctx.nchw else _as_cl(dout)
        g, sums = ops.nb_tail_bwd(a, ctx.edge, dout, ctx.nchw)
        ctx.edge.sums = sums
        c = a.shape[1]
        dgamma = dbeta = None
        if ctx.needs_input_grad[1] or ctx.needs_input_grad[2]:
            grp = ctx.edge.groups
            dgb = sums.float() if grp == 1 else sums.view(grp, 2 * c).sum(0).float()
            dgamma = dgb[c:] if ctx.needs_input_grad[1] else None
            dbeta = dgb[:c] if ctx.needs_input_grad[2] else None
        return g, dgamma, dbeta, None, None, None, None, None, None


class _tf32_matmul:
    """cuBLAS TF32 for the GEMMs inside the block (a plain library GEMM: dcgan.py:50, Linear(100, 128 * 16 * 16))."""

    def __enter__(self):
        self.prev = torch.backends.cuda.matmul.allow_tf32
        torch.backends.cuda.matmul.allow_tf32 = True

    def __exit__(self, *exc):
        torch.backends.cuda.matmul.allow_tf32 = self.prev


class LinearWideFn(torch.autograd.Function):
    """nn.Linear with a wide output (the generator's first layer, dcgan.py:50: 0.84 GFLOP, 16.8 MB written) as TF32
    library GEMMs; torch's default for matmul is fp32 SIMT (30 us per GEMM here), while every convolution after it is
    TF32 anyway."""

    @staticmethod
    def forward(ctx, x, weight, bias):
        ctx.save_for_backward(x, weight)
        ctx.has_bias = bias is not None
        with _tf32_matmul():
            return torch.addmm(bias, x, weight.t()) if bias is not None else x @ weight.t()

    @staticmethod
    def backward(ctx, dy):
        x, weight = ctx.saved_tensors
        dx = dw = db = None
        with _tf32_matmul():
            if ctx.needs_input_grad[0]:
                dx = dy @ weight
            if ctx.needs_input_grad[1]:
                dw = dy.t() @ x
        if ctx.has_bias and ctx.needs_input_grad[2]:
            db = dy.sum(0)
        return dx, dw, db


class Linear1Fn(torch.autograd.Function):
    """nn.Linear(K, 1) [+ Sigmoid/Tanh/...] on a 2-D CUDA tensor: the discriminator head (dcgan.py:92)."""

    @staticmethod
    def forward(ctx, x, weight, bias, act):
        ops._require_cuda(x, "linear input")
        x = x.contiguous()
        y = ops.linear1_fwd(x, weight.detach().contiguous(), None if bias is None else bias.detach(), act)
        ctx.act, ctx.has_bias = act, bias is not None
        ctx.save_for_backward(x, weight, y)
        return y

    @staticmethod
    def backward(ctx, dy):
        x, weight, y = ctx.saved_tensors
        if torch.is_grad_enabled():  # create_graph=True: stay differentiable (plain torch ops on the saved tensors)
            if ctx.act == ACT_SIGMOID:
                dl = dy * y * (1 - y)
            elif ctx.act == ACT_TANH:
                dl = dy * (1 - y * y)
            else:
                dl = dy
            return dl @ weight, dl.t() @ x, (dl.sum(0) if ctx.has_bias else None), None
        dx, dw, db = ops.linear1_bwd(x, weight.detach().contiguous(), y, dy.contiguous(), ctx.act,
                                     ctx.needs_input_grad[0], ctx.has_bias and ctx.needs_input_grad[2])
        return dx, dw if ctx.needs_input_grad[1] else None, db, None


class BCEMeanFn(torch.autograd.Function):
    """torch.nn.BCELoss() (reduction 'mean') forward and backward as one kernel each (dcgan.py:103,166)."""

    @staticmethod
    def forward(ctx, v, t):
        v, t = v.contiguous(), t.contiguous()
        ctx.save_for_backward(v, t)
        return ops.bce_fwd(v, t)

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, gout):
        v, t = ctx.saved_tensors
        return ops.bce_bwd(v, t, gout.contiguous()), None


def conv_block(x, weight, bias, chan_scale, spec, cache):
    return ConvFn.apply(x, weight, bias, chan_scale, spec, cache)


def norm_block(x, gamma, beta, stats, running_mean, running_var, nbt, spec):
    return NormFn.apply(x, gamma, beta, stats, running_mean, running_var, nbt, spec)


class GradientPenaltyMLPFn(torch.autograd.Function):
    """lambda * mean((||dD/dx||_2 - 1)^2) for the MLP critic D = L3(lrelu(L2(lrelu(L1 x)))) with the
    gradient w.r.t. the weights produced in the same kernel (closed-form double backward)."""

    @staticmethod
    def forward(ctx, xi, w1, b1, w2, b2, w3, slope, lambda_gp):
        gp, dw1, dw2, dw3 = ops.gp_mlp_fwd_bwd(xi.detach(), w1.detach().contiguous(), b1.detach().contiguous(),
                                               w2.detach().contiguous(), b2.detach().contiguous(),
                                               w3.detach().contiguous(), slope, lambda_gp)
        ctx.save_for_backward(dw1, dw2, dw3)
        return gp

    @staticmethod
    def backward(ctx, g):
        dw1, dw2, dw3 = ctx.saved_tensors
        # the penalty does not depend on the biases; the interpolates are constants (.data in the reference)
        return None, g * dw1, None, g * dw2, None, g * dw3, None, None


def gradient_penalty_mlp(critic_layers, xi, lambda_gp):
    """critic_layers: the nn.Sequential(Linear, LeakyReLU, Linear, LeakyReLU, Linear) of wgan_gp.py:72-78."""
    mods = list(critic_layers)
    if not (len(mods) == 5 and all(isinstance(mods[i], torch.nn.Linear) for i in (0, 2, 4)) and
            all(isinstance(mods[i], torch.nn.LeakyReLU) for i in (1, 3)) and mods[4].out_features == 1 and
            mods[1].negative_slope == mods[3].negative_slope):
        raise NotImplementedError("b200gan: fused gradient penalty expects Linear-LReLU-Linear-LReLU-Linear(->1)")
    l1, l2, l3 = mods[0], mods[2], mods[4]
    return GradientPenaltyMLPFn.apply(xi, l1.weight, l1.bias, l2.weight, l2.bias, l3.weight, float(mods[1].negative_slope),
                                      float(lambda_gp))


class CriticStepMLPFn(torch.autograd.Function):
    """d_loss = -mean(D(real)) + mean(D(fake)) + lambda * gp(D, interpolates) of wgan_gp.py:164-171 for the MLP critic,
    with every parameter gradient produced by the same kernel (first-order backward + closed-form double backward)."""

    @staticmethod
    def forward(ctx, real, fake, alpha, w1, b1, w2, b2, w3, b3, slope, lambda_gp):
        out = ops.critic_step_mlp(real.detach(), fake.detach(), alpha, *[t.detach().contiguous() for t in
                                                                        (w1, b1, w2, b2, w3, b3)], slope, lambda_gp)
        losses, grads = out[0], out[1:]
        ctx.save_for_backward(*grads)
        ctx.mark_non_differentiable(losses[1:])
        return losses[0], losses[1]

    @staticmethod
    def backward(ctx, g, _g_gp):
        return (None, None, None) + tuple(g * t for t in ctx.saved_tensors) + (None, None)


def critic_step_mlp(critic_layers, real, fake, alpha, lambda_gp):
    """critic_layers: nn.Sequential(Linear, LeakyReLU, Linear, LeakyReLU, Linear(-> 1)) (wgan_gp.py:72-78).
    Returns (d_loss, lambda * gradient penalty); d_loss.backward() fills the gradients of all six parameters."""
    mods = list(critic_layers)
    if not (len(mods) == 5 and all(isinstance(mods[i], torch.nn.Linear) for i in (0, 2, 4)) and
            all(isinstance(mods[i], torch.nn.LeakyReLU) for i in (1, 3)) and mods[4].out_features == 1 and
            mods[1].negative_slope == mods[3].negative_slope and all(mods[i].bias is not None for i in (0, 2, 4))):
        raise NotImplementedError("b200gan: fused critic step expects Linear-LReLU-Linear-LReLU-Linear(->1) with biases")
    l1, l2, l3 = mods[0], mods[2], mods[4]
    return CriticStepMLPFn.apply(real, fake, alpha, l1.weight, l1.bias, l2.weight, l2.bias, l3.weight, l3.bias,
                                 float(mods[1].negative_slope), float(lambda_gp))
