"""Tensor-level wrappers over the C ABI (include/b200gan.h).

Activations are torch tensors of logical shape [N, C, H, W] whose memory is NHWC
(`torch.channels_last`).  Nothing here differentiates; autograd lives in functional.py.
PyTorch is used for device memory (caching allocator), streams and tensor plumbing only.
"""
import ctypes
import os

import torch

from . import _lib
from ._lib import (ACT_NONE, ALGO_SIMT, ALGO_TC, PAD_REFLECT, PAD_ZERO, ConvGeom, Epilogue, GpMlpDesc, NbBn, NormDesc,
                   TailDesc)

CL = torch.channels_last


class Config:
    """Global switches. `algo`: 'auto' (tcgen05 where the geometry qualifies) or 'simt'."""
    algo = os.environ.get("B200GAN_ALGO", "auto")
    weight_cache = True
    # a fused Sequential fed an NCHW-contiguous tensor returns an NCHW-contiguous tensor (what a script may .view,
    # dcgan.py:96) only for feature maps of at most this many pixels; larger maps stay channels_last
    contiguous_hw_limit = 64
    # BatchNorm2d -> act -> Conv2d(C, K<=3, 3, 1, 1) -> act as the fused tail kernels (csrc/tail.cu)
    fuse_tail = os.environ.get("B200GAN_FUSE_TAIL", "1") not in ("", "0")
    # [Conv2d -> LeakyReLU -> Dropout2d -> BatchNorm2d] runs of narrow layers as the fused chain (csrc/narrow_block.cu)
    fuse_narrow_chain = os.environ.get("B200GAN_FUSE_CHAIN", "1") not in ("", "0")
    # train.dcgan_step: discriminator(real) and discriminator(fake) as ONE grouped pass through the fused chain
    batch_d_passes = os.environ.get("B200GAN_BATCH_D", "1") not in ("", "0")
    # norm kernels: fixed-channel-group fast paths (csrc/norm.cu) and activation mask recomputed from x in backward
    norm_fast = os.environ.get("B200GAN_NORM_FAST", "1") not in ("", "0")


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _ptr(t):
    return 0 if t is None else t.data_ptr()


def _require_cuda(t, name="tensor"):
    if not t.is_cuda:
        raise RuntimeError(f"b200gan: {name} is on {t.device}; the b200gan product path runs on CUDA only "
                           "(no CPU fallback)")
    if t.dtype != torch.float32:
        raise RuntimeError(f"b200gan: {name} has dtype {t.dtype}; fp32 expected")


def is_cl(x):
    return x.dim() == 4 and x.is_contiguous(memory_format=CL)


def empty_cl(n, c, h, w, device):
    return torch.empty((n, c, h, w), device=device, dtype=torch.float32, memory_format=CL)


def to_cl(x):
    """NCHW-contiguous -> NHWC memory (our transpose kernel); no-op if already channels_last."""
    _require_cuda(x, "input")
    if is_cl(x):
        return x
    if x.dim() == 4 and x.stride(1) == 1 and not x.is_contiguous():
        # channel-innermost but not dense: a channel slice of a channels_last tensor (the gradient of one input of
        # torch.cat(..., 1), pix2pix/models.py:50,132).  One strided copy, coalesced along C -- not a round trip
        # through NCHW.
        y = empty_cl(*x.shape, x.device)
        y.copy_(x)
        return y
    if not x.is_contiguous():
        x = x.contiguous()
    n, c, h, w = x.shape
    y = empty_cl(n, c, h, w, x.device)
    if x.numel() == 0:
        return y
    _lib.check(_lib.load().b200gan_nchw_to_nhwc(x.data_ptr(), y.data_ptr(), n, c, h * w, _stream()), "nchw_to_nhwc")
    return y


def to_nchw(x):
    """NHWC memory -> NCHW-contiguous tensor (needed where scripts call .view, dcgan.py:96)."""
    _require_cuda(x, "input")
    if x.is_contiguous():
        return x
    if not is_cl(x):
        return x.contiguous()
    n, c, h, w = x.shape
    y = torch.empty((n, c, h, w), device=x.device, dtype=torch.float32)
    if x.numel() == 0:
        return y
    _lib.check(_lib.load().b200gan_nhwc_to_nchw(x.data_ptr(), y.data_ptr(), n, c, h * w, _stream()), "nhwc_to_nchw")
    return y


# ---- convolution -------------------------------------------------------------------------------
def make_geom(x_shape, weight_shape, stride, pads, pad_mode=PAD_ZERO, up=1, transposed=False):
    """pads = (top, left, bottom, right) of the virtual input. Returns (ConvGeom, out_shape)."""
    n, c, h, w = x_shape
    g = ConvGeom()
    g.N, g.H, g.W, g.C = n, h, w, c
    if transposed:
        cin, cout, r, s = weight_shape
    else:
        cout, cin, r, s = weight_shape
    if cin != c:
        raise RuntimeError(f"b200gan conv: input has {c} channels, weight expects {cin}")
    g.K, g.R, g.S, g.stride = cout, r, s, stride
    g.pad_t, g.pad_l, g.pad_b, g.pad_r = pads
    g.pad_mode, g.up, g.transposed = pad_mode, up, int(transposed)
    if transposed:
        g.P = (h - 1) * stride - 2 * pads[0] + r
        g.Q = (w - 1) * stride - 2 * pads[1] + s
    else:
        g.P = (h * up + pads[0] + pads[2] - r) // stride + 1
        g.Q = (w * up + pads[1] + pads[3] - s) // stride + 1
    return g, (n, cout, g.P, g.Q)


def tc_supported(g, pas):
    if Config.algo == "simt":
        return False
    return bool(_lib.load().b200gan_conv2d_supported(ctypes.byref(g), pas, ALGO_TC))


def pack_weights(g, w, kind, out=None):
    lib = _lib.load()
    if out is None:
        n = lib.b200gan_packed_weight_floats(ctypes.byref(g), kind)
        out = torch.empty(n, device=w.device, dtype=torch.float32)
    _lib.check(lib.b200gan_pack_weights(ctypes.byref(g), kind, w.data_ptr(), out.data_ptr(), _stream()), "pack_weights")
    return out


def pack_weights_multi(jobs):
    """jobs: [(ConvGeom, kind, weight tensor, packed buffer)] -- one launch for all of them."""
    table = (_lib.PackJob * len(jobs))()
    for i, (g, kind, w, packed) in enumerate(jobs):
        table[i].w, table[i].packed, table[i].geom, table[i].pack = w.data_ptr(), packed.data_ptr(), g, kind
    _lib.check(_lib.load().b200gan_pack_weights_multi(table, len(jobs), _stream()), "pack_weights_multi")


def conv_fprop(g, x, packed, algo, bias=None, act=ACT_NONE, slope=0.0, chan_scale=None, stats=None,
               stats_per_sample=False, round_tf32=False):
    y = empty_cl(g.N, g.K, g.P, g.Q, x.device)
    if g.N == 0:
        return y
    ep = Epilogue()
    ep.bias, ep.act, ep.slope = _ptr(bias), act, slope
    ep.chan_scale, ep.stats = _ptr(chan_scale), _ptr(stats)
    ep.stats_per_sample, ep.round_tf32 = int(stats_per_sample), int(round_tf32)
    _lib.check(_lib.load().b200gan_conv2d_fprop(ctypes.byref(g), ctypes.byref(ep), x.data_ptr(), packed.data_ptr(),
                                                y.data_ptr(), algo, _stream()), "conv2d_fprop")
    return y


def conv_dgrad(g, dy, packed, algo):
    lib = _lib.load()
    dx = empty_cl(g.N, g.C, g.H, g.W, dy.device)
    nws = lib.b200gan_conv2d_dgrad_workspace_floats(ctypes.byref(g), algo)
    ws = torch.empty(nws, device=dy.device, dtype=torch.float32) if nws else None
    _lib.check(lib.b200gan_conv2d_dgrad(ctypes.byref(g), dy.data_ptr(), packed.data_ptr(), dx.data_ptr(), _ptr(ws),
                                        algo, _stream()), "conv2d_dgrad")
    return dx


def conv_wgrad(g, x, dy, weight_shape, need_bias, algo):
    lib = _lib.load()
    dw = torch.empty(weight_shape, device=x.device, dtype=torch.float32)
    db = torch.empty(g.K, device=x.device, dtype=torch.float32) if need_bias else None
    nws = lib.b200gan_conv2d_wgrad_workspace_floats(ctypes.byref(g), algo)
    ws = torch.empty(nws, device=x.device, dtype=torch.float32) if nws else None
    _lib.check(lib.b200gan_conv2d_wgrad(ctypes.byref(g), x.data_ptr(), dy.data_ptr(), dw.data_ptr(), _ptr(db),
                                        _ptr(ws), algo, _stream()), "conv2d_wgrad")
    return dw, db


def epilogue_bwd(dy, y, chan_scale, act, slope, round_tf32=False):
    n, k, p, q = dy.shape
    dz = torch.empty_like(dy, memory_format=CL)
    _lib.check(_lib.load().b200gan_epilogue_bwd(dy.data_ptr(), _ptr(y), _ptr(chan_scale), act, slope, dy.numel(), k,
                                                p * q, int(round_tf32), dz.data_ptr(), _stream()), "epilogue_bwd")
    return dz


def bias_grad(dy, y, chan_scale, act, slope):
    """Bias gradient of a fused conv block from unrounded values (see include/b200gan.h)."""
    n, k, p, q = dy.shape
    db = torch.empty(k, device=dy.device, dtype=torch.float32)
    _lib.check(_lib.load().b200gan_bias_grad(dy.data_ptr(), _ptr(y), _ptr(chan_scale), act, slope, n * p * q, k, p * q,
                                             db.data_ptr(), _stream()), "bias_grad")
    return db


# ---- normalisation -----------------------------------------------------------------------------
def _norm_desc(x, per_sample, eps, momentum, act, slope, round_tf32):
    n, c, h, w = x.shape
    d = NormDesc()
    d.N, d.HW, d.C, d.per_sample = n, h * w, c, int(per_sample)
    d.eps, d.momentum, d.act, d.slope, d.round_tf32 = eps, momentum, act, slope, int(round_tf32)
    return d


_zero_scratch = {}


def zero_scratch(device, numel):
    """Persistent fp64 accumulator that is zero whenever it is handed out: every kernel that consumes it
    (norm_finalize, norm_bwd) zeroes it again, so no fill kernel is launched per use.  One buffer per
    (device, size) suffices because producer -> consumer pairs never interleave on the stream."""
    key = (device, numel)
    t = _zero_scratch.get(key)
    if t is None:
        t = torch.zeros(numel, device=device, dtype=torch.float64)
        _zero_scratch[key] = t
    return t


def reset_scratch():
    """Re-zero the accumulators (only needed after an exception interrupted a producer/consumer pair)."""
    for t in _zero_scratch.values():
        t.zero_()


def new_stats(x, per_sample):
    n, c = x.shape[0], x.shape[1]
    return zero_scratch(x.device, 2 * (n * c if per_sample else c))


def norm_forward(x, gamma, beta, running_mean, running_var, nbt, per_sample, eps, momentum, act=ACT_NONE, slope=0.0,
                 stats=None, round_tf32=False, return_scale_shift=False):
    """Training-mode BatchNorm2d / InstanceNorm2d.  Returns (y, mean_rstd)."""
    lib = _lib.load()
    d = _norm_desc(x, per_sample, eps, momentum, act, slope, round_tf32)
    st = _stream()
    if stats is None:
        stats = new_stats(x, per_sample)
        _lib.check(lib.b200gan_norm_stats(ctypes.byref(d), x.data_ptr(), stats.data_ptr(), st), "norm_stats")
    groups = stats.numel() // 2
    mean_rstd = torch.empty(2 * groups, device=x.device, dtype=torch.float32)
    scale_shift = torch.empty(2 * groups, device=x.device, dtype=torch.float32)
    _lib.check(lib.b200gan_norm_finalize(ctypes.byref(d), stats.data_ptr(), _ptr(gamma), _ptr(beta),
                                         mean_rstd.data_ptr(), scale_shift.data_ptr(), _ptr(running_mean),
                                         _ptr(running_var), _ptr(nbt), st), "norm_finalize")
    y = torch.empty_like(x, memory_format=CL)
    _lib.check(lib.b200gan_norm_apply(ctypes.byref(d), x.data_ptr(), scale_shift.data_ptr(), y.data_ptr(), st),
               "norm_apply")
    if return_scale_shift:
        return y, mean_rstd, scale_shift
    return y, mean_rstd


def norm_finalize(x_shape, stats, gamma, beta, running_mean, running_var, nbt, per_sample, eps, momentum, device):
    """Batch statistics -> (mean_rstd, scale_shift); updates the running statistics.  `stats` is consumed (zeroed)."""
    n, c, h, w = x_shape
    d = NormDesc()
    d.N, d.HW, d.C, d.per_sample = n, h * w, c, int(per_sample)
    d.eps, d.momentum, d.act, d.slope, d.round_tf32 = eps, momentum, ACT_NONE, 0.0, 0
    groups = stats.numel() // 2
    mean_rstd = torch.empty(2 * groups, device=device, dtype=torch.float32)
    scale_shift = torch.empty(2 * groups, device=device, dtype=torch.float32)
    _lib.check(_lib.load().b200gan_norm_finalize(ctypes.byref(d), stats.data_ptr(), _ptr(gamma), _ptr(beta),
                                                 mean_rstd.data_ptr(), scale_shift.data_ptr(), _ptr(running_mean),
                                                 _ptr(running_var), _ptr(nbt), _stream()), "norm_finalize")
    return mean_rstd, scale_shift


def norm_stats(x, per_sample):
    d = _norm_desc(x, per_sample, 0.0, 0.0, ACT_NONE, 0.0, False)
    stats = new_stats(x, per_sample)
    _lib.check(_lib.load().b200gan_norm_stats(ctypes.byref(d), x.data_ptr(), stats.data_ptr(), _stream()), "norm_stats")
    return stats


# ---- Generator tail: BatchNorm2d -> act -> Conv2d(C, K<=3, 3, 1, 1) -> act (csrc/tail.cu) -------------------
def tail_desc(a_shape, k, act_mid, slope, act_out):
    n, c, h, w = a_shape
    d = TailDesc()
    d.N, d.H, d.W, d.C, d.K = n, h, w, c, k
    d.act_mid, d.slope, d.act_out = act_mid, slope, act_out
    return d


def tail_supported(a_shape, k, act_mid, slope, act_out):
    if Config.algo == "simt" or not Config.fuse_tail:
        return False
    return bool(_lib.load().b200gan_tail_supported(ctypes.byref(tail_desc(a_shape, k, act_mid, slope, act_out))))


def tail_fprop(d, a, scale_shift, w, bias):
    out = empty_cl(d.N, d.K, d.H, d.W, a.device)
    _lib.check(_lib.load().b200gan_tail_fprop(ctypes.byref(d), a.data_ptr(), scale_shift.data_ptr(), w.data_ptr(),
                                              _ptr(bias), out.data_ptr(), _stream()), "tail_fprop")
    return out


def tail_bwd(d, a, mean_rstd, scale_shift, w, g, need_affine, need_bias, round_tf32):
    lib = _lib.load()
    nws = lib.b200gan_tail_bwd_workspace_bytes(ctypes.byref(d))
    ws = torch.empty((nws + 7) // 8, device=a.device, dtype=torch.float64)
    da = torch.empty_like(a, memory_format=CL)
    dgb = torch.empty(2 * d.C, device=a.device, dtype=torch.float32) if need_affine else None
    dw = torch.empty((d.K, d.C, 3, 3), device=a.device, dtype=torch.float32)
    db = torch.empty(d.K, device=a.device, dtype=torch.float32) if need_bias else None
    _lib.check(lib.b200gan_tail_bwd(ctypes.byref(d), a.data_ptr(), mean_rstd.data_ptr(), scale_shift.data_ptr(),
                                    w.data_ptr(), g.data_ptr(), ws.data_ptr(), da.data_ptr(), _ptr(dgb), dw.data_ptr(),
                                    _ptr(db), int(round_tf32), _stream()), "tail_bwd")
    return da, dgb, dw, db


def norm_apply_affine(x, scale_shift, per_sample, act=ACT_NONE, slope=0.0):
    """y = act(x * scale + shift) with precomputed per-group scale/shift (eval-mode BatchNorm)."""
    d = _norm_desc(x, per_sample, 0.0, 0.0, act, slope, False)
    y = torch.empty_like(x, memory_format=CL)
    _lib.check(_lib.load().b200gan_norm_apply(ctypes.byref(d), x.data_ptr(), scale_shift.data_ptr(), y.data_ptr(),
                                              _stream()), "norm_apply")
    return y


def norm_backward(dy, x, y, mean_rstd, gamma, per_sample, eps, act=ACT_NONE, slope=0.0, need_params=False,
                  round_tf32=False, scale_shift=None):
    lib = _lib.load()
    d = _norm_desc(x, per_sample, eps, 0.0, act, slope, round_tf32)
    groups = mean_rstd.numel() // 2
    sums = zero_scratch(x.device, 2 * groups)
    dx = torch.empty_like(x, memory_format=CL)
    dgb = torch.empty(2 * groups, device=x.device, dtype=torch.float32) if need_params else None
    _lib.check(lib.b200gan_norm_bwd(ctypes.byref(d), dy.data_ptr(), x.data_ptr(), _ptr(y), mean_rstd.data_ptr(),
                                    _ptr(scale_shift), _ptr(gamma), sums.data_ptr(), dx.data_ptr(), _ptr(dgb), _stream()),
               "norm_bwd")
    return dx, dgb


def norm_backward_backward(dy, x, u, mean_rstd, scale_shift, gamma, gg_gamma, gg_beta, eps, act=ACT_NONE, slope=0.0,
                           need_dgamma=False):
    """Double backward of training-mode BatchNorm2d [+ LeakyReLU / ReLU]: given u = dL/d(dx) and (optionally) dL/d(dgamma),
    dL/d(dbeta) for the outputs of norm_backward(dy, x, ...), returns (dL/dx, dL/d(dy), dL/dgamma or None).  All of dy, x,
    u are NHWC; scale_shift carries the activation mask (required with an activation)."""
    for t_ in (dy, x, u):
        if not is_cl(t_):
            raise RuntimeError("b200gan norm_backward_backward: NHWC (channels_last) tensors expected")
    lib = _lib.load()
    d = _norm_desc(x, False, eps, 0.0, act, slope, False)
    c = x.shape[1]
    sums = zero_scratch(x.device, 5 * c)
    gx = torch.empty_like(x, memory_format=CL)
    gdy = torch.empty_like(x, memory_format=CL)
    dgamma = torch.empty(c, device=x.device, dtype=torch.float32) if need_dgamma else None
    _lib.check(lib.b200gan_norm_bwd_bwd(ctypes.byref(d), dy.data_ptr(), x.data_ptr(), u.data_ptr(), mean_rstd.data_ptr(),
                                        _ptr(scale_shift), _ptr(gamma), _ptr(gg_gamma), _ptr(gg_beta), sums.data_ptr(),
                                        gx.data_ptr(), gdy.data_ptr(), _ptr(dgamma), _stream()), "norm_bwd_bwd")
    return gx, gdy, dgamma


# ---- shape ops ------------------------------------------------------------------------------------
def upsample2x(x):
    n, c, h, w = x.shape
    y = empty_cl(n, c, 2 * h, 2 * w, x.device)
    _lib.check(_lib.load().b200gan_upsample2x_fwd(x.data_ptr(), y.data_ptr(), n, h, w, c, _stream()), "upsample2x_fwd")
    return y


def upsample2x_bwd(dy):
    n, c, h2, w2 = dy.shape
    dx = empty_cl(n, c, h2 // 2, w2 // 2, dy.device)
    _lib.check(_lib.load().b200gan_upsample2x_bwd(dy.data_ptr(), dx.data_ptr(), n, h2 // 2, w2 // 2, c, _stream()),
               "upsample2x_bwd")
    return dx


def pad2d(x, pads, mode, round_tf32=False):
    n, c, h, w = x.shape
    t, l, b, r = pads
    y = empty_cl(n, c, h + t + b, w + l + r, x.device)
    _lib.check(_lib.load().b200gan_pad2d_fwd(x.data_ptr(), y.data_ptr(), n, h, w, c, t, l, b, r, mode, int(round_tf32),
                                             _stream()), "pad2d_fwd")
    return y


def pad2d_bwd(dy, pads, mode):
    n, c, ho, wo = dy.shape
    t, l, b, r = pads
    h, w = ho - t - b, wo - l - r
    dx = empty_cl(n, c, h, w, dy.device)
    _lib.check(_lib.load().b200gan_pad2d_bwd(dy.data_ptr(), dx.data_ptr(), n, h, w, c, t, l, b, r, mode, _stream()),
               "pad2d_bwd")
    return dx


def act_forward(x, act, slope, mask=None, mask_per_channel=False):
    n, c, h, w = x.shape
    y = torch.empty_like(x, memory_format=CL)
    _lib.check(_lib.load().b200gan_act_fwd(x.data_ptr(), _ptr(mask), int(mask_per_channel), act, slope, x.numel(), c,
                                           h * w, y.data_ptr(), _stream()), "act_fwd")
    return y


# ---- Discriminator conv blocks as a fused chain (csrc/narrow_block.cu) ------------------------------------------
class BnEdge:
    """A training-mode BatchNorm2d between two fused convs: its batch statistics (fp64 sums of the producer's output)
    and parameters.  `sums` is filled by the consumer's backward (sum g, sum g * ahat) for the producer's backward.
    `grad_of_stored` is set by the consumer's backward when it runs under create_graph: from then on every backward
    through this edge hands the producer a gradient w.r.t. the stored tensor a (the BatchNorm backward already done);
    while it is False the gradient is w.r.t. the virtual normalised tensor and `sums` completes it."""

    def __init__(self, stats, gamma, beta, eps, count, groups=1):
        """stats: [groups][2][C] fp64; count: elements per channel and group (see b200gan_nb_bn in include/b200gan.h)."""
        self.stats, self.gamma, self.beta, self.eps, self.count = stats, gamma, beta, float(eps), float(count)
        self.groups = int(groups)
        self.sums = None
        self.grad_of_stored = False

    def c_struct(self):
        b = NbBn()
        b.stats, b.gamma, b.beta = self.stats.data_ptr(), _ptr(self.gamma), _ptr(self.beta)
        b.eps, b.count, b.groups, b.reserved = self.eps, self.count, self.groups, 0
        return b


class bn_groups:
    """`with ops.bn_groups(G):` -- the batch entering the drop-in modules is G equal runs of images that are to be treated
    as G separate forward passes of the reference sharing the weights: independent BatchNorm batch statistics (running
    statistics updated G times, in order), Dropout2d masks drawn in the order of G separate passes, parameter gradients
    summed.  Used by train.dcgan_step to run discriminator(real_imgs) and discriminator(gen_imgs.detach())
    (dcgan.py:178-179) as one launch per layer.  Only the fused chain honours it: every other normalisation /
    dropout module raises while it is active (train.py checks eligibility first)."""

    active = 1

    def __init__(self, groups):
        self.groups = int(groups)

    def __enter__(self):
        self.prev = bn_groups.active
        bn_groups.active = self.groups
        return self

    def __exit__(self, *exc):
        bn_groups.active = self.prev


def nb_supported(g):
    if not Config.fuse_narrow_chain:
        return False
    lib = _lib.load()
    if bn_groups.active > 1:
        return bool(lib.b200gan_nb_groups_supported(ctypes.byref(g), bn_groups.active))
    return bool(lib.b200gan_nb_supported(ctypes.byref(g)))


def _bn_ref(edge):
    return ctypes.byref(edge.c_struct()) if edge is not None else None


def nb_fprop(g, x, packed, bias, act, slope, chan_scale, in_edge, running_mean, running_var, nbt, momentum, want_stats,
             groups=1):
    y = empty_cl(g.N, g.K, g.P, g.Q, x.device)
    stats = torch.empty(groups * 2 * g.K, device=x.device, dtype=torch.float64) if want_stats else None
    _lib.check(_lib.load().b200gan_nb_fprop(ctypes.byref(g), _bn_ref(in_edge), _ptr(running_mean), _ptr(running_var),
                                            _ptr(nbt), float(momentum), x.data_ptr(), packed.data_ptr(), _ptr(bias),
                                            act, slope, _ptr(chan_scale), y.data_ptr(), _ptr(stats), int(groups),
                                            _stream()), "nb_fprop")
    return y, stats


def nb_dz(g_in, a, chan_scale, act, slope, out_edge, want_db):
    n, k, p, q = a.shape
    dz = torch.empty_like(a, memory_format=CL)
    db = torch.empty(k, device=a.device, dtype=torch.float32) if want_db else None
    sums = out_edge.sums if out_edge is not None else None
    _lib.check(_lib.load().b200gan_nb_dz(n, p * q, k, g_in.data_ptr(), a.data_ptr(), _ptr(chan_scale), act, slope,
                                         _bn_ref(out_edge), _ptr(sums), dz.data_ptr(), _ptr(db), _stream()), "nb_dz")
    return dz, db


def nb_wgrad(g, x, dz, in_edge, weight_shape):
    dw = torch.empty(weight_shape, device=x.device, dtype=torch.float32)
    lib = _lib.load()
    nws = int(lib.b200gan_nb_wgrad_workspace_floats(ctypes.byref(g)))
    ws = torch.empty(nws, device=x.device, dtype=torch.float32) if nws else None
    _lib.check(lib.b200gan_nb_wgrad(ctypes.byref(g), _bn_ref(in_edge), x.data_ptr(), dz.data_ptr(), dw.data_ptr(), _ptr(ws),
                                    _stream()), "nb_wgrad")
    return dw


def nb_dgrad(g, dz, packed, in_edge, a_prev):
    gout = empty_cl(g.N, g.C, g.H, g.W, dz.device)
    sums = (torch.empty(in_edge.groups * 2 * g.C, device=dz.device, dtype=torch.float64)
            if in_edge is not None else None)
    _lib.check(_lib.load().b200gan_nb_dgrad(ctypes.byref(g), dz.data_ptr(), packed.data_ptr(), _bn_ref(in_edge),
                                            _ptr(a_prev) if in_edge is not None else 0, gout.data_ptr(), _ptr(sums),
                                            _stream()), "nb_dgrad")
    return gout, sums


def nb_tail_fwd(a, edge, running_mean, running_var, nbt, momentum, nchw):
    n, c, h, w = a.shape
    if nchw:
        out = torch.empty((n, c, h, w), device=a.device, dtype=torch.float32)
    else:
        out = torch.empty_like(a, memory_format=CL)
    _lib.check(_lib.load().b200gan_nb_tail_fwd(n, h * w, c, _bn_ref(edge), _ptr(running_mean), _ptr(running_var), _ptr(nbt),
                                               float(momentum), a.data_ptr(), out.data_ptr(), int(nchw), _stream()),
               "nb_tail_fwd")
    return out


def nb_tail_bwd(a, edge, dout, nchw):
    n, c, h, w = a.shape
    g = torch.empty_like(a, memory_format=CL)
    sums = torch.empty(edge.groups * 2 * c, device=a.device, dtype=torch.float64)
    _lib.check(_lib.load().b200gan_nb_tail_bwd(n, h * w, c, _bn_ref(edge), a.data_ptr(), dout.data_ptr(), int(nchw),
                                               g.data_ptr(), sums.data_ptr(), _stream()), "nb_tail_bwd")
    return g, sums


# ---- Discriminator head / adversarial loss (csrc/head.cu) ----------------------------------------------------
def linear1_fwd(x, w, b, act):
    n, k = x.shape
    y = torch.empty((n, 1), device=x.device, dtype=torch.float32)
    _lib.check(_lib.load().b200gan_linear1_fwd(x.data_ptr(), w.data_ptr(), _ptr(b), y.data_ptr(), n, k, act, _stream()),
               "linear1_fwd")
    return y


def linear1_bwd(x, w, y, dy, act, need_dx, need_db):
    n, k = x.shape
    dx = torch.empty_like(x) if need_dx else None
    dw = torch.empty((1, k), device=x.device, dtype=torch.float32)
    db = torch.empty(1, device=x.device, dtype=torch.float32) if need_db else None
    _lib.check(_lib.load().b200gan_linear1_bwd(x.data_ptr(), w.data_ptr(), y.data_ptr(), dy.data_ptr(), _ptr(dx),
                                               dw.data_ptr(), _ptr(db), n, k, act, _stream()), "linear1_bwd")
    return dx, dw, db


def bce_fwd(v, t):
    loss = torch.empty((), device=v.device, dtype=torch.float32)
    _lib.check(_lib.load().b200gan_bce_fwd(v.data_ptr(), t.data_ptr(), loss.data_ptr(), v.numel(), _stream()), "bce_fwd")
    return loss


def bce_bwd(v, t, gout):
    dv = torch.empty_like(v)
    _lib.check(_lib.load().b200gan_bce_bwd(v.data_ptr(), t.data_ptr(), gout.data_ptr(), dv.data_ptr(), v.numel(),
                                           _stream()), "bce_bwd")
    return dv


def adam_step(p, g, m, v, lr, beta1, beta2, eps, grad_scale, step):
    _lib.check(_lib.load().b200gan_adam_step(p.data_ptr(), g.data_ptr(), m.data_ptr(), v.data_ptr(), p.numel(), lr,
                                             beta1, beta2, eps, grad_scale, step.data_ptr(), _stream()), "adam_step")


def gp_mlp_fwd_bwd(xi, w1, b1, w2, b2, w3, slope, lambda_gp):
    """Gradient penalty of the 3-layer MLP critic and its weight gradients in one kernel
    (wgan_gp.py:119-138 + the double backward at wgan_gp.py:173).  Returns (gp, dW1, dW2, dW3)."""
    for t_ in (xi, w1, b1, w2, b2, w3):
        _require_cuda(t_, "gp_mlp operand")
    lib = _lib.load()
    xi = xi.contiguous().view(xi.shape[0], -1)
    d = GpMlpDesc()
    d.N, d.Din, d.H1, d.H2 = xi.shape[0], xi.shape[1], w1.shape[0], w2.shape[0]
    d.slope, d.lambda_gp = slope, lambda_gp
    if w1.shape[1] != d.Din or w2.shape[1] != d.H1 or w3.numel() != d.H2:
        raise RuntimeError("b200gan gp_mlp: layer shapes do not chain")
    ws = torch.empty(lib.b200gan_gp_mlp_workspace_floats(ctypes.byref(d)), device=xi.device, dtype=torch.float32)
    gp = torch.empty((), device=xi.device, dtype=torch.float32)
    dw1, dw2, dw3 = torch.empty_like(w1), torch.empty_like(w2), torch.empty_like(w3)
    _lib.check(lib.b200gan_gp_mlp_fwd_bwd(ctypes.byref(d), xi.data_ptr(), w1.data_ptr(), b1.data_ptr(), w2.data_ptr(),
                                          b2.data_ptr(), w3.data_ptr(), gp.data_ptr(), dw1.data_ptr(), dw2.data_ptr(),
                                          dw3.data_ptr(), ws.data_ptr(), _stream()), "gp_mlp_fwd_bwd")
    return gp, dw1, dw2, dw3


def critic_step_mlp(real, fake, alpha, w1, b1, w2, b2, w3, b3, slope, lambda_gp):
    """wgan_gp.py:164-173 for the MLP critic in one kernel.  Returns (losses[2], dW1, db1, dW2, db2, dW3, db3)."""
    for t_ in (real, fake, alpha, w1, b1, w2, b2, w3, b3):
        _require_cuda(t_, "critic_step operand")
    lib = _lib.load()
    n = real.shape[0]
    real, fake = real.contiguous().view(n, -1), fake.contiguous().view(n, -1)
    alpha = alpha.contiguous().view(-1)
    d = GpMlpDesc()
    d.N, d.Din, d.H1, d.H2 = n, real.shape[1], w1.shape[0], w2.shape[0]
    d.slope, d.lambda_gp = slope, lambda_gp
    if (fake.shape != real.shape or alpha.numel() != n or w1.shape[1] != d.Din or w2.shape[1] != d.H1
            or w3.numel() != d.H2):
        raise RuntimeError("b200gan critic_step_mlp: shapes do not chain")
    dev = real.device
    ws = torch.empty(lib.b200gan_critic_step_workspace_floats(ctypes.byref(d)), device=dev, dtype=torch.float32)
    losses = torch.empty(2, device=dev, dtype=torch.float32)
    grads = [torch.empty_like(t_) for t_ in (w1, b1, w2, b2, w3, b3)]
    _lib.check(lib.b200gan_critic_step_mlp(ctypes.byref(d), real.data_ptr(), fake.data_ptr(), alpha.data_ptr(),
                                           w1.data_ptr(), b1.data_ptr(), w2.data_ptr(), b2.data_ptr(), w3.data_ptr(),
                                           b3.data_ptr(), losses.data_ptr(), *[g.data_ptr() for g in grads],
                                           ws.data_ptr(), _stream()), "critic_step_mlp")
    return (losses, *grads)
