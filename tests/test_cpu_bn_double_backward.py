"""The closed form of the double backward of a training-mode BatchNorm2d [+ LeakyReLU / ReLU] that
csrc/norm.cu:b200gan_norm_bwd_bwd implements, restated in numpy float64 and checked against torch's own double
backward of act(batch_norm(x)) on the CPU.  The GPU kernel is checked against the same torch reference in
test_gpu_bn_double_backward.py."""
import numpy as np
import pytest
import torch
import torch.nn.functional as tF


def bn_double_backward(x, gamma, dy, u, gg_gamma, gg_beta, eps, slope, beta=None):
    """numpy float64, NCHW.  The first backward of y = act(BN(x)) maps dy to (dx, dgamma, dbeta); given u = dL/d(dx),
    gg_gamma = dL/d(dgamma), gg_beta = dL/d(dbeta), returns (dL/dx, dL/dgamma, dL/d(dy)).
    slope: None = no activation, 0.0 = ReLU, else LeakyReLU slope.  gamma None = no affine parameters."""
    c = x.shape[1]
    m_count = x.size // c
    axes = (0, 2, 3)

    def v(t):
        return np.asarray(t, dtype=np.float64).reshape(1, c, 1, 1)

    def mean(t):
        return t.mean(axis=axes)

    ga = np.ones(c) if gamma is None else gamma
    be = np.zeros(c) if beta is None else beta
    ggg = np.zeros(c) if gg_gamma is None else gg_gamma
    ggb = np.zeros(c) if gg_beta is None else gg_beta
    mu = mean(x)
    r = 1.0 / np.sqrt(mean((x - v(mu)) ** 2) + eps)
    xh = (x - v(mu)) * v(r)
    if slope is None:
        mask = np.ones_like(x)
    else:
        mask = np.where(xh * v(ga) + v(be) > 0, 1.0, float(slope))
    g = dy * mask
    a, b = mean(g), mean(g * xh)
    uu, cu, d = mean(u), mean(u * xh), mean(u * g)
    e = d - uu * a - cu * b
    t = g - v(a) - xh * v(b)
    w = u - v(uu) - xh * v(cu)
    gr = ga * r
    gx = v(r) * (v(ggg - gr * cu) * t - v(gr * b) * w - v(gr) * xh * v(e))
    dgamma = r * m_count * e
    gdy = mask * (v(gr) * w + v(ggg) * xh + v(ggb))
    return gx, dgamma, gdy


def torch_double_backward(x, gamma, beta, dy, u, gg_gamma, gg_beta, eps, slope):
    """Reference: torch autograd twice through act(batch_norm(x, training=True)), float64."""
    x = x.clone().requires_grad_(True)
    dy = dy.clone().requires_grad_(True)
    params = []
    if gamma is not None:
        gamma = gamma.clone().requires_grad_(True)
        beta = beta.clone().requires_grad_(True)
        params = [gamma, beta]
    y = tF.batch_norm(x, None, None, gamma, beta, training=True, eps=eps)
    if slope is not None:
        y = tF.leaky_relu(y, slope) if slope > 0 else tF.relu(y)
    first = torch.autograd.grad(y, [x] + params, dy, create_graph=True)
    loss = (first[0] * u).sum()
    if params:
        loss = loss + (first[1] * gg_gamma).sum() + (first[2] * gg_beta).sum()
    out = torch.autograd.grad(loss, [x, dy] + params[:1])
    return out[0], (out[2] if params else None), out[1]


@pytest.mark.parametrize("shape", [(4, 3, 5, 5), (3, 12, 7, 6), (2, 5, 3, 9)])
@pytest.mark.parametrize("slope", [0.2, 0.0, None])
@pytest.mark.parametrize("eps", [0.8, 1e-5])
@pytest.mark.parametrize("affine", [True, False])
def test_closed_form_matches_torch_double_backward(shape, slope, eps, affine):
    gen = torch.Generator().manual_seed(hash((shape, slope, eps, affine)) % 2 ** 31)
    c = shape[1]

    def rnd(*s):
        return torch.randn(*s, generator=gen, dtype=torch.float64)

    x, dy, u = rnd(*shape) * 2 + 0.5, rnd(*shape), rnd(*shape)
    gamma = rnd(c) if affine else None
    beta = rnd(c) if affine else None
    ggg = rnd(c) if affine else None
    ggb = rnd(c) if affine else None
    gx_t, dg_t, gdy_t = torch_double_backward(x, gamma, beta, dy, u, ggg, ggb, eps, slope)
    npy = (lambda t: None if t is None else t.numpy())
    gx, dg, gdy = bn_double_backward(x.numpy(), npy(gamma), dy.numpy(), u.numpy(), npy(ggg), npy(ggb), eps, slope,
                                     npy(beta))

    def rel(a, b):
        return np.linalg.norm(a - b.numpy()) / np.linalg.norm(b.numpy())

    assert rel(gx, gx_t) < 1e-10
    assert rel(gdy, gdy_t) < 1e-10
    if affine:
        assert rel(dg, dg_t) < 1e-10
