"""Gradient penalties through training-mode BatchNorm2d (SURVEY.md section 8f, N2, BatchNorm critics):
the double-backward kernel (b200gan_norm_bwd_bwd) against torch float64, and the critics of DRAGAN
(dragan.py:144-167, the DCGAN discriminator as a fused chain or not) and DualGAN (dualgan.py:116-135, BatchNorm with a
fused LeakyReLU and a ZeroPad2d((1, 0, 1, 0)) patch head) against stock torch on the same GPU."""
import copy
import os

import pytest
import torch

from conftest import rel_err
from test_cpu_bn_double_backward import torch_double_backward

pytestmark = pytest.mark.gpu


def _set_tf32(on):
    torch.backends.cudnn.allow_tf32 = on
    torch.backends.cuda.matmul.allow_tf32 = on


def _grad_bound(algo, ours_tf32_dev):
    """Gradients of a penalty through BatchNorm (eps 0.8) are ill-conditioned: with algo 'simt' the project's bound for
    fp32 re-association through BatchNorm backward (test_gpu_dcgan.py, 5e-3); with 'auto' the bound of the TF32 conv
    double backward (test_gpu_n2.py, 2e-2) or 1.5x what stock torch TF32 shows on the same inputs."""
    return 5e-3 if algo == "simt" else max(2e-2, 1.5 * ours_tf32_dev)


# ---- the kernel --------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("c", [16, 128, 256, 12])
@pytest.mark.parametrize("act", ["lrelu", "relu", "none"])
@pytest.mark.parametrize("with_gg", [True, False])
def test_norm_backward_backward_kernel_vs_torch_float64(c, act, with_gg):
    from b200gan import ops
    from b200gan._lib import ACT_LRELU, ACT_NONE, ACT_RELU
    code, slope = {"lrelu": (ACT_LRELU, 0.2), "relu": (ACT_RELU, 0.0), "none": (ACT_NONE, 0.0)}[act]
    eps = 0.8
    gen = torch.Generator(device="cuda").manual_seed(c * 7 + code)
    shape = (4, c, 9, 7)
    cl = torch.channels_last

    def rnd(*s):
        return torch.randn(*s, device="cuda", generator=gen)

    x = (rnd(*shape) * 2 + 0.3).contiguous(memory_format=cl)
    dy, u = rnd(*shape).contiguous(memory_format=cl), rnd(*shape).contiguous(memory_format=cl)
    gamma, beta = rnd(c), rnd(c)
    ggg, ggb = (rnd(c), rnd(c)) if with_gg else (None, None)
    _, mean_rstd, scale_shift = ops.norm_forward(x, gamma, beta, None, None, None, False, eps, 0.0, code, slope,
                                                 return_scale_shift=True)
    # elements whose pre-activation sits within rounding of 0 may take either side of the mask in fp32 vs fp64:
    # give them no incoming gradient and leave them out of the dL/d(dy) comparison
    xd = x.double()
    pre = (xd - xd.mean((0, 2, 3), keepdim=True)) / torch.sqrt(xd.var((0, 2, 3), unbiased=False, keepdim=True) + eps)
    pre = pre * gamma.double().view(1, c, 1, 1) + beta.double().view(1, c, 1, 1)
    keep = pre.abs() > 1e-4 if code != ACT_NONE else torch.ones_like(pre, dtype=torch.bool)
    dy = (dy * keep).contiguous(memory_format=cl)
    gx, gdy, dg = ops.norm_backward_backward(dy, x, u, mean_rstd, scale_shift, gamma, ggg, ggb, eps, code, slope,
                                             need_dgamma=True)
    ref_slope = None if code == ACT_NONE else slope
    gx_r, dg_r, gdy_r = torch_double_backward(
        xd, gamma.double(), beta.double(), dy.double(), u.double(),
        ggg.double() if with_gg else torch.zeros(c, device="cuda", dtype=torch.float64),
        ggb.double() if with_gg else torch.zeros(c, device="cuda", dtype=torch.float64), eps, ref_slope)
    assert rel_err(gx, gx_r) < 1e-4
    assert rel_err(gdy * keep, gdy_r * keep) < 1e-4
    assert rel_err(dg, dg_r) < 1e-4
    torch.cuda.synchronize()
    assert int((ops.zero_scratch(x.device, 5 * c) != 0).sum()) == 0   # workspace handed back zeroed


@pytest.mark.parametrize("c,act", [(64, "lrelu"), (64, "none"), (12, "lrelu")])
@pytest.mark.parametrize("norm_fast", [True, False])
def test_norm_first_order_gradient_is_the_same_under_create_graph(c, act, norm_fast):
    """NormFn under create_graph returns its input gradient from the same kernel as without: bit-identical."""
    import b200gan
    from b200gan import functional as F
    from b200gan._lib import ACT_LRELU, ACT_NONE
    prev = b200gan.Config.norm_fast
    b200gan.Config.norm_fast = norm_fast
    try:
        torch.manual_seed(5)
        spec = F.NormSpec(eps=0.8, momentum=0.0, act=ACT_LRELU if act == "lrelu" else ACT_NONE, slope=0.2)
        x = torch.randn(8, c, 6, 6, device="cuda").contiguous(memory_format=torch.channels_last).requires_grad_(True)
        gamma = torch.randn(c, device="cuda", requires_grad=True)
        beta = torch.randn(c, device="cuda", requires_grad=True)
        dy = torch.randn(8, c, 6, 6, device="cuda").contiguous(memory_format=torch.channels_last)
        res = []
        for create in (False, True):
            y = F.norm_block(x, gamma, beta, None, None, None, None, spec)
            res.append(torch.autograd.grad(y, (x, gamma, beta), dy, create_graph=create))
        for a, b in zip(*res):
            assert torch.equal(a.detach(), b.detach())
    finally:
        b200gan.Config.norm_fast = prev


# ---- DRAGAN: the DCGAN discriminator (dragan.py:73-100), penalty of dragan.py:144-167 ----------------------------
def _dragan_gp(d, x, noise, alpha):
    interpolates = alpha * x + ((1 - alpha) * (x + 0.5 * x.std() * noise))
    interpolates = interpolates.detach().requires_grad_(True)
    d_int = d(interpolates)
    ones = torch.ones(x.shape[0], 1, device=x.device)
    grads = torch.autograd.grad(outputs=d_int, inputs=interpolates, grad_outputs=ones, create_graph=True,
                                retain_graph=True, only_inputs=True)[0]
    return 10 * ((grads.norm(2, dim=1) - 1) ** 2).mean()


def _dragan_d_iteration(d, real, fake, noise, alpha, seed):
    """One D iteration of dragan.py:199-217: D(real), D(fake), the penalty, and only gradient_penalty.backward()."""
    torch.manual_seed(seed)
    bce = torch.nn.BCELoss()
    ones = torch.ones(real.shape[0], 1, device=real.device)
    d.zero_grad()
    d_loss = (bce(d(real), ones) + bce(d(fake), ones * 0)) / 2
    gp = _dragan_gp(d, real, noise, alpha)
    gp.backward()
    return dict(gp=gp.detach(), d_loss=d_loss.detach(),
                grads={k: p.grad.detach().clone() for k, p in d.named_parameters()},
                bufs={k: b.detach().clone() for k, b in d.named_buffers() if b.dtype == torch.float32})


@pytest.mark.parametrize("fuse", [True, False])
@pytest.mark.parametrize("algo", ["simt", "auto"])
def test_dragan_critic_gradient_penalty_vs_stock(fuse, algo):
    import b200gan
    from b200gan import zoo
    prev = (b200gan.Config.algo, b200gan.Config.fuse_narrow_chain)
    b200gan.Config.algo, b200gan.Config.fuse_narrow_chain = algo, fuse
    try:
        torch.manual_seed(0)
        ref = zoo.DCGANDiscriminator(img_size=32, channels=1, nn=zoo.namespace(stock=True))
        ref.apply(zoo.weights_init_normal)
        ours = zoo.DCGANDiscriminator(img_size=32, channels=1)
        ours.load_state_dict(ref.state_dict())
        ref, ours = ref.cuda(), ours.cuda()
        ref_t = copy.deepcopy(ref)
        n = 64
        g = torch.Generator(device="cuda").manual_seed(1)
        real = torch.rand(n, 1, 32, 32, device="cuda", generator=g) * 2 - 1
        fake = torch.tanh(torch.randn(n, 1, 32, 32, device="cuda", generator=g))
        noise = torch.rand(n, 1, 32, 32, device="cuda", generator=g)
        alpha = torch.rand(n, 1, 32, 32, device="cuda", generator=g)
        _set_tf32(False)
        r32 = _dragan_d_iteration(ref, real, fake, noise, alpha, seed=7)
        _set_tf32(True)
        rtf = _dragan_d_iteration(ref_t, real, fake, noise, alpha, seed=7)
        _set_tf32(False)
        o = _dragan_d_iteration(ours, real, fake, noise, alpha, seed=7)
        if fuse:
            assert any(type(s).__name__ == "_ChainStep" for s in ours.model._plan())

        def bound(a, b):
            return 1e-4 if algo == "simt" else max(2e-3, 1.5 * rel_err(a, b))

        assert abs(o["gp"].item() - r32["gp"].item()) <= bound(rtf["gp"], r32["gp"]) * abs(r32["gp"].item())
        assert abs(o["d_loss"].item() - r32["d_loss"].item()) <= (bound(rtf["d_loss"], r32["d_loss"])
                                                                     * abs(r32["d_loss"].item()))
        errs = {k: rel_err(o["grads"][k], gr) for k, gr in r32["grads"].items()}
        print("dragan", fuse, algo, {k: f"{e:.2e}" for k, e in errs.items()})
        for k, gr in r32["grads"].items():
            assert errs[k] < _grad_bound(algo, rel_err(rtf["grads"][k], gr)), (k, errs[k])
        for k, b in r32["bufs"].items():   # running statistics: updated once per forward, never by the penalty
            e = rel_err(o["bufs"][k], b)
            assert e < (1e-5 if algo == "simt" else max(1e-5, 1.5 * rel_err(rtf["bufs"][k], b))), (k, e)
    finally:
        b200gan.Config.algo, b200gan.Config.fuse_narrow_chain = prev
        _set_tf32(False)


# ---- DualGAN: two BatchNorm critics, WGAN-GP (dualgan.py:116-135, 180-191) -----------------------------------------
def _dualgan_gp(d, real, fake, alpha):
    interpolates = (alpha * real + ((1 - alpha) * fake)).requires_grad_(True)
    validity = d(interpolates)
    grads = torch.autograd.grad(outputs=validity, inputs=interpolates, grad_outputs=torch.ones_like(validity),
                                create_graph=True, retain_graph=True, only_inputs=True)[0]
    grads = grads.view(grads.size(0), -1)
    return ((grads.norm(2, dim=1) - 1) ** 2).mean()


def _dualgan_d_step(d_a, d_b, data):
    a, b, fa, fb, al_a, al_b = data
    opts = [torch.optim.Adam(m.parameters(), lr=1e-4, betas=(0.5, 0.999)) for m in (d_a, d_b)]
    for o_ in opts:
        o_.zero_grad()
    gp_a = _dualgan_gp(d_a, a, fa, al_a)
    loss_a = -torch.mean(d_a(a)) + torch.mean(d_a(fa)) + 10 * gp_a
    gp_b = _dualgan_gp(d_b, b, fb, al_b)
    loss_b = -torch.mean(d_b(b)) + torch.mean(d_b(fb)) + 10 * gp_b
    loss = loss_a + loss_b
    loss.backward()
    grads = {f"{i}.{k}": p.grad.detach().clone() for i, m in enumerate((d_a, d_b)) for k, p in m.named_parameters()}
    for o_ in opts:
        o_.step()
    params = {f"{i}.{k}": p.detach().clone() for i, m in enumerate((d_a, d_b)) for k, p in m.named_parameters()}
    return dict(loss=loss.detach(), gp=(gp_a + gp_b).detach(), grads=grads, params=params)


@pytest.mark.parametrize("algo", ["simt", "auto"])
def test_dualgan_critic_step_vs_stock(algo):
    import b200gan
    from b200gan import zoo
    prev = b200gan.Config.algo
    b200gan.Config.algo = algo
    try:
        torch.manual_seed(3)
        refs = [zoo.DualGANDiscriminator(3, nn=zoo.namespace(stock=True)) for _ in range(2)]
        ours = [zoo.DualGANDiscriminator(3) for _ in range(2)]
        for o_, r_ in zip(ours, refs):
            o_.load_state_dict(r_.state_dict())
        refs = [m.cuda() for m in refs]
        ours = [m.cuda() for m in ours]
        refs_t = copy.deepcopy(refs)
        g = torch.Generator(device="cuda").manual_seed(4)
        n = 8
        imgs = [torch.rand(n, 3, 128, 128, device="cuda", generator=g) * 2 - 1 for _ in range(4)]
        alphas = [torch.rand(n, 1, 1, 1, device="cuda", generator=g) for _ in range(2)]
        data = (*imgs, *alphas)
        _set_tf32(False)
        r32 = _dualgan_d_step(*refs, data)
        _set_tf32(True)
        rtf = _dualgan_d_step(*refs_t, data)
        _set_tf32(False)
        o = _dualgan_d_step(*ours, data)

        def bound(a, b):
            return 1e-4 if algo == "simt" else max(2e-3, 1.5 * rel_err(a, b))

        assert abs(o["gp"].item() - r32["gp"].item()) <= bound(rtf["gp"], r32["gp"]) * abs(r32["gp"].item())
        assert abs(o["loss"].item() - r32["loss"].item()) <= bound(rtf["loss"], r32["loss"]) * abs(r32["loss"].item())
        # Parameters whose gradient is zero by construction: the bias of a conv feeding BatchNorm directly
        # (models.py:106-108) cannot change the loss, and the head bias (models.py:119) gets -1 from -mean(D(real)) and
        # +1 from mean(D(fake)) while the penalty does not depend on it.  Their computed gradients are rounding noise,
        # which Adam (eps 1e-8) turns into a step of up to lr whose size depends on the noise, so their updated values
        # are not compared.  The head bias must come out zero to fp32 rounding of those two unit terms.
        skip = {f"{i}.model.{j}.bias" for i in (0, 1) for j in (2, 5, 9)}
        for i in (0, 1):
            head = o["grads"][f"{i}.model.9.bias"].abs().max().item()
            assert head < 1e-5, (i, head)
        for key in ("grads", "params"):
            errs = {k: rel_err(o[key][k], ref) for k, ref in r32[key].items() if k not in skip}
            print("dualgan", algo, key, {k: f"{e:.2e}" for k, e in errs.items()})
            for k, e in errs.items():
                assert e < _grad_bound(algo, rel_err(rtf[key][k], r32[key][k])), (key, k, e)
    finally:
        b200gan.Config.algo = prev
        _set_tf32(False)


# ---- a DRAGAN-style script through the launcher --------------------------------------------------------------------
def test_mini_dragan_under_the_launcher_matches_stock():
    from b200gan import launch
    script = os.path.join(os.path.dirname(os.path.abspath(__file__)), "scripts", "mini_dragan", "mini_dragan.py")
    args = ["--n_epochs", "1", "--batch_size", "16", "--img_size", "32"]
    _set_tf32(False)
    ref = launch.run(script, args, iters=3, seed=5, stock=True, quiet=True)
    ours = launch.run(script, args, iters=3, seed=5, stock=False, quiet=True)
    assert any(type(s).__name__ == "_ChainStep" for s in ours["discriminator"].model._plan())
    assert len(ref["history"]) == 3 and len(ours["history"]) == 3
    for r_, o_ in zip(ref["history"], ours["history"]):
        for a, b in zip(o_, r_):
            assert abs(a - b) < 2e-3 * abs(b), (ref["history"], ours["history"])
