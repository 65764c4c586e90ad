"""CPU suite (-m "not gpu"): the oracle against the golden vectors produced by the reference
itself, the numpy operator oracle against stock torch, the C ABI surface, and the host logic."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

from conftest import ROOT, rel_err
from oracle import np_ops, ref_models


def test_oracle_matches_reference_golden(golden_dir):
    fix = torch.load(os.path.join(golden_dir, "dcgan_32_b8.pt"), weights_only=False)
    g, d = ref_models.build_dcgan(fix["img_size"], seed=fix["seed"])
    for m in d.modules():
        if isinstance(m, torch.nn.Dropout2d):
            m.p = 0.0
    gen = g(fix["z"])
    assert rel_err(gen, fix["gen"]) < 1e-6
    validity = d(gen)
    assert rel_err(validity, fix["validity"]) < 1e-6
    loss = torch.nn.BCELoss()(validity, torch.ones(fix["batch"], 1))
    assert abs(loss.item() - fix["g_loss"].item()) < 1e-6
    loss.backward()
    for k, p in g.named_parameters():
        ref = fix["g_grads"][k]
        assert abs(p.grad.double().norm().item() - ref["norm"]) <= 1e-5 * max(ref["norm"], 1e-12) + 1e-12, k
        assert torch.allclose(p.grad.flatten()[:64], ref["head"], rtol=1e-4, atol=1e-9), k
    for k, v in fix["bn_running"].items():
        assert torch.allclose(g.state_dict()[k].float(), v.float(), rtol=1e-5, atol=1e-7), k


def test_batchnorm_second_positional_arg_is_eps():
    # SURVEY.md section 0.4: nn.BatchNorm2d(C, 0.8) sets eps, dcgan.py:56
    g, _ = ref_models.build_dcgan(32)
    bn = g.conv_blocks[3]
    assert bn.eps == 0.8 and bn.momentum == 0.1
    assert g.conv_blocks[0].eps == 1e-5


def test_numpy_conv_oracle_against_torch_golden(golden_dir):
    cases = torch.load(os.path.join(golden_dir, "ops_conv.pt"), weights_only=False)
    assert len(cases) == 7
    for c in cases:
        x, w, b = (c[k].double().numpy() for k in ("x", "w", "b"))
        if c["transposed"]:
            y = np_ops.conv_transpose2d(x, w, b, c["stride"], c["pad"])
        else:
            y = np_ops.conv2d(x, w, b, c["stride"], c["pad"])
        assert y.shape == tuple(c["y"].shape), c["name"]
        assert rel_err(torch.from_numpy(y), c["y"]) < 1e-5, c["name"]


def test_numpy_shape_ops_bit_exact_against_torch():
    x = torch.randn(2, 3, 5, 4)
    xn = x.double().numpy()
    assert np.array_equal(np_ops.upsample2x(xn), torch.nn.Upsample(scale_factor=2)(x).double().numpy())
    assert np.array_equal(np_ops.pad2d(xn, (1, 1, 0, 0)), torch.nn.ZeroPad2d((1, 0, 1, 0))(x).double().numpy())
    assert np.array_equal(np_ops.pad2d(xn, (3, 3, 3, 3), "reflect"),
                          torch.nn.ReflectionPad2d(3)(x).double().numpy())
    y, mean, uvar = np_ops.batch_norm_train(xn, np.ones(3), np.zeros(3), 0.8)
    bn = torch.nn.BatchNorm2d(3, 0.8)
    yt = bn(x)
    assert rel_err(torch.from_numpy(y), yt) < 1e-5
    assert np.allclose(bn.running_mean.numpy(), 0.1 * mean, atol=1e-6)
    assert np.allclose(bn.running_var.numpy(), 0.9 + 0.1 * uvar, atol=1e-6)
    assert rel_err(torch.from_numpy(np_ops.instance_norm(xn)), torch.nn.InstanceNorm2d(3)(x)) < 1e-5


# ---- C ABI surface ----------------------------------------------------------------------------
def _declared_symbols():
    hdr = open(os.path.join(ROOT, "include", "b200gan.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    return sorted(set(re.findall(r"\b(b200gan_[a-z0-9_]+)\s*\(", hdr)))


def test_library_loads_and_exports_every_declared_symbol():
    import b200gan
    from b200gan import _lib
    lib = b200gan.load_library()
    names = _declared_symbols()
    assert len(names) >= 25
    for n in names:
        assert hasattr(lib, n), f"libb200gan.so does not export {n}"
        assert n in _lib.SIGNATURES, f"{n} missing from the ctypes signature table"
    assert sorted(_lib.SIGNATURES) == names
    assert lib.b200gan_version() == 100


def test_struct_layouts_match_the_header():
    from b200gan import _lib
    assert ctypes.sizeof(_lib.ConvGeom) == 17 * 4
    assert ctypes.sizeof(_lib.Epilogue) == 40
    assert ctypes.sizeof(_lib.NormDesc) == 9 * 4
    assert ctypes.sizeof(_lib.GpMlpDesc) == 6 * 4
    assert ctypes.sizeof(_lib.TailDesc) == 8 * 4
    assert ctypes.sizeof(_lib.NbBn) == 48 and ctypes.sizeof(_lib.AdamTensor) == 40
    assert ctypes.sizeof(_lib.PackJob) == 16 + 17 * 4 + 4


def test_geometry_helper_matches_torch_shapes():
    from b200gan import ops
    g, out = ops.make_geom((2, 3, 10, 8), (7, 3, 3, 3), 2, (1, 1, 1, 1))
    assert out == (2, 7, 5, 4)
    g, out = ops.make_geom((2, 6, 5, 6), (6, 4, 4, 4), 2, (1, 1, 1, 1), transposed=True)
    assert out == (2, 4, 10, 12)
    g, out = ops.make_geom((1, 128, 16, 16), (64, 128, 3, 3), 1, (1, 1, 1, 1), up=2)
    assert out == (1, 64, 32, 32)
    # pix2pix final: Upsample -> ZeroPad2d((1,0,1,0)) -> Conv(k4, p1)  (pix2pix/models.py:76-81)
    g, out = ops.make_geom((1, 128, 128, 128), (3, 128, 4, 4), 1, (2, 2, 1, 1), up=2)
    assert out == (1, 3, 256, 256)


# ---- host logic -------------------------------------------------------------------------------
def test_drop_in_modules_keep_names_params_and_state_dict():
    from b200gan import zoo
    torch.manual_seed(0)
    g = zoo.DCGANGenerator(32)
    d = zoo.DCGANDiscriminator(32)
    g.apply(zoo.weights_init_normal)
    d.apply(zoo.weights_init_normal)
    go, do = ref_models.build_dcgan(32, seed=0)
    for ours, ref in ((g, go), (d, do)):
        so, sr = ours.state_dict(), ref.state_dict()
        assert list(so.keys()) == list(sr.keys())
        for k in so:  # same RNG consumption order of .apply(init) => identical parameters
            assert torch.equal(so[k], sr[k]), k
        for mo, mr in zip(ours.modules(), ref.modules()):
            assert type(mo).__name__ == type(mr).__name__
            assert mo is ours or isinstance(mo, type(mr))
    ours_bn = g.conv_blocks[3]
    assert ours_bn.eps == 0.8 and ours_bn.momentum == 0.1


def test_patch_rebinds_and_restores_torch_nn():
    import torch.nn as tnn
    import b200gan
    from b200gan import nn as bnn
    stock = tnn.Conv2d
    with b200gan.patched():
        assert tnn.Conv2d is bnn.Conv2d and tnn.Sequential is bnn.Sequential
        m = tnn.Conv2d(3, 4, 3, 2, 1)
        assert m.__class__.__name__ == "Conv2d" and isinstance(m, stock)
    assert tnn.Conv2d is stock


def test_fusion_plan_for_dcgan():
    from b200gan import nn as bnn, zoo
    g, d = zoo.DCGANGenerator(64), zoo.DCGANDiscriminator(64)
    kinds = [type(s).__name__ for s in bnn._build_plan(list(g.conv_blocks))]
    # BatchNorm2d(64, .8) + LeakyReLU + Conv2d(64, 1, 3, 1, 1) + Tanh (dcgan.py:60-63) is the fused tail node
    assert kinds == ["_NormStep", "_ConvStep", "_NormStep", "_ConvStep", "_TailStep"]
    steps = bnn._build_plan(list(g.conv_blocks))
    tail = steps[4]
    assert steps[1].up == 2 and steps[3].up == 2 and tail.conv_step.up == 1
    assert steps[1].stats is False and steps[3].stats is False and steps[3].next_norm is g.conv_blocks[7]
    assert tail.norm_step.takes_stats and tail.norm_step.act == 1 and tail.norm_step.rtf_dx
    assert tail.conv_step.stats is None and tail.conv_step.act == 3
    # the four discriminator blocks (dcgan.py:77-88) form one fused chain; its constituent steps stay available
    plan = bnn._build_plan(list(d.model))
    assert [type(s).__name__ for s in plan] == ["_ChainStep"]
    dsteps = plan[0].steps
    assert [type(s).__name__ for s in dsteps] == ["_ConvStep", "_ConvStep", "_NormStep", "_ConvStep", "_NormStep",
                                                  "_ConvStep", "_NormStep"]
    assert all(s.dropout2d is not None for s in dsteps if isinstance(s, bnn._ConvStep))
    assert dsteps[0].stats is None and dsteps[1].stats is False
    assert [(type(a).__name__, type(b).__name__) for a, b in plan[0].layers] == [
        ("_ConvStep", "NoneType"), ("_ConvStep", "_NormStep"), ("_ConvStep", "_NormStep"), ("_ConvStep", "_NormStep")]


def test_no_cpu_fallback():
    from b200gan import nn as bnn
    conv = bnn.Conv2d(3, 4, 3, 1, 1)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        conv(torch.randn(1, 3, 8, 8))
    bn = bnn.BatchNorm2d(3)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        bn(torch.randn(2, 3, 4, 4))


def test_mlp_modules_run_stock_on_cpu():
    # BASELINE config 0 (gan.py): MLP on CPU uses stock torch ops through the same classes
    from b200gan import nn as bnn
    net = bnn.Sequential(torch.nn.Linear(10, 8), bnn.LeakyReLU(0.2, inplace=True), torch.nn.Linear(8, 1),
                         bnn.Sigmoid())
    y = net(torch.randn(4, 10))
    assert y.shape == (4, 1) and bool((y > 0).all())


def test_wgan_gp_oracle_and_closed_form_against_reference_golden(golden_dir):
    """The golden file holds the reference's own compute_gradient_penalty output and the D gradients of
    lambda*gp (oracle/make_golden.py).  Check (a) the torch restatement, (b) the closed form the CUDA kernel
    implements (numpy float64)."""
    fix = torch.load(os.path.join(golden_dir, "wgan_gp_32_b64.pt"), weights_only=False)
    _, d = ref_models.build_wgan_gp(fix["img_size"], seed=fix["seed"])
    gp = ref_models.compute_gradient_penalty(d, fix["real"], fix["fake"], fix["alpha"])
    assert abs(gp.item() - fix["gp"].item()) < 1e-6
    (fix["lambda_gp"] * gp).backward()
    assert rel_err(d.model[4].weight.grad, fix["dW3"]) < 1e-5
    assert fix["bias_grads_zero"]
    xi = (fix["alpha"] * fix["real"] + (1 - fix["alpha"]) * fix["fake"]).double().numpy()
    w = [p.detach().double().numpy() for p in d.parameters()]
    gp_c, dw1, dw2, dw3 = np_ops.gp_mlp_closed_form(xi, w[0], w[1], w[2], w[3], w[4], 0.2, fix["lambda_gp"])
    assert abs(gp_c - fix["lambda_gp"] * fix["gp"].item()) < 1e-5 * abs(gp_c)
    assert rel_err(torch.from_numpy(dw3.reshape(1, -1)), fix["dW3"]) < 1e-5
    assert rel_err(torch.from_numpy(dw1[:4]), fix["dW1_head"]) < 1e-5
    assert rel_err(torch.from_numpy(dw2[:8]), fix["dW2_head"]) < 1e-5
    assert abs(np.linalg.norm(dw1) - fix["dW1_norm"]) < 1e-5 * fix["dW1_norm"]
    assert abs(np.linalg.norm(dw2) - fix["dW2_norm"]) < 1e-5 * fix["dW2_norm"]


SCRIPTS = os.path.join(ROOT, "tests", "scripts")


def test_launcher_runs_unmodified_gan_script_on_cpu_config0():
    """BASELINE config 0: an MLP GAN script in the reference's idiom (tests/scripts/mini_mlpgan), 28x28 synthetic,
    batch 64, CPU -- the unmodified script under the launcher with the drop-in classes patched in (MLP: stock ops
    through the same classes) prints the same losses as the stock run."""
    from b200gan import launch
    script = os.path.join(SCRIPTS, "mini_mlpgan", "mini_mlpgan.py")
    args = ["--epochs", "1", "--batch_size", "64"]
    ours = launch.run(script, args, iters=3, seed=0, stock=False, quiet=True)
    stock = launch.run(script, args, iters=3, seed=0, stock=True, quiet=True)
    lines = [l for l in ours["__b200_stdout__"].splitlines() if "[D loss" in l]
    assert len(lines) == 3
    assert ours["__b200_stdout__"] == stock["__b200_stdout__"]
    assert type(ours["generator"].model[1]).__name__ == "LeakyReLU"
    from b200gan import nn as bnn
    assert isinstance(ours["generator"].model, bnn.Sequential)
    assert not isinstance(stock["generator"].model, bnn.Sequential)


def test_launcher_builds_dcgan_with_drop_in_modules():
    """A DCGAN-style script in the reference's idiom (tests/scripts/mini_convgan), built under the launcher: the
    drop-in classes are patched in and draw the same initial weights as the stock run of the same script."""
    from b200gan import launch, nn as bnn
    script = os.path.join(SCRIPTS, "mini_convgan", "mini_convgan.py")
    args = ["--epochs", "0", "--side", "32"]
    ours = launch.run(script, args, iters=1, seed=0, quiet=True)
    stock = launch.run(script, args, iters=1, seed=0, stock=True, quiet=True)
    gen, ref = ours["G"], stock["G"]
    assert isinstance(gen.body, bnn.Sequential) and isinstance(gen.body[2], bnn.Conv2d)
    assert not isinstance(ref.body, bnn.Sequential)
    for k, v in ref.state_dict().items():
        assert torch.equal(gen.state_dict()[k].cpu(), v.cpu()), k


def test_pix2pix_and_cyclegan_oracle_against_reference_golden(golden_dir):
    fix = torch.load(os.path.join(golden_dir, "cyclegan_64_b2.pt"), weights_only=False)
    shape = (3, fix["size"], fix["size"])
    g_ab, g_ba, d_a, d_b = ref_models.build_cyclegan(shape, fix["blocks"], fix["seed"])
    real_a = ref_models.synthetic_images(fix["batch"], 3, fix["size"], fix["size"], seed=fix["seed"] + 1)
    with torch.no_grad():
        fake_b = g_ab(real_a)
    assert rel_err(fake_b[..., ::4, ::4], fix["fake_b"]) < 1e-6
    fixp = torch.load(os.path.join(golden_dir, "pix2pix_256_b1.pt"), weights_only=False)
    _, d = ref_models.build_pix2pix(fixp["seed"])
    assert sorted(d.state_dict().keys()) == sorted(k for k in fixp["d_grad_norms"].keys())
