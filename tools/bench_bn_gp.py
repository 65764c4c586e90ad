"""Gradient penalties through BatchNorm critics on the GPU: the two critic iterations, patched (b200gan drop-ins and
Adam) vs stock torch (cuDNN, TF32 allowed) in the same process, and the double-backward kernels of
b200gan_norm_bwd_bwd alone against the bytes they must move.

    python tools/bench_bn_gp.py [--iters 30] [--out profiles/r3_bn_gp_bench.json]

  * DRAGAN D iteration (dragan.py:199-217): batch 64, 1x32x32, DCGAN discriminator: D(real), D(fake), D(interpolates)
    + autograd.grad(create_graph=True), gradient_penalty.backward(), Adam step.
  * DualGAN critic iteration (dualgan.py:116-135, 180-191): batch 8, 3x128x128, two critics: gp_A + gp_B + Wasserstein
    terms, D_loss.backward(), two Adam steps.
  * Kernels: the reduction reads dy, x, u (12 B/element), the element-wise pass reads them again and writes two
    outputs (20 B/element); at the DualGAN shapes [8,128,32,32], [8,256,16,16] (L2-resident) and at [64,128,64,64]
    (134 MB per tensor set, larger than the 126 MB L2; the inputs are rotated over three sets so that each timed launch
    reads from HBM).
Times are CUDA-event times of steady-state iterations after warm-up.  The card name and power limit are read in the
same run and written beside the numbers."""
import argparse
import copy
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "pytorch-gan_b200")]


def _card():
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        info["power_limit_and_max_sm_clock"] = out[0] if out else "unavailable"
    except (OSError, subprocess.SubprocessError):
        info["power_limit_and_max_sm_clock"] = "unavailable"
    return info


def _time(fn, iters, warmup):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for _ in range(iters):
        fn()
    end.record()
    torch.cuda.synchronize()
    return start.elapsed_time(end) / iters


def _dragan_iteration(d, opt, real, fake):
    def step():
        bce = torch.nn.BCELoss()
        ones = torch.ones(real.shape[0], 1, device=real.device)
        opt.zero_grad()
        d_loss = (bce(d(real), ones) + bce(d(fake), ones * 0)) / 2
        alpha = torch.rand_like(real)
        interpolates = alpha * real + ((1 - alpha) * (real + 0.5 * real.std() * torch.rand_like(real)))
        interpolates.requires_grad_(True)
        d_int = d(interpolates)
        grads = torch.autograd.grad(d_int, interpolates, torch.ones_like(d_int), create_graph=True,
                                    retain_graph=True, only_inputs=True)[0]
        gp = 10 * ((grads.norm(2, dim=1) - 1) ** 2).mean()
        gp.backward()
        opt.step()
        return d_loss
    return step


def _dualgan_iteration(d_a, d_b, opts, a, b, fa, fb):
    def gp(d, real, fake_):
        alpha = torch.rand(real.shape[0], 1, 1, 1, device=real.device)
        interpolates = (alpha * real + ((1 - alpha) * fake_)).requires_grad_(True)
        v = d(interpolates)
        g = torch.autograd.grad(v, interpolates, torch.ones_like(v), create_graph=True, retain_graph=True,
                                only_inputs=True)[0]
        return ((g.view(g.size(0), -1).norm(2, dim=1) - 1) ** 2).mean()

    def step():
        for o in opts:
            o.zero_grad()
        loss_a = -torch.mean(d_a(a)) + torch.mean(d_a(fa)) + 10 * gp(d_a, a, fa)
        loss_b = -torch.mean(d_b(b)) + torch.mean(d_b(fb)) + 10 * gp(d_b, b, fb)
        (loss_a + loss_b).backward()
        for o in opts:
            o.step()
    return step


def bench_models(iters, warmup):
    import b200gan
    from b200gan import optim as boptim, zoo
    torch.backends.cudnn.allow_tf32 = True
    torch.backends.cuda.matmul.allow_tf32 = True
    torch.backends.cudnn.benchmark = True
    res = {}
    torch.manual_seed(0)
    ref = zoo.DCGANDiscriminator(img_size=32, channels=1, nn=zoo.namespace(stock=True))
    ref.apply(zoo.weights_init_normal)
    ours = zoo.DCGANDiscriminator(img_size=32, channels=1)
    ours.load_state_dict(ref.state_dict())
    ref, ours = ref.cuda(), ours.cuda()
    real = torch.rand(64, 1, 32, 32, device="cuda") * 2 - 1
    fake = torch.rand(64, 1, 32, 32, device="cuda") * 2 - 1
    runs = {"stock": _dragan_iteration(ref, torch.optim.Adam(ref.parameters(), 2e-4, (0.5, 0.999)), real, fake),
            "patched": _dragan_iteration(ours, boptim.Adam(ours.parameters(), 2e-4, (0.5, 0.999)), real, fake)}
    res["dragan_d_iteration_b64_32px_ms"] = _alternate(runs, iters, warmup)

    torch.manual_seed(1)
    refs = [zoo.DualGANDiscriminator(3, nn=zoo.namespace(stock=True)).cuda() for _ in range(2)]
    ours = [zoo.DualGANDiscriminator(3).cuda() for _ in range(2)]
    for o, r in zip(ours, refs):
        o.load_state_dict(r.state_dict())
    imgs = [torch.rand(8, 3, 128, 128, device="cuda") * 2 - 1 for _ in range(4)]
    runs = {"stock": _dualgan_iteration(*refs, [torch.optim.Adam(m.parameters(), 2e-4, (0.5, 0.999)) for m in refs],
                                        *imgs),
            "patched": _dualgan_iteration(*ours, [boptim.Adam(m.parameters(), 2e-4, (0.5, 0.999)) for m in ours],
                                          *imgs)}
    res["dualgan_critic_iteration_b8_128px_ms"] = _alternate(runs, iters, warmup)
    res["config"] = {"algo": b200gan.Config.algo, "fuse_narrow_chain": b200gan.Config.fuse_narrow_chain}
    return res


def _alternate(runs, iters, warmup, rounds=3):
    """Best of `rounds` alternating windows per variant (other work shares the host)."""
    out = {k: [] for k in runs}
    for _ in range(rounds):
        for k, fn in runs.items():
            out[k].append(_time(fn, iters, warmup))
    best = {k: min(v) for k, v in out.items()}
    return {"stock_ms": best["stock"], "patched_ms": best["patched"], "speedup": best["stock"] / best["patched"],
            "windows_ms": out}


def bench_kernels(iters, warmup):
    from b200gan import ops
    from b200gan._lib import ACT_LRELU, ACT_NONE
    cl = torch.channels_last
    res = {}
    for shape, act in (((8, 128, 32, 32), ACT_LRELU), ((8, 256, 16, 16), ACT_LRELU), ((64, 128, 64, 64), ACT_NONE)):
        n, c, h, w = shape
        elems = n * c * h * w
        sets = []
        for _ in range(3 if elems * 12 > 64e6 else 1):
            x = torch.randn(shape, device="cuda").contiguous(memory_format=cl)
            dy = torch.randn(shape, device="cuda").contiguous(memory_format=cl)
            u = torch.randn(shape, device="cuda").contiguous(memory_format=cl)
            gam, bet = torch.randn(c, device="cuda"), torch.randn(c, device="cuda")
            _, mr, ss = ops.norm_forward(x, gam, bet, None, None, None, False, 0.8, 0.0, act, 0.2,
                                         return_scale_shift=True)
            sets.append((dy, x, u, mr, ss, gam, torch.randn(c, device="cuda"), torch.randn(c, device="cuda")))
        k = [0]

        def call():
            s = sets[k[0] % len(sets)]
            k[0] += 1
            ops.norm_backward_backward(*s, 0.8, act, 0.2, True)

        # kernel times from the profiler (one run of its own), whole-call time from events
        call_ms = _time(call, iters, warmup)
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(iters):
                call()
            torch.cuda.synchronize()
        kt = {}
        for e in prof.key_averages():
            if "norm_bwd_bwd" in e.key:
                dev_us = getattr(e, "device_time_total", None)
                if dev_us is None:
                    dev_us = e.cuda_time_total
                kt[e.key] = dev_us / max(e.count, 1)
        red = sum(v for kk, v in kt.items() if "reduce" in kk)
        app = sum(v for kk, v in kt.items() if "apply" in kk)
        entry = {"elements": elems, "call_us_events": call_ms * 1e3, "kernel_us": kt,
                 "reduce_GBps": 12 * elems / (red * 1e-6) / 1e9 if red else None,
                 "apply_GBps": 20 * elems / (app * 1e-6) / 1e9 if app else None,
                 "input_sets_rotated": len(sets)}
        res["x".join(map(str, shape))] = entry
    res["hbm_datasheet_GBps"] = 7700
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3_bn_gp_bench.json"))
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_bn_gp: needs a CUDA device")
    import b200gan
    b200gan.load_library()
    res = {"card": _card(), "models": bench_models(a.iters, a.warmup), "kernels": bench_kernels(200, 20)}
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
