#!/usr/bin/env python
"""bench.py -- the GAN training step of the reference's hot path on B200, one JSON line per run.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|stock|reference]
                    [--config dcgan|wgan_gp|pix2pix|cyclegan] [--dump-outputs DIR]

Default: BASELINE configs[1] -- DCGAN 64x64, batch 128 per GPU, the full G+D step of dcgan.py:146-183, images/sec.
N > 1 is launched by torchrun (one rank per GPU, NCCL, weak scaling).  Rank 0 prints ONE JSON line.

  --impl ours       the b200gan drop-in modules (libb200gan.so), b200gan.optim.Adam, step replayed from a CUDA graph
  --impl stock      the SAME step on stock torch.nn / cuDNN / cuBLAS with TF32 allowed (the reference's own GPU path,
                    BASELINE.md section 5), same CUDA-graph runner, same inputs: the GPU baseline
  --impl reference  the reference's CPU path (oracle port of the step, stock torch CPU) on the host cores

Keys of the line (DESIGN.md section 5):
  value          device-resident inputs, step loop replayed from a CUDA graph
  e2e            the same step driven from pinned HOST buffers: H2D of the inputs every step, D2H of the losses
  gpu_reference  (N = 1, --impl ours) the stock arm measured in the same process on the same GPU
  roofline       the time-dominant kernel group of the step timed alone with CUDA events against its bound, plus the
                 tcgen05 conv kernels against the TF32 peak and the whole step in reference-form FLOPs
  cpu_baseline   the oracle restatement of the reference step on the host cores (N = 1 only)
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "pytorch-gan_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

LATENT = 100
# SURVEY.md section 8(d): useful conv/linear GFLOP of one step per GPU (reference formulation), batch per GPU, image
CONFIGS = {
    "dcgan": dict(batch=128, img=64, ch=1, gflop=359.0, unit="images/s", metric="DCGAN 64x64 images/sec (full G+D step)",
                  workload="DCGAN 64x64 synthetic, batch 128 per GPU (BASELINE configs[1])"),
    "wgan_gp": dict(batch=64, img=32, ch=1, gflop=1.5, unit="images/s",
                    metric="WGAN-GP 32x32 images/sec (critic iteration incl. gradient penalty)",
                    workload="WGAN-GP 32x32 synthetic, batch 64, one critic iteration (BASELINE configs[2])"),
    "pix2pix": dict(batch=16, img=256, ch=3, gflop=1048.0, unit="images/s", metric="Pix2Pix 256x256 images/sec (full G+D step)",
                    workload="Pix2Pix U-Net 256x256 paired synthetic, batch 16 per GPU (BASELINE configs[3])"),
    "cyclegan": dict(batch=8, img=256, ch=3, gflop=16784.0, unit="image pairs/s",
                     metric="CycleGAN 256x256 image pairs/sec (two-G/two-D step)",
                     workload="CycleGAN ResNet-9 256x256 unpaired synthetic, batch 8 per GPU (BASELINE configs[4])"),
}


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "stock", "reference"])
    ap.add_argument("--config", default="dcgan", choices=sorted(CONFIGS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-gpu-reference", action="store_true")
    ap.add_argument("--no-roofline", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="eager step loop (debugging)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the losses of the last timed step and the state of the networks it trained to DIR/*.npy")
    a = ap.parse_args()
    if a.dump_outputs and a.impl == "reference":
        ap.error("--dump-outputs needs --impl ours or stock: the reference leg shrinks its batch to fit a time budget")
    if a.steps is None:
        a.steps = {"dcgan": 50, "wgan_gp": 200, "pix2pix": 20, "cyclegan": 10}[a.config]
    return a


# ---------------------------------------------------------------------------------------------------
class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.path = tempfile.mktemp(prefix="b200gan_clocks_", suffix=".csv")
        self.proc = None
        self.index = index

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits",
                 "-lms", "100"], stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except OSError:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in open(self.path):
            parts = [p.strip() for p in line.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0]))
                mx.append(float(parts[1]))
            except ValueError:
                continue
            for nm, v in zip(names, parts[3:7]):
                if v.lower() == "active":
                    reasons.add(nm)
        try:
            os.unlink(self.path)
        except OSError:
            pass
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        d = json.load(open(path))
        return d.get("hbm_gbs", 6650.0), d.get("bf16_tflops", 1590.0), "measured (MEASURED_PEAKS.json)"
    return 6650.0, 1590.0, "fallback (B200_PROFILING.md)"


# ---------------------------------------------------------------------------------------------------
# the reference's CPU path (oracle port; the one place bench.py executes oracle/)
# ---------------------------------------------------------------------------------------------------
def cpu_step_throughput(config, steps, warmup, threads=None, budget_s=150.0):
    """Oracle restatement of the reference step with stock torch.nn on the host cores.  Bounded sample: if `steps`
    full-batch steps would not fit in `budget_s`, every step processes a smaller batch of the same workload (per-image
    CPU cost is batch-insensitive); units/s is reported either way."""
    import itertools
    import torch
    from oracle import ref_models
    cfg = CONFIGS[config]
    threads = threads or min(os.cpu_count() or 1, 32)   # more threads than that only add contention on this path
    torch.set_num_threads(threads)
    full = cfg["batch"]
    img = cfg["img"]
    if config == "dcgan":
        g, d = ref_models.build_dcgan(img, seed=0)
        og, od = ref_models.make_adam(g.parameters()), ref_models.make_adam(d.parameters())
        data = (ref_models.synthetic_images(full, 1, img, img, seed=0), ref_models.synthetic_z(full, seed=0))
        run = lambda a, z: ref_models.dcgan_step(g, d, og, od, a, z)  # noqa: E731
        floor = 8
    elif config == "wgan_gp":
        from b200gan import train
        g, d = ref_models.build_wgan_gp(img, seed=0)
        od = ref_models.make_adam(d.parameters())
        data = (ref_models.synthetic_images(full, 1, img, img, seed=0), ref_models.synthetic_z(full, seed=0),
                ref_models.synthetic_alpha(full, seed=0))
        run = lambda a, z, al: train.wgan_gp_critic_step(g, d, od, a, z, al, 10.0, fused_gp=False)  # noqa: E731
        floor = 8
    elif config == "pix2pix":
        from b200gan import train
        g, d = ref_models.build_pix2pix(0)
        og, od = ref_models.make_adam(g.parameters()), ref_models.make_adam(d.parameters())
        data = (ref_models.synthetic_images(full, 3, img, img, seed=1), ref_models.synthetic_images(full, 3, img, img, seed=2))
        run = lambda a, b: train.pix2pix_step(g, d, og, od, a, b)  # noqa: E731
        floor = 1
    else:
        from b200gan import train
        nets = ref_models.build_cyclegan((3, img, img), 9, 0)
        og = ref_models.make_adam(itertools.chain(nets[0].parameters(), nets[1].parameters()))
        oa, ob = ref_models.make_adam(nets[2].parameters()), ref_models.make_adam(nets[3].parameters())
        data = (ref_models.synthetic_images(full, 3, img, img, seed=1), ref_models.synthetic_images(full, 3, img, img, seed=2))
        run = lambda a, b: train.cyclegan_step(*nets, og, oa, ob, a, b)  # noqa: E731
        floor = 1
    batch = full
    probe_n = min(full, max(floor, 2)) if config in ("pix2pix", "cyclegan") else full
    t0 = time.perf_counter()
    run(*[t[:probe_n] for t in data])          # first warm-up step doubles as the probe
    t_probe = (time.perf_counter() - t0) * full / probe_n
    n_steps = steps + max(warmup - 1, 0)
    if n_steps * t_probe > budget_s:
        batch = int(full * budget_s / (n_steps * t_probe))
        batch = max(floor, min(full, batch // floor * floor))
    data = [t[:batch] for t in data]
    for _ in range(max(warmup - 1, 0)):
        run(*data)
    t0 = time.perf_counter()
    for _ in range(steps):
        run(*data)
    dt = time.perf_counter() - t0
    return batch * steps / dt, dt / steps, threads, batch


def run_reference(args):
    if int(os.environ.get("RANK", "0")) != 0:
        return
    cfg = CONFIGS[args.config]
    ups, spstep, threads, batch = cpu_step_throughput(args.config, args.steps, max(args.warmup, 1))
    sample = (f"{args.steps} steps of the reference step on {batch} of the {cfg['batch']} samples per step "
              f"({cfg['img']}x{cfg['img']}) after {args.warmup} warm-up, oracle port (pinned bit-exact against the "
              f"unmodified reference scripts by oracle/make_golden.py), stock torch CPU, {threads} threads")
    print(json.dumps({
        "impl": "reference", "metric": cfg["metric"], "value": ups, "unit": cfg["unit"],
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": spstep * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": cfg["workload"], "global_batch": cfg["batch"],
                   "path": "reference CPU path (oracle port)"},
        "cpu_baseline": {"value": ups, "unit": cfg["unit"], "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": ups, "unit": cfg["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }))


# ---------------------------------------------------------------------------------------------------
# kernels timed alone (roofline leg)
# ---------------------------------------------------------------------------------------------------
def _event_time(torch, fn, iters, warm=3):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def dcgan_kernel_groups(torch, batch, hbm_peak, tf32_peak, iters=20):
    """Every heavy kernel of the DCGAN Generator at the bench size, alone, CUDA events; tensors > L2 so no flush is
    needed (the small discriminator kernels are launch-bound and are reported through the step's launch list).
    Returns a list of dicts; `per_step` = launches of that kernel in one training step."""
    from b200gan import ops
    from b200gan._lib import ACT_LRELU, ACT_TANH, ALGO_TC, PACK_TC_DGRAD_UP2, PACK_TC_FPROP_UP2
    CL = torch.channels_last
    out = []

    def conv_up2(name, cin, cout, hw):
        x = torch.randn(batch, cin, hw, hw, device="cuda").contiguous(memory_format=CL)
        w = torch.randn(cout, cin, 3, 3, device="cuda") * 0.02
        g, oshape = ops.make_geom(tuple(x.shape), tuple(w.shape), 1, (1, 1, 1, 1), 0, 2, False)
        if not ops.tc_supported(g, 0):
            return
        dy = torch.randn(oshape, device="cuda").contiguous(memory_format=CL)
        pf, pd = ops.pack_weights(g, w, PACK_TC_FPROP_UP2), ops.pack_weights(g, w, PACK_TC_DGRAD_UP2)
        flops = 2.0 * batch * hw * hw * 4 * cout * cin * 4   # executed: 4 phases x 4 taps (2.25x fewer than reference form)
        nbytes = (x.numel() + dy.numel() + pf.numel()) * 4
        for pas, fn in (("fprop", lambda: ops.conv_fprop(g, x, pf, ALGO_TC)),
                        ("dgrad", lambda: ops.conv_dgrad(g, dy, pd, ALGO_TC)),
                        ("wgrad", lambda: ops.conv_wgrad(g, x, dy, tuple(w.shape), False, ALGO_TC))):
            ms = _event_time(torch, fn, iters)
            out.append({"kernel": f"{name} {pas} (tcgen05 TF32, Upsample x2 folded)", "bound": "tensor", "ms": ms,
                        "achieved": flops / ms / 1e9, "peak": tf32_peak, "unit": "TFLOP/s", "frac": flops / ms / 1e9 / tf32_peak,
                        "algorithmic_mbytes": nbytes / 1e6, "executed_gflop": flops / 1e9, "per_step": 1})

    conv_up2("G conv1 128->128 @16->32", 128, 128, 16)
    conv_up2("G conv2 128->64 @32->64", 128, 64, 32)

    # the fused tail: BN(64, .8) + LeakyReLU + Conv 64->1 + Tanh on the 134 MB conv2 output (dcgan.py:60-63)
    img = 64
    a = torch.randn(batch, 64, img, img, device="cuda").contiguous(memory_format=CL)
    if ops.tail_supported(tuple(a.shape), 1, ACT_LRELU, 0.2, ACT_TANH):
        d = ops.tail_desc(tuple(a.shape), 1, ACT_LRELU, 0.2, ACT_TANH)
        ss = torch.cat([torch.rand(64, device="cuda") + 0.5, torch.randn(64, device="cuda") * 0.1])
        mr = torch.cat([torch.randn(64, device="cuda") * 0.1, torch.rand(64, device="cuda") + 0.5])
        w3 = torch.randn(1, 64, 3, 3, device="cuda") * 0.02
        b3 = torch.zeros(1, device="cuda")
        gimg = torch.randn(batch, 1, img, img, device="cuda")
        ms = _event_time(torch, lambda: ops.tail_fprop(d, a, ss, w3, b3), iters)
        nb = a.numel() * 4 + gimg.numel() * 4
        out.append({"kernel": "G tail fprop: BN+LReLU+Conv 64->1+Tanh (tcgen05 on transformed tiles)", "bound": "hbm",
                    "ms": ms, "achieved": nb / ms / 1e6, "peak": hbm_peak, "unit": "GB/s", "frac": nb / ms / 1e6 / hbm_peak,
                    "algorithmic_mbytes": nb / 1e6, "per_step": 1})
        ms = _event_time(torch, lambda: ops.tail_bwd(d, a, mr, ss, w3, gimg, True, True, True), iters)
        nb = 3 * a.numel() * 4 + 2 * gimg.numel() * 4   # reduce pass reads a; apply pass reads a, writes da
        out.append({"kernel": "G tail backward: recomputed dgrad + BN backward + wgrad (2 passes over a)", "bound": "hbm",
                    "ms": ms, "achieved": nb / ms / 1e6, "peak": hbm_peak, "unit": "GB/s", "frac": nb / ms / 1e6 / hbm_peak,
                    "algorithmic_mbytes": nb / 1e6, "per_step": 1})
    # BatchNorm over the 67 MB conv1 output (training mode, eps 0.8, + LeakyReLU): forward and backward
    x = torch.randn(batch, 128, 32, 32, device="cuda").contiguous(memory_format=CL)
    gamma, beta = torch.ones(128, device="cuda"), torch.zeros(128, device="cuda")
    y, mr = ops.norm_forward(x, gamma, beta, None, None, None, False, 0.8, 0.1, 1, 0.2)
    dy = torch.randn_like(x)
    ms = _event_time(torch, lambda: ops.norm_forward(x, gamma, beta, None, None, None, False, 0.8, 0.1, 1, 0.2), iters)
    nb = 3 * x.numel() * 4
    out.append({"kernel": "BatchNorm2d(128)+LeakyReLU forward on 67 MB (stats + apply)", "bound": "hbm", "ms": ms,
                "achieved": nb / ms / 1e6, "peak": hbm_peak, "unit": "GB/s", "frac": nb / ms / 1e6 / hbm_peak,
                "algorithmic_mbytes": nb / 1e6, "per_step": 1})
    ms = _event_time(torch, lambda: ops.norm_backward(dy, x, y, mr, gamma, False, 0.8, 1, 0.2, True), iters)
    nb = 5 * x.numel() * 4   # algorithmic: reduce reads dy, x; apply reads dy, x, writes dx (the mask is a function of x)
    out.append({"kernel": "BatchNorm2d(128)+LeakyReLU backward on 67 MB (reduce + apply)", "bound": "hbm", "ms": ms,
                "achieved": nb / ms / 1e6, "peak": hbm_peak, "unit": "GB/s", "frac": nb / ms / 1e6 / hbm_peak,
                "algorithmic_mbytes": nb / 1e6, "per_step": 1})
    return out


def cublas_tf32_tflops(torch):
    torch.backends.cuda.matmul.allow_tf32 = True
    a = torch.randn(8192, 8192, device="cuda")
    ms = _event_time(torch, lambda: a @ a, 5)
    torch.backends.cuda.matmul.allow_tf32 = False
    return 2 * 8192.0 ** 3 / ms / 1e9


# ---------------------------------------------------------------------------------------------------
# the step under test
# ---------------------------------------------------------------------------------------------------
def build_job(torch, config, stock, dev, world, rank):
    """Returns (step_fn(*inputs) -> tensor of losses, host input pools, D2H bytes per step, {name: network the step
    trains})."""
    import itertools
    from b200gan import optim, train, zoo
    cfg = CONFIGS[config]
    ns = zoo.namespace(stock=stock)
    B, img = cfg["batch"], cfg["img"]

    def adam(params):
        if stock:
            return torch.optim.Adam(params, lr=2e-4, betas=(0.5, 0.999), capturable=True)
        return optim.Adam(params, lr=2e-4, betas=(0.5, 0.999))

    def reducer(params, opt):
        if world == 1:
            return None
        from b200gan import ddp
        return ddp.GradReducer(list(params), world, None if stock else opt)

    torch.manual_seed(0)  # identical init on every rank
    gen = torch.Generator(device="cpu").manual_seed(1234 + rank)  # per-rank data streams
    pool_n = 8 if config in ("dcgan", "wgan_gp") else 3

    def images(c):
        return [(torch.rand(B, c, img, img, generator=gen) * 2 - 1).pin_memory() for _ in range(pool_n)]

    if config == "dcgan":
        g = zoo.DCGANGenerator(img, nn=ns).to(dev)
        d = zoo.DCGANDiscriminator(img, nn=ns).to(dev)
        g.apply(zoo.weights_init_normal)
        d.apply(zoo.weights_init_normal)
        og, od = adam(g.parameters()), adam(d.parameters())
        rg, rd = reducer(g.parameters(), og), reducer(d.parameters(), od)
        loss = ns.BCELoss()
        valid, fake = torch.ones(B, 1, device=dev), torch.zeros(B, 1, device=dev)

        def step(imgs, z):
            gl, dl, _ = train.dcgan_step(g, d, og, od, imgs, z, loss, valid, fake, rg, rd)
            return torch.stack([gl, dl])
        pools = [images(1), [torch.randn(B, LATENT, generator=gen).pin_memory() for _ in range(pool_n)]]
        nets = {"generator": g, "discriminator": d}
    elif config == "wgan_gp":
        g = zoo.WGANGPGenerator((1, img, img), nn=ns).to(dev)
        d = zoo.WGANGPDiscriminator((1, img, img), nn=ns).to(dev)
        od = adam(d.parameters())
        rd = reducer(d.parameters(), od)

        def step(imgs, z, alpha):
            dl, gp = train.wgan_gp_critic_step(g, d, od, imgs, z, alpha, 10.0, fused_gp=False if stock else "step",
                                                 reduce_d=rd)
            return torch.stack([dl, gp])
        pools = [images(1), [torch.randn(B, LATENT, generator=gen).pin_memory() for _ in range(pool_n)],
                 [torch.rand(B, 1, 1, 1, generator=gen).pin_memory() for _ in range(pool_n)]]
        nets = {"discriminator": d}
    elif config == "pix2pix":
        g, d = zoo.GeneratorUNet(nn=ns).to(dev), zoo.Pix2PixDiscriminator(nn=ns).to(dev)
        g.apply(zoo.weights_init_normal)
        d.apply(zoo.weights_init_normal)
        og, od = adam(g.parameters()), adam(d.parameters())
        rg, rd = reducer(g.parameters(), og), reducer(d.parameters(), od)

        def step(a, b):
            lg, ld = train.pix2pix_step(g, d, og, od, a, b, reduce_g=rg, reduce_d=rd)
            return torch.stack([lg, ld])
        pools = [images(3), images(3)]
        nets = {"generator": g, "discriminator": d}
    else:
        shape = (3, img, img)
        nets = [zoo.GeneratorResNet(shape, 9, nn=ns), zoo.GeneratorResNet(shape, 9, nn=ns),
                zoo.CycleGANDiscriminator(shape, nn=ns), zoo.CycleGANDiscriminator(shape, nn=ns)]
        for m in nets:
            m.to(dev).apply(zoo.weights_init_normal_cyclegan)
        og = adam(itertools.chain(nets[0].parameters(), nets[1].parameters()))
        oa, ob = adam(nets[2].parameters()), adam(nets[3].parameters())
        rg = reducer(itertools.chain(nets[0].parameters(), nets[1].parameters()), og)
        ra, rb = reducer(nets[2].parameters(), oa), reducer(nets[3].parameters(), ob)

        def step(a, b):
            # replay buffers (cyclegan/utils.py:19-33) hand back the incoming fakes while they fill (the first
            # 50 / batch steps): the timed step is that steady state, free of host-side randomness
            lg, ld = train.cyclegan_step(*nets, og, oa, ob, a, b, None, None, reduce_g=rg, reduce_d_a=ra, reduce_d_b=rb)
            return torch.stack([lg, ld])
        pools = [images(3), images(3)]
        nets = dict(zip(("G_AB", "G_BA", "D_A", "D_B"), nets))
    return step, pools, 8, nets


DUMP_FLOATS = 3_000_000  # per trained network: the four of CycleGAN stay under 64 MB


def snapshot_outputs(torch, losses, nets):
    """What a step hands back: its losses, and the state (weights, running statistics) of every network it trains,
    flattened in state_dict order.  A network of more than DUMP_FLOATS values is cut to a fixed, seeded sample.
    Split reductions add their partial sums in no fixed order, so two runs agree to rounding, not bit for bit."""
    out = {"losses": losses.detach().float().cpu().numpy()}
    for name, net in nets.items():
        flat = torch.cat([v.detach().float().flatten() for v in net.state_dict().values() if v.is_floating_point()])
        flat = flat.cpu()
        if flat.numel() > DUMP_FLOATS:
            pick = torch.randperm(flat.numel(), generator=torch.Generator().manual_seed(0))[:DUMP_FLOATS]
            flat = flat[pick.sort().values]
        out[name] = flat.numpy()
    return out


def time_job(torch, dist, args, stock, dev, world, rank, local, steps, warmup, clocks=False, dump=False):
    from b200gan import _lib, train
    step, pools, d2h, nets = build_job(torch, args.config, stock, dev, world, rank)
    pool_n = len(pools[0])
    dev_pools = [[t.to(dev) for t in p] for p in pools]
    torch.manual_seed(99 + rank)  # dropout streams differ per rank
    calls0 = _lib.CALLS
    graph_error = None
    if args.no_graph:
        runner = lambda *xs: step(*[x.to(dev, non_blocking=True) for x in xs])  # noqa: E731
        for _ in range(3):
            runner(*[p[0] for p in dev_pools])
        calls_per_step = (_lib.CALLS - calls0) // 3
    else:
        try:
            runner = train.GraphedStep(step, [p[0] for p in dev_pools], warmup=3)
            calls_per_step = (_lib.CALLS - calls0) // 4  # 3 warm-up + 1 captured executions
        except Exception as e:  # a step that cannot be captured is still measured (eagerly) and says so
            graph_error = f"{type(e).__name__}: {e}"[:300]
            torch.cuda.synchronize()
            runner = lambda *xs: step(*[x.to(dev, non_blocking=True) for x in xs])  # noqa: E731
            c1 = _lib.CALLS
            runner(*[p[0] for p in dev_pools])
            calls_per_step = _lib.CALLS - c1

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for i in range(max(warmup, 3)):
        runner(*[p[i % pool_n] for p in dev_pools])
    sampler = ClockSampler(local) if clocks else None
    barrier()
    if sampler and rank == 0:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(steps):
        out = runner(*[p[i % pool_n] for p in dev_pools])
    e1.record()
    barrier()
    clk = sampler.stop() if (sampler and rank == 0) else None
    ms = e0.elapsed_time(e1)
    losses = out.tolist()
    outputs = snapshot_outputs(torch, out, nets) if dump else None  # before the e2e leg trains further
    # e2e: host buffers in, losses out, every step
    for i in range(3):
        runner(*[p[i % pool_n] for p in pools])
    barrier()
    e2, e3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e2.record()
    for i in range(steps):
        out = runner(*[p[i % pool_n] for p in pools])
        _ = out.cpu()  # D2H read of the step's losses: the reference's per-step .item() (dcgan.py:185-188)
    e3.record()
    barrier()
    ms_e2e = e2.elapsed_time(e3)
    t = torch.tensor([ms, ms_e2e], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms, ms_e2e = t.tolist()
    h2d = sum(p[0].numel() * 4 for p in pools)
    res = dict(ms_per_step=ms / steps, ms_per_step_e2e=ms_e2e / steps, losses=losses, clocks=clk, h2d=h2d, d2h=d2h,
               calls_per_step=calls_per_step, graph_error=graph_error, outputs=outputs)
    del runner, step
    return res


def _finish(world):
    """Leave without tearing NCCL down: destroy_process_group() can block while CUDA graphs that captured
    collectives are still alive, and the measurement is already printed."""
    sys.stdout.flush()
    sys.stderr.flush()
    if world > 1:
        os._exit(0)


def run_gpu(args):
    import torch
    import torch.distributed as dist
    import b200gan

    cfg = CONFIGS[args.config]
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py --impl ours/stock needs a GPU (no CPU fallback)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    stock = args.impl == "stock"
    if not stock:
        b200gan.load_library()

    def set_stock_flags(on):
        # the reference's own GPU path: stock torch.nn on cuDNN/cuBLAS with TF32 convolutions (torch's default)
        torch.backends.cudnn.allow_tf32 = True
        torch.backends.cuda.matmul.allow_tf32 = bool(on)
        torch.backends.cudnn.benchmark = bool(on)

    gpu_ref = None
    if not stock and world == 1 and not args.no_gpu_reference:
        set_stock_flags(True)
        r = time_job(torch, dist, args, True, dev, world, rank, local, max(5, args.steps // 2), 3)
        gpu_ref = {"impl": "stock torch.nn + cuDNN/cuBLAS, TF32 allowed, same CUDA-graph runner and inputs",
                   "ms_per_step": r["ms_per_step"], "value": cfg["batch"] / r["ms_per_step"] * 1e3, "unit": cfg["unit"],
                   "e2e_ms_per_step": r["ms_per_step_e2e"]}
        torch.cuda.empty_cache()
    set_stock_flags(stock)
    res = time_job(torch, dist, args, stock, dev, world, rank, local, args.steps, args.warmup, clocks=True,
                   dump=bool(args.dump_outputs) and rank == 0)
    if rank != 0:
        _finish(world)
        return
    if args.dump_outputs:
        import numpy as np
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, arr in res["outputs"].items():
            np.save(os.path.join(args.dump_outputs, f"{name}.npy"), arr)

    hbm_peak, bf16_peak, peak_src = measured_peaks()
    tf32_peak = bf16_peak / 2.0  # kind::tf32 issues at half the kind::f16 rate (guide: 1.13 vs 2.25 PF nominal)
    step_ms = res["ms_per_step"]
    roofline = None
    if not stock and not args.no_roofline and args.config == "dcgan":
        groups = dcgan_kernel_groups(torch, cfg["batch"], hbm_peak, tf32_peak)
        for g_ in groups:
            g_["share_of_step"] = g_["ms"] * g_["per_step"] / step_ms
        dom = max(groups, key=lambda g_: g_["share_of_step"])
        # dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed `ncu --set full` capture of the same
        # kernels (profiles/r2_ncu_full_tail_kernels_c3.txt; the kernels' traffic is set by the algorithm, not the timing)
        ncu_traffic = {"G tail fprop": 145.4e6, "G tail backward": 141.6e6 + 218.7e6}
        dom_traffic = next((v for k_, v in ncu_traffic.items() if dom["kernel"].startswith(k_)), None)
        tc = [g_ for g_ in groups if g_["bound"] == "tensor"]
        roofline = {"kernel": dom["kernel"], "bound": dom["bound"], "achieved": dom["achieved"], "peak": dom["peak"],
                    "unit": dom["unit"], "frac": dom["frac"], "ms_per_launch": dom["ms"],
                    "share_of_step": dom["share_of_step"], "traffic": dom_traffic,
                    "traffic_source": "profiles/r2_ncu_full_tail_kernels_c3.txt (bytes per launch)" if dom_traffic else None,
                    "peak_source": peak_src + ("; TF32 = bf16/2" if dom["bound"] == "tensor" else ""),
                    "step_tensor_fraction_reference_form": cfg["gflop"] / step_ms / tf32_peak,
                    "step_gflop_reference_form": cfg["gflop"],
                    "tcgen05_kernels_exec_tflops": {g_["kernel"]: round(g_["achieved"], 1) for g_ in tc},
                    "cublas_tf32_gemm_8192_tflops": cublas_tf32_tflops(torch),
                    "groups": groups}
    elif not stock:
        roofline = {"kernel": "whole step, reference-form conv FLOPs", "bound": "tensor",
                    "achieved": cfg["gflop"] / step_ms, "peak": tf32_peak, "unit": "TFLOP/s",
                    "frac": cfg["gflop"] / step_ms / tf32_peak, "traffic": None,
                    "peak_source": peak_src + "; TF32 = bf16/2"}

    cpu = None
    if not args.no_cpu_baseline and world == 1 and not stock:
        ups, spstep, threads, batch = cpu_step_throughput(args.config, 2, 1, budget_s=25.0)
        cpu = {"value": ups, "unit": cfg["unit"], "cores": threads, "kind": "port",
               "sample": f"2 steps on {batch} of the {cfg['batch']} samples per step after 1 warm-up, oracle port of the "
                         f"reference step, stock torch CPU"}

    B = cfg["batch"]
    line = {
        "impl": args.impl, "metric": cfg["metric"],
        "value": B * world / step_ms * 1e3, "unit": cfg["unit"], "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": step_ms, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "tf32 (fp32 storage, fp32 accumulate)", "data": "synthetic",
        "config": {"workload": cfg["workload"], "global_batch": B * world, "parallelism": f"dp{world}",
                   "cuda_graph": not args.no_graph and res["graph_error"] is None,
                   "cuda_graph_error": res["graph_error"],
                   "l2": "per-step working set of activations exceeds the 126 MB L2; a pool of distinct input batches; "
                         "no explicit flush",
                   "algo": "stock" if stock else b200gan.Config.algo},
        "e2e": {"value": B * world / res["ms_per_step_e2e"] * 1e3, "unit": cfg["unit"], "h2d_bytes_per_step": res["h2d"],
                "d2h_bytes_per_step": res["d2h"], "ms_per_step": res["ms_per_step_e2e"]},
        "gpu_launches": 0 if stock else res["calls_per_step"] * args.steps,
        "gpu_launches_note": "C-ABI launches of libb200gan kernels per step x steps (replayed from a CUDA graph)",
        "clocks": res["clocks"],
        "roofline": roofline,
        "gpu_reference": gpu_ref,
        "speedup_vs_gpu_reference": (gpu_ref["ms_per_step"] / step_ms) if gpu_ref else None,
        "cpu_baseline": cpu,
        "final_losses": res["losses"],
    }
    print(json.dumps(line), flush=True)
    _finish(world)


if __name__ == "__main__":
    a = parse_args()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_gpu(a)
