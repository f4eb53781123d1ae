"""bench.py — BigGAN-Deep 256x256 G+D step throughput (BASELINE.json config 4) on N B200s, one JSON line on rank 0.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--batch B] [--config yaml] [--dump-outputs DIR]

step     = WORKER.train_discriminator (d_updates_per_step = 2 discriminator updates) + WORKER.train_generator
           (one generator update + EMA), i.e. one iteration of the reference loop (src/loader.py:392-398).
metric   = images/s = global batch x acml_steps / step time, whole job over all ranks (strong scaling: the global
           batch is fixed at 256, each rank takes 256/N).
value    = synthetic real images already resident in HBM.
e2e      = the same step driven from pinned HOST buffers: the basket's H2D copy and a D2H read of both losses are inside
           the timed region.
--impl reference : the CPU path (oracle port of the reference step) on the host cores, bounded sample, rank 0 only.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "pytorch-studiogan_b200")
for p in (ROOT, PKG):
    if p not in sys.path:
        sys.path.insert(0, p)
sys.dont_write_bytecode = True       # the benchmark leaves the tree it runs from untouched (it may be read-only)

import numpy as np  # noqa: E402
import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

# conv + linear + attention-bmm FLOPs per image (2 x MAC), BASELINE.md section 3 / SURVEY.md 8(d)
# WGAN-GP-128res (SURVEY a7: G 18.2 / D 9.4 GF per image forward): 5 D updates x (G fwd + 2 D fwd + 2 D bwd + penalty ~ 7 D fwd)
# + 1 G update (G fwd + D fwd + D dgrad + G bwd) ~ 775 GF per batch image per step
# SNGAN / BigGAN CIFAR10 (SURVEY 8d table): 44.3 / 101.1 GF per batch image per step (5 D updates + 1 G update)
STEP_GFLOP_PER_IMAGE = {"BigGAN-Deep-256res": 1141.0, "WGAN-GP-128res": 775.0, "SNGAN-CIFAR10-b256": 44.3, "BigGAN-CIFAR10-b512": 101.1}
METRIC_NAME = {"BigGAN-Deep-256res": "BigGAN-Deep 256x256 G+D step images/sec",
               "WGAN-GP-128res": "WGAN-GP ResNetGAN 128x128 G+D step images/sec (5 D updates with gradient penalty + 1 G update)",
               "SNGAN-CIFAR10-b256": "SNGAN CIFAR10 32x32 G+D step images/sec (5 D updates + 1 G update)",
               "BigGAN-CIFAR10-b512": "BigGAN CIFAR10 32x32 G+D step images/sec (5 D updates + 1 G update + EMA, sync-BN when N > 1)"}
# BASELINE.json configs 2 / 3 / 5, measured after the headline config and reported under config.also_measured:
# (yaml, the world sizes it is run at)
ALSO = [("SNGAN-CIFAR10-b256", (1,)), ("BigGAN-CIFAR10-b512", (1, 2, 4)), ("WGAN-GP-128res", (1, 2))]
G_FWD_GF, D_FWD_GF = 58.80, 60.50


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=0, help="override the global batch (diagnostics only)")
    ap.add_argument("--config", default=os.path.join(PKG, "configs", "BigGAN-Deep-256res.yaml"))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--graphs", default="auto", choices=["auto", "on", "off"],
                    help="capture each training phase in a CUDA graph; auto = on when the per-GPU batch is <= 64 (launch-bound regime)")
    ap.add_argument("--no-fid", action="store_true", help="skip the FID-50k evaluation timing")
    ap.add_argument("--no-also", action="store_true", help="skip BASELINE configs 2 / 3 / 5 (config.also_measured)")
    ap.add_argument("--fid-num", type=int, default=50000)
    ap.add_argument("--cpu-batch", type=int, default=4, help="images per CPU-baseline step (4 -> ~15 s of CPU work on 32 threads)")
    ap.add_argument("--cpu-threads", type=int, default=0, help="0 = min(32, host cores): more threads only add contention for these layer sizes")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last one computed to DIR/<name>.npy")
    ap.add_argument("--kernel-breakdown", metavar="PATH", help="write the per-kernel accounting step to this JSON file")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


class Logger:
    def info(self, *a, **k):
        pass


class SyntheticBasketLoader:
    """Infinite loader with the reference basket contract (src/loader.py:178-193): one item = batch x acml x d_updates
    images in [-1, 1] fp32 NCHW + int64 labels.  ``device`` None -> pinned host memory (the e2e leg), else HBM-resident."""

    def __init__(self, per_rank_batch, n_items, img_size, num_classes, seed, device=None, pool=2):
        g = torch.Generator().manual_seed(seed)
        self.items = []
        for _ in range(pool):
            img = torch.rand(per_rank_batch * n_items, 3, img_size, img_size, generator=g) * 2 - 1
            lab = torch.randint(0, num_classes, (per_rank_batch * n_items,), generator=g)
            if device is None:
                img, lab = img.pin_memory(), lab.pin_memory()
            else:
                img, lab = img.to(device), lab.to(device)
            self.items.append((img, lab))
        self.i = 0

    def __iter__(self):
        return self

    def __next__(self):
        self.i += 1
        return self.items[self.i % len(self.items)]


class ClockSampler(threading.Thread):
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        super().__init__(daemon=True)
        self.gpu_index = gpu_index
        self.rows = []
        self.stop_flag = False

    def run(self):
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.gpu_index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.split(",")])
            except Exception:
                pass
            time.sleep(0.2)

    def summary(self):
        sm = [float(r[1]) for r in self.rows if len(r) > 8 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) > 8 and r[2].replace(".", "").isdigit()]
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            if len(r) > 8:
                for n, v in zip(names, r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def build_worker(args, rank, world, device, config_path=None):
    from sgb200 import config as C
    from sgb200.models import model as M
    from sgb200.utils import misc
    from sgb200.worker import WORKER
    cfgs = C.Configurations(config_path or args.config)
    if args.batch and config_path is None:
        cfgs.OPTIMIZATION.batch_size = args.batch
    global_batch = cfgs.OPTIMIZATION.batch_size
    assert global_batch % world == 0
    cfgs.OPTIMIZATION.batch_size = global_batch // world           # per-rank batch, as src/loader.py:162
    cfgs.RUN.cuda_graphs = args.graphs == "on" or (args.graphs == "auto" and cfgs.OPTIMIZATION.batch_size <= 64)
    cfgs.OPTIMIZATION.world_size = world
    cfgs.RUN.distributed_data_parallel = world > 1
    cfgs.RUN.synchronized_bn = world > 1
    misc.fix_seed(0 + rank)                                         # seed + rank (src/loader.py:99)
    Gen, _, _, Dis, Gen_ema, _, _, ema = M.load_generator_discriminator(cfgs.DATA, cfgs.OPTIMIZATION, cfgs.MODEL, cfgs.STYLEGAN,
                                                                        cfgs.MODULES, cfgs.RUN, device, Logger())
    if world > 1:
        Gen, _, _, Dis, Gen_ema, _, _ = M.prepare_parallel_training(Gen, None, None, Dis, Gen_ema, None, None, cfgs.MODEL, world,
                                                                    True, True, cfgs.MODEL.apply_g_ema, device)
    cfgs.define_optimizer(Gen, Dis)
    worker = WORKER(cfgs=cfgs, run_name="bench", Gen=Gen, Gen_mapping=None, Gen_synthesis=None, Dis=Dis, Gen_ema=Gen_ema,
                    Gen_ema_mapping=None, Gen_ema_synthesis=None, ema=ema, eval_model=None, train_dataloader=None,
                    eval_dataloader=None, global_rank=rank, local_rank=device, mu=None, sigma=None, real_feats=None, logger=Logger())
    return cfgs, worker, global_batch


def run_steps(worker, n, read_losses):
    out = None
    for s in range(n):
        _, d_loss = worker.train_discriminator(s)
        g_loss = worker.train_generator(s)
        out = (d_loss, g_loss)
        if read_losses:
            out = (float(d_loss.detach()), float(g_loss.detach()))      # D2H read of the step's results
    return out


DUMP_SAMPLE = 1 << 22      # elements kept per network state: three states of 16 MB (float32) and the losses stay under 64 MB


def dump_outputs(worker, losses, out_dir):
    """What the last timed step hands back: both losses and the generator, discriminator and EMA-generator states it
    leaves (every floating-point tensor of each state_dict, flattened in key order).  A state of more than DUMP_SAMPLE
    elements is reduced to the elements at DUMP_SAMPLE sorted indices drawn from a fixed seed, so that two builds of the
    same model dump the same positions."""
    os.makedirs(out_dir, exist_ok=True)
    for name, v in zip(("d_loss", "g_loss"), losses):
        np.save(os.path.join(out_dir, name + ".npy"), torch.as_tensor(v).detach().float().reshape(1).cpu().numpy())
    for name, net in (("G_state", worker.Gen), ("D_state", worker.Dis), ("G_ema_state", worker.Gen_ema)):
        if net is None:
            continue
        flat = torch.cat([t.detach().float().flatten() for t in net.state_dict().values() if t.is_floating_point()])
        if flat.numel() > DUMP_SAMPLE:
            idx = torch.randint(0, flat.numel(), (DUMP_SAMPLE,), generator=torch.Generator().manual_seed(0)).sort().values
            flat = flat[idx.to(flat.device)]
        np.save(os.path.join(out_dir, name + ".npy"), flat.cpu().numpy())


def timed(worker, steps, world, read_losses):
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    losses = run_steps(worker, steps, read_losses)
    e1.record()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    ms = torch.tensor([e0.elapsed_time(e1)], device="cuda")
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    return float(ms) / steps, losses


def fid_eval_seconds(worker, cfgs, device, num_eval, batch, world=1):
    """BASELINE metric, second half: wall seconds of one FID-N evaluation (WORKER.evaluate: N generated images through
    G_ema -> quantise/resize/normalise -> InceptionV3 -> IS + FID), preceded by the reference-statistics pass over N
    synthetic uint8-valued reference images.  Inception weights are seeded (the pretrained file cannot be downloaded
    here), which changes no shape or FLOP."""
    from sgb200.metrics import features, fid
    from sgb200.metrics.preparation import LoadEvalModel
    ev = LoadEvalModel("InceptionV3_tf", "legacy", 1, False, device)
    gen = torch.Generator(device=device).manual_seed(1234)
    S = cfgs.DATA.img_size

    def ref_batches():
        for i in range(0, num_eval, batch * world):          # N > 1: each rank extracts its share, features are all-gathered
            n = min(batch, max(0, num_eval - i - batch * (dist.get_rank() if world > 1 else 0)))
            if n > 0:
                yield torch.randint(0, 256, (n, 3, S, S), generator=gen, device=device).float()
    # load cuSOLVER (the Frechet distance's two symmetric eigendecompositions) before anything is timed: on a fresh box the first
    # call pages the library in from disk, measured at 0.2 s to 30 s for the same code (profiles/r02_fid_n2_eval_phases.txt)
    _a = torch.randn(2048, 2048, dtype=torch.float64, device=device)
    _a = _a @ _a.t()
    torch.linalg.eigh(_a)
    torch.linalg.eigvalsh(_a)
    del _a
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    rf, _ = features.stack_real_features(ref_batches(), ev, False, device)
    if world > 1:
        sizes = [torch.zeros(1, dtype=torch.long, device=device) for _ in range(world)]
        dist.all_gather(sizes, torch.tensor([rf.shape[0]], device=device))
        mx = int(max(int(s) for s in sizes))
        pad = torch.zeros((mx, rf.shape[1]), device=device, dtype=rf.dtype)
        pad[:rf.shape[0]] = rf
        parts = [torch.empty_like(pad) for _ in range(world)]
        dist.all_gather(parts, pad)
        rf = torch.cat([p[:int(n)] for p, n in zip(parts, sizes)], 0)
    mu, sigma = fid.calculate_moments(rf)
    torch.cuda.synchronize()
    t_ref = time.perf_counter() - t0
    worker.eval_model, worker.mu, worker.sigma, worker.num_eval = ev, mu, sigma, num_eval
    bs = cfgs.OPTIMIZATION.batch_size
    cfgs.OPTIMIZATION.batch_size = batch
    try:
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        worker.evaluate(step=0, metrics=["is", "fid"], writing=False, training=True)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        t_eval = time.perf_counter() - t0
    finally:
        cfgs.OPTIMIZATION.batch_size = bs
    m = worker.last_metrics or {}
    return {"seconds": t_eval, "ref_stats_seconds": t_ref, "num_eval": num_eval, "batch": batch, "img_per_s": num_eval / t_eval,
            "FID": m.get("FID"), "IS": m.get("IS"), "n_gpus": world, "inception_weights": "seeded (pretrained FID weights unavailable offline)"}


def cpu_step_images_per_sec(config_path, batch, threads, n_steps=1):
    """The reference step restated by the oracle (fp32 CPU torch): 2 discriminator updates + 1 generator update with Adam,
    BigGAN-Deep 256x256, on ``threads`` host threads.  A bounded sample: ``batch`` images per step."""
    import yaml
    from oracle import studiogan_oracle as O
    from sgb200 import config as C
    from sgb200.models import model as M
    torch.set_num_threads(threads)
    cfgs = C.Configurations(config_path)
    torch.manual_seed(0)
    Gen, _, _, Dis, _, _, _, _ = M.load_generator_discriminator(cfgs.DATA, cfgs.OPTIMIZATION, _no_ema(cfgs.MODEL), cfgs.STYLEGAN,
                                                                 cfgs.MODULES, cfgs.RUN, "cpu", Logger())
    m = cfgs.MODEL
    sdG = {k: v.detach().clone() for k, v in Gen.state_dict().items()}
    sdD = {k: v.detach().clone() for k, v in Dis.state_dict().items()}
    pG = [k for k, _ in Gen.named_parameters()]
    pD = [k for k, _ in Dis.named_parameters()]
    del Gen, Dis
    kw_g = dict(img_size=cfgs.DATA.img_size, g_conv_dim=m.g_conv_dim, g_depth=m.g_depth, attn_g_loc=tuple(m.attn_g_loc), apply_attn=m.apply_attn)
    kw_d = dict(img_size=cfgs.DATA.img_size, d_conv_dim=m.d_conv_dim, d_depth=m.d_depth, attn_d_loc=tuple(m.attn_d_loc), apply_attn=m.apply_attn)
    optG = torch.optim.Adam([sdG[k].requires_grad_(True) for k in pG], lr=cfgs.OPTIMIZATION.g_lr, betas=(cfgs.OPTIMIZATION.beta1, cfgs.OPTIMIZATION.beta2), eps=1e-6)
    optD = torch.optim.Adam([sdD[k].requires_grad_(True) for k in pD], lr=cfgs.OPTIMIZATION.d_lr, betas=(cfgs.OPTIMIZATION.beta1, cfgs.OPTIMIZATION.beta2), eps=1e-6)
    S, nc = cfgs.DATA.img_size, cfgs.DATA.num_classes
    samples = []
    for it in range(n_steps + 1):           # iteration 0 warms the allocator / thread pool / oneDNN primitive caches, untimed
        t0 = time.perf_counter()
        for _ in range(cfgs.OPTIMIZATION.d_updates_per_step):
            optD.zero_grad()
            real, yr = torch.rand(batch, 3, S, S) * 2 - 1, torch.randint(0, nc, (batch,))
            yf = torch.randint(0, nc, (batch,))
            z = torch.randn(batch, m.z_dim)
            with torch.no_grad():
                fake = O.deep_generator(sdG, z, yf, track=False, **kw_g)
            a, _ = O.deep_discriminator(sdD, real, yr, **kw_d)
            b, _ = O.deep_discriminator(sdD, fake, yf, **kw_d)
            O.d_hinge(a, b).backward()
            optD.step()
        optG.zero_grad()
        yf = torch.randint(0, nc, (batch,))
        z = torch.randn(batch, m.z_dim)
        fake = O.deep_generator(sdG, z, yf, **kw_g)
        a, _ = O.deep_discriminator({k: v.detach() for k, v in sdD.items()}, fake, yf, **kw_d)
        O.g_hinge(a).backward()
        optG.step()
        if it > 0:
            samples.append(time.perf_counter() - t0)
    dt = float(np.sum(samples))
    return batch * len(samples) / dt, dt, [batch / t for t in samples]


def _no_ema(MODEL):
    import copy
    m = copy.copy(MODEL)
    m.apply_g_ema = False
    return m


def shutdown(worker, world):
    """Leave without hanging: captured CUDA graphs that contain NCCL kernels must die before the process group does, and a
    watchdog hard-exits if the teardown still blocks (the JSON line is already flushed by then)."""
    sys.stdout.flush()
    if world <= 1:
        return

    def _hard_exit():
        time.sleep(20.0)
        os._exit(0)
    threading.Thread(target=_hard_exit, daemon=True).start()
    if worker is not None:
        for name in ("_d_graph", "_g_graph"):
            if getattr(worker, name, None) is not None:
                setattr(worker, name, None)
    import gc
    gc.collect()
    torch.cuda.synchronize()
    try:
        dist.barrier()
        dist.destroy_process_group()
    except Exception:
        pass
    os._exit(0)


def config_dict(workload, cfgs_or_none, global_batch, world, graphs, S, d_updates, acml):
    per_rank = global_batch // world
    return {"workload": workload, "global_batch": global_batch, "per_gpu_batch": per_rank, "img_size": S,
            "d_updates_per_step": d_updates, "acml_steps": acml, "parallelism": "dp%d" % world, "cuda_graphs": bool(graphs),
            "l2": "per-step working set (tens of GB of activations) >> 126 MB L2; no explicit flush needed"}


def graphs_wanted(args, per_rank):
    return args.graphs == "on" or (args.graphs == "auto" and per_rank <= 64)


def reference_arm(args, workload):
    """The reference step on the host cores (oracle port: /root/reference does not travel to the GPU box), on OUR arm's
    config / metric / unit: each step is a bounded sample of the workload -- ``cpu_batch`` images of the 256-image batch
    through the full step (2 D updates + 1 G update, forward + backward + Adam) -- W warm-up steps, K timed steps."""
    import yaml
    from sgb200 import config as C
    cfgs = C.Configurations(args.config)
    threads = args.cpu_threads or min(32, os.cpu_count() or 1)
    global_batch = args.batch or cfgs.OPTIMIZATION.batch_size
    K, W = max(1, args.steps), max(1, args.warmup)
    # size the per-step sample so that W + K steps end within ~4 minutes: one probe step at the requested sample size
    batch = args.cpu_batch
    _, t_probe, _ = cpu_step_images_per_sec(args.config, batch, threads, n_steps=1)
    while batch > 1 and t_probe * (batch / args.cpu_batch) * (K + W) > 240.0:
        batch //= 2
    v, dt, per = cpu_step_images_per_sec(args.config, batch, threads, n_steps=K + W - 1)   # its iteration 0 is warm-up 1 of W
    per = per[W - 1:]
    v = float(len(per) / sum(1.0 / x for x in per))            # images / total seconds of the K timed steps
    cfg = config_dict(workload, cfgs, global_batch, args.gpus, graphs_wanted(args, global_batch // args.gpus), cfgs.DATA.img_size,
                      cfgs.OPTIMIZATION.d_updates_per_step, cfgs.OPTIMIZATION.acml_steps)
    sample = ("%d of the %d images of each step (full step: 2 D updates + 1 G update, fwd + bwd + Adam) on %d host threads; %d warm-up + "
              "%d timed steps; per-step img/s min %.3f max %.3f" % (batch, global_batch, threads, W, len(per), min(per), max(per)))
    return {"impl": "reference", "metric": METRIC_NAME.get(workload, workload), "value": v, "unit": "img/s", "n_gpus": args.gpus,
            "steps": len(per), "warmup": W, "ms_per_step": 1000.0 * batch / v, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": cfg,
            "cpu_baseline": {"value": v, "unit": "img/s", "cores": threads, "kind": "port", "sample": sample},
            "e2e": {"value": v, "unit": "img/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}


def measure(args, rank, world, device, config_path, steps, warmup, want_e2e, want_profile, dump_dir=None):
    """Warm-up + timed steps of one workload (device-resident baskets), optional output dump of the last timed step,
    per-kernel accounting step and e2e leg."""
    from sgb200 import _lib
    cfgs, worker, global_batch = build_worker(args, rank, world, device, config_path)
    opt = cfgs.OPTIMIZATION
    per_rank = opt.batch_size
    n_items = opt.acml_steps * opt.d_updates_per_step
    S = cfgs.DATA.img_size
    dev_loader = SyntheticBasketLoader(per_rank, n_items, S, cfgs.DATA.num_classes, 100 + rank, device=device)
    worker.train_dataloader, worker.train_iter = dev_loader, iter(dev_loader)
    run_steps(worker, warmup, False)
    sampler = ClockSampler(device.index)
    if rank == 0:
        sampler.start()
    launches0 = _lib.LAUNCHES[0]
    ms_step, losses = timed(worker, steps, world, False)
    launches = (_lib.LAUNCHES[0] - launches0)
    sampler.stop_flag = True
    if dump_dir and rank == 0:               # before the accounting step and the e2e leg train any further
        dump_outputs(worker, losses, dump_dir)
    res = {"cfgs": cfgs, "worker": worker, "global_batch": global_batch, "per_rank": per_rank, "S": S, "ms_step": ms_step,
           "value": global_batch * opt.acml_steps / (ms_step * 1e-3), "launches": launches, "clocks": sampler.summary() if rank == 0 else None,
           "graphs_captured": {n: bool(getattr(getattr(worker, n, None), "graph", None) is not None) for n in ("_d_graph", "_g_graph")},
           "prof": None, "prof_by_tag": None, "e2e": None}
    if want_profile:
        try:
            _lib.PROFILE["events"] = []
            _lib.PROFILE["enabled"] = True
            graphs_on, cfgs.RUN.cuda_graphs = cfgs.RUN.cuda_graphs, False      # the accounting step runs eagerly (events per call)
            torch.cuda.synchronize()
            w0 = time.perf_counter()
            run_steps(worker, 1, False)
            torch.cuda.synchronize()
            prof_wall_ms = (time.perf_counter() - w0) * 1e3
            _lib.PROFILE["enabled"] = False
            cfgs.RUN.cuda_graphs = graphs_on
            agg, by_tag = {}, {}
            for tag, flops, e0, e1, nbytes in _lib.PROFILE["events"]:
                ms = e0.elapsed_time(e1)
                for key, store in ((tag.split(" ")[0], agg), (tag, by_tag)):
                    a = store.setdefault(key, [0.0, 0.0, 0, 0.0])
                    a[0] += ms; a[1] += flops; a[2] += 1; a[3] += nbytes
            _lib.PROFILE["events"] = []
            res["prof"] = {k: {"ms": v[0], "tflops": (v[1] / (v[0] * 1e-3) * 1e-12) if v[0] > 0 and v[1] > 0 else None, "launches": v[2],
                               "flop": v[1], "gbytes": v[3] * 1e-9, "gb_per_s": (v[3] / (v[0] * 1e-3) * 1e-9) if v[0] > 0 and v[3] > 0 else None}
                           for k, v in agg.items()}
            res["prof_by_tag"] = by_tag
            if rank == 0 and args.kernel_breakdown:
                with open(args.kernel_breakdown, "w") as fh:
                    json.dump({"wall_ms_of_profiled_step": prof_wall_ms, "sum_ms": sum(v[0] for v in agg.values()), "by_kind": res["prof"],
                               "by_tag": [{"tag": k, "ms": v[0], "n": v[2], "flop": v[1], "bytes": v[3]} for k, v in
                                          sorted(by_tag.items(), key=lambda kv: -kv[1][0])]}, fh, indent=1)
        except Exception as ex:  # accounting must never take the bench line down
            _lib.PROFILE["enabled"] = False
            res["prof"] = {"error": repr(ex)}
    if want_e2e:
        # the product data path (sgb200/data_util.py): a uint8 NHWC dataset in host memory (synthetic, 3 baskets), baskets gathered
        # into pinned staging buffers, H2D on a side stream, flip + ToTensor + Normalize on the device; both losses read back
        from sgb200 import data_util
        rs = np.random.RandomState(200 + rank)
        basket = per_rank * n_items
        ds = data_util.Dataset_.from_arrays(rs.randint(0, 256, size=(3 * basket, S, S, 3), dtype=np.uint8),
                                            rs.randint(0, cfgs.DATA.num_classes, size=3 * basket), random_flip=True)
        host_loader = data_util.DeviceBasketLoader(ds, basket, device, shuffle=True, seed=200 + rank)
        worker.train_dataloader, worker.train_iter = host_loader, iter(host_loader)
        run_steps(worker, 1, True)
        ms_e2e, _ = timed(worker, steps, world, True)
        res["e2e"] = {"value": global_batch * opt.acml_steps / (ms_e2e * 1e-3), "unit": "img/s",
                      "h2d_bytes_per_step": world * host_loader.h2d_bytes, "d2h_bytes_per_step": 8 * world, "ms_per_step": ms_e2e,
                      "input": "uint8 NHWC baskets from pinned host memory (%d B/step/rank), device-side flip + normalise" % host_loader.h2d_bytes}
        worker.train_dataloader = worker.train_iter = None
        host_loader.close()
        del host_loader, ds
    return res


def release(res):
    """Drop a measured workload (graphs first: they pin their memory pools) so the next one starts from an empty allocator."""
    w = res.pop("worker", None)
    if w is not None:
        for name in ("_d_graph", "_g_graph"):
            if getattr(w, name, None) is not None:
                setattr(w, name, None)
    res.pop("cfgs", None)
    del w
    import gc
    gc.collect()
    torch.cuda.empty_cache()


def main():
    args = parse()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    workload = os.path.splitext(os.path.basename(args.config))[0]

    if args.impl == "reference":
        if rank != 0:
            return
        print(json.dumps(reference_arm(args, workload)))
        return

    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=device)
    from sgb200 import _lib
    _lib.check(_lib.load().sgb_device_check(), "sgb_device_check")
    # N > 1: numeric check of the data-parallel path before anything is timed (N ranks x 4 images == 1 rank x 4N images:
    # sync-BN forward / backward exchanges, arena gradient all-reduce, running statistics); reported in the JSON line
    mr_check = None
    if world > 1:
        try:
            from sgb200.utils.ddp_check import multirank_parity_check
            mr_check = multirank_parity_check(device)
        except Exception as ex:  # noqa: BLE001
            mr_check = {"ok": False, "error": repr(ex)}

    res = measure(args, rank, world, device, None, args.steps, args.warmup, not args.no_e2e, True, args.dump_outputs)
    cfgs, worker, global_batch, per_rank, S = res["cfgs"], res["worker"], res["global_batch"], res["per_rank"], res["S"]
    opt = cfgs.OPTIMIZATION
    ms_step, value, prof = res["ms_step"], res["value"], res["prof"]

    fid50k = None
    if not args.no_fid:                       # every rank takes part (features are all-gathered when N > 1)
        try:
            fid50k = fid_eval_seconds(worker, cfgs, device, args.fid_num, min(256, per_rank), world)
        except Exception as ex:  # the evaluation timing must never take the bench line down
            fid50k = {"error": repr(ex)}
    release(res)

    # ---- BASELINE configs 2 / 3 / 5 at the world sizes they are defined for (same timing rules, no accounting step)
    also = {}
    if not args.no_also and not args.batch:
        for name, worlds in ALSO:
            if world not in worlds or name == workload:
                continue
            try:
                r = measure(args, rank, world, device, os.path.join(PKG, "configs", name + ".yaml"), max(3, min(args.steps, 10)), 3,
                            True, False)
                gf = STEP_GFLOP_PER_IMAGE.get(name, 0.0) * 1e9 * r["global_batch"]
                also[name] = {"metric": METRIC_NAME[name], "value": r["value"], "unit": "img/s", "ms_per_step": r["ms_step"],
                              "global_batch": r["global_batch"], "img_size": r["S"], "d_updates_per_step": r["cfgs"].OPTIMIZATION.d_updates_per_step,
                              "e2e": r["e2e"], "gpu_launches": r["launches"], "cuda_graphs_captured": r["graphs_captured"],
                              "step_tflops_per_gpu": gf / (r["ms_step"] * 1e-3) * 1e-12 / world}
                release(r)
            except Exception as ex:  # noqa: BLE001
                also[name] = {"error": repr(ex)}

    if rank != 0:
        shutdown(None, world)
        return

    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak_tf = peaks.get("bf16_tflops_sustained", 1400.0)
    peak_src = "MEASURED_PEAKS.json bf16_tflops_sustained" if "bf16_tflops_sustained" in peaks else "fallback 1.4 PFLOP/s sustained"
    step_flop = STEP_GFLOP_PER_IMAGE.get(workload, 0.0) * 1e9 * global_batch
    # roofline.traffic: DRAM bytes per launch of the dominant kernel from this round's committed `ncu --set full` captures
    # (profiles/r02_ncu_traffic.json, one record per conv kernel kind, written from the .ncu-rep files of profiles/ncu_target.py)
    traffic_db = {}
    try:
        traffic_db = json.load(open(os.path.join(ROOT, "profiles", "r02_ncu_traffic.json")))
    except Exception:
        pass
    traffic, traffic_note = None, "no ncu capture of the current kernel committed"
    roof = {"bound": "tensor", "unit": "TFLOP/s", "peak": peak_tf, "peak_source": peak_src, "traffic": traffic, "traffic_note": traffic_note,
            "step_algorithmic_tflop": step_flop * 1e-12,
            "step_achieved": step_flop / (ms_step * 1e-3) * 1e-12 / world,
            "step_frac": step_flop / (ms_step * 1e-3) * 1e-12 / world / peak_tf}
    CONV_KINDS = ("conv3x3_rows", "conv_fprop_kxk", "conv_fprop_1x1", "conv_wgrad")
    if isinstance(prof, dict) and any(kk in prof for kk in CONV_KINDS):
        hbm = peaks.get("hbm_gbs", 6500.0)
        # every conv kernel class is listed under roofline.kernels with both of its rates (TFLOP/s and GB/s) and its share of the step
        kname = {"conv3x3_rows": "conv3x3_rows_kernel (3x3 fprop + dgrad, halo rows, tcgen05)",
                 "conv_fprop_kxk": "conv_fprop_kernel on k x k filters (fprop + dgrad, tcgen05)",
                 "conv_fprop_1x1": "conv_fprop_kernel on 1x1 filters / GEMMs (fprop + dgrad, tcgen05; HBM bound)",
                 "conv_wgrad": "conv_wgrad_kernel + wgrad3x3_c64_kernel (weight gradients, tcgen05)"}
        # dominant = the conv kernel class with the most time in the accounting step.  The 1x1 launches of conv_fprop_kernel are
        # HBM bound (K = 32..128 channels: a few FLOP per byte), the others tensor bound; the roofline is reported accordingly.
        dom = max((kk for kk in CONV_KINDS if kk in prof), key=lambda kk: prof[kk]["ms"])
        k = prof[dom]
        if dom in traffic_db:
            traffic, traffic_note = traffic_db[dom]["dram_bytes_per_launch"], traffic_db[dom]["note"]
            roof["traffic_algorithmic_bytes_of_that_launch"] = traffic_db[dom]["algorithmic_bytes"]
        roof["traffic"], roof["traffic_note"] = traffic, traffic_note
        if dom == "conv_fprop_1x1":
            roof.update({"bound": "hbm", "unit": "GB/s", "peak": hbm, "peak_source": "MEASURED_PEAKS.json hbm_gbs (copy)"})
        ew = {kk: vv for kk, vv in prof.items() if kk not in CONV_KINDS and vv.get("gbytes")}
        ew_ms = sum(v["ms"] for v in ew.values())
        ew_gb = sum(v["gbytes"] for v in ew.values())
        ach = k["gb_per_s"] if roof["bound"] == "hbm" else k["tflops"]
        roof.update({"kernel": kname[dom], "achieved": ach, "frac": ach / roof["peak"],
                     "kernel_ms_per_step": k["ms"], "kernel_share_of_step": k["ms"] / ms_step,
                     "kernel_algorithmic_gbytes_per_step": k["gbytes"], "kernel_gb_per_s": k["gb_per_s"],
                     "kernels": {kname[kk]: dict(prof[kk], frac_of_tensor_peak=(prof[kk]["tflops"] or 0.0) / peak_tf,
                                                 frac_of_hbm_copy_peak=(prof[kk]["gb_per_s"] or 0.0) / hbm,
                                                 share_of_step=prof[kk]["ms"] / ms_step)
                                 for kk in CONV_KINDS if kk in prof},
                     "streaming_kernels": {"ms_per_step": ew_ms, "algorithmic_gbytes_per_step": ew_gb,
                                           "gb_per_s": ew_gb / (ew_ms * 1e-3) if ew_ms > 0 else None, "hbm_peak_gb_per_s": hbm,
                                           "frac_of_hbm_copy_peak": (ew_gb / (ew_ms * 1e-3) / hbm) if ew_ms > 0 else None}})
    else:
        roof.update({"achieved": roof["step_achieved"], "frac": roof["step_frac"], "kernels": prof})

    cpu = None
    if not args.no_cpu_baseline and world == 1:
        threads = args.cpu_threads or min(32, os.cpu_count() or 1)
        try:
            v, dt, per = cpu_step_images_per_sec(args.config, args.cpu_batch, threads, n_steps=3)
            cpu = {"value": v, "unit": "img/s", "cores": threads, "kind": "port",
                   "sample": "%d of the %d images of each step (2 D updates + 1 G update, fwd+bwd+Adam); 1 warm-up + 3 timed steps, %.1f s; "
                             "per-step img/s min %.3f max %.3f" % (args.cpu_batch, global_batch, dt, min(per), max(per))}
        except Exception as ex:
            cpu = {"value": None, "unit": "img/s", "cores": threads, "kind": "port", "sample": "failed: %r" % (ex,)}

    cfg = config_dict(workload, cfgs, global_batch, world, graphs_wanted(args, per_rank), S, opt.d_updates_per_step, opt.acml_steps)
    cfg["cuda_graphs_captured"] = res["graphs_captured"]
    cfg["also_measured"] = also
    e2e = res["e2e"]
    if e2e is not None and isinstance(fid50k, dict) and "seconds" in fid50k:
        e2e["fid50k_eval_seconds"] = fid50k["seconds"]                 # second half of BASELINE's metric
        e2e["fid50k_ref_stats_seconds"] = fid50k["ref_stats_seconds"]
    line = {"metric": METRIC_NAME.get(workload, workload + " G+D step images/sec"), "value": value, "unit": "img/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "bf16", "data": "synthetic", "config": cfg,
            "e2e": e2e, "gpu_launches": res["launches"], "roofline": roof, "cpu_baseline": cpu, "fid50k": fid50k, "multirank_check": mr_check,
            "clocks": res["clocks"]}
    print(json.dumps(line))
    shutdown(None, world)


if __name__ == "__main__":
    main()
