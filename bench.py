#!/usr/bin/env python
"""Benchmark of the DGOD hot path (BASELINE.json `metric`): DG training images/s of the detector step.

    python bench.py --gpus N --steps K --warmup W                      # this repo's CUDA path (DGFRCNN dg, configs[1])
    python bench.py --model fcos ...                                   # DGFCOS dg (configs[2])
    python bench.py --exp non_dg ...                                   # mode 0 only (DGFRCNN.py:128)
    python bench.py --impl reference --gpus N --steps K --warmup W     # the reference's own code on the host CPU
    python bench.py ... --dump-outputs DIR                             # also save the last timed step's results (.npy)

A *step* is one pass of the reference's 8-training-step mode cycle (0,1,0,2,0,3,0,4 — DGFRCNN.py:125-199,
DGFCOS.py:164-243; `non_dg`: eight mode-0 steps) over synthetic 3x800x1333 batches: 8*B images per GPU, optimizer
step included in every training step.  Rank 0 prints ONE JSON line.
  value        whole-job images/s with the batches resident in HBM, CUDA-event timed, max over ranks
  e2e          the same loop fed from pinned host memory (H2D of images + targets and D2H of the loss inside the
               timed region)
  roofline     the dominant dgod_b200 kernel: algorithmic bytes / CUDA-event time of its launches in the timed
               region vs the measured HBM copy peak (MEASURED_PEAKS.json); `traffic` from the committed ncu capture
  cpu_baseline (N=1) the reference's own modules (baseline/_ref, else the oracle port) on the host cores, bounded sample
  extras       (N=1, --model frcnn --exp dg) the same step with 3 source domains (the D of the multi-GPU runs, so
               that the scaling curve has an identical-D point at N=1), mode-0-only img/s (`non_dg`), and `tv_cuda`:
               the UNMODIFIED reference modules with stock torchvision CUDA ops on the same GPU — what the step costs
               without this repo's kernels and host mirror
"""
from __future__ import annotations

import argparse
import gc
import json
import os
import statistics
import subprocess
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

IMG_H, IMG_W, N_GT = 800, 1333, 20
REG_WEIGHTS = [0.5, 0.5, 0.5, 0.05, 0.0001]
CYCLE = (0, 1, 0, 2, 0, 3, 0, 4)
# The reference fine-tunes COCO-pretrained weights at lr 2e-3 (DGFRCNN.py:81,85,99) / 1e-4 (DGFCOS.py); those weights
# cannot be downloaded here.  A random-init detector at 2e-3 diverges to NaN within a few steps whatever the sampler
# does (it is the backbone / RPN that blows up), after which the proposals — and with them the work of the hot path —
# disappear.  All arms therefore run the same optimizer kernels with a tiny rate (override with --lr) so that every
# timed step does the full, representative work.
BENCH_LR = 1e-5
FALLBACK_HBM_GBS = 6650.0  # /opt/skills/guides/B200_PROFILING.md


def parse():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=3)
    p.add_argument("--warmup", type=int, default=3)
    p.add_argument("--impl", default="b200", choices=["b200", "reference"])
    p.add_argument("--model", default="frcnn", choices=["frcnn", "fcos"], help="DGFRCNN (configs[1]) or DGFCOS (configs[2])")
    p.add_argument("--exp", default="dg", choices=["dg", "non_dg"])
    p.add_argument("--batch", type=int, default=8, help="images per GPU per training step")
    p.add_argument("--domains", type=int, default=0, help="source domains (default 2 at N=1, 3 at N>1: configs[1] / configs[4])")
    p.add_argument("--lr", type=float, default=BENCH_LR)
    p.add_argument("--no-cpu-baseline", action="store_true")
    p.add_argument("--no-e2e", action="store_true")
    p.add_argument("--no-extras", action="store_true", help="skip the D=3 / non_dg / tv_cuda side measurements at N=1")
    p.add_argument("--no-graph-backbone", action="store_true",
                   help="run the backbone eagerly (default: its forward and backward are captured as CUDA graphs)")
    p.add_argument("--no-fold-bn", action="store_true",
                   help="keep FrozenBatchNorm2d as separate elementwise passes (default: folded into the conv, utils.py)")
    p.add_argument("--memory-format", default="channels_last", choices=["channels_last", "contiguous"],
                   help="memory format of the detector's convolutions / FPN features")
    p.add_argument("--dump-outputs", metavar="DIR",
                   help="write what the last timed step computed to DIR/*.npy (see dump_outputs), to compare two builds")
    return p.parse_args()


# --------------------------------------------------------------------------------------------- helpers
class ClockSampler:
    """nvidia-smi clocks + throttle reasons sampled every 200 ms while the timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.rows, self.proc, self.thread, self.gpu = [], None, None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            self.proc = None
            return
        self.thread = threading.Thread(target=self._read, daemon=True)
        self.thread.start()

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

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
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
            except (ValueError, IndexError):
                continue
            for n, v in zip(names, r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def synthetic_batches(n_batches, batch, n_domains, seed0, pin=False):
    """DrivingDataset-shaped tuples (DrivingDataset.py:71 / DGcommon.collate_fn): images float
    [3,800,1333] in [0,1), boxes, labels 1..8, domain = i mod D.  Seeds 1000*rank + batch index."""
    from dgod_b200 import synth
    out = []
    for j in range(n_batches):
        imgs = synth.random_images(batch, IMG_H, IMG_W, seed0 + j)
        targets, dom = synth.random_targets(batch, N_GT, IMG_H, IMG_W, seed0 + j, n_domains)
        boxes = [t["boxes"] for t in targets]
        labels = [t["labels"] for t in targets]
        if pin:
            imgs = [i.pin_memory() for i in imgs]
            boxes = [b.pin_memory() for b in boxes]
            labels = [l.pin_memory() for l in labels]
        out.append((imgs, boxes, labels, dom))
    return out


def to_device(batch, dev):
    """Images and targets to the device; the domain ids stay on the host as in the reference (DGcommon.collate_fn builds
    them with torch.tensor(domain), DGFRCNN.py:150 moves them inside training_step)."""
    imgs, boxes, labels, dom = batch
    return ([i.to(dev, non_blocking=True) for i in imgs], [b.to(dev, non_blocking=True) for b in boxes],
            [l.to(dev, non_blocking=True) for l in labels], dom)


def batch_bytes(batch):
    imgs, boxes, labels, dom = batch
    return sum(t.numel() * t.element_size() for t in (*imgs, *boxes, *labels, dom))


def measured_hbm_peak():
    f = ROOT / "MEASURED_PEAKS.json"
    if f.exists():
        try:
            return float(json.loads(f.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return FALLBACK_HBM_GBS, "fallback (B200_PROFILING.md)"


def calibrate(detector, imgs):
    """Random init with calibrated frozen-BN statistics (dgod_b200/utils.py) — every arm."""
    import torch
    from dgod_b200.utils import calibrate_frozen_bn
    with torch.no_grad():
        image_list, _ = detector.transform([i for i in imgs[:2]], None)
        calibrate_frozen_bn(detector.backbone, image_list.tensors)


def cycle_modes(exp):
    return CYCLE if exp == "dg" else (0,) * len(CYCLE)


DUMP_PER_TENSOR = 1 << 15


def dump_outputs(out_dir, model, losses):
    """Writes what one timed step hands back to its caller, in float32:
      losses.npy  the loss returned by each training step of the step, in schedule order
      params.npy  every parameter after the step's last optimizer update, concatenated in named_parameters() order
    A tensor of more than DUMP_PER_TENSOR elements contributes a fixed sample of them (positions drawn by a generator
    seeded with the parameter's name), so that runs and builds are compared entry for entry (about 10 MB for either
    model).  Gradients are left out: after a few cycles the nondeterministic order of GPU reductions has changed which
    proposals survive NMS, and the last backward's gradients are mostly run-to-run noise (two runs of the same build,
    --steps 3 --warmup 3 on one B200 at 1000 W: gradients 49 % apart in relative L2 norm, losses at most 0.6 %,
    parameters 1e-5)."""
    import zlib

    import numpy as np
    import torch
    out = Path(out_dir)
    out.mkdir(parents=True, exist_ok=True)
    params = []
    for name, p in model.named_parameters():
        n = p.numel()
        idx = (np.arange(n) if n <= DUMP_PER_TENSOR else
               np.sort(np.random.default_rng(zlib.crc32(name.encode())).choice(n, DUMP_PER_TENSOR, replace=False)))
        params.append(p.detach().flatten()[torch.from_numpy(idx).to(p.device)])
    np.save(out / "losses.npy", torch.stack(losses).float().cpu().numpy())
    np.save(out / "params.npy", torch.cat(params).float().cpu().numpy())


# --------------------------------------------------------------------------------------------- CUDA arm
class B200Run:
    """One model instance of this repo on the current device + the loops that time it."""

    def __init__(self, args, model_name, exp, n_dom, dev, rank, world, graph_backbone=True):
        import torch
        import torch.distributed as dist
        self.torch, self.dist = torch, dist
        self.args, self.exp, self.n_dom, self.dev, self.world = args, exp, n_dom, dev, world
        B = args.batch
        torch.manual_seed(0)
        if model_name == "frcnn":
            from dgod_b200.dg import DGFRCNN
            model = DGFRCNN(9, B, exp, REG_WEIGHTS, n_dom)
        else:
            from dgod_b200.dg_fcos import DGFCOS
            model = DGFCOS(9, B, exp, REG_WEIGHTS, n_dom)
        model = model.to(dev).train()
        if args.memory_format == "channels_last":
            # NHWC is what cuDNN's tensor-core convolutions run natively; the FPN maps then reach the RoIAlign kernels
            # channels-last (lanes = channels, no staging)
            model = model.to(memory_format=torch.channels_last)
        self.model = model
        self.host = synthetic_batches(4, B, n_dom, 1000 * rank, pin=True)
        self.resident = [to_device(b, dev) for b in self.host]
        calibrate(model.detector, self.resident[0][0])
        self.n_folded = 0
        if not args.no_fold_bn:
            from dgod_b200.utils import fold_frozen_bn
            self.n_folded = fold_frozen_bn(model.detector.backbone)
        if world > 1:
            for t in list(model.parameters()) + list(model.buffers()):
                dist.broadcast(t.data, 0)
        self.graphed = False
        if graph_backbone and not args.no_graph_backbone and model_name == "frcnn":
            # The ResNet-50-FPN forward and backward are ~4 000 small PyTorch/cuDNN launches per training step with static
            # shapes (every batch is padded to the same size): capture them as two CUDA graphs.  The hot-path kernels, the
            # heads and the losses stay eager (data-dependent proposal counts).
            det = model.detector
            with torch.no_grad():
                shape = det.transform([i for i in self.resident[0][0]], None)[0].tensors.shape
            sample = torch.rand(shape, device=dev)
            det.backbone = torch.cuda.make_graphed_callables(det.backbone, (sample,), num_warmup_iters=3)
            self.graphed = True
        self.opt = model.configure_optimizer(lr=args.lr)
        self.sync = None
        if world > 1:
            from dgod_b200.ddp import GradSync
            self.sync = GradSync(list(model.parameters()), world, bucket_bytes=int(os.environ.get("DGOD_BUCKET_MB", "32")) << 20)
        self.copy_stream = torch.cuda.Stream(device=dev)
        self.modes = cycle_modes(exp)
        torch.cuda.synchronize()

    def train_step(self, batch):
        mode = self.model.mode
        loss = self.model.training_step(batch)
        if self.sync is not None:
            # gradients are views of one flat buffer; buckets are all-reduced from backward hooks while backward runs
            self.sync.begin(mode)
            loss.backward()
            self.sync.finish()          # the synthetic domain ids are i mod D on every rank: the touched heads agree
        else:
            self.opt.zero_grad(set_to_none=True)
            loss.backward()
        self.opt.step()
        return loss

    def prefetch(self, b):
        """H2D copy of one step's inputs from pinned host memory on the copy stream (as a DataLoader with pin_memory +
        non_blocking does); the returned event orders it before the step that uses it."""
        torch = self.torch
        main = torch.cuda.current_stream()
        with torch.cuda.stream(self.copy_stream):
            d = to_device(b, self.dev)
            for t in (*d[0], *d[1], *d[2]):
                t.record_stream(main)
            ev = torch.cuda.Event()
            ev.record(self.copy_stream)
        return d, ev

    def cycle(self, from_host: bool):
        torch = self.torch
        n = len(self.modes)
        if not from_host:
            # detached: the losses outlive the cycle for dump_outputs, their autograd graphs do not
            self.losses = [self.train_step(self.resident[(s // 2) % 4]).detach() for s in range(n)]
            return self.losses[-1]
        # end to end: every step's inputs come from the host and every step's loss goes back to it.  The copy of step s+1
        # overlaps the compute of step s, and the loss of step s is read while step s+1 is queued (the host stays one step
        # ahead instead of draining the GPU after every step).
        nxt = self.prefetch(self.host[0])
        pending = None
        for s in range(n):
            cur, ev = nxt
            torch.cuda.current_stream().wait_event(ev)
            if s + 1 < n:
                nxt = self.prefetch(self.host[((s + 1) // 2) % 4])
            loss = self.train_step(cur)
            if pending is not None:
                pending.item()              # D2H read of the previous step's result
            pending = loss
        return pending.item()

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def timed(self, n_cycles: int, from_host: bool):
        torch = self.torch
        self.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n_cycles):
            self.cycle(from_host)
        e1.record()
        self.barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=self.dev)
        if self.world > 1:
            self.dist.all_reduce(ms, op=self.dist.ReduceOp.MAX)
        return float(ms.item())

    def reset_schedule(self):
        self.model.mode = self.model.sub_mode = 0

    def img_per_cycle(self):
        return len(self.modes) * self.args.batch * self.world

    def release(self):
        self.model = self.opt = self.sync = self.resident = self.host = None
        gc.collect()
        self.torch.cuda.empty_cache()


def side_measure(args, model_name, exp, n_dom, dev, steps):
    """img/s of another configuration of this repo's path on the same GPU (N=1 extras)."""
    run = B200Run(args, model_name, exp, n_dom, dev, 0, 1)
    for _ in range(max(1, min(args.warmup, 2))):
        run.cycle(False)
    ms = run.timed(steps, False)
    v = steps * run.img_per_cycle() / (ms / 1e3)
    run.release()
    return {"value": round(v, 2), "unit": "img/s", "ms_per_step": round(ms / steps, 2), "domains": n_dom, "exp": exp,
            "steps": steps}


def tv_cuda_measure(args, model_name, n_dom, dev, steps):
    """The UNMODIFIED reference modules (baseline/_ref) with stock torchvision CUDA ops on this GPU: same synthetic
    batches, same schedule, same optimizer kernels and learning rate.  None when the reference is not installed."""
    import torch
    from oracle import ref_real
    if not ref_real.available():
        return {"unavailable": "baseline/_ref is not installed (python -m oracle.install_ref)"}
    B = args.batch
    torch.manual_seed(0)
    build = ref_real.build_dgfrcnn if model_name == "frcnn" else ref_real.build_dgfcos
    model = build(9, B, "dg", REG_WEIGHTS, n_dom).to(dev).train()
    host = synthetic_batches(4, B, n_dom, 0)
    resident = [(torch.stack(b[0]).to(dev), [x.to(dev) for x in b[1]], [x.to(dev) for x in b[2]], b[3]) for b in host]
    calibrate(model.detector, list(resident[0][0]))
    opt = model.configure_optimizers()[0][0]
    for g in opt.param_groups:
        g["lr"] = args.lr

    def step(b, i):
        loss = model.training_step(b, i)["loss"]
        opt.zero_grad(set_to_none=True)
        loss.backward()
        opt.step()
        return loss

    def cycle():
        for s in range(len(CYCLE)):
            step(resident[(s // 2) % 4], s)

    cycle()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        cycle()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    out = {"value": round(steps * len(CYCLE) * B / (ms / 1e3), 2), "unit": "img/s", "ms_per_step": round(ms / steps, 2),
           "steps": steps, "domains": n_dom,
           "what": "unmodified reference modules (baseline/_ref) + stock torchvision CUDA ops, eager, fp32, same GPU"}
    del model, opt, resident
    gc.collect()
    torch.cuda.empty_cache()
    return out


def run_b200(args):
    import torch
    import torch.distributed as dist
    from dgod_b200 import _lib, ops

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the dgod_b200 path has no CPU fallback")
    rank = int(os.environ.get("RANK", 0))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    n_dom = args.domains or (2 if world == 1 else 3)
    B = args.batch
    torch.backends.cudnn.benchmark = True
    run = B200Run(args, args.model, args.exp, n_dom, dev, rank, world)

    for _ in range(args.warmup):
        run.cycle(False)
    clocks = ClockSampler(local_rank)
    if rank == 0 and not os.environ.get("DGOD_BENCH_NO_CLOCKS"):
        clocks.start()
    ops.KernelTimer.enabled = True
    ops.KernelTimer.reset()
    launches0 = _lib.launch_count()
    torch.cuda.profiler.start()      # `ncu --profile-from-start off` then lists exactly the timed region
    ms = run.timed(args.steps, False)
    torch.cuda.profiler.stop()
    launches = _lib.launch_count() - launches0
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, run.model, run.losses)
    final_loss = float(run.train_step(run.resident[0]).item())   # untimed: is the run still numerically sane?
    run.reset_schedule()
    ops.KernelTimer.enabled = False
    kern = ops.KernelTimer.summary()
    clk = clocks.stop() if rank == 0 else None
    imgs_per_cycle = run.img_per_cycle()
    value = args.steps * imgs_per_cycle / (ms / 1e3)

    e2e = None
    if not args.no_e2e:
        run.cycle(True)
        run.reset_schedule()
        ms_e = run.timed(args.steps, True)
        n = len(run.modes)
        h2d = sum(batch_bytes(run.host[(s // 2) % 4]) for s in range(n))
        e2e = {"value": round(args.steps * imgs_per_cycle / (ms_e / 1e3), 3), "unit": "img/s",
               "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4 * n, "ms_per_step": round(ms_e / args.steps, 3)}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    peak, peak_src = measured_hbm_peak()
    roof, kernels = None, {}
    for name, (n, tot_ms, tot_bytes) in kern.items():
        gbs = tot_bytes / 1e9 / (tot_ms / 1e3) if tot_ms > 0 else 0.0
        kernels[name] = {"launches": n, "avg_us": round(1e3 * tot_ms / max(n, 1), 2), "GB/s": round(gbs, 1),
                         "share_of_step": round(tot_ms / ms, 4)}
    if kern:
        pick = [k for k in kern if k.startswith("msroi")] or list(kern)
        top = max(pick, key=lambda k: kern[k][1])
        n, tot_ms, tot_bytes = kern[top]
        ach = tot_bytes / 1e9 / (tot_ms / 1e3)
        traffic = None
        tf = ROOT / "profiles" / "roofline_traffic.json"
        if tf.exists():
            try:
                traffic = json.loads(tf.read_text()).get(top)
            except Exception:
                traffic = None
        roof = {"kernel": top, "bound": "hbm", "achieved": round(ach, 1), "peak": peak, "unit": "GB/s",
                "frac": round(ach / peak, 4), "traffic": traffic, "peak_source": peak_src,
                "launches": n, "avg_launch_us": round(1e3 * tot_ms / n, 2)}
    n_folded, graphed = run.n_folded, run.graphed
    model_title = "DGFRCNN" if args.model == "frcnn" else "DGFCOS"
    out = {
        "metric": f"{model_title} {args.exp} train img/s", "value": round(value, 3), "unit": "img/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(ms / args.steps, 3),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"{model_title} {args.exp} mode, {n_dom} synthetic source domains, instance+image domain "
                               f"classifiers with GRL, batch {B}/GPU, R50-FPN random init (stem + layer1 frozen as with the "
                               f"reference's pretrained=True), 3x{IMG_H}x{IMG_W} images (detector min/max 600/1200 -> 608x1024), "
                               f"{N_GT} GT/img; step = one 8-training-step mode cycle "
                               f"{','.join(map(str, run.modes))} incl. optimizer steps ({len(run.modes) * B} img/GPU)",
                   "model": args.model, "exp": args.exp,
                   "batch_per_gpu": B, "domains": n_dom, "parallelism": f"dp{world}",
                   "cache": "per-step working set (>1 GB of activations) exceeds the 126 MB L2; no flush needed",
                   "optimizer": (f"SGD wd 5e-4 as DGFRCNN.py:98-104" if args.model == "frcnn" else "Adam wd 1e-4 as DGFCOS.py:140-146")
                                + f", lr {args.lr} (random init diverges at the reference's rate: bench.py BENCH_LR)",
                   "gradient_sync": "none (1 GPU)" if world == 1 else
                                    "NCCL all-reduce (avg) per 32 MB bucket of one flat gradient buffer, launched from backward hooks (dgod_b200/ddp.py)",
                   "memory_format": args.memory_format,
                   "backbone_math": "PyTorch defaults (cuDNN conv may use TF32, matmul fp32); hot-path kernels fp32",
                   "frozen_bn": (f"{n_folded} FrozenBatchNorm2d layers evaluated as the epilogue of their conv "
                                 "(conv(x, w*s) + shift, same function and parameters; dgod_b200/utils.py)") if n_folded
                   else "separate elementwise passes (torchvision default)",
                   "backbone_launch": "forward and backward captured as CUDA graphs (torch.cuda.make_graphed_callables)"
                   if graphed else "eager"},
        "e2e": e2e, "gpu_launches": launches, "clocks": clk, "roofline": roof, "kernels": kernels,
        "loss_finite": bool(torch.isfinite(torch.as_tensor(final_loss)).all()),
    }
    if world == 1:
        run.release()
        if not args.no_extras and args.model == "frcnn" and args.exp == "dg":
            steps = max(1, min(args.steps, 2))
            extras = {}
            try:
                if n_dom != 3:
                    extras["dg_3_domains"] = side_measure(args, "frcnn", "dg", 3, dev, steps)
                extras["non_dg"] = side_measure(args, "frcnn", "non_dg", n_dom, dev, steps)
                extras["tv_cuda"] = tv_cuda_measure(args, "frcnn", n_dom, dev, steps)
            except Exception as e:                      # a side measurement must never cost the headline line
                extras["error"] = f"{type(e).__name__}: {e}"
            out["extras"] = extras
        if not args.no_cpu_baseline:
            out["cpu_baseline"] = cpu_reference_sample(args.model, args.exp, 1, 1, 2, n_dom, args.lr)["cpu_baseline"]
    print(json.dumps(out), flush=True)
    if world > 1:
        dist.destroy_process_group()


# --------------------------------------------------------------------------------------------- CPU arm
def cpu_reference_sample(model_name: str, exp: str, steps: int, warmup: int, batch: int, n_dom: int, lr: float):
    """The reference's CPU path on all host threads, bounded: one step = one full mode cycle at `batch` images per
    training step.  Runs the reference's OWN modules from baseline/_ref (kind "reference": DGFRCNN.training_step /
    DGFCOS.training_step unmodified, `.cuda()` made a no-op on the host); without that install, the oracle port
    (oracle/ref_dgfrcnn.py, FRCNN only, kind "port")."""
    import torch
    from oracle import ref_real
    cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    torch.set_num_threads(cores)
    torch.manual_seed(0)
    batches = synthetic_batches(4, batch, n_dom, 0)
    modes = cycle_modes(exp)
    if ref_real.available():
        kind = "reference"
        ref_real.load(cpu_shims=True)       # on a GPU box too: this arm is the reference on the HOST cores
        build = ref_real.build_dgfrcnn if model_name == "frcnn" else ref_real.build_dgfcos
        model = build(9, batch, exp, REG_WEIGHTS, n_dom).train()
        calibrate(model.detector, batches[0][0] + batches[1][0])
        opt = model.configure_optimizers()[0][0]
        for g in opt.param_groups:
            g["lr"] = lr
        batches = [(torch.stack(b[0]), b[1], b[2], b[3]) for b in batches]      # DGcommon.collate_fn stacks the images

        def step(b, i):
            loss = model.training_step(b, i)["loss"]
            opt.zero_grad(set_to_none=True)
            loss.backward()
            opt.step()

        def reset():
            model.mode = model.sub_mode = 0
        what = "the reference's own modules (baseline/_ref) on torchvision CPU ops"
    else:
        if model_name != "frcnn":
            raise SystemExit("bench.py: the DGFCOS CPU arm needs the reference install (python -m oracle.install_ref)")
        from oracle.ref_dgfrcnn import RefDGFRCNN
        kind = "port"
        model = RefDGFRCNN(9, batch, REG_WEIGHTS, n_dom).train()
        if exp != "dg":
            model.CYCLE = (0,)
        calibrate(model.detector, batches[0][0] + batches[1][0])
        opt = model.configure_optimizer(lr=lr)

        def step(b, i):
            loss = model.training_step(b)
            opt.zero_grad(set_to_none=True)
            loss.backward()
            opt.step()

        def reset():
            model.step_index = 0
        what = "oracle/ref_dgfrcnn.py (port of the reference step) on torchvision CPU ops"

    for _ in range(warmup):            # one untimed mode-0 step is enough to warm the allocator
        step(batches[0], 0)
        reset()
    t0 = time.perf_counter()
    for _ in range(steps):
        for s in range(len(modes)):
            step(batches[(s // 2) % 4], s)
    dt = time.perf_counter() - t0
    n_img = steps * len(modes) * batch
    v = n_img / dt
    return {"value": v, "ms_per_step": 1e3 * dt / steps,
            "cpu_baseline": {"value": round(v, 4), "unit": "img/s", "cores": cores, "kind": kind,
                             "sample": f"{steps} {exp} mode cycle(s) at batch {batch} ({n_img} images of 3x{IMG_H}x{IMG_W}), "
                                       f"{what}, {cores} threads, {dt:.1f} s"}}


def run_reference(args):
    rank = int(os.environ.get("RANK", 0))
    if rank != 0:
        return
    # the GPU arm's workload (same model, schedule, batch per training step and domain count); steps / warm-up capped
    # so that the run ends within a few minutes on the host cores (one cycle at batch 8 is 64 images, about a minute)
    steps, warmup = min(args.steps, 1), min(args.warmup, 1)
    n_dom = args.domains or (2 if args.gpus == 1 else 3)        # same rule as the CUDA arm
    r = cpu_reference_sample(args.model, args.exp, steps, warmup, args.batch, n_dom, args.lr)
    model_title = "DGFRCNN" if args.model == "frcnn" else "DGFCOS"
    out = {
        "impl": "reference", "metric": f"{model_title} {args.exp} train img/s", "value": round(r["value"], 4), "unit": "img/s",
        "n_gpus": args.gpus, "steps": steps, "warmup": warmup, "ms_per_step": round(r["ms_per_step"], 1),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"{model_title} {args.exp} mode on the host CPU: step = one 8-training-step mode cycle at batch "
                               f"{args.batch} (the GPU arm's per-GPU workload: same 3x{IMG_H}x{IMG_W} synthetic images, same detector, "
                               "schedule, optimizer and learning rate); steps/warmup capped at 1/1 to stay within minutes",
                   "model": args.model, "exp": args.exp, "batch_per_gpu": args.batch, "domains": n_dom, "parallelism": "cpu"},
        "cpu_baseline": r["cpu_baseline"],
        "e2e": {"value": round(r["value"], 4), "unit": "img/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(out), flush=True)


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_b200(a)
