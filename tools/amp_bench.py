"""fp32 against bf16 autocast on bench.py's workload: the DGFRCNN dg 8-step cycle at batch 8, synthetic 3x800x1333 images,
folded backbone, channels_last, the backbone's forward and backward captured as CUDA graphs in both arms (the bf16 arm
captures under torch.autocast(cache_enabled=False), the mode make_graphed_callables requires).  The two arms are timed
alternately in one process, ROUNDS rounds each, and the median img/s and the spread of each arm are reported.  Then the
native backbone epilogues are timed in isolation at the bench's shapes, fp32 and bf16, with CUDA events: bytes moved over
kernel time, against bench.measured_hbm_peak().  The card's name and power limit are read in the same run.

    python tools/amp_bench.py [--rounds 3] [--steps 3] [--out /tmp/amp_bench.json]

Prints one JSON line (and writes it to --out when given)."""
from __future__ import annotations

import argparse
import contextlib
import json
import statistics
import subprocess
import sys
import types
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

import torch  # noqa: E402

import bench  # noqa: E402
from dgod_b200 import ops  # noqa: E402

BF = torch.bfloat16


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clock = [s.strip() for s in out.split(",")]
        return {"name": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:                       # the numbers are still reported, marked as unattributed
        return {"name": torch.cuda.get_device_name(0), "power_limit": f"unknown ({type(e).__name__})"}


def make_run(amp: bool, dev):
    """bench.B200Run without its own graph capture; the backbone is captured here, under autocast for the bf16 arm."""
    args = types.SimpleNamespace(batch=8, memory_format="channels_last", no_fold_bn=False, no_graph_backbone=True,
                                 lr=bench.BENCH_LR)
    run = bench.B200Run(args, "frcnn", "dg", 2, dev, 0, 1, graph_backbone=False)
    det = run.model.detector
    with torch.no_grad():
        shape = det.transform([i for i in run.resident[0][0]], None)[0].tensors.shape
    ctx = torch.autocast("cuda", dtype=BF, cache_enabled=False) if amp else contextlib.nullcontext()
    with ctx:
        det.backbone = torch.cuda.make_graphed_callables(det.backbone, (torch.rand(shape, device=dev),),
                                                         num_warmup_iters=3)
    if amp:
        step = run.model.training_step

        def training_step(batch):
            with torch.autocast("cuda", dtype=BF, cache_enabled=False):
                return step(batch)
        run.model.training_step = training_step
    torch.cuda.synchronize()
    return run


def time_epilogues(peak):
    """(kernel, dtype) -> CUDA-event time per launch and bytes / time at the bench's shapes (batch 8, 608x1024 input)."""
    g = torch.Generator(device="cuda").manual_seed(0)
    cl = torch.channels_last

    def m(shape, dt):
        return torch.randn(shape, generator=g, device="cuda").to(dt).contiguous(memory_format=cl)

    out = {}
    for dt in (torch.float32, BF):
        c256, r256 = m((8, 256, 152, 256), dt), m((8, 256, 152, 256), dt)
        s256 = torch.randn(256, generator=g, device="cuda")
        lat, coarse = m((8, 256, 152, 256), dt), m((8, 256, 76, 128), dt)
        g_lb = m((8, 256, 76, 128), dt)
        stem, s64 = m((8, 64, 304, 512), dt), torch.randn(64, generator=g, device="cuda")
        cases = {
            "shift_relu (8x256x152x256, plain)": lambda: ops._shift_relu_fwd(c256, s256, None, None),
            "shift_relu (8x256x152x256, downsample tail)": lambda: ops._shift_relu_fwd(c256, s256, r256, s256),
            "fpn_merge_fwd (P2 <- P3)": lambda: ops.fpn_merge(lat, s256, coarse),
            "fpn_merge_bwd (P3 <- P2)": lambda: ops.fpn_merge_backward(lat, g_lb, coarse.shape),
            "stem_pool (8x64x304x512)": lambda: ops.stem_pool(stem, s64),
        }
        for name, fn in cases.items():
            ops.KernelTimer.enabled = True
            for _ in range(5):
                fn()
            ops.KernelTimer.reset()
            for _ in range(50):
                fn()
            torch.cuda.synchronize()
            (launches, ms, nbytes), = ops.KernelTimer.summary().values()
            ops.KernelTimer.enabled = False
            gbs = nbytes / 1e9 / (ms / 1e3)
            out[f"{name} {'bf16' if dt == BF else 'fp32'}"] = {
                "us": round(1e3 * ms / launches, 2), "MB": round(nbytes / launches / 1e6, 1), "GB/s": round(gbs, 1),
                "of_peak": round(gbs / peak, 3)}
    return out


def main():
    p = argparse.ArgumentParser()
    p.add_argument("--rounds", type=int, default=3)
    p.add_argument("--steps", type=int, default=3, help="8-step cycles per timed round")
    p.add_argument("--warmup", type=int, default=2)
    p.add_argument("--out")
    a = p.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("amp_bench.py: no CUDA device")
    dev = torch.device("cuda", 0)
    torch.backends.cudnn.benchmark = True
    runs = {"fp32": make_run(False, dev), "bf16_autocast": make_run(True, dev)}
    for run in runs.values():
        for _ in range(a.warmup):
            run.cycle(False)
    rates = {k: [] for k in runs}
    for _ in range(a.rounds):
        for k, run in runs.items():
            ms = run.timed(a.steps, False)
            rates[k].append(a.steps * run.img_per_cycle() / (ms / 1e3))
    finite = {k: bool(torch.isfinite(torch.stack(run.losses)).all()) for k, run in runs.items()}
    for run in runs.values():
        run.release()
    peak, peak_src = bench.measured_hbm_peak()
    arms = {k: {"median_img_s": round(statistics.median(v), 2), "min": round(min(v), 2), "max": round(max(v), 2),
                "spread": round((max(v) - min(v)) / statistics.median(v), 4), "rounds": [round(x, 2) for x in v],
                "losses_finite": finite[k]} for k, v in rates.items()}
    out = {"what": "DGFRCNN dg 8-step cycle, batch 8, 3x800x1333 synthetic (608x1024 padded), folded backbone, "
                   "channels_last, backbone forward+backward as CUDA graphs in both arms; arms alternated",
           "card": card(), "steps_per_round": a.steps, "arms": arms,
           "bf16_over_fp32": round(arms["bf16_autocast"]["median_img_s"] / arms["fp32"]["median_img_s"], 4),
           "epilogue_kernels": time_epilogues(peak), "hbm_peak_GBs": peak, "hbm_peak_source": peak_src}
    line = json.dumps(out)
    print(line, flush=True)
    if a.out:
        Path(a.out).parent.mkdir(parents=True, exist_ok=True)
        Path(a.out).write_text(line + "\n")


if __name__ == "__main__":
    main()
