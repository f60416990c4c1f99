#!/usr/bin/env python
"""The RPN head after its 3x3 conv at bench.py's shapes (batch 8, P2-P6 of a 608x1024 batch, 256 channels, 3 anchors):
ops.rpn_head against the stock composition (ATen bias add_, relu_, two biased 1x1 cuDNN convs and autograd's backward
of them), forward, backward and both, CUDA events over --iters repetitions after a warm-up.  Byte model of the native
passes: forward reads c and writes 15 outputs per pixel; backward reads c and the 15 incoming gradients and writes c's
gradient.  Rates are set against the copy bandwidth measured in the same run (a 2 GB device-to-device copy: read +
write bytes over time).  Prints one JSON line per measurement.  Usage: python tools/rpn_head_bench.py [--iters 20]
"""
import argparse, json, subprocess, sys
from pathlib import Path
import torch
import torch.nn.functional as F
sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
from dgod_b200 import ops

ap = argparse.ArgumentParser()
ap.add_argument("--iters", type=int, default=20)
args = ap.parse_args()
dev = torch.device("cuda")
torch.backends.cudnn.benchmark = True
card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                      capture_output=True, text=True).stdout.strip()
print(json.dumps({"card": card}))
LEVELS, N = ((152, 256), (76, 128), (38, 64), (19, 32), (10, 16)), 8
g = torch.Generator(device=dev).manual_seed(0)
cs = [torch.randn(N, 256, h, w, device=dev, generator=g).to(memory_format=torch.channels_last).requires_grad_(True)
      for h, w in LEVELS]
params = [(torch.randn(*s, device=dev, generator=g) * 0.05).requires_grad_(True)
          for s in ((256,), (3, 256, 1, 1), (3,), (12, 256, 1, 1), (12,))]
g_out = [torch.randn(N, k, h, w, device=dev, generator=g) for k in (3, 12) for h, w in LEVELS]


def stock(cs, bias, w_cls, b_cls, w_bbox, b_bbox):
    obj, dl = [], []
    for c in cs:
        t = torch.relu_(c + bias.view(1, -1, 1, 1))
        obj.append(F.conv2d(t, w_cls, b_cls))
        dl.append(F.conv2d(t, w_bbox, b_bbox))
    return obj, dl


def timed(fn):
    for _ in range(3):
        fn()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(args.iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / args.iters


src = torch.empty(2 ** 29, device=dev)
dst = torch.empty_like(src)
copy_gbs = 2 * src.numel() * 4 / timed(lambda: dst.copy_(src)) / 1e6
del src, dst
print(json.dumps({"copy_peak_GBps": round(copy_gbs, 1)}))
S = sum(c.numel() for c in cs) * 4
small = sum(c[:, 0].numel() for c in cs) * 4 * 15
model = {"fwd": S + small, "bwd": 2 * S + small, "fwd+bwd": 3 * S + 2 * small}


def fwd(f):
    with torch.no_grad():
        f(cs, *params)


def bwd_of(f):
    obj, dl = f(cs, *params)
    outs = obj + dl
    return lambda: torch.autograd.grad(outs, cs + params, g_out, retain_graph=True)


def both(f):
    obj, dl = f(cs, *params)
    torch.autograd.grad(obj + dl, cs + params, g_out)


for name, f in (("native", ops.rpn_head), ("stock", stock)):
    for what, run in (("fwd", lambda: fwd(f)), ("bwd", bwd_of(f)), ("fwd+bwd", lambda: both(f))):
        ms = timed(run)
        print(json.dumps({"impl": name, "pass": what, "ms": round(ms, 4), "model_MB": round(model[what] / 1e6, 1),
                          "GBps": round(model[what] / ms / 1e6, 1),
                          "share_of_copy_peak": round(model[what] / ms / 1e6 / copy_gbs, 3)}))
