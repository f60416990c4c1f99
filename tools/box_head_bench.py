#!/usr/bin/env python
"""The box head's six matrix products (fc6 / fc7 x forward / dgrad / wgrad) at bench.py's shapes: dgod_linear_tc
(3xTF32 on tcgen05, split pass included) against cuBLAS's fp32 SGEMM on the same inputs, CUDA events over --iters
launches after a warm-up.  Useful work = 2*m*n*k fp32 FLOP.  Also prints each product's error against a float64
matmul, |C - C64| / (|A| @ |B|), max and RMS, for both.  Usage: python tools/box_head_bench.py [--rois 4096] [--iters 50]
"""
import argparse, json, subprocess, sys
from pathlib import Path
import torch
sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
from dgod_b200 import ops

ap = argparse.ArgumentParser()
ap.add_argument("--rois", type=int, default=4096)
ap.add_argument("--iters", type=int, default=50)
args = ap.parse_args()
dev = torch.device("cuda")
torch.backends.cuda.matmul.allow_tf32 = False
card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                      capture_output=True, text=True).stdout.strip()
print(json.dumps({"card": card}))
g = torch.Generator(device=dev).manual_seed(0)
M = args.rois


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


def err(c, a, b):
    """max and RMS of |C - C64| / (|A| @ |B|^T) with A [m, k], B [n, k] (float64)."""
    a64, b64 = a.double(), b.double()
    ref = a64 @ b64.t()
    den = a64.abs() @ b64.abs().t()
    e = (c.double() - ref).abs() / den.clamp_min(1e-300)
    return float(e.max()), float(e.square().mean().sqrt())


for layer, (n_out, k_in) in (("fc6", (1024, 256 * 7 * 7)), ("fc7", (1024, 1024))):
    x = torch.randn(M, k_in, device=dev, generator=g)
    w = torch.randn(n_out, k_in, device=dev, generator=g) * k_in ** -0.5
    dy = torch.randn(M, n_out, device=dev, generator=g)
    cases = {
        # name: (tc call, cuBLAS call, A [m, k], B [n, k])
        "forward": (lambda: ops.linear_tc(x, w), lambda: x @ w.t(), x, w),
        "dgrad": (lambda: ops.linear_tc(dy, w, b_trans=True), lambda: dy @ w, dy, w.t()),
        "wgrad": (lambda: ops.linear_tc(dy, x, a_trans=True, b_trans=True), lambda: dy.t() @ x, dy.t(), x.t()),
    }
    for prod, (tc, blas, a, b) in cases.items():
        m, k = a.shape
        n = b.shape[0]
        flop = 2.0 * m * n * k
        t_tc, t_blas = timed(tc), timed(blas)
        e_tc, e_blas = err(tc(), a, b), err(blas(), a, b)
        print(json.dumps({"layer": layer, "product": prod, "m": m, "n": n, "k": k,
                          "tc_ms": round(t_tc, 4), "tc_tflops": round(flop / t_tc / 1e9, 1),
                          "sgemm_ms": round(t_blas, 4), "sgemm_tflops": round(flop / t_blas / 1e9, 1),
                          "speedup": round(t_blas / t_tc, 2), "tc_err_max_rms": e_tc, "sgemm_err_max_rms": e_blas}))
