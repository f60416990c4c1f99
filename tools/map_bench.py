"""Times the GPU validation mAP (dgod_b200.metrics.MeanAveragePrecision) against the numpy restatement of pycocotools'
arithmetic (oracle/coco_map.py) on one synthetic validation set, and checks that their precision / recall tables are
bitwise equal.

Workload: --images synthetic images (default 5 000), 100 detections and on average 8 ground truths each over 9
classes, fed to update() in batches of --batch images; both torchmetrics threshold sets ([0.5], the reference's
setting, and the default 10 IoU thresholds).  About half of the detections are jittered copies of a ground truth, the
rest are random boxes, so precision and recall both vary.  The GPU time covers every update() plus compute(),
bracketed by CUDA events after one untimed warm-up pass over the same set; the host time is the oracle's.
Prints one JSON line with the GPU's name and power limit read in the same run.

    python tools/map_bench.py [--images 5000] [--batch 8] [--out results/map_bench.json]
"""
from __future__ import annotations

import argparse
import json
import subprocess
import sys
import time
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

from dgod_b200 import synth  # noqa: E402
from dgod_b200.metrics import MeanAveragePrecision  # noqa: E402
from oracle import coco_map  # noqa: E402

H, W = 600, 1200


def make_set(n_img: int, seed: int = 0):
    g = synth.gen(seed)
    preds, targets = [], []
    for _ in range(n_img):
        m = int(torch.randint(4, 13, (1,), generator=g))              # 4..12 ground truths, mean 8
        gt = synth.random_boxes(m, H, W, g)
        glab = torch.randint(1, 10, (m,), generator=g)
        det = synth.random_boxes(100, H, W, g)
        lab = torch.randint(1, 10, (100,), generator=g)
        use = torch.rand(100, generator=g) < 0.5
        pick = torch.randint(0, m, (100,), generator=g)
        det[use] = gt[pick[use]] + torch.randn(int(use.sum()), 4, generator=g) * 4
        lab[use] = glab[pick[use]]
        preds.append({"boxes": det, "scores": torch.rand(100, generator=g), "labels": lab})
        targets.append({"boxes": gt, "labels": glab})
    return preds, targets


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                           capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
        name, power = [s.strip() for s in q.split(",")]
    except Exception:                         # no nvidia-smi: the name from torch, the limit unknown
        name, power = torch.cuda.get_device_name(), "unknown"
    return name, power


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--images", type=int, default=5000)
    ap.add_argument("--batch", type=int, default=8)
    ap.add_argument("--out", type=str, default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("map_bench.py needs a CUDA device")
    preds, targets = make_set(args.images)
    dp = [{k: v.cuda() for k, v in p.items()} for p in preds]
    dt = [{k: v.cuda() for k, v in t.items()} for t in targets]
    hp = [{k: v.numpy() for k, v in p.items()} for p in preds]
    ht = [{k: v.numpy() for k, v in t.items()} for t in targets]
    name, power = gpu_info()
    result = {"tool": "map_bench", "gpu": name, "power_limit": power, "images": args.images, "batch": args.batch,
              "dets_per_image": 100, "gts": sum(len(t["labels"]) for t in targets), "classes": 9, "runs": []}
    for iou in ([0.5], torch.linspace(0.5, 0.95, 10).tolist()):
        metric = MeanAveragePrecision(iou_thresholds=iou, class_metrics=True)

        def run():
            metric.reset()
            for b in range(0, len(dp), args.batch):
                metric.update(dp[b:b + args.batch], dt[b:b + args.batch])
            e_mid.record()
            return metric.compute()

        e0, e_mid, e1 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
        run()                                                    # warm-up: allocator, pinned staging, module load
        torch.cuda.synchronize()
        t_host = time.perf_counter()
        e0.record()
        out = run()
        e1.record()
        torch.cuda.synchronize()
        wall = time.perf_counter() - t_host
        t0 = time.perf_counter()
        ref = coco_map.mean_average_precision(hp, ht, iou, metric.rec_thresholds, metric.max_det)
        t_oracle = time.perf_counter() - t0
        equal = bool(np.array_equal(metric.precision.cpu().numpy().view(np.int64), ref["precision"].view(np.int64))
                     and np.array_equal(metric.recall.cpu().numpy().view(np.int64), ref["recall"].view(np.int64)))
        result["runs"].append({
            "iou_thresholds": len(iou), "gpu_update_ms": round(e0.elapsed_time(e_mid), 3),
            "gpu_update_compute_ms": round(e0.elapsed_time(e1), 3), "host_wall_ms": round(wall * 1e3, 3),
            "oracle_host_ms": round(t_oracle * 1e3, 1), "tables_bitwise_equal": equal,
            "map": float(out["map"]), "map_50": float(out["map_50"]),
            "map_diff_vs_oracle": abs(float(metric.stats64["map"]) - ref["map"])})
    line = json.dumps(result)
    print(line)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(line + "\n")
    if not all(r["tables_bitwise_equal"] for r in result["runs"]):
        raise SystemExit("map_bench: the GPU tables differ from the oracle's")


if __name__ == "__main__":
    main()
