"""Validation mAP on the GPU: torchmetrics' `MeanAveragePrecision` (bbox, xyxy, pycocotools arithmetic) for the subset
the reference uses (DGcommon.py:127,154-172), with the matching and accumulation in `csrc/map_eval.cu`.

`update()` enqueues one `dgod_map_match` launch per call and keeps its per-detection records on the device: it never
reads anything back, so a validation loop does not wait on the host.  `compute()` reads back the class list and a NaN
flag, orders the records with one stable sort and runs `dgod_map_accumulate`.  The precision / recall tables are
bit-identical with pycocotools'; the means are float64 sums in another order (within 1e-12), returned as float32 like
torchmetrics.  Not supported (rejected): crowd ground truths, box formats other than xyxy, segmentation IoU; area
ranges and `mar_1` / `mar_10` are not computed.  Boxes are expected with x2 >= x1, y2 >= y1 and an area below 1e10
(pycocotools' "all" range), as the detectors produce them.
"""
from __future__ import annotations

import ctypes as C
from typing import Dict, List, Optional, Sequence

import torch
from torch import Tensor

from ._lib import check, load

MAX_DETS_PER_IMAGE = 4096       # DGOD_MAP_MAX_DETS_PER_IMAGE: one image's detections sort in shared memory
MAX_GTS_PER_IMAGE = 1024        # DGOD_MAP_MAX_GTS_PER_IMAGE
MAX_IOU_THRESHOLDS = 32         # a detection's matches are one 32-bit mask


def _p(t: Tensor) -> C.c_void_p:
    return C.c_void_p(t.data_ptr())


def _to_device(values, dtype, device) -> Tensor:
    """A small host-built tensor moved without blocking the host (pinned staging, asynchronous copy)."""
    return torch.tensor(values, dtype=dtype).pin_memory().to(device, non_blocking=True)


def _mean_valid(x: Tensor, dims=None) -> Tensor:
    """COCOeval.summarize: mean of the entries > -1, -1 where there are none (no host read)."""
    valid = x > -1
    n = valid.sum() if dims is None else valid.sum(dims)
    s = torch.where(valid, x, torch.zeros_like(x))
    s = s.sum() if dims is None else s.sum(dims)
    return torch.where(n > 0, s / n.clamp(min=1), torch.full_like(s, -1.0))


class MeanAveragePrecision:
    """torchmetrics.detection.MeanAveragePrecision with the same names, on CUDA tensors only.

    Only the last (largest) of `max_detection_thresholds` is used.  `compute()` returns `map`, `map_50`, `map_75`,
    `mar_100` (named after torchmetrics' default 100 whatever the value), `map_per_class`, `mar_100_per_class` and
    `classes`; the float64 tables of the last `compute()` stay on the object as `precision` [T, R, K] and
    `recall` [T, K]."""

    def __init__(self, box_format: str = "xyxy", iou_type: str = "bbox",
                 iou_thresholds: Optional[Sequence[float]] = None, rec_thresholds: Optional[Sequence[float]] = None,
                 max_detection_thresholds: Optional[Sequence[int]] = None, class_metrics: bool = False):
        if box_format != "xyxy":
            raise ValueError(f"MeanAveragePrecision: only box_format='xyxy' is supported, got {box_format!r}")
        if iou_type != "bbox":
            raise ValueError(f"MeanAveragePrecision: only iou_type='bbox' is supported, got {iou_type!r}")
        # torchmetrics builds its defaults with float32 linspace on the CPU; the recall grid is not k / 100
        self.iou_thresholds = [float(t) for t in iou_thresholds] if iou_thresholds is not None else \
            torch.linspace(0.5, 0.95, round((0.95 - 0.5) / 0.05) + 1).tolist()
        self.rec_thresholds = [float(r) for r in rec_thresholds] if rec_thresholds is not None else \
            torch.linspace(0.0, 1.00, round(1.00 / 0.01) + 1).tolist()
        if not 1 <= len(self.iou_thresholds) <= MAX_IOU_THRESHOLDS:
            raise ValueError(f"MeanAveragePrecision: 1..{MAX_IOU_THRESHOLDS} IoU thresholds, got {len(self.iou_thresholds)}")
        if not self.rec_thresholds:
            raise ValueError("MeanAveragePrecision: at least one recall threshold is needed")
        self.max_detection_thresholds = sorted(int(m) for m in (max_detection_thresholds or [1, 10, 100]))
        self.max_det = self.max_detection_thresholds[-1]
        if self.max_det < 1:
            raise ValueError("MeanAveragePrecision: max_detection_thresholds must be positive")
        self.class_metrics = bool(class_metrics)
        self.precision: Optional[Tensor] = None
        self.recall: Optional[Tensor] = None
        self._thr: Dict[str, Tensor] = {}
        self.reset()

    def reset(self) -> None:
        self._scores: List[Tensor] = []
        self._labels: List[Tensor] = []
        self._tp: List[Tensor] = []
        self._kept: List[Tensor] = []
        self._gt_labels: List[Tensor] = []

    def _thresholds(self, device) -> Tensor:
        key = str(device)
        if key not in self._thr:
            self._thr[key] = _to_device(self.iou_thresholds, torch.float64, device)
        return self._thr[key]

    def update(self, preds: List[Dict[str, Tensor]], target: List[Dict[str, Tensor]]) -> None:
        """Matches one batch: `preds` of dicts boxes [n,4] / scores [n] / labels [n], `target` of dicts boxes [m,4] /
        labels [m], CUDA tensors.  Enqueues one launch; reads nothing back."""
        if len(preds) != len(target):
            raise ValueError(f"MeanAveragePrecision.update: {len(preds)} predictions for {len(target)} targets")
        if not preds:
            return
        boxes, scores, labels, g_boxes, g_labels, nd, ng = [], [], [], [], [], [], []
        for p, t in zip(preds, target):
            if "iscrowd" in t:
                raise ValueError("MeanAveragePrecision: crowd ground truths ('iscrowd') are not supported")
            for name, d, keys in (("preds", p, ("boxes", "scores", "labels")), ("target", t, ("boxes", "labels"))):
                for k in keys:
                    if k not in d:
                        raise ValueError(f"MeanAveragePrecision.update: {name} entry without '{k}'")
                    if not isinstance(d[k], Tensor) or not d[k].is_cuda:
                        raise RuntimeError(f"MeanAveragePrecision.update: {name}['{k}'] must be a CUDA tensor "
                                           "(there is no CPU fallback)")
            n, m = p["boxes"].shape[0] if p["boxes"].numel() else 0, t["boxes"].shape[0] if t["boxes"].numel() else 0
            if p["scores"].numel() != n or p["labels"].numel() != n or t["labels"].numel() != m:
                raise ValueError("MeanAveragePrecision.update: boxes, scores and labels disagree in length")
            if n > MAX_DETS_PER_IMAGE or m > MAX_GTS_PER_IMAGE:
                raise ValueError(f"MeanAveragePrecision.update: an image has {n} detections and {m} ground truths; "
                                 f"at most {MAX_DETS_PER_IMAGE} and {MAX_GTS_PER_IMAGE} are supported")
            boxes.append(p["boxes"].reshape(n, 4))
            scores.append(p["scores"].reshape(n))
            labels.append(p["labels"].reshape(n))
            g_boxes.append(t["boxes"].reshape(m, 4))
            g_labels.append(t["labels"].reshape(m))
            nd.append(n)
            ng.append(m)
        dev = boxes[0].device
        boxes = torch.cat(boxes).float().contiguous()
        scores = torch.cat(scores).float().contiguous()
        labels = torch.cat(labels).long().contiguous()
        g_boxes = torch.cat(g_boxes).float().contiguous()
        g_labels = torch.cat(g_labels).long().contiguous()
        tp = torch.zeros(scores.shape[0], dtype=torch.int32, device=dev)
        kept = torch.zeros(scores.shape[0], dtype=torch.uint8, device=dev)
        if sum(nd):
            d_off, g_off = [0], [0]
            for a, b in zip(nd, ng):
                d_off.append(d_off[-1] + a)
                g_off.append(g_off[-1] + b)
            d_off = _to_device(d_off, torch.int32, dev)
            g_off = _to_device(g_off, torch.int32, dev)
            st = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
            check(load().dgod_map_match(_p(boxes), _p(scores), _p(labels), _p(d_off), _p(g_boxes), _p(g_labels),
                                        _p(g_off), len(nd), max(nd), max(ng), _p(self._thresholds(dev)),
                                        len(self.iou_thresholds), self.max_det, _p(tp), _p(kept), st), ValueError)
        self._scores.append(scores)
        self._labels.append(labels)
        self._tp.append(tp)
        self._kept.append(kept)
        self._gt_labels.append(g_labels)

    def compute(self) -> Dict[str, Tensor]:
        T, R = len(self.iou_thresholds), len(self.rec_thresholds)
        if not self._scores:
            raise RuntimeError("MeanAveragePrecision.compute: update() was never called")
        scores = torch.cat(self._scores)
        labels = torch.cat(self._labels)
        tp = torch.cat(self._tp)
        kept = torch.cat(self._kept).bool()
        g_labels = torch.cat(self._gt_labels)
        dev = scores.device
        classes = torch.unique(torch.cat([labels, g_labels]))                 # sorted
        if bool(torch.isnan(scores).any()):
            raise ValueError("MeanAveragePrecision.compute: NaN detection scores")
        K = int(classes.numel())
        precision = torch.full((T, R, K), -1.0, dtype=torch.float64, device=dev)
        recall = torch.full((T, K), -1.0, dtype=torch.float64, device=dev)
        if K:
            # records grouped by class, descending score; the stable sort keeps (update, image, detection) order on
            # ties, which is pycocotools' order.  -0.0 + 0.0 = +0.0: the two zeros share one key, as numpy sees them.
            bits = (scores + 0.0).view(torch.int32).to(torch.int64) & 0xFFFFFFFF
            ordered = torch.where(bits >= 0x80000000, bits ^ 0xFFFFFFFF, bits | 0x80000000)
            cls = torch.where(kept, torch.searchsorted(classes, labels), torch.full_like(labels, K))
            key, perm = torch.sort(cls * (1 << 32) + (0xFFFFFFFF - ordered), stable=True)
            tp_sorted = tp[perm].contiguous()
            seg = torch.searchsorted(key, torch.arange(K + 1, device=dev, dtype=torch.int64) * (1 << 32)).to(torch.int32)
            gt_count = torch.zeros(K, dtype=torch.int32, device=dev)
            gt_count.index_add_(0, torch.searchsorted(classes, g_labels),
                                torch.ones(g_labels.shape[0], dtype=torch.int32, device=dev))
            rec = _to_device(self.rec_thresholds, torch.float64, dev)
            lib = load()
            n = int(tp_sorted.numel())
            ws = torch.empty(max(int(lib.dgod_map_accumulate_workspace_bytes(n, T)), 1), dtype=torch.uint8, device=dev)
            st = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
            check(lib.dgod_map_accumulate(_p(tp_sorted) if n else None, _p(seg), _p(gt_count), K, n, _p(rec), R, T,
                                          _p(precision), _p(recall), _p(ws), ws.numel(), st))
        self.precision, self.recall = precision, recall

        def at(thr: float) -> Tensor:
            idx = [i for i, v in enumerate(self.iou_thresholds) if v == thr]
            return _mean_valid(precision[idx]) if idx else torch.tensor(-1.0, dtype=torch.float64, device=dev)

        self.stats64 = {"map": _mean_valid(precision), "map_50": at(0.5), "map_75": at(0.75),
                        "mar_100": _mean_valid(recall)}
        if self.class_metrics:
            self.stats64["map_per_class"] = _mean_valid(precision, (0, 1))
            self.stats64["mar_100_per_class"] = _mean_valid(recall, 0)
        else:
            self.stats64["map_per_class"] = torch.tensor(-1.0, dtype=torch.float64, device=dev)
            self.stats64["mar_100_per_class"] = torch.tensor(-1.0, dtype=torch.float64, device=dev)
        out = {k: v.float() for k, v in self.stats64.items()}
        out["classes"] = classes.to(torch.int32)
        return out


class DetectionValidation:
    """The validation hooks of the reference's DGModel (DGcommon.py:154-172) for a DG module holding `self.detector`:
    every validation batch updates a mAP@0.5 metric, the epoch end reports `val_acc` (map_50, what the reference's
    checkpointing monitors) and the per-class mAP, then resets."""

    def _val_metric(self) -> MeanAveragePrecision:
        if getattr(self, "_map_metric", None) is None:
            self._map_metric = MeanAveragePrecision(iou_thresholds=[0.5], class_metrics=True)   # DGcommon.py:127
        return self._map_metric

    def validation_step(self, batch) -> List[Dict[str, Tensor]]:
        """batch = (images, boxes, labels, domain) as in training, on the device.  Runs the detector in eval mode
        without gradients, feeds its original-size detections to the metric and returns them."""
        imgs, boxes, labels = list(batch[0]), batch[1], batch[2]
        was_training = self.detector.training
        self.detector.eval()
        try:
            with torch.no_grad():
                preds = self.detector(imgs)
        finally:
            self.detector.train(was_training)
        targets = [{"boxes": b.float(), "labels": l.long()} for b, l in zip(boxes, labels)]
        self._val_metric().update([{k: p[k] for k in ("boxes", "scores", "labels")} for p in preds], targets)
        return preds

    def on_validation_epoch_end(self) -> Dict[str, Tensor]:
        m = self._val_metric()
        out = m.compute()
        m.reset()
        return {"val_acc": out["map_50"], "map_per_class": out["map_per_class"], "classes": out["classes"]}
