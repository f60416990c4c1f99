"""The GPU MeanAveragePrecision (dgod_b200.metrics, csrc/map_eval.cu) against the numpy restatement of pycocotools
(oracle/coco_map.py): precision and recall tables bit for bit on seeded sets built to hit every rule — score ties,
duplicate GTs, IoU exactly at a threshold, more than max_det detections of one class, empty images — plus the
sync-free update, the input checks, the DG models' validation hooks and the patch() rebinding."""
import sys
import types

import numpy as np
import pytest
import torch

from dgod_b200 import synth
from oracle import coco_map as M

REC = torch.linspace(0.0, 1.0, 101).tolist()
IOU10 = torch.linspace(0.5, 0.95, 10).tolist()
H, W = 200, 300


def _int_boxes(n, g):
    return synth.random_boxes(n, H, W, g).round()


def _random_set(seed, n_img):
    """Integer-valued boxes (so IoU = t can be exact), scores quantised to eighths (ties everywhere)."""
    g = synth.gen(seed)
    preds, targets = [], []
    for i in range(n_img):
        kind = i % 7
        m = 0 if kind == 3 else int(torch.randint(1, 12, (1,), generator=g))
        gt = _int_boxes(m, g)
        glab = torch.randint(1, 4, (m,), generator=g)
        if kind == 1 and m >= 2:                       # duplicate GTs
            gt[1], glab[1] = gt[0], glab[0]
        n = 0 if kind == 5 else (260 if kind == 2 else int(torch.randint(1, 60, (1,), generator=g)))
        det = _int_boxes(n, g)
        lab = torch.randint(1, 4, (n,), generator=g)
        if m:
            pick = torch.randint(0, m, (n,), generator=g)
            use = torch.rand(n, generator=g) < 0.6
            jit = torch.randint(-3, 4, (n, 4), generator=g).float()
            det[use] = gt[pick[use]] + jit[use]
            lab[use] = glab[pick[use]]
            if kind == 4 and n >= 2:                   # IoU exactly 0.5 and exactly 0.75 with GT 0
                x1, y1, x2, y2 = gt[0].tolist()
                w = max(x2 - x1, 1.0)
                gt[0] = torch.tensor([x1, y1, x1 + 4 * w, y2])
                det[:2] = torch.tensor([[x1, y1, x1 + 2 * w, y2], [x1, y1, x1 + 3 * w, y2]])
                lab[:2] = glab[0]
        if kind == 6 and n:
            lab[0] = 7                                 # a class without ground truth
        sc = torch.randint(0, 8, (n,), generator=g).float() / 8
        sc[(sc == 0) & (torch.rand(n, generator=g) < 0.5)] = -0.0
        preds.append({"boxes": det, "scores": sc, "labels": lab})
        targets.append({"boxes": gt, "labels": glab})
    return preds, targets


def _np(d):
    return {k: v.numpy() for k, v in d.items()}


def _gpu(d):
    return {k: v.cuda() for k, v in d.items()}


def _bitwise(a, b):
    return a.shape == b.shape and torch.equal(a.cpu().view(torch.int64), torch.from_numpy(np.ascontiguousarray(b)).view(torch.int64))


def _check_against_oracle(metric, out, preds, targets):
    ref = M.mean_average_precision([_np(p) for p in preds], [_np(t) for t in targets], metric.iou_thresholds,
                                   metric.rec_thresholds, metric.max_det)
    assert out["classes"].cpu().tolist() == ref["classes"].tolist()
    assert _bitwise(metric.precision, ref["precision"]), "precision table differs from pycocotools' arithmetic"
    assert _bitwise(metric.recall, ref["recall"]), "recall table differs from pycocotools' arithmetic"
    for k in ("map", "map_50", "map_75", "mar_100"):
        assert abs(float(metric.stats64[k]) - ref[k]) <= 1e-12, k
        assert float(out[k]) == np.float32(metric.stats64[k].item()), k
    if metric.class_metrics:
        np.testing.assert_allclose(metric.stats64["map_per_class"].cpu().numpy(), ref["map_per_class"], rtol=0, atol=1e-12)
        np.testing.assert_allclose(metric.stats64["mar_100_per_class"].cpu().numpy(), ref["mar_100_per_class"], rtol=0,
                                   atol=1e-12)
    return ref


@pytest.mark.gpu
@pytest.mark.parametrize("iou", [[0.5], IOU10], ids=["T1", "T10"])
@pytest.mark.parametrize("seed", [0, 1, 2])
def test_random_sets_match_pycocotools_bitwise(seed, iou):
    from dgod_b200.metrics import MeanAveragePrecision
    preds, targets = _random_set(seed, 60)
    metric = MeanAveragePrecision(iou_thresholds=iou, class_metrics=True)
    dp, dt = [_gpu(p) for p in preds], [_gpu(t) for t in targets]
    first = 5
    metric.update(dp[:first], dt[:first])                   # warm-up: pinned staging, thresholds on the device
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        for b in range(first, len(preds), 6):
            metric.update(dp[b:b + 6], dt[b:b + 6])
    finally:
        torch.cuda.set_sync_debug_mode(0)
    out = metric.compute()
    ref = _check_against_oracle(metric, out, preds, targets)
    assert (ref["precision"] == -1).any() and (ref["precision"] > 0).any()    # the set covers both kinds of class


@pytest.mark.gpu
def test_max_det_and_thresholds_of_the_constructor():
    from dgod_b200.metrics import MeanAveragePrecision
    preds, targets = _random_set(5, 21)
    for max_dets, rec in (([1, 10, 3], REC), ([100], [0.0, 0.3, 0.5, 0.9999])):
        metric = MeanAveragePrecision(iou_thresholds=[0.3, 0.5, 0.75], rec_thresholds=rec,
                                      max_detection_thresholds=max_dets)
        metric.update([_gpu(p) for p in preds], [_gpu(t) for t in targets])
        out = metric.compute()
        assert metric.max_det == max(max_dets)
        _check_against_oracle(metric, out, preds, targets)
        metric.reset()
        metric.update([_gpu(p) for p in preds[:3]], [_gpu(t) for t in targets[:3]])
        _check_against_oracle(metric, metric.compute(), preds[:3], targets[:3])


@pytest.mark.gpu
def test_input_errors():
    from dgod_b200.metrics import MeanAveragePrecision
    metric = MeanAveragePrecision()
    ok_p = {"boxes": torch.zeros(1, 4), "scores": torch.ones(1), "labels": torch.ones(1, dtype=torch.int64)}
    ok_t = {"boxes": torch.tensor([[0.0, 0.0, 1.0, 1.0]]), "labels": torch.ones(1, dtype=torch.int64)}
    with pytest.raises(RuntimeError, match="CUDA"):
        metric.update([ok_p], [_gpu(ok_t)])
    with pytest.raises(ValueError, match="iscrowd"):
        metric.update([_gpu(ok_p)], [dict(_gpu(ok_t), iscrowd=torch.zeros(1, device="cuda"))])
    big = {"boxes": torch.zeros(4097, 4), "scores": torch.ones(4097), "labels": torch.ones(4097, dtype=torch.int64)}
    with pytest.raises(ValueError, match="4096"):
        metric.update([_gpu(big)], [_gpu(ok_t)])
    many = {"boxes": torch.zeros(1025, 4), "labels": torch.ones(1025, dtype=torch.int64)}
    with pytest.raises(ValueError, match="1024"):
        metric.update([_gpu(ok_p)], [_gpu(many)])
    with pytest.raises(ValueError):
        MeanAveragePrecision(iou_thresholds=[0.5] * 33)
    with pytest.raises(ValueError):
        MeanAveragePrecision(box_format="xywh")
    with pytest.raises(ValueError):
        MeanAveragePrecision(iou_type="segm")
    nan_p = dict(ok_p, scores=torch.tensor([float("nan")]))
    metric.update([_gpu(nan_p)], [_gpu(ok_t)])              # update() cannot see the NaN without a host read
    with pytest.raises(ValueError, match="NaN"):
        metric.compute()


def _validate(model, n_batches, B, seed):
    """Runs validation_step over synthetic batches; returns (hook output, host copies of preds and targets, metric)."""
    preds_h, targets_h = [], []
    for b in range(n_batches):
        imgs = [i.cuda() for i in synth.random_images(B, 320, 416, seed + b)]
        tg, dom = synth.random_targets(B, 6, 320, 416, seed + b)
        preds = model.validation_step((imgs, [t["boxes"].cuda() for t in tg], [t["labels"].cuda() for t in tg], dom))
        preds_h += [{k: p[k].detach().cpu() for k in ("boxes", "scores", "labels")} for p in preds]
        targets_h += tg
    metric = model._val_metric()
    return model.on_validation_epoch_end(), preds_h, targets_h, metric


@pytest.mark.gpu
@pytest.mark.parametrize("arch", ["frcnn", "fcos"])
def test_dg_validation_hooks_match_the_oracle(arch):
    from dgod_b200 import dg, dg_fcos
    torch.manual_seed(0)
    cls = dg.DGFRCNN if arch == "frcnn" else dg_fcos.DGFCOS
    model = cls(9, 2, "dg", [0.5, 0.5, 0.5, 0.05, 0.0001], num_domains=2).cuda().train()
    if arch == "fcos":
        model.detector.score_thresh = 0.0                   # the random-init head's scores sit below the 0.2 default
    out, preds, targets, metric = _validate(model, 3, 2, 11)
    assert model.detector.training                          # the hook restores the mode it found
    assert sum(len(p["scores"]) for p in preds) > 0
    ref = M.mean_average_precision([_np(p) for p in preds], [_np(t) for t in targets], [0.5], REC, 100)
    assert _bitwise(metric.precision, ref["precision"]) and _bitwise(metric.recall, ref["recall"])
    assert abs(float(out["val_acc"]) - ref["map_50"]) <= 1e-6
    np.testing.assert_allclose(out["map_per_class"].cpu().numpy(), ref["map_per_class"], rtol=0, atol=1e-6)
    assert out["classes"].cpu().tolist() == ref["classes"].tolist()
    assert not metric._scores                               # reset for the next epoch


@pytest.mark.gpu
def test_patch_rebinds_the_metric_in_the_reference_namespaces():
    from dgod_b200 import metrics, ops, patch

    class Stub:
        pass

    def grad_reverse(x):
        return x

    mods = {name: types.ModuleType(name) for name in ("DGcommon", "DGFRCNN")}
    for m in mods.values():
        m.MeanAveragePrecision, m.grad_reverse = Stub, grad_reverse
    saved = {n: sys.modules.get(n) for n in mods}
    sys.modules.update(mods)
    try:
        patch.patch()
        try:
            for m in mods.values():
                assert m.MeanAveragePrecision is metrics.MeanAveragePrecision
                assert m.grad_reverse is ops.grad_reverse
            assert isinstance(mods["DGcommon"].MeanAveragePrecision(iou_thresholds=[0.5]), metrics.MeanAveragePrecision)
        finally:
            patch.unpatch()
        for m in mods.values():
            assert m.MeanAveragePrecision is Stub and m.grad_reverse is grad_reverse
    finally:
        for n, m in saved.items():
            if m is None:
                sys.modules.pop(n, None)
            else:
                sys.modules[n] = m
