"""COCO-style bbox mAP, restated in numpy float64.  TEST INFRASTRUCTURE — see oracle/__init__.py.

The arithmetic of torchmetrics' `MeanAveragePrecision(box_format="xyxy", iou_type="bbox")` with its pycocotools
backend (`COCOeval.evaluateImg` / `accumulate` / `summarize` and `maskApi.c:bbIou`), restated line for line for the
subset the product implements: no crowd ground truths, the "all" area range, one max-detections value.  Images are
numbered 0.. in the order they are given, which is what torchmetrics hands pycocotools.

preds:   list of dicts {"boxes": [n,4] fp32 xyxy, "scores": [n] fp32, "labels": [n] int}
targets: list of dicts {"boxes": [m,4] fp32 xyxy, "labels": [m] int}
"""
from __future__ import annotations

import numpy as np

EPS = np.spacing(1)          # 2.220446049250313e-16, COCOeval.accumulate


def _xywh(boxes) -> np.ndarray:
    """torchvision box_convert xyxy -> xywh in fp32 (w = x2 - x1 rounded to fp32), then handed over as doubles."""
    b = np.asarray(boxes, dtype=np.float32).reshape(-1, 4)
    return np.stack([b[:, 0], b[:, 1], b[:, 2] - b[:, 0], b[:, 3] - b[:, 1]], axis=1).astype(np.float64)


def bb_iou(dt: np.ndarray, gt: np.ndarray) -> np.ndarray:
    """maskApi.c:bbIou without crowd: [len(dt), len(gt)] in double."""
    o = np.zeros((len(dt), len(gt)))
    for g in range(len(gt)):
        G = gt[g]
        ga = G[2] * G[3]
        for d in range(len(dt)):
            D = dt[d]
            da = D[2] * D[3]
            w = min(D[2] + D[0], G[2] + G[0]) - max(D[0], G[0])
            if w <= 0:
                continue
            h = min(D[3] + D[1], G[3] + G[1]) - max(D[1], G[1])
            if h <= 0:
                continue
            i = w * h
            u = da + ga - i
            o[d, g] = i / u
    return o


def evaluate_img(dt_boxes, dt_scores, gt_boxes, iou_thrs, max_det):
    """COCOeval.computeIoU + evaluateImg for one (image, class).  None when the pair has neither detections nor GTs."""
    G, Dn = len(gt_boxes), len(dt_scores)
    if G == 0 and Dn == 0:
        return None
    gt_ignore = np.zeros(G, dtype=np.int64)                       # no crowd, area range "all"
    gtind = np.argsort(gt_ignore, kind="mergesort")
    dtind = np.argsort([-s for s in dt_scores], kind="mergesort")
    dtind = dtind[0:max_det]
    dt = dt_boxes[dtind]
    gt = gt_boxes[gtind]
    ious = bb_iou(dt, gt) if G > 0 else np.zeros((0, 0))
    T, D = len(iou_thrs), len(dt)
    gtm = np.zeros((T, G))
    dtm = np.zeros((T, D))
    gtIg = gt_ignore[gtind]
    dtIg = np.zeros((T, D))
    gt_ids = gtind + 1                                          # annotation ids start at 1
    if ious.size != 0:
        for tind, t in enumerate(iou_thrs):
            for dind in range(D):
                iou = min([t, 1 - 1e-10])
                m = -1
                for gind in range(G):
                    if gtm[tind, gind] > 0:
                        continue
                    if m > -1 and gtIg[m] == 0 and gtIg[gind] == 1:
                        break
                    if ious[dind, gind] < iou:
                        continue
                    iou = ious[dind, gind]
                    m = gind
                if m == -1:
                    continue
                dtIg[tind, dind] = gtIg[m]
                dtm[tind, dind] = gt_ids[m]
                gtm[tind, m] = dind + 1
    return {"dtMatches": dtm, "dtScores": [float(dt_scores[i]) for i in dtind], "gtIgnore": gtIg,
            "dtIgnore": dtIg.astype(bool)}


def accumulate(evals, iou_thrs, rec_thrs, max_det):
    """COCOeval.accumulate for one class over its per-image evaluations (update order).
    Returns (precision [T, R], recall [T]) with -1 where the class has no ground truth."""
    T, R = len(iou_thrs), len(rec_thrs)
    precision = -np.ones((T, R))
    recall = -np.ones(T)
    E = [e for e in evals if e is not None]
    if len(E) == 0:
        return precision, recall
    dtScores = np.concatenate([e["dtScores"][0:max_det] for e in E])
    inds = np.argsort(-dtScores, kind="mergesort")
    dtm = np.concatenate([e["dtMatches"][:, 0:max_det] for e in E], axis=1)[:, inds]
    dtIg = np.concatenate([e["dtIgnore"][:, 0:max_det] for e in E], axis=1)[:, inds]
    gtIg = np.concatenate([e["gtIgnore"] for e in E])
    npig = np.count_nonzero(gtIg == 0)
    if npig == 0:
        return precision, recall
    tps = np.logical_and(dtm, np.logical_not(dtIg))
    fps = np.logical_and(np.logical_not(dtm), np.logical_not(dtIg))
    tp_sum = np.cumsum(tps, axis=1).astype(dtype=float)
    fp_sum = np.cumsum(fps, axis=1).astype(dtype=float)
    for t, (tp, fp) in enumerate(zip(tp_sum, fp_sum)):
        tp = np.array(tp)
        fp = np.array(fp)
        nd = len(tp)
        rc = tp / npig
        pr = tp / (fp + tp + EPS)
        q = np.zeros((R,))
        recall[t] = rc[-1] if nd else 0
        pr = pr.tolist()
        q = q.tolist()
        for i in range(nd - 1, 0, -1):
            if pr[i] > pr[i - 1]:
                pr[i - 1] = pr[i]
        inds_r = np.searchsorted(rc, rec_thrs, side="left")
        try:
            for ri, pi in enumerate(inds_r):
                q[ri] = pr[pi]
        except IndexError:
            pass
        precision[t] = np.array(q)
    return precision, recall


def _mean_valid(s: np.ndarray) -> float:
    """COCOeval.summarize: the mean of the entries > -1, or -1 when there are none."""
    return -1.0 if len(s[s > -1]) == 0 else float(np.mean(s[s > -1]))


def mean_average_precision(preds, targets, iou_thresholds, rec_thresholds, max_det: int = 100):
    """Runs the whole evaluation.  Returns float64 numpy values: precision [T, R, K], recall [T, K], classes [K],
    map, map_50, map_75, mar_100, map_per_class [K], mar_100_per_class [K]."""
    iou_thresholds = [float(t) for t in iou_thresholds]
    rec_thresholds = np.asarray([float(r) for r in rec_thresholds], dtype=np.float64)
    P = [{k: np.asarray(v) for k, v in p.items()} for p in preds]
    G = [{k: np.asarray(v) for k, v in t.items()} for t in targets]
    labels = [p["labels"].reshape(-1) for p in P] + [g["labels"].reshape(-1) for g in G]
    classes = np.unique(np.concatenate(labels).astype(np.int64)) if labels else np.zeros(0, np.int64)
    T, R, K = len(iou_thresholds), len(rec_thresholds), len(classes)
    precision = -np.ones((T, R, K))
    recall = -np.ones((T, K))
    for k, c in enumerate(classes):
        evals = []
        for p, g in zip(P, G):
            dsel = p["labels"].reshape(-1) == c
            gsel = g["labels"].reshape(-1) == c
            scores = np.asarray(p["scores"], dtype=np.float32).reshape(-1)[dsel].astype(np.float64)
            evals.append(evaluate_img(_xywh(p["boxes"])[dsel], scores, _xywh(g["boxes"])[gsel], iou_thresholds, max_det))
        precision[:, :, k], recall[:, k] = accumulate(evals, iou_thresholds, rec_thresholds, max_det)

    def at(thr):
        t = [i for i, v in enumerate(iou_thresholds) if v == thr]
        return _mean_valid(precision[t]) if t else -1.0

    return {
        "precision": precision, "recall": recall, "classes": classes,
        "map": _mean_valid(precision), "map_50": at(0.5), "map_75": at(0.75), "mar_100": _mean_valid(recall),
        "map_per_class": np.array([_mean_valid(precision[:, :, k]) for k in range(K)]),
        "mar_100_per_class": np.array([_mean_valid(recall[:, k]) for k in range(K)]),
    }
