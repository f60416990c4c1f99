"""Known answers of the COCO bbox mAP restatement (oracle/coco_map.py), each worked out by hand from pycocotools'
rules: greedy matching by descending score, the later GT winning an IoU tie, per-class max-detection truncation,
cross-image ties to the earlier image, the float32 recall grid torchmetrics builds, and the `tp / (tp + fp + eps)`
precision.  These pin the oracle that the GPU metric is compared against bit for bit."""
import numpy as np
import pytest
import torch

from oracle import coco_map as M

REC = torch.linspace(0.0, 1.0, 101).tolist()          # torchmetrics' recall grid: float32 values as doubles
ONE_GT = 1.0 / (1.0 + np.spacing(1))                  # 0.9999999999999998: precision of a lone first TP


def _img(det_boxes, scores, det_labels, gt_boxes, gt_labels):
    p = {"boxes": np.asarray(det_boxes, np.float32).reshape(-1, 4), "scores": np.asarray(scores, np.float32),
         "labels": np.asarray(det_labels, np.int64)}
    t = {"boxes": np.asarray(gt_boxes, np.float32).reshape(-1, 4), "labels": np.asarray(gt_labels, np.int64)}
    return p, t


def _run(images, iou=(0.5,), max_det=100):
    preds, targets = zip(*images)
    return M.mean_average_precision(list(preds), list(targets), list(iou), REC, max_det)


HIT, MISS = [0, 0, 10, 10], [50, 50, 60, 60]          # a detection on / far away from the GT [0, 0, 10, 10]


def test_recall_grid_is_float32():
    assert REC[7] == 0.07000000029802322 and REC[50] == 0.5 and REC[25] == 0.25
    assert sum(r != k / 100 for k, r in enumerate(REC)) == 96


def test_fp_then_tp_is_one_half():
    r = _run([_img([MISS, HIT], [0.9, 0.8], [1, 1], [[0, 0, 10, 10]], [1])])
    assert r["map"] == 0.5 and r["map_50"] == 0.5 and r["mar_100"] == 1.0


def test_tp_fp_tp_over_two_gts():
    r = _run([_img([HIT, MISS, [20, 20, 30, 30]], [0.9, 0.8, 0.7], [1, 1, 1], [[0, 0, 10, 10], [20, 20, 30, 30]], [1, 1])])
    # recall 0.5 on 51 grid points (precision 1/(1+eps)), 1.0 on 50 (precision 2/(3+eps))
    assert r["map"] == pytest.approx(0.834983498349835, abs=1e-15, rel=0)


def test_tp_fp_fp_tp_over_four_gts():
    gts = [[0, 0, 10, 10], [20, 20, 30, 30], [40, 0, 50, 10], [0, 40, 10, 50]]
    dets = [HIT, MISS, [70, 70, 80, 80], [20, 20, 30, 30]]
    r = _run([_img(dets, [0.9, 0.8, 0.7, 0.6], [1] * 4, gts, [1] * 4)])
    assert r["map"] == pytest.approx(0.38118811881188114, abs=1e-15, rel=0)
    assert r["mar_100"] == 0.5


def test_iou_exactly_one_half_matches():
    dt, gt = M._xywh([[0, 0, 2, 1]]), M._xywh([[0, 0, 1, 1]])
    assert M.bb_iou(dt, gt)[0, 0] == 0.5                # i = 1, u = 2
    r = _run([_img([[0, 0, 2, 1]], [0.5], [3], [[0, 0, 1, 1]], [3])])
    assert (r["precision"] == ONE_GT).all()
    r = _run([_img([[0, 0, 2, 1]], [0.5], [3], [[0, 0, 1, 1]], [3])], iou=(0.55,))
    assert r["map"] == 0.0


def test_equal_iou_goes_to_the_later_gt():
    e = M.evaluate_img(M._xywh([HIT, HIT]), [0.9, 0.8], M._xywh([HIT, HIT]), [0.5], 100)
    assert e["dtMatches"].tolist() == [[2.0, 1.0]]     # annotation ids: the first detection takes the second GT


def test_max_det_truncates_per_class():
    dets = [MISS] * 100 + [HIT]
    scores = [0.9 - 0.001 * i for i in range(101)]
    img = _img(dets + [HIT], scores + [0.05], [1] * 101 + [2], [[0, 0, 10, 10], [0, 0, 10, 10]], [1, 2])
    r = _run([img])
    # the 101st detection of class 1 is its only TP and is dropped; class 2's lone detection is not affected by class 1
    assert (r["precision"][0, :, 0] == 0).all() and (r["precision"][0, :, 1] == ONE_GT).all()
    assert r["recall"][0].tolist() == [0.0, 1.0]
    r = _run([img], max_det=101)
    assert r["recall"][0].tolist() == [1.0, 1.0]


def test_score_ties_across_images_go_to_the_earlier_image():
    a = _img([MISS], [0.5], [1], [], [])
    b = _img([HIT], [0.5], [1], [[0, 0, 10, 10]], [1])
    assert _run([a, b])["map"] == 0.5                   # FP (image 0) ranks first
    assert (_run([b, a])["precision"] == ONE_GT).all()  # TP (image 0) ranks first


def test_class_without_gt_is_excluded():
    img = _img([HIT, HIT], [0.9, 0.9], [1, 2], [[0, 0, 10, 10]], [1])
    r = _run([img])
    assert r["classes"].tolist() == [1, 2]
    assert r["map_per_class"][1] == -1.0 and r["mar_100_per_class"].tolist() == [1.0, -1.0]
    assert (r["precision"][:, :, 1] == -1).all() and (r["precision"][:, :, 0] == ONE_GT).all()
    assert r["map"] == r["map_per_class"][0] == pytest.approx(ONE_GT, abs=2e-16, rel=0)


def test_class_without_detections_scores_zero():
    img = _img([HIT], [0.9], [1], [[0, 0, 10, 10], [20, 20, 30, 30]], [1, 4])
    r = _run([img])
    assert (r["precision"][0, :, 0] == ONE_GT).all() and r["map_per_class"][1] == 0.0
    assert r["recall"][0].tolist() == [1.0, 0.0]
    assert r["map"] == pytest.approx(ONE_GT / 2, abs=2e-16, rel=0)


def test_predictions_equal_to_targets():
    gts = [[0, 0, 10, 10], [20, 20, 30, 30], [5, 40, 25, 70]]
    r = _run([_img(gts, [0.7, 0.7, 0.7], [1, 1, 2], gts, [1, 1, 2])], iou=torch.linspace(0.5, 0.95, 10).tolist())
    # k / (k + eps) rounds to 1 for k >= 2, but 1 / (1 + eps) does not
    assert (r["precision"][:, :, 0] == 1.0).all() and (r["precision"][:, :, 1] == ONE_GT).all()
    assert r["map_per_class"][0] == 1.0 and r["map_75"] == pytest.approx((1.0 + ONE_GT) / 2, abs=2e-16, rel=0)


def test_empty_images():
    e = _img([], [], [], [], [])
    hit = _img([HIT], [0.9], [1], [[0, 0, 10, 10]], [1])
    only_gt = _img([], [], [], [[0, 0, 10, 10]], [1])
    r = _run([e, hit, e, only_gt, e])
    assert r["recall"][0].tolist() == [0.5]
    # precision 1/(1+eps) up to recall 0.5 (51 grid points), 0 after it
    assert r["map"] == pytest.approx(51 * ONE_GT / 101, abs=2e-16, rel=0)
    r = _run([e, e])
    assert r["classes"].size == 0 and r["map"] == -1.0 and r["mar_100"] == -1.0


def test_signed_zero_scores_tie():
    img = _img([MISS, HIT], [-0.0, 0.0], [1, 1], [[0, 0, 10, 10]], [1])
    assert _run([img])["map"] == 0.5                    # stable: the FP at -0.0 stays in front of the TP at +0.0


def test_map_50_and_75_lookup_by_equality():
    img = _img([HIT], [0.9], [1], [[0, 0, 10, 10]], [1])
    r = _run([img], iou=(0.55,))
    assert r["map_50"] == -1.0 and r["map_75"] == -1.0 and r["map"] == pytest.approx(ONE_GT, abs=2e-16, rel=0)
