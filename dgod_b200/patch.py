"""Rebinds the reference's call sites to the sm_100a kernels (SURVEY.md §8b).

`patch()` swaps the module attributes torchvision's detection glue looks up at call time
(TV models/detection/rpn.py:277-289, roi_heads.py:595-728, fcos.py:597,608 of the reference) and
`patch_model()` swaps what was bound early on an already-built detector: the RoI pooler
(fasterrcnn.py:412-416), the two Matchers (TV rpn.py:169, roi_heads.py:538), RPN box similarity
(TV rpn.py:167), `filter_proposals` / target assignment (fused, sync-free variants) and, for
FCOS, the location->target assignment inside `compute_loss` (fcos.py:503-550).
`patch()` also binds the GPU `MeanAveragePrecision` in the reference's DG namespaces.
`unpatch()` restores every binding.  After patching the ops require CUDA tensors.
"""
from __future__ import annotations

import sys
import types
from typing import Dict, List, Tuple

import torch

from . import metrics, ops
from .poolers import MultiScaleRoIAlign

_saved: List[Tuple[object, str, object]] = []


def _set(obj, name, value):
    _saved.append((obj, name, getattr(obj, name)))
    setattr(obj, name, value)


def patch(grad_reverse: bool = True) -> None:
    """Module-level rebinding; idempotent."""
    if _saved:
        return
    import torchvision
    from torchvision.models.detection import _utils as det_utils
    from torchvision.ops import boxes as box_ops
    from torchvision.ops import poolers as tv_poolers

    for mod in (box_ops, torchvision.ops):
        _set(mod, "nms", ops.nms)
        _set(mod, "batched_nms", ops.batched_nms)
        _set(mod, "box_iou", ops.box_iou)
    _set(tv_poolers, "roi_align", ops.roi_align)
    _set(torchvision.ops, "roi_align", ops.roi_align)
    _set(torchvision.ops, "MultiScaleRoIAlign", MultiScaleRoIAlign)
    _set(det_utils, "Matcher", ops.Matcher)
    # DGFRCNN.py:1 / DGFCOS.py:1 do `from DGcommon import *`: rebind in every namespace.  The metric is looked up when
    # a DGModel is constructed (DGcommon.py:127), so models built after patch() validate on the GPU metric.
    for name in ("DGcommon", "DGFRCNN", "DGFCOS"):
        mod = sys.modules.get(name)
        if mod is None:
            continue
        if grad_reverse and hasattr(mod, "grad_reverse"):
            _set(mod, "grad_reverse", ops.grad_reverse)
        if hasattr(mod, "MeanAveragePrecision"):
            _set(mod, "MeanAveragePrecision", metrics.MeanAveragePrecision)


def unpatch() -> None:
    while _saved:
        obj, name, value = _saved.pop()
        setattr(obj, name, value)


# ------------------------------------------------------------------------------------ instance level
def _image_sizes_tensor(image_shapes, device):
    return torch.tensor([[float(h), float(w)] for h, w in image_shapes], dtype=torch.float32, device=device)


def _fused_filter_proposals(self, proposals, objectness, image_shapes, num_anchors_per_level):
    """TV models/detection/rpn.py:242-297 in one pipeline; one D2H read (the kept counts)."""
    n_img = proposals.shape[0]
    sizes = _image_sizes_tensor(image_shapes, proposals.device)
    boxes, scores, counts = ops.rpn_filter_proposals(
        proposals, objectness.reshape(n_img, -1), sizes, list(num_anchors_per_level),
        self.pre_nms_top_n(), self.post_nms_top_n(), self.nms_thresh, self.min_size, self.score_thresh)
    cnt = counts.tolist()
    return [boxes[i, :c] for i, c in enumerate(cnt)], [scores[i, :c] for i, c in enumerate(cnt)]


def _fused_assign_targets_to_anchors(self, anchors, targets):
    """TV models/detection/rpn.py:193-229 for the whole batch in two launches."""
    m = self.proposal_matcher
    out = ops.match_boxes([t["boxes"] for t in targets], anchors[0], m.high_threshold, m.low_threshold,
                          m.allow_low_quality_matches, want=("labels_f32", "matched_boxes"))
    return list(out["labels_f32"].unbind(0)), list(out["matched_boxes"].unbind(0))


def _fused_assign_targets_to_proposals(self, proposals, gt_boxes, gt_labels):
    """TV models/detection/roi_heads.py:580-613 for the whole batch in one launch."""
    m = self.proposal_matcher
    out = ops.match_boxes(gt_boxes, proposals, m.high_threshold, m.low_threshold, m.allow_low_quality_matches,
                          gt_labels=gt_labels, want=("labels_i64", "clamped_idx"))
    sizes = [p.shape[0] for p in proposals]
    return list(out["clamped_idx"].split(sizes)), list(out["labels_i64"].split(sizes))


def _fused_fcos_compute_loss(self, targets, head_outputs, anchors, num_anchors_per_level):
    """fcos.py:503-550: assignment in one launch, then the reference's own head loss."""
    idx = ops.fcos_assign(anchors[0], [t["boxes"] for t in targets], list(num_anchors_per_level),
                          self.center_sampling_radius)
    return self.head.compute_loss(targets, head_outputs, anchors, list(idx.unbind(0)))


def patch_model(model, fused: bool = True):
    """Swap the early-bound pieces of a built Faster R-CNN / FCOS detector (reference
    `fasterrcnn.FastWILDS`, `fcos.FCOS` or torchvision's own classes).  Returns the model."""
    rpn = getattr(model, "rpn", None)
    roi_heads = getattr(model, "roi_heads", None)
    if rpn is not None:
        m = rpn.proposal_matcher
        rpn.proposal_matcher = ops.Matcher(m.high_threshold, m.low_threshold, m.allow_low_quality_matches)
        rpn.box_similarity = ops.box_iou
        if fused:
            rpn.filter_proposals = types.MethodType(_fused_filter_proposals, rpn)
            rpn.assign_targets_to_anchors = types.MethodType(_fused_assign_targets_to_anchors, rpn)
    if roi_heads is not None:
        m = roi_heads.proposal_matcher
        roi_heads.proposal_matcher = ops.Matcher(m.high_threshold, m.low_threshold, m.allow_low_quality_matches)
        pool = roi_heads.box_roi_pool
        if pool is not None and not isinstance(pool, MultiScaleRoIAlign):
            roi_heads.box_roi_pool = MultiScaleRoIAlign.from_torchvision(pool)
        if fused:
            roi_heads.assign_targets_to_proposals = types.MethodType(_fused_assign_targets_to_proposals, roi_heads)
    if fused and hasattr(model, "center_sampling_radius") and hasattr(model, "head"):
        model.compute_loss = types.MethodType(_fused_fcos_compute_loss, model)
    return model
