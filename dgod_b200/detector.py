"""Faster R-CNN (R50-FPN) with per-image losses — host-side mirror of the reference's
`fasterrcnn.FastWILDS` (fasterrcnn.py:354-499) whose detection-head hot path runs on the
sm_100a kernels.

What stays PyTorch/cuDNN (SURVEY.md L-1): image transform, ResNet-50 + FPN convolutions, the RPN head's 3x3 conv,
TwoMLPHead / FastRCNNPredictor, the loss arithmetic.  What is replaced (SURVEY.md §8a):
  A1-A4  anchors + decode + per-level top-k + clip/filters + batched NMS   -> ops.rpn_proposals
  A5     assign_targets_to_anchors (box_iou + Matcher + labels)            -> ops.match_boxes
  A6     assign_targets_to_proposals                                        -> ops.match_boxes
  A7/A8  MultiScaleRoIAlign forward / backward                              -> poolers.MultiScaleRoIAlign
  A9     postprocess_detections candidates + per-class NMS                  -> ops.detect_candidates + ops.nms_segments
Module and parameter names follow the reference so its checkpoints load unchanged
(train_driving_dg.py:154-155): backbone.*, rpn.head.*, roi_heads.box_head.fc6/fc7,
roi_heads.box_predictor.cls_score/bbox_pred.

The positive/negative samplers (TV models/detection/_utils.py:11-71) draw the same uniform
subsets as upstream but with fixed output shapes (masks instead of `torch.where`), and the RoI heads
take the RPN's proposals padded with their counts on the device, so a training step reads nothing
back to the host.
"""
from __future__ import annotations

import math
from collections import OrderedDict
from typing import Dict, List, Optional, Sequence, Tuple

import torch
import torch.nn.functional as F
from torch import Tensor, nn
from torchvision.models.detection.backbone_utils import resnet_fpn_backbone
from torchvision.models.detection.faster_rcnn import FastRCNNPredictor
from torchvision.models.detection import rpn as tv_rpn
from torchvision.models.detection.transform import GeneralizedRCNNTransform
from torchvision.ops.feature_pyramid_network import FeaturePyramidNetwork

from . import ops
from .poolers import MultiScaleRoIAlign

BBOX_XFORM_CLIP = math.log(1000.0 / 16)


# ------------------------------------------------------------------------------------ small host helpers
def make_cell_anchors(sizes: Sequence[Sequence[int]], aspect_ratios: Sequence[Sequence[float]]) -> List[Tensor]:
    """Zero-centred base anchors per level, rounded (TV models/detection/anchor_utils.py:58-74)."""
    cells = []
    for scales, ratios in zip(sizes, aspect_ratios):
        s = torch.as_tensor(scales, dtype=torch.float32)
        r = torch.as_tensor(ratios, dtype=torch.float32)
        h_r = torch.sqrt(r)
        w_r = 1 / h_r
        ws = (w_r[:, None] * s[None, :]).view(-1)
        hs = (h_r[:, None] * s[None, :]).view(-1)
        cells.append((torch.stack([-ws, -hs, ws, hs], dim=1) / 2).round())
    return cells


def grid_anchors(cells: Sequence[Tensor], grids: Sequence[Tuple[int, int]], strides: Sequence[Tuple[int, int]],
                 device) -> Tensor:
    """All anchors of one image in torchvision's (level, y, x, a) order (anchor_utils.py:84-113)."""
    out = []
    for cell, (h, w), (sh, sw) in zip(cells, grids, strides):
        sx = torch.arange(0, w, dtype=torch.int32, device=device) * sw
        sy = torch.arange(0, h, dtype=torch.int32, device=device) * sh
        yy, xx = torch.meshgrid(sy, sx, indexing="ij")
        shifts = torch.stack((xx.reshape(-1), yy.reshape(-1), xx.reshape(-1), yy.reshape(-1)), dim=1)
        out.append((shifts.view(-1, 1, 4) + cell.to(device).view(1, -1, 4)).reshape(-1, 4))
    return torch.cat(out)


def encode_boxes(reference: Tensor, proposals: Tensor, weights: Tuple[float, float, float, float]) -> Tensor:
    """BoxCoder.encode_single (TV models/detection/_utils.py:75-119) on [...,4] tensors."""
    wx, wy, ww, wh = weights
    ex_w = proposals[..., 2] - proposals[..., 0]
    ex_h = proposals[..., 3] - proposals[..., 1]
    ex_cx = proposals[..., 0] + 0.5 * ex_w
    ex_cy = proposals[..., 1] + 0.5 * ex_h
    gt_w = reference[..., 2] - reference[..., 0]
    gt_h = reference[..., 3] - reference[..., 1]
    gt_cx = reference[..., 0] + 0.5 * gt_w
    gt_cy = reference[..., 1] + 0.5 * gt_h
    return torch.stack((wx * (gt_cx - ex_cx) / ex_w, wy * (gt_cy - ex_cy) / ex_h,
                        ww * torch.log(gt_w / ex_w), wh * torch.log(gt_h / ex_h)), dim=-1)


class BalancedSampler:
    """Fixed-shape BalancedPositiveNegativeSampler (TV models/detection/_utils.py:11-71).

    Given labels [B,N] (>=1 positive, 0 negative, <0 ignored) picks a uniformly random subset of
    min(#pos, P) positives and min(#neg, S - #picked_pos) negatives per image, exactly like
    upstream's two `randperm`s, but returns index tensors of static shape plus validity masks.
    `keys` ([B,N] uniform numbers) can be injected to force a selection (tests).  On the device the selection is
    `ops.balanced_sample` (csrc/sampler.cu, one launch per batch); the two-`topk` torch formulation below is the host
    form of the same rule (CPU tests of the host logic)."""

    def __init__(self, batch_size_per_image: int, positive_fraction: float):
        self.batch_size_per_image = batch_size_per_image
        self.num_pos = int(batch_size_per_image * positive_fraction)

    def __call__(self, labels: Tensor, keys: Optional[Tensor] = None):
        B, N = labels.shape
        if keys is None:
            keys = torch.rand((B, N), device=labels.device)
        if labels.is_cuda:
            # one launch for the batch: radix select of the smallest keys per class, survivors in ascending index
            pos_idx, pos_valid, neg_idx, neg_valid, _ = ops.balanced_sample(labels, keys, self.num_pos, self.batch_size_per_image)
            return pos_idx, pos_valid, neg_idx, neg_valid
        P, S = min(self.num_pos, N), min(self.batch_size_per_image, N)
        pk = torch.where(labels >= 1, keys, torch.full_like(keys, 2.0))
        nk = torch.where(labels == 0, keys, torch.full_like(keys, 2.0))
        pv, pos_idx = torch.topk(pk, P, dim=1, largest=False)
        pos_valid = pv < 2.0
        n_pos = pos_valid.sum(1, keepdim=True)
        nv, neg_idx = torch.topk(nk, S, dim=1, largest=False)
        neg_valid = (nv < 2.0) & (torch.arange(S, device=labels.device)[None, :] < (S - n_pos))
        return pos_idx, pos_valid, neg_idx, neg_valid


class TwoMLPHead(nn.Module):
    """fasterrcnn.py:331-352: fc6/fc7 with the extra (unused) labels argument DGFRCNN's forward
    hook reads (DGFRCNN.py:89-91)."""

    def __init__(self, in_channels: int, representation_size: int):
        super().__init__()
        self.fc6 = nn.Linear(in_channels, representation_size)
        self.fc7 = nn.Linear(representation_size, representation_size)

    def forward(self, x: Tensor, box_labels=None) -> Tensor:
        x = x.flatten(start_dim=1)
        if ops.box_head_mlp_supported(x, self.fc6.weight, self.fc7.weight):
            return ops.box_head_mlp(x, self.fc6.weight, self.fc6.bias, self.fc7.weight, self.fc7.bias)
        return F.relu(self.fc7(F.relu(self.fc6(x))))


# ------------------------------------------------------------------------------------ RPN
class RPNHead(tv_rpn.RPNHead):
    """torchvision's RPNHead (same modules, parameters and state-dict keys) whose bias, ReLU and 1x1 predictors run as
    `ops.rpn_head`, one native pass over all levels each way, after the 3x3 conv (cuDNN, without its bias).  On CUDA
    fp32 NHWC maps with autocast off; anything else (CPU, NCHW, bf16 autocast) is torchvision's forward."""

    def forward(self, x: List[Tensor]) -> Tuple[List[Tensor], List[Tensor]]:
        block = self.conv[0] if len(self.conv) == 1 else None
        conv = block[0] if block is not None and len(block) == 2 and isinstance(block[1], nn.ReLU) else None
        if conv is None or not ops.rpn_head_supported(x, conv, self.cls_logits.weight, self.bbox_pred.weight):
            return super().forward(x)
        cs = [conv._conv_forward(f, conv.weight, None) for f in x]
        return ops.rpn_head(cs, conv.bias, self.cls_logits.weight, self.cls_logits.bias, self.bbox_pred.weight,
                            self.bbox_pred.bias)


class RegionProposalNetwork(nn.Module):
    """fasterrcnn.py:90-196 (RegionProposalNetworkWILDS) on the fused kernels."""

    def __init__(self, in_channels: int, anchor_sizes, aspect_ratios, fg_iou_thresh=0.7, bg_iou_thresh=0.3,
                 batch_size_per_image=256, positive_fraction=0.5, pre_nms_top_n=None, post_nms_top_n=None,
                 nms_thresh=0.7, score_thresh=0.0):
        super().__init__()
        self.cells = make_cell_anchors(anchor_sizes, aspect_ratios)
        self.head = RPNHead(in_channels, len(self.cells[0]))
        self.fg_iou_thresh, self.bg_iou_thresh = fg_iou_thresh, bg_iou_thresh
        self.sampler = BalancedSampler(batch_size_per_image, positive_fraction)
        self._pre_nms_top_n = pre_nms_top_n or dict(training=2000, testing=1000)
        self._post_nms_top_n = post_nms_top_n or dict(training=2000, testing=1000)
        self.nms_thresh, self.score_thresh, self.min_size = nms_thresh, score_thresh, 1e-3
        self._anchor_cache: Dict[tuple, Tensor] = {}

    def pre_nms_top_n(self):
        return self._pre_nms_top_n["training" if self.training else "testing"]

    def post_nms_top_n(self):
        return self._post_nms_top_n["training" if self.training else "testing"]

    def anchors_for(self, grids, strides, device) -> Tensor:
        key = (tuple(grids), tuple(strides), str(device))
        if key not in self._anchor_cache:
            self._anchor_cache[key] = grid_anchors(self.cells, grids, strides, device)
        return self._anchor_cache[key]

    def forward(self, image_tensor_shape, image_sizes: List[Tuple[int, int]], features: Dict[str, Tensor],
                targets: Optional[List[Dict[str, Tensor]]] = None, sampler_keys: Optional[Tensor] = None):
        feats = list(features.values())
        objectness, deltas = self.head(feats)                              # fasterrcnn.py:165 (cuDNN)
        dev = feats[0].device
        grids = [tuple(o.shape[-2:]) for o in objectness]
        ph, pw = image_tensor_shape[-2:]
        strides = [(ph // g[0], pw // g[1]) for g in grids]                # TV anchor_utils.py:119-125
        sizes = ops.device_constant(tuple((float(h), float(w)) for h, w in image_sizes), torch.float32, dev)
        boxes, scores, counts = ops.rpn_proposals(                          # fasterrcnn.py:166-182
            objectness, deltas, sizes, strides, [c.tolist() for c in self.cells],
            self.pre_nms_top_n(), self.post_nms_top_n(), self.nms_thresh, self.min_size, self.score_thresh)
        losses = {}
        if self.training:
            assert targets is not None
            anchors = self.anchors_for(grids, strides, dev)
            m = ops.match_boxes([t["boxes"] for t in targets], anchors, self.fg_iou_thresh, self.bg_iou_thresh,
                                True, want=("labels_f32", "matched_boxes"))  # fasterrcnn.py:187
            losses = self.compute_loss(objectness, deltas, m["labels_f32"], m["matched_boxes"], anchors, sampler_keys)
            self.last_anchor_labels = m["labels_f32"]          # [B, A] 1 / 0 / -1 (tests compare them with the golden)
        return (boxes, scores, counts), losses

    def compute_loss(self, objectness, deltas, labels, matched_gt_boxes, anchors, sampler_keys=None):
        """Per-image RPN losses (fasterrcnn.py:105-140), regression targets encoded only where the
        sampler picked a positive (identical values, TV _utils.py:139-160)."""
        B = labels.shape[0]
        obj = torch.cat([o.permute(0, 2, 3, 1).reshape(B, -1) for o in objectness], dim=1)        # TV rpn.py:81-110
        dl = torch.cat([d.view(B, -1, 4, d.shape[-2], d.shape[-1]).permute(0, 3, 4, 1, 2).reshape(B, -1, 4)
                        for d in deltas], dim=1)
        pos_idx, pos_valid, neg_idx, neg_valid = self.sampler(labels, sampler_keys)
        n_sampled = (pos_valid.sum(1) + neg_valid.sum(1)).to(obj.dtype)
        pred = torch.gather(dl, 1, pos_idx[..., None].expand(-1, -1, 4))
        tgt = encode_boxes(torch.gather(matched_gt_boxes, 1, pos_idx[..., None].expand(-1, -1, 4)),
                           anchors[pos_idx], (1.0, 1.0, 1.0, 1.0))
        tgt = torch.where(pos_valid[..., None], tgt, torch.zeros_like(tgt))
        box = F.smooth_l1_loss(pred, tgt, beta=1 / 9, reduction="none").sum(-1)
        loss_box = (box * pos_valid).sum(1) / n_sampled
        lp = torch.gather(obj, 1, pos_idx)
        ln = torch.gather(obj, 1, neg_idx)
        bce = (F.binary_cross_entropy_with_logits(lp, torch.ones_like(lp), reduction="none") * pos_valid).sum(1) + \
              (F.binary_cross_entropy_with_logits(ln, torch.zeros_like(ln), reduction="none") * neg_valid).sum(1)
        return {"loss_objectness": bce / n_sampled, "loss_rpn_box_reg": loss_box}


# ------------------------------------------------------------------------------------ RoI heads
class RoIHeads(nn.Module):
    """fasterrcnn.py:238-305 (RoIHeadsWILDS) on the fused kernels."""

    def __init__(self, out_channels: int, num_classes: int, fg_iou_thresh=0.5, bg_iou_thresh=0.5,
                 batch_size_per_image=512, positive_fraction=0.25, bbox_reg_weights=None, score_thresh=0.05,
                 nms_thresh=0.5, detections_per_img=100):
        super().__init__()
        self.box_roi_pool = MultiScaleRoIAlign(["0", "1", "2", "3"], 7, 2)          # fasterrcnn.py:412-416
        self.box_head = TwoMLPHead(out_channels * 7 * 7, 1024)
        self.box_predictor = FastRCNNPredictor(1024, num_classes)
        self.fg_iou_thresh, self.bg_iou_thresh = fg_iou_thresh, bg_iou_thresh
        self.batch_size_per_image = batch_size_per_image
        self.sampler = BalancedSampler(batch_size_per_image, positive_fraction)
        self.weights = tuple(bbox_reg_weights or (10.0, 10.0, 5.0, 5.0))
        self.score_thresh, self.nms_thresh, self.detections_per_img = score_thresh, nms_thresh, detections_per_img

    def select_training_samples(self, proposals, targets, sampler_keys=None):
        """TV models/detection/roi_heads.py:642-678 with exactly batch_size_per_image rows per
        image (what fasterrcnn.py:211-212 and DGFRCNN.py:152-153 assume).

        `proposals` is the RPN's padded output (boxes [B,cap,4], device counts [B]) or a list of per-image [n_i,4]
        boxes.  The candidates of image i are its proposals followed by its ground truths (add_gt_proposals), in slots
        [0, N) with N = cap + the largest ground-truth count (known from the shapes), unused slots ignored; matcher,
        sampler and the sample epilogue all read the counts on the device, so no step waits on the host.  Returns
        (s_props [B,S,4], s_labels int64 [B,S], reg_targets [B,S,4]).  An image with fewer than S candidates leaves
        slots empty: the reference would mis-split its batch there (fasterrcnn.py:211-212 hard-codes 512 rows per
        image); this mirror keeps the [B, S] shape DGFRCNN.py:152-153 relies on and marks the empty slots with label
        -100 (cross_entropy's ignore_index, also inside the DG heads) and a zero box, excluded from both loss
        denominators."""
        if isinstance(proposals, tuple):
            boxes, counts = proposals
        else:
            boxes = torch.nn.utils.rnn.pad_sequence(list(proposals), batch_first=True)
            counts = ops.device_constant(tuple(p.shape[0] for p in proposals), torch.int32, boxes.device)
        gt_boxes = [t["boxes"].to(boxes.dtype) for t in targets]
        m = ops.match_boxes(gt_boxes, (boxes, counts), self.fg_iou_thresh, self.bg_iou_thresh, False,
                            gt_labels=[t["labels"] for t in targets], want=("labels_i64", "clamped_idx"))
        labels = m["labels_i64"]
        B, N = labels.shape
        if sampler_keys is not None and sampler_keys.shape[1] < N:   # the padding slots are never picked (label -1)
            sampler_keys = F.pad(sampler_keys, (0, N - sampler_keys.shape[1]), value=1.0)
        pos_idx, pos_valid, neg_idx, neg_valid = self.sampler(labels, sampler_keys)
        return ops.sample_rois(pos_idx, pos_valid, neg_idx, neg_valid, labels, m["clamped_idx"], boxes, counts,
                               gt_boxes, self.batch_size_per_image, self.weights)

    def losses(self, class_logits, box_regression, labels, regression_targets):
        """fastrcnn_loss per image (fasterrcnn.py:198-236)."""
        B, S = labels.shape
        C = class_logits.shape[-1]
        n_valid = (labels >= 0).sum(1).clamp(min=1).to(class_logits.dtype)      # == S unless slots are empty
        cls = F.cross_entropy(class_logits, labels.reshape(-1), reduction="none").view(B, S).sum(1) / n_valid
        pos = labels > 0
        reg = box_regression.view(B, S, C, 4)
        picked = torch.gather(reg, 2, labels.clamp(min=0)[..., None, None].expand(-1, -1, 1, 4)).squeeze(2)
        tgt = torch.where(pos[..., None], regression_targets, torch.zeros_like(regression_targets))
        box = (F.smooth_l1_loss(picked, tgt, beta=1 / 9, reduction="none").sum(-1) * pos).sum(1) / n_valid
        return {"loss_classifier": cls, "loss_box_reg": box}

    def postprocess_detections(self, class_logits, box_regression, proposals, boxes_per_image, image_sizes_t):
        """TV models/detection/roi_heads.py:680-737 for the batch: candidates in one launch, per-class
        NMS of all images in one call.  Returns padded [B,100] results + counts (no host sync)."""
        cb, cs, cl, cv = ops.detect_candidates(class_logits, box_regression, proposals, boxes_per_image,
                                               image_sizes_t, self.weights, self.score_thresh, 1e-2)
        nc = cb.shape[1]
        seg = [n * nc for n in boxes_per_image]
        keep, info = ops.nms_segments(cb.view(-1, 4), cs.view(-1), cl.view(-1), seg, self.nms_thresh,
                                      valid=cv.view(-1), max_out_per_seg=self.detections_per_img)
        off = ops.device_constant(tuple(sum(seg[:i]) for i in range(len(seg))), torch.int64, cb.device)
        flat = keep + off[:, None]
        return (cb.view(-1, 4)[flat], cs.view(-1)[flat], cl.view(-1)[flat], info[:-1])

    def forward(self, features, proposals, image_sizes: List[Tuple[int, int]], targets=None, sampler_keys=None):
        """`proposals`: in training the RPN's (boxes [B,cap,4], counts [B]) or a list of [n_i,4]; in eval a list."""
        dev = proposals[0].device
        sizes_t = ops.device_constant(tuple((float(h), float(w)) for h, w in image_sizes), torch.float32, dev)
        labels = reg_targets = label_list = None
        if self.training:
            props, labels, reg_targets = self.select_training_samples(proposals, targets, sampler_keys)
            B, S = labels.shape
            box_features = self.box_roi_pool(features, props, image_sizes)                # fasterrcnn.py:278
            label_list = list(labels.unbind(0))
            props, per_image = props.view(-1, 4), [S] * B
        else:
            box_features = self.box_roi_pool(features, proposals, image_sizes)
            props, per_image = torch.cat(proposals), [p.shape[0] for p in proposals]
        box_features = self.box_head(box_features, label_list)                            # fasterrcnn.py:279
        class_logits, box_regression = self.box_predictor(box_features)
        losses = {}
        if self.training:
            losses = self.losses(class_logits, box_regression, labels, reg_targets)
        det = self.postprocess_detections(class_logits, box_regression, props, per_image, sizes_t)
        return det, losses, box_features, label_list


# ------------------------------------------------------------------------------------ input side
class FusedTransform(GeneralizedRCNNTransform):
    """GeneralizedRCNNTransform (TV models/detection/transform.py:102-153; fasterrcnn.py:439-441, fcos.py:483)
    with normalize + resize + batch in ONE launch (`ops.image_batch`, SURVEY.md §8f rank 4) instead of ~50, and
    the box targets rescaled by one multiply per image.  `postprocess` (eval) is torchvision's."""

    def forward(self, images: List[Tensor], targets: Optional[List[Dict[str, Tensor]]] = None):
        images = list(images)
        if targets is not None and any(("masks" in t or "keypoints" in t) for t in targets):
            return super().forward(images, targets)        # not on DGOD's path (boxes and labels only)
        if self.training and len(self.min_size) > 1:       # transform.py:168-175: random scale choice in training
            k = int(torch.empty(1).uniform_(0.0, float(len(self.min_size))).item())
            size = self.min_size[k]
        else:
            size = self.min_size[-1]
        batched, sizes = ops.image_batch(images, self.image_mean, self.image_std, size, self.max_size, self.size_divisible)
        if targets is not None:
            out_targets = []
            for img, t, (oh, ow) in zip(images, targets, sizes):
                t = dict(t)                                # transform.py:112-120 copies the dicts
                t["boxes"] = t["boxes"] * self._ratios(int(img.shape[-2]), int(img.shape[-1]), oh, ow, t["boxes"])
                out_targets.append(t)
            targets = out_targets
        from torchvision.models.detection.image_list import ImageList
        return ImageList(batched, [(int(h), int(w)) for h, w in sizes]), targets

    def _ratios(self, h: int, w: int, oh: int, ow: int, like: Tensor) -> Tensor:
        """resize_boxes (transform.py:305-316): fp32 ratios new/orig per axis, cached on the device."""
        key = (h, w, oh, ow, like.device, like.dtype)
        cache = self.__dict__.setdefault("_ratio_cache", {})
        r = cache.get(key)
        if r is None:
            rh = torch.tensor(float(oh), dtype=torch.float32) / torch.tensor(float(h), dtype=torch.float32)
            rw = torch.tensor(float(ow), dtype=torch.float32) / torch.tensor(float(w), dtype=torch.float32)
            r = torch.stack([rw, rh, rw, rh]).to(device=like.device, dtype=like.dtype)
            cache[key] = r
        return r


# ------------------------------------------------------------------------------------ FPN
class FusedFPN(FeaturePyramidNetwork):
    """torchvision's FeaturePyramidNetwork (TV ops/feature_pyramid_network.py; fasterrcnn.py:317) whose top-down merge
    runs natively on CUDA: the lateral 1x1 convs run without their bias, and `ops.fpn_top_down` adds the bias, the
    nearest-upsampled coarser level and the lateral in one pass per level (one pass per level backward as well),
    instead of a bias-add pass, a full-size upsampled copy and an add.  The 3x3 layer blocks run their conv without the
    bias and `ops.bias_add` adds it (under autocast they are the stock modules).  The coarsest lateral conv and
    LastLevelMaxPool are the stock modules.  Same parameters, state-dict keys and results, bit for bit.  On CPU it is
    torchvision's forward."""

    def forward(self, x: Dict[str, Tensor]) -> Dict[str, Tensor]:
        names, feats = list(x.keys()), list(x.values())
        if not feats[-1].is_cuda:
            return super().forward(x)
        convs = [blk[0] for blk in self.inner_blocks]
        top = self.inner_blocks[-1](feats[-1])
        if torch.is_autocast_enabled("cuda"):
            # Under autocast F.interpolate runs in fp32 (upsample_nearest2d is on autocast's fp32 list), so the stock
            # merge adds a bf16 lateral, bias included, to an fp32 map: every merged level but the top is fp32.  The fp32
            # merge on the upcast laterals computes exactly that; their bias is already in, so it adds -0.0 (an exact
            # identity).  The top feeds its layer block as the bf16 map the stock forward uses.
            laterals = [conv(f).float() for conv, f in zip(convs[:-1], feats[:-1])]
            no_bias = [torch.full((conv.out_channels,), -0.0, device=top.device) for conv in convs[:-1]]
            inners = ops.fpn_top_down(laterals, no_bias, top.float())
            inners[-1] = top
            results = [blk(t) for blk, t in zip(self.layer_blocks, inners)]
        else:
            laterals = [conv._conv_forward(f, conv.weight, None) for conv, f in zip(convs[:-1], feats[:-1])]
            inners = ops.fpn_top_down(laterals, [conv.bias for conv in convs[:-1]], top)
            # each 3x3 layer block as ATen runs a cuDNN conv: the conv without its bias, then the bias add (natively)
            layers = [blk[0] for blk in self.layer_blocks]
            results = [ops.bias_add(conv._conv_forward(t, conv.weight, None), conv.bias) for conv, t in zip(layers, inners)]
        if self.extra_blocks is not None:
            results, names = self.extra_blocks(results, feats, names)
        return OrderedDict(zip(names, results))


def fuse_fpn(fpn: FeaturePyramidNetwork) -> None:
    """Rebinds a stock FeaturePyramidNetwork without norm layers (each inner and layer block a single biased Conv2d) to
    FusedFPN."""
    if type(fpn) is not FeaturePyramidNetwork:
        raise TypeError(f"fuse_fpn expects a torchvision FeaturePyramidNetwork, got {type(fpn).__name__}")
    for blk in (*fpn.inner_blocks, *fpn.layer_blocks):
        if len(blk) != 1 or type(blk[0]) is not nn.Conv2d or blk[0].bias is None:
            raise TypeError("fuse_fpn: every inner and layer block must be one Conv2d with a bias (no norm layer)")
    fpn.__class__ = FusedFPN


# ------------------------------------------------------------------------------------ detector
class FasterRCNN(nn.Module):
    def __init__(self, num_classes: int = 9, min_size: int = 800, max_size: int = 1333,
                 trainable_backbone_layers: int = 5, rpn_batch_size_per_image=256, box_batch_size_per_image=512):
        super().__init__()
        self.transform = FusedTransform(min_size, max_size, [0.0, 0.0, 0.0], [1.0, 1.0, 1.0])  # fasterrcnn.py:439-441
        self.backbone = resnet_fpn_backbone(backbone_name="resnet50", weights=None,
                                            trainable_layers=trainable_backbone_layers)   # fasterrcnn.py:317
        fuse_fpn(self.backbone.fpn)
        oc = self.backbone.out_channels
        self.rpn = RegionProposalNetwork(oc, ((32,), (64,), (128,), (256,), (512,)), ((0.5, 1.0, 2.0),) * 5,
                                         batch_size_per_image=rpn_batch_size_per_image)
        self.roi_heads = RoIHeads(oc, num_classes, batch_size_per_image=box_batch_size_per_image)
        self.last: Dict[str, object] = {}

    def forward(self, images: List[Tensor], targets: Optional[List[Dict[str, Tensor]]] = None,
                sampler_keys: Optional[Dict[str, Tensor]] = None):
        """Returns a list of per-image dicts: 'boxes', 'scores', 'labels' (padded to
        detections_per_img rows in training, 'num' = valid rows) and, in training, 'losses'
        (fasterrcnn.py:492-497)."""
        if self.training and targets is None:
            raise ValueError("In training mode, targets should be passed")
        original_sizes = [tuple(img.shape[-2:]) for img in images]
        image_list, targets = self.transform(images, targets)
        if targets is not None:
            for ti, t in enumerate(targets):
                b = t["boxes"]
                if b.dim() != 2 or b.shape[-1] != 4:
                    raise ValueError(f"Expected target boxes to be a tensor of shape [N, 4], got {b.shape}.")
        features = self.backbone(image_list.tensors)
        keys = sampler_keys or {}
        (pb, ps, pc), rpn_losses = self.rpn(image_list.tensors.shape, image_list.image_sizes, features, targets,
                                            keys.get("rpn"))
        if self.training:
            proposals = (pb, pc)                               # padded + device counts: training never reads them back
        else:
            proposals = [pb[i, :c] for i, c in enumerate(pc.tolist())]
        det, roi_losses, box_features, box_labels = self.roi_heads(features, proposals, image_list.image_sizes,
                                                                   targets, keys.get("roi"))
        self.last = {"features": features, "box_features": box_features, "box_labels": box_labels,
                     "proposals": proposals}
        boxes, scores, labels, num = det
        out = []
        for i in range(len(images)):
            d = {"boxes": boxes[i], "scores": scores[i], "labels": labels[i], "num": num[i]}
            if self.training:
                d["losses"] = {k: v[i] for k, v in {**rpn_losses, **roi_losses}.items()}
            out.append(d)
        if not self.training:
            nums = num.tolist()
            for i, d in enumerate(out):
                n = nums[i]
                b = d["boxes"][:n]
                oh, ow = original_sizes[i]
                h, w = image_list.image_sizes[i]
                ratio = torch.tensor([ow / w, oh / h, ow / w, oh / h], dtype=b.dtype, device=b.device)
                out[i] = {"boxes": b * ratio, "scores": d["scores"][:n], "labels": d["labels"][:n]}
        return out
