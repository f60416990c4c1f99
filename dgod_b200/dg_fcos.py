"""Host-side mirror of the reference's FCOS detector and DGFCOS training step (BASELINE configs[2]).

`fcos.py` of the reference is torchvision's FCOS with three changes — the `len(labels) <= 1`
rule (fcos.py:139), the `(y1-x1)*(y2-y1)` area (fcos.py:543) and the one-hot `gt_classes` handed
back in the loss dict (fcos.py:201) — and `DGFCOS.py` drives it through the same five-mode
schedule as DGFRCNN.  Here the backbone / heads stay torchvision modules on PyTorch/cuDNN; the
per-location work of the path runs on the sm_100a kernels:

  * location -> GT assignment + target gather (fcos.py:510-548, 136-158): ONE `dgod_fcos_assign`
    launch per batch (rows A10/A11 of SURVEY.md §8a) instead of ~25 ATen kernels per image;
  * eval post-processing (fcos.py:552-619): `ops.clip_boxes_to_image` / `ops.batched_nms` (row A12);
  * gradient reversal in front of the DG heads (DGcommon.py:33-45, row A13): fused into the first layer's input gradient
    (`ops.grl_conv2d` for ImageDA.Conv1, `ops.grl_linear` for the per-location heads).

Names, arguments and the contents of the returned dicts follow the reference so that the parity
tests read like its own code.
"""
from __future__ import annotations

from typing import Dict, List, Optional, Sequence

import torch
import torch.nn.functional as F
from torch import Tensor, nn
from torchvision.models.detection.backbone_utils import _resnet_fpn_extractor
from torchvision.models.detection.fcos import FCOS as _TVFCOS, FCOSHead as _TVFCOSHead
from torchvision.models.resnet import resnet50
from torchvision.ops import generalized_box_iou_loss, sigmoid_focal_loss
from torchvision.ops import misc as misc_nn_ops
from torchvision.ops.feature_pyramid_network import LastLevelP6P7

from . import ops
from .detector import FusedTransform
from .metrics import DetectionValidation


# --------------------------------------------------------------------------------- detector
class FCOSHead(_TVFCOSHead):
    """fcos.py:103-213.  `compute_loss` takes the targets the assignment kernel already gathered and, by
    default, evaluates the focal / GIoU / centre-ness tail (fcos.py:149-202) with the fused `ops.fcos_loss`
    kernels (forward 2 launches, backward 1, no host sync); `fused_loss = False` keeps the ATen chain."""

    fused_loss = True

    def compute_loss(self, targets, head_outputs: Dict[str, Tensor], anchors: List[Tensor], assigned) -> Dict[str, Tensor]:
        if self.fused_loss:
            _, cls_t, box_t, onehot = assigned
            out = ops.fcos_loss(head_outputs["cls_logits"], head_outputs["bbox_regression"], head_outputs["bbox_ctrness"],
                                anchors[0], cls_t, box_t)
            return {"classification": out[0], "bbox_regression": out[1], "bbox_ctrness": out[2], "gt_classes": onehot}
        cls_logits = head_outputs["cls_logits"]            # [B, N, C]
        bbox_regression = head_outputs["bbox_regression"]  # [B, N, 4]
        bbox_ctrness = head_outputs["bbox_ctrness"]        # [B, N, 1]
        _, all_gt_classes_targets, all_gt_boxes_targets, gt_classes_targets = assigned
        foregroud_mask = all_gt_classes_targets >= 0
        num_foreground = foregroud_mask.sum()              # stays on the device: no .item() sync (fcos.py:154)
        denom = num_foreground.clamp(min=1).to(cls_logits.dtype)

        loss_cls = sigmoid_focal_loss(cls_logits, gt_classes_targets, reduction="sum")            # fcos.py:159
        anchors_b = torch.stack(anchors)                                                         # [B, N, 4]
        pred_boxes = self.box_coder.decode(bbox_regression, anchors_b)                           # fcos.py:165-168
        loss_bbox_reg = generalized_box_iou_loss(pred_boxes[foregroud_mask].float(),
                                                 all_gt_boxes_targets[foregroud_mask], reduction="sum")
        bbox_reg_targets = self.box_coder.encode(anchors_b, all_gt_boxes_targets)                # fcos.py:178-182
        left_right = bbox_reg_targets[:, :, [0, 2]]
        top_bottom = bbox_reg_targets[:, :, [1, 3]]
        gt_ctrness_targets = torch.sqrt((left_right.min(dim=-1)[0] / left_right.max(dim=-1)[0])
                                        * (top_bottom.min(dim=-1)[0] / top_bottom.max(dim=-1)[0]))
        pred_centerness = bbox_ctrness.squeeze(dim=2)
        loss_bbox_ctrness = F.binary_cross_entropy_with_logits(pred_centerness[foregroud_mask],
                                                               gt_ctrness_targets[foregroud_mask], reduction="sum")
        return {
            "classification": loss_cls / denom,
            "bbox_regression": loss_bbox_reg / denom,
            "bbox_ctrness": loss_bbox_ctrness / denom,
            "gt_classes": gt_classes_targets,              # fcos.py:201 — what DGFCOS.py:211,222,237 consume
        }


class FCOS(_TVFCOS):
    """fcos.py:346-690 on the fused kernels."""

    def __init__(self, backbone, num_classes, **kwargs):
        super().__init__(backbone, num_classes, **kwargs)
        # same construction order and shapes as TV's head: parameters initialise identically under one seed
        head = FCOSHead(backbone.out_channels, self.anchor_generator.num_anchors_per_location()[0], num_classes)
        head.load_state_dict(self.head.state_dict())
        self.head = head
        self.num_classes = num_classes
        t = self.transform                                   # fcos.py:483 -> the one-launch transform
        self.transform = FusedTransform(t.min_size, t.max_size, t.image_mean, t.image_std, size_divisible=t.size_divisible,
                                        fixed_size=t.fixed_size)

    def compute_loss(self, targets, head_outputs, anchors, num_anchors_per_level):
        # fcos.py:503-550: anchors are identical for every image of a batch (one padded size)
        assigned = ops.fcos_assign(anchors[0], [t["boxes"] for t in targets], list(num_anchors_per_level),
                                   self.center_sampling_radius, gt_labels=[t["labels"] for t in targets],
                                   num_classes=self.num_classes)
        return self.head.compute_loss(targets, head_outputs, anchors, assigned)

    def postprocess_detections(self, head_outputs, anchors, image_shapes):
        """fcos.py:552-619 for the batch: candidates (score, threshold, top-k, decode, clip) of every image and level in ONE
        launch, the per-class NMS of all images in ONE segmented call (vanilla mode; the reference switches to the
        coordinate trick below 4 000 candidates, same keeps up to rounding-edge pairs), one device->host read for the
        detection counts that TV's list-of-dicts result needs."""
        class_logits, box_regression, box_ctrness = (head_outputs["cls_logits"], head_outputs["bbox_regression"],
                                                     head_outputs["bbox_ctrness"])
        npl = [a.shape[0] for a in anchors[0]]
        cl, rg, ct = torch.cat(list(class_logits), dim=1), torch.cat(list(box_regression), dim=1), torch.cat(list(box_ctrness), dim=1)
        dev = cl.device
        sizes = ops.device_constant(tuple((float(h), float(w)) for h, w in image_shapes), torch.float32, dev)
        boxes, scores, labels, valid, _ = ops.fcos_candidates(cl, rg, ct, torch.cat(list(anchors[0])), npl, sizes,
                                                               self.score_thresh, self.topk_candidates)
        B, per = boxes.shape[0], boxes.shape[1]
        keep, info = ops.nms_segments(boxes.view(-1, 4), scores.view(-1), labels.view(-1), [per] * B, self.nms_thresh,
                                      valid=valid.view(-1), max_out_per_seg=self.detections_per_img)
        nums = info[:-1].tolist()
        detections: List[Dict[str, Tensor]] = []
        for i in range(B):
            k = keep[i, :nums[i]]
            detections.append({"boxes": boxes[i][k], "scores": scores[i][k], "labels": labels[i][k]})
        return detections


def fcos_resnet50_fpn(num_classes: int = 9, trainable_backbone_layers: int = 3, **kwargs) -> FCOS:
    """fcos.py:702-788 without the downloads (random init, as bench.py's synthetic runs need)."""
    backbone = resnet50(weights=None, norm_layer=misc_nn_ops.FrozenBatchNorm2d)
    backbone = _resnet_fpn_extractor(backbone, trainable_backbone_layers, returned_layers=[2, 3, 4],
                                     extra_blocks=LastLevelP6P7(256, 256))
    return FCOS(backbone, num_classes, **kwargs)


# --------------------------------------------------------------------------------- DG heads
class ImageDA(nn.Module):
    """DGcommon.py:86-113: image-level domain classifier on C5 (2048 channels) behind the GRL."""

    def __init__(self, num_domains: int):
        super().__init__()
        self.num_domains = num_domains
        self.Conv1 = nn.Conv2d(2048, 1024, 3, stride=(2, 4))
        self.Conv2 = nn.Conv2d(1024, 512, 3, stride=2)
        self.Conv3 = nn.Conv2d(512, 256, 3, stride=2)
        self.flatten = nn.Flatten()
        self.linear1 = nn.Linear(256, 128)
        self.linear2 = nn.Linear(128, num_domains)
        self.reLu = nn.ReLU(inplace=False)
        for conv in (self.Conv1, self.Conv2, self.Conv3):
            torch.nn.init.normal_(conv.weight, std=0.001)
            torch.nn.init.constant_(conv.bias, 0)

    def forward(self, x: Tensor) -> Tensor:
        x = self.reLu(ops.grl_conv2d(x, self.Conv1))        # grad_reverse fused into Conv1's input gradient (DGcommon.py:106-107)
        x = self.reLu(self.Conv2(x))
        x = self.reLu(self.Conv3(x))
        x = self.reLu(self.linear1(self.flatten(x)))
        return torch.sigmoid(self.linear2(x))


class InstanceDA(nn.Module):
    """DGFCOS.py:4-17: per-location domain classifier on the 256-channel head input."""

    def __init__(self, num_domains: int):
        super().__init__()
        self.dc_ip1 = nn.Linear(256, 128)
        self.dc_relu1 = nn.ReLU()
        self.classifer = nn.Linear(128, num_domains)

    def forward(self, x: Tensor) -> Tensor:
        x = ops.grl_linear(x, self.dc_ip1.weight, self.dc_ip1.bias)      # grad_reverse fused into dc_ip1's dgrad (DGFCOS.py:14-15)
        return torch.sigmoid(self.classifer(self.dc_relu1(x)))


class _InsCls(nn.Module):
    """DGFCOS.py:19-56: per-location class heads (InsClsPrime sits behind the GRL, InsCls does not)."""

    def __init__(self, num_cls: int, reverse: bool):
        super().__init__()
        self.reverse = reverse
        self.dc_ip1 = nn.Linear(256, 128)
        self.dc_relu1 = nn.ReLU()
        self.dc_ip2 = nn.Linear(128, 64)
        self.dc_relu2 = nn.ReLU()
        self.classifer = nn.Linear(64, num_cls)

    def forward(self, x: Tensor) -> Tensor:
        if self.reverse:
            x = ops.grl_linear(x, self.dc_ip1.weight, self.dc_ip1.bias)  # DGFCOS.py:34-35
        else:
            x = self.dc_ip1(x)
        x = self.dc_ip2(self.dc_relu1(x))
        return torch.sigmoid(self.classifer(x))


class InsClsPrime(_InsCls):
    def __init__(self, num_cls: int):
        super().__init__(num_cls, True)


class InsCls(_InsCls):
    def __init__(self, num_cls: int):
        super().__init__(num_cls, False)


# --------------------------------------------------------------------------------- DGFCOS
class DGFCOS(DetectionValidation, nn.Module):
    """DGFCOS.py:115-243 without the Lightning trainer: `training_step(batch)` returns the loss of
    the current mode and advances the 0,1,0,2,0,3,0,4 schedule.  batch = (images, boxes, labels,
    domain) as the reference's collate_fn yields them (DGcommon.py:14-31), tensors on the device.
    `validation_step` / `on_validation_epoch_end` score the detector with mAP@0.5 (metrics.DetectionValidation)."""

    def __init__(self, n_classes: int, batch_size: int, exp: str, reg_weights: Sequence[float], num_domains: int,
                 min_size: int = 600, max_size: int = 1200):
        super().__init__()
        self.n_classes, self.batch_size, self.exp = n_classes, batch_size, exp
        self.reg_weights, self.num_domains = list(reg_weights), num_domains
        self.mode = 0
        self.sub_mode = 0
        self.InsDA = InstanceDA(num_domains)
        self.InsClsPrime = nn.ModuleList([InsClsPrime(n_classes) for _ in range(num_domains)])
        self.InsCls = nn.ModuleList([InsCls(n_classes) for _ in range(num_domains)])
        self.detector = fcos_resnet50_fpn(num_classes=n_classes, trainable_backbone_layers=3,
                                          min_size=min_size, max_size=max_size)                  # DGFCOS.py:119
        self.detector.backbone.body.register_forward_hook(self._store_backbone_out)              # DGFCOS.py:120
        self.detector.head.register_forward_hook(self._store_head_input)                         # DGFCOS.py:121
        self.ImageDA = ImageDA(num_domains)
        self.base_lr, self.weight_decay = 1e-4, 0.0001
        self.base_feat: Optional[Tensor] = None
        self.ins_feat: Optional[Tensor] = None

    def _store_backbone_out(self, module, inputs, output):
        self.base_feat = output["2"]                       # C5: the image-level feature (DGFCOS.py:128-129)

    def _store_head_input(self, module, inputs, output):
        # the five FPN maps the head sees, flattened to [B, sum(HW), 256] (DGFCOS.py:131-137)
        self.ins_feat = torch.cat([f.flatten(2) for f in inputs[0]], dim=-1).permute(0, 2, 1)

    def configure_optimizer(self, lr: Optional[float] = None):
        lr = self.base_lr if lr is None else lr
        groups = [self.detector, self.ImageDA, self.InsDA, self.InsCls, self.InsClsPrime]       # DGFCOS.py:140-146
        return torch.optim.Adam([{"params": m.parameters(), "lr": lr, "weight_decay": self.weight_decay} for m in groups])

    def _advance_after_mode0(self):
        if self.exp != "dg":
            return
        if self.sub_mode in (0, 1, 2, 3):                  # DGFCOS.py:166-180
            self.sub_mode += 1
            self.mode = self.sub_mode
        else:
            self.sub_mode = 0
            self.mode = 0

    def training_step(self, batch) -> Tensor:
        imgs = list(batch[0])
        targets = [{"boxes": b.float(), "labels": l.long()} for b, l in zip(batch[1], batch[2])]
        # batch[3] is a host tensor in the reference (DGcommon.collate_fn; `.to(device=0)` at DGFCOS.py:186): the per-image
        # loops of modes 2-4 read the ids from it for free; a device tensor costs one device->host read there
        dom_src = batch[3]
        domain = dom_src.to(imgs[0].device, non_blocking=True)
        if self.mode == 0:
            loss_dict = self.detector(imgs, targets)
            loss = loss_dict["classification"] + loss_dict["bbox_regression"] + loss_dict["bbox_ctrness"]
            self._advance_after_mode0()
            return loss
        if self.mode == 1:                                 # DGFCOS.py:182-194
            self.detector(imgs, targets)
            img_scores = self.ImageDA(self.base_feat)
            loss = self.reg_weights[0] * F.cross_entropy(img_scores, domain)
            ida = self.InsDA(self.ins_feat)                # [B, N, D]
            n_loc = ida.shape[1]
            loss = loss + self.reg_weights[1] * F.cross_entropy(ida.permute(0, 2, 1),
                                                                domain.unsqueeze(-1).repeat(1, n_loc).long())
            loss = loss + self.reg_weights[2] * F.mse_loss(img_scores.unsqueeze(1).repeat(1, n_loc, 1), ida)
            self.mode = 0
            return loss
        dom = dom_src.tolist()
        losses = []
        if self.mode == 2:                                 # DGFCOS.py:196-208: detector frozen, InsCls learn
            for head in self.InsCls:
                for p in head.parameters():
                    p.requires_grad = True
            for i in range(len(imgs)):
                with torch.no_grad():
                    out = self.detector([imgs[i]], [targets[i]])
                # the reference feeds [1,N,C] scores and the [1,N,C] one-hot to cross_entropy as they are:
                # dim 1 (the locations) is the "class" axis and the target is read as probabilities
                losses.append(F.cross_entropy(self.InsCls[dom[i]](self.ins_feat), out["gt_classes"]))
            weight = self.reg_weights[4]
        elif self.mode == 3:                               # DGFCOS.py:210-219
            for i in range(len(imgs)):
                out = self.detector([imgs[i]], [targets[i]])
                losses.append(F.cross_entropy(self.InsClsPrime[dom[i]](self.ins_feat), out["gt_classes"]))
            weight = self.reg_weights[3]
        else:                                              # mode 4, DGFCOS.py:221-236
            for head in self.InsCls:
                for p in head.parameters():
                    p.requires_grad = False
            for i in range(len(imgs)):
                out = self.detector([imgs[i]], [targets[i]])
                for d in range(len(self.InsCls)):
                    if d != dom[i]:
                        losses.append(F.cross_entropy(self.InsCls[d](self.ins_feat), out["gt_classes"]))
            weight = self.reg_weights[4]
            self.sub_mode = 0
        self.mode = 0
        return weight * torch.mean(torch.stack(losses))
