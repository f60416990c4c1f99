"""DG-mode training logic of the reference's DGFRCNN (DGFRCNN.py:73-201, DGcommon.py:33-172) as a
plain nn.Module + explicit step function (pytorch_lightning is not a dependency of the hot path).

Same heads, same 5-mode schedule (0,1,0,2,0,3,0,4), same per-image detector passes in modes 2-4,
same optimizer (SGD lr 2e-3, wd 5e-4).  Every gradient-reversal layer is fused into the input-gradient
of the layer behind it: the instance-level heads start with a Linear (DGFRCNN.py:8,19-20,29,40-41:
ops.grl_linear, the scale is the GEMM's alpha), the image-level head with a Conv2d (DGcommon.py:53,73-74:
ops.grl_conv2d, cuDNN's dgrad on the pre-scaled weight).  `ops.grad_reverse` (the stand-alone kernel)
remains what `patch()` binds to the reference's own `grad_reverse` call sites.
"""
from __future__ import annotations

from typing import Dict, List, Optional, Sequence

import torch
import torch.distributed as dist
import torch.nn.functional as F
from torch import Tensor, nn

from . import ops
from .detector import FasterRCNN
from .metrics import DetectionValidation


class ImageDAFPN(nn.Module):
    """DGcommon.py:48-81: GRL -> 4 strided convs -> Linear(256,128) -> Linear(128,D) -> sigmoid."""

    def __init__(self, num_domains: int):
        super().__init__()
        self.Conv1 = nn.Conv2d(256, 256, 3, stride=(2, 4))
        self.Conv2 = nn.Conv2d(256, 256, 3, stride=4)
        self.Conv3 = nn.Conv2d(256, 256, 3, stride=4)
        self.Conv4 = nn.Conv2d(256, 256, 3, stride=3)
        self.linear1 = nn.Linear(256, 128)
        self.linear2 = nn.Linear(128, num_domains)
        for conv in (self.Conv1, self.Conv2, self.Conv3, self.Conv4):
            nn.init.normal_(conv.weight, std=0.001)
            nn.init.constant_(conv.bias, 0)

    def forward(self, x: Tensor) -> Tensor:
        x = F.relu(ops.grl_conv2d(x, self.Conv1))           # grad_reverse fused into Conv1's input gradient (DGcommon.py:73-74)
        for conv in (self.Conv2, self.Conv3, self.Conv4):
            x = F.relu(conv(x))
        x = F.relu(self.linear1(x.flatten(1)))
        return torch.sigmoid(self.linear2(x))


class _InstanceMLP(nn.Module):
    """Linear(1024,512)-ReLU-Linear(512,256)-Linear(256,out)-sigmoid (DGFRCNN.py:4-64)."""

    def __init__(self, n_out: int, reverse: bool):
        super().__init__()
        self.dc_ip1 = nn.Linear(1024, 512)
        self.dc_ip2 = nn.Linear(512, 256)
        self.classifer = nn.Linear(256, n_out)
        self.reverse = reverse

    def forward(self, x: Tensor) -> Tensor:
        if self.reverse:
            x = ops.grl_linear(x, self.dc_ip1.weight, self.dc_ip1.bias)   # grad_reverse fused into dc_ip1's dgrad
        else:
            x = self.dc_ip1(x)
        x = self.dc_ip2(F.relu(x))
        return torch.sigmoid(self.classifer(x))


class InstanceDA(_InstanceMLP):
    def __init__(self, num_domains: int):
        super().__init__(num_domains, reverse=True)


class InsClsPrime(_InstanceMLP):
    def __init__(self, num_cls: int):
        super().__init__(num_cls, reverse=True)


class InsCls(_InstanceMLP):
    def __init__(self, num_cls: int):
        super().__init__(num_cls, reverse=False)


class DGFRCNN(DetectionValidation, nn.Module):
    """DGFRCNN.py:73-201.  `training_step(batch)` returns the loss and advances the mode schedule;
    `batch` = (images list, boxes list, labels list, domain tensor) like DGcommon.collate_fn.  `validation_step` /
    `on_validation_epoch_end` score the detector with mAP@0.5 (metrics.DetectionValidation)."""

    def __init__(self, n_classes: int, batch_size: int, exp: str, reg_weights: Sequence[float], num_domains: int,
                 min_size: int = 600, max_size: int = 1200, batched_modes: bool = True,
                 trainable_backbone_layers: int = 3):
        super().__init__()
        self.n_classes, self.batch_size, self.exp = n_classes, batch_size, exp
        # Modes 2-4 of the reference run B separate batch-1 detector passes (DGFRCNN.py:165,177,190).
        # Every term of those losses is per image (frozen BatchNorm, per-image RPN / RoI heads), so one
        # batched pass + per-image slices of box_features / box_labels gives the same losses and
        # gradients with 1/B of the launches (SURVEY.md §8f rank 2).  False = the reference's loop.
        self.batched_modes = batched_modes
        # modes 2-4, batched: evaluate only the heads whose domain occurs in the batch (needs the domain ids on the
        # host).  With the ids on the device and this flag off, every head is evaluated and masked instead (no host
        # read; heads without a matching image then receive zero gradients rather than none).
        self.exact_head_set = True
        self.reg_weights, self.num_domains = list(reg_weights), num_domains
        self.mode = 0
        self.sub_mode = 0
        self.InsDA = InstanceDA(num_domains)
        self.InsClsPrime = nn.ModuleList([InsClsPrime(n_classes) for _ in range(num_domains)])
        self.InsCls = nn.ModuleList([InsCls(n_classes) for _ in range(num_domains)])
        # DGFRCNN.py:81 -> fasterrcnn.py:307-329: the factory builds FastRCNNPredictor(in_features, num_classes + 1) (10 logits,
        # 40 box outputs for the 9 of DGOD) and, with pretrained=True, keeps trainable_backbone_layers=3 (conv1 / layer1 frozen)
        self.detector = FasterRCNN(num_classes=n_classes + 1, min_size=min_size, max_size=max_size,
                                   trainable_backbone_layers=trainable_backbone_layers)
        self.ImageDA = ImageDAFPN(num_domains)
        self.base_lr, self.weight_decay = 2e-3, 0.0005

    def configure_optimizer(self, lr: Optional[float] = None):
        """SGD as in DGFRCNN.py:98-104; `lr` overrides the reference's 2e-3 (bench.py uses a tiny
        rate: random-init weights diverge at 2e-3, the reference starts from pretrained ones)."""
        groups = [{"params": m.parameters(), "lr": self.base_lr if lr is None else lr, "weight_decay": self.weight_decay}
                  for m in (self.detector, self.ImageDA, self.InsDA, self.InsCls, self.InsClsPrime)]
        return torch.optim.SGD(groups)                                     # DGFRCNN.py:98-104

    # hooks of DGFRCNN.py:89-94 become plain reads of what the detector just produced
    @property
    def box_features(self):
        return self.detector.last["box_features"]

    @property
    def box_labels(self):
        return self.detector.last["box_labels"]

    @property
    def base_feat(self):
        return self.detector.last["features"]

    def _advance_after_mode0(self):
        if self.exp != "dg":
            return
        if self.sub_mode < 4:                                              # DGFRCNN.py:128-143
            self.sub_mode += 1
            self.mode = self.sub_mode
        else:
            self.sub_mode = 0
            self.mode = 0

    def _instance_losses_batched(self, heads, domain: Tensor, own_domain: bool, dom_list=None) -> Tensor:
        """Per-(image, head) cross-entropy terms of modes 2-4 from ONE batched detector pass.
        A head scores every image's 512 RoI features; a device-side mask then keeps head domain[i] for image i
        (own_domain) or all the other heads (mode 4).  Only the heads the reference's per-image loop would touch are
        evaluated (`dom_list`, the domain ids on the host — the reference reads them with `.item()` per image,
        DGFRCNN.py:165,177,193), so the untouched heads keep `.grad is None` and the optimizer skips them exactly as
        it does for the reference.  Returns the mean over the kept terms (DGFRCNN.py:170,181,196)."""
        feats = self.box_features                                           # [B*S, 1024]
        B = len(self.box_labels)
        labels = torch.stack(self.box_labels).reshape(-1)                   # [B*S]
        S = labels.numel() // B
        D = len(heads)
        if dom_list is None:
            used = list(range(D))
        elif own_domain:
            used = sorted(set(dom_list))
        else:
            used = [j for j in range(D) if any(d != j for d in dom_list)]
        per = []
        for j in used:
            ce = F.cross_entropy(heads[j](feats), labels, reduction="none").view(B, S)
            n = (labels.view(B, S) >= 0).sum(1).clamp(min=1)                # == S unless the sampler left slots empty
            per.append(ce.sum(1) / n)
        if dom_list is not None:
            # the kept (image, head) terms in the reference loop's order; views + one stack, no host->device traffic
            terms = [per[k][i] for i, d in enumerate(dom_list) for k, j in enumerate(used) if (j == d) == own_domain]
            return torch.stack(terms).mean()
        per = torch.stack(per, dim=1)                                       # [B, D]
        own = F.one_hot(domain.long(), D).to(per.dtype)
        keep = own if own_domain else 1.0 - own
        return (per * keep).sum() / keep.sum()

    def training_step(self, batch) -> Tensor:
        imgs, boxes, labels, domain = batch
        dev = imgs[0].device
        targets = [{"boxes": b.float(), "labels": l.long()} for b, l in zip(boxes, labels)]
        # batch[3] is a host tensor in the reference (DGcommon.collate_fn; `.to(device=0)` at DGFRCNN.py:150): reading
        # the ids there costs nothing.  A device tensor works too, at the price of one device->host read in modes 2-4.
        dom_host = domain.tolist() if (self.mode >= 2 and (not domain.is_cuda or not self.batched_modes or self.exact_head_set)) else None
        domain = domain.to(dev, non_blocking=True)
        if self.batched_modes and self.mode >= 2:
            if self.mode == 2:
                for head in self.InsCls:
                    for p in head.parameters():
                        p.requires_grad = True
                with torch.no_grad():
                    self.detector(imgs, targets)
                loss = self.reg_weights[4] * self._instance_losses_batched(self.InsCls, domain, True, dom_host)
            elif self.mode == 3:
                self.detector(imgs, targets)
                loss = self.reg_weights[3] * self._instance_losses_batched(self.InsClsPrime, domain, True, dom_host)
            else:
                for head in self.InsCls:
                    for p in head.parameters():
                        p.requires_grad = False
                self.detector(imgs, targets)
                loss = self.reg_weights[4] * self._instance_losses_batched(self.InsCls, domain, False, dom_host)
                self.sub_mode = 0
            self.mode = 0
            return loss
        dom_list = dom_host
        if self.mode == 0:
            det = self.detector(imgs, targets)
            loss = sum(v for d in det for v in d["losses"].values())      # DGFRCNN.py:126-127
            self._advance_after_mode0()
        elif self.mode == 1:
            self.detector(imgs, targets)
            img_scores = self.ImageDA(self.base_feat["0"])
            l_img = self.reg_weights[0] * F.cross_entropy(img_scores, domain)
            ida = self.InsDA(self.box_features)
            rep = int(ida.shape[0] / self.batch_size)
            ins_labels = domain.reshape(self.batch_size, 1).repeat(1, rep).reshape(ida.shape[0])
            l_ins = self.reg_weights[1] * F.cross_entropy(ida, ins_labels)
            exp_scores = img_scores.repeat(1, rep).reshape(ida.shape[0], self.num_domains)
            l_cst = self.reg_weights[2] * F.mse_loss(ida, exp_scores)
            loss = l_img + l_ins + l_cst                                   # DGFRCNN.py:146-157
            self.mode = 0
        elif self.mode == 2:
            for head in self.InsCls:
                for p in head.parameters():
                    p.requires_grad = True
            per = []
            for i in range(len(imgs)):
                with torch.no_grad():
                    self.detector([imgs[i]], [targets[i]])
                scores = self.InsCls[dom_list[i]](self.box_features)
                per.append(F.cross_entropy(scores, self.box_labels[0]))
            loss = self.reg_weights[4] * torch.mean(torch.stack(per))      # DGFRCNN.py:159-171
            self.mode = 0
        elif self.mode == 3:
            per = []
            for i in range(len(imgs)):
                self.detector([imgs[i]], [targets[i]])
                scores = self.InsClsPrime[dom_list[i]](self.box_features)
                per.append(F.cross_entropy(scores, self.box_labels[0]))
            loss = self.reg_weights[3] * torch.mean(torch.stack(per))      # DGFRCNN.py:173-182
            self.mode = 0
        else:
            for head in self.InsCls:
                for p in head.parameters():
                    p.requires_grad = False
            per = []
            for i in range(len(imgs)):
                self.detector([imgs[i]], [targets[i]])
                for j in range(self.num_domains):
                    if j != dom_list[i]:
                        scores = self.InsCls[j](self.box_features)
                        per.append(F.cross_entropy(scores, self.box_labels[0]))
            loss = self.reg_weights[4] * torch.mean(torch.stack(per))      # DGFRCNN.py:184-199
            self.mode = 0
            self.sub_mode = 0
        return loss


from .ddp import GradSync, allreduce_gradients  # noqa: E402,F401  (data-parallel gradient sync lives in ddp.py)
