"""MultiScaleRoIAlign with the four-level pooling done by ONE kernel launch.

Subclass of torchvision's module (fasterrcnn.py:380 asserts the type), same constructor and
`forward(x, boxes, image_shapes)` contract as TV ops/poolers.py:230-327.  Scale inference and
the LevelMapper parameters stay on the host exactly as upstream (TV ops/poolers.py:98-134);
the level mapping itself, the per-level gather and the result scatter of
TV ops/poolers.py:147-227 are fused into the kernel.
"""
from __future__ import annotations

from typing import Dict, List, Tuple, Union

import torch
from torch import Tensor
from torchvision.ops import poolers as tv_poolers

from . import ops


class MultiScaleRoIAlign(tv_poolers.MultiScaleRoIAlign):
    def forward(self, x: Dict[str, Tensor], boxes: Union[List[Tensor], Tensor],
                image_shapes: List[Tuple[int, int]]) -> Tensor:
        """`boxes`: a list of per-image [n_i,4] tensors, or one [B,S,4] tensor (S boxes for every image)."""
        x_filtered = tv_poolers._filter_input(x, self.featmap_names)
        if self.scales is None or self.map_levels is None:
            self.scales, self.map_levels = tv_poolers._setup_scales(
                x_filtered, image_shapes, self.canonical_scale, self.canonical_level)
        if isinstance(boxes, Tensor):
            B, S = boxes.shape[:2]
            ids = torch.arange(B, dtype=boxes.dtype, device=boxes.device).view(B, 1, 1).expand(B, S, 1)
            rois = torch.cat((ids, boxes), dim=2).view(B * S, 5)
            counts = [S] * B
        else:
            rois = ops._convert_to_roi_format(boxes)
            counts = [b.shape[0] for b in boxes]
        offsets = ops._offsets(counts, rois.device) if len(counts) == x_filtered[0].shape[0] else None
        m = self.map_levels
        return ops.multiscale_roi_align(
            x_filtered, rois, self.scales, tuple(self.output_size), self.sampling_ratio,
            k_min=m.k_min, k_max=m.k_max, canonical_scale=float(m.s0), canonical_level=float(m.lvl0),
            aligned=False, roi_img_offsets=offsets)

    @classmethod
    def from_torchvision(cls, pool: tv_poolers.MultiScaleRoIAlign) -> "MultiScaleRoIAlign":
        new = cls(pool.featmap_names, tuple(pool.output_size), pool.sampling_ratio,
                  canonical_scale=pool.canonical_scale, canonical_level=pool.canonical_level)
        return new
