"""torchvision-signature operators backed by the sm_100a kernels (via the C ABI).

Drop-in surface (SURVEY.md §8b): `nms`, `batched_nms`, `box_iou`, `roi_align`,
`multiscale_roi_align`, `Matcher`, `match_boxes`, `fcos_assign`, `grad_reverse`,
`rpn_proposals`, `rpn_filter_proposals`, `detect_candidates`.  Same names, argument meaning and
error behaviour as the functions they replace (torchvision 0.26.0 `ops/boxes.py`,
`ops/roi_align.py`, `ops/poolers.py`, `models/detection/_utils.py`; `fcos.py:510-548`;
`DGcommon.py:33-45`).  Every function requires CUDA tensors — there is no CPU path.

The compute entry points are also registered as PyTorch custom ops in the `dgod_b200::`
namespace (CUDA + fake/meta + autograd registrations), which is what `torch.ops.dgod_b200.*`
resolves to.
"""
from __future__ import annotations

import ctypes as C
import math
from typing import List, Optional, Sequence, Tuple

import torch
from torch import Tensor

from . import _lib
from ._lib import RoiConfig, RpnConfig, check

# torchvision's CPU rule for batched_nms (TV ops/boxes.py:80): more than this many box
# coordinates -> per-group NMS, else the coordinate-offset trick.  The oracle is the CPU path.
BATCHED_NMS_TRICK_MAX_NUMEL = 4000


# --------------------------------------------------------------------------------- helpers
def _stream() -> C.c_void_p:
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _p(t: Optional[Tensor]) -> Optional[C.c_void_p]:
    return None if t is None else C.c_void_p(t.data_ptr())


def _need_cuda(*ts: Optional[Tensor]):
    for t in ts:
        if t is not None and not t.is_cuda:
            raise RuntimeError("dgod_b200 ops need CUDA tensors (sm_100a); there is no CPU fallback")


# Per-call host overhead matters as much as the kernels for the latency-bound ops (a 20 us kernel behind 100 us of
# wrapper), so the small things a call needs are cached instead of rebuilt:
#   * scratch workspaces: one growing buffer per (device, stream) — kernels of one stream run in order, so the next
#     call may reuse the bytes of the previous one; nothing in a workspace outlives the call that filled it;
#   * offset vectors (`gt_offsets`, `seg_offsets`, `roi_img_offsets`) and other tiny host-built tensors: keyed by
#     their values — the counts repeat from step to step (512 RoIs per image, 20 boxes per image, ...), and a
#     `torch.tensor(list, device=cuda)` is a pageable host->device copy that stalls the launching thread.
_WS_CACHE: dict = {}
_CONST_CACHE: dict = {}
_CONST_CACHE_MAX = 4096


def _ws(nbytes: int, device) -> Tensor:
    n = max(int(nbytes), 1)
    key = (device.index if device.index is not None else torch.cuda.current_device(), torch.cuda.current_stream(device).cuda_stream)
    buf = _WS_CACHE.get(key)
    if buf is None or buf.numel() < n:
        buf = torch.empty(max(n, 1 << 20) * 5 // 4, dtype=torch.uint8, device=device)
        _WS_CACHE[key] = buf
    return buf


def _f32c(t: Tensor) -> Tensor:
    return t.contiguous() if t.dtype == torch.float32 else t.float().contiguous()


def device_constant(values, dtype, device) -> Tensor:
    """A small read-only device tensor holding `values` (nested tuples / lists of numbers), cached by value."""
    key = (repr(values), dtype, str(device))
    t = _CONST_CACHE.get(key)
    if t is None:
        if len(_CONST_CACHE) >= _CONST_CACHE_MAX:
            _CONST_CACHE.clear()
        t = torch.tensor(values, dtype=dtype, device=device)
        _CONST_CACHE[key] = t
    return t


def _offsets(counts: Sequence[int], device) -> Tensor:
    off = [0]
    for c in counts:
        off.append(off[-1] + int(c))
    return device_constant(tuple(off), torch.int32, device)


def _eager(op):
    """The Python body of a `torch.library.custom_op`.  The ops stay registered (`torch.ops.dgod_b200.*`: CUDA kernel,
    fake / meta kernel, autograd) for dispatcher users and torch.compile; the eager entry points of this module call the
    body directly — the custom_op wrapper costs 60-100 us per call (schema checks, dispatcher round trip, autograd
    bookkeeping), more than most of the kernels behind it."""
    if torch.compiler.is_compiling():
        return op
    return getattr(op, "_init_fn", op)


class KernelTimer:
    """Optional CUDA-event timing of individual kernels on the launching stream (bench.py's
    roofline leg).  Disabled by default: zero overhead."""
    enabled = False
    records: dict = {}

    @classmethod
    def reset(cls):
        cls.records = {}

    @classmethod
    def start(cls, name: str, nbytes: int):
        if not cls.enabled:
            return None
        e0 = torch.cuda.Event(enable_timing=True)
        e1 = torch.cuda.Event(enable_timing=True)
        e0.record()
        return (name, nbytes, e0, e1)

    @classmethod
    def stop(cls, tok):
        if tok is None:
            return
        name, nbytes, e0, e1 = tok
        e1.record()
        cls.records.setdefault(name, []).append((nbytes, e0, e1))

    @classmethod
    def summary(cls):
        """name -> (launches, total_ms, total_bytes); call after torch.cuda.synchronize()."""
        out = {}
        for name, recs in cls.records.items():
            ms = sum(e0.elapsed_time(e1) for _, e0, e1 in recs)
            out[name] = (len(recs), ms, sum(b for b, _, _ in recs))
        return out


# --------------------------------------------------------------------------------- box_iou
@torch.library.custom_op("dgod_b200::box_iou", mutates_args=())
def _box_iou_op(boxes1: Tensor, boxes2: Tensor) -> Tensor:
    _need_cuda(boxes1, boxes2)
    b1, b2 = _f32c(boxes1), _f32c(boxes2)
    out = torch.empty((b1.shape[0], b2.shape[0]), dtype=torch.float32, device=b1.device)
    check(_lib.load().dgod_box_iou(_p(b1), b1.shape[0], _p(b2), b2.shape[0], _p(out), _stream()))
    return out


@_box_iou_op.register_fake
def _(boxes1, boxes2):
    return boxes1.new_empty((boxes1.shape[0], boxes2.shape[0]), dtype=torch.float32)


def box_iou(boxes1: Tensor, boxes2: Tensor) -> Tensor:
    """TV ops/boxes.py:344-370 (xyxy only): [N,4] x [M,4] -> [N,M] IoU, fp32 bit-exact."""
    if boxes1.dim() != 2 or boxes2.dim() != 2 or boxes1.shape[-1] != 4 or boxes2.shape[-1] != 4:
        raise ValueError("box_iou expects boxes of shape [N, 4] and [M, 4]")
    return _eager(_box_iou_op)(boxes1, boxes2)


# --------------------------------------------------------------------------------- NMS
@torch.library.custom_op("dgod_b200::nms_batched", mutates_args=())
def _nms_batched_op(boxes: Tensor, scores: Tensor, groups: Optional[Tensor], valid: Optional[Tensor],
                    seg_offsets: Tensor, max_seg_len: int, iou_threshold: float, offset_mode: bool,
                    max_out_per_seg: int) -> Tuple[Tensor, Tensor]:
    _need_cuda(boxes, scores, groups, valid, seg_offsets)
    lib = _lib.load()
    n_total, n_seg = boxes.shape[0], seg_offsets.shape[0] - 1
    dev = boxes.device
    boxes, scores = _f32c(boxes), _f32c(scores)
    if groups is not None:
        groups = groups.to(torch.int64).contiguous()
    if valid is not None:
        valid = valid.to(torch.uint8).contiguous()
    seg_offsets = seg_offsets.to(torch.int32).contiguous()
    out_stride = max_out_per_seg if max_out_per_seg > 0 else max_seg_len
    keep = torch.zeros((n_seg, max(out_stride, 0)), dtype=torch.int64, device=dev)
    info = torch.zeros(n_seg + 1, dtype=torch.int32, device=dev)  # counts..., status
    ws_bytes = lib.dgod_nms_workspace_bytes(n_total, n_seg, max_seg_len)
    ws = _ws(ws_bytes, dev)
    tok = KernelTimer.start("nms_batched", 28 * n_total + 8 * keep.numel())
    check(lib.dgod_nms_batched(_p(boxes), _p(scores), _p(groups), _p(valid), _p(seg_offsets), n_seg,
                               n_total, max_seg_len, float(iou_threshold), int(offset_mode),
                               int(max_out_per_seg), _p(keep), _p(info),
                               C.c_void_p(info.data_ptr() + 4 * n_seg), _p(ws), ws_bytes, _stream()))
    KernelTimer.stop(tok)
    return keep, info


@_nms_batched_op.register_fake
def _(boxes, scores, groups, valid, seg_offsets, max_seg_len, iou_threshold, offset_mode, max_out_per_seg):
    n_seg = seg_offsets.shape[0] - 1
    stride = max_out_per_seg if max_out_per_seg > 0 else max_seg_len
    return (boxes.new_empty((n_seg, stride), dtype=torch.int64),
            boxes.new_empty((n_seg + 1,), dtype=torch.int32))


def nms_segments(boxes: Tensor, scores: Tensor, groups: Optional[Tensor], seg_counts: Sequence[int],
                 iou_threshold: float, *, valid: Optional[Tensor] = None, offset_mode: bool = False,
                 max_out_per_seg: int = 0) -> Tuple[Tensor, Tensor]:
    """NMS of several independent segments (images) in one call, no host synchronisation.
    Returns (keep [n_seg, stride] segment-relative indices, info int32 [n_seg+1] = counts + status)."""
    seg_offsets = _offsets(seg_counts, boxes.device)
    max_len = max([int(c) for c in seg_counts], default=0)
    return _eager(_nms_batched_op)(boxes, scores, groups, valid, seg_offsets, max_len, float(iou_threshold),
                           bool(offset_mode), int(max_out_per_seg))


def nms(boxes: Tensor, scores: Tensor, iou_threshold: float) -> Tensor:
    """TV ops/boxes.py:20-48: indices kept by NMS, descending score (stable), int64."""
    n = boxes.shape[0]
    if n == 0:
        return torch.empty((0,), dtype=torch.int64, device=boxes.device)
    keep, info = nms_segments(boxes, scores, None, [n], iou_threshold)
    cnt = int(info[0].item())
    return keep[0, :cnt]


def batched_nms(boxes: Tensor, scores: Tensor, idxs: Tensor, iou_threshold: float) -> Tensor:
    """TV ops/boxes.py:51-120 with the CPU path's mode rule (coordinate trick up to 1000 boxes,
    per-group NMS above).  Equal scores are ordered by ascending index."""
    n = boxes.shape[0]
    if n == 0:
        return torch.empty((0,), dtype=torch.int64, device=boxes.device)
    trick = boxes.numel() <= BATCHED_NMS_TRICK_MAX_NUMEL
    keep, info = nms_segments(boxes, scores, idxs, [n], iou_threshold, offset_mode=trick)
    cnt, status = info.tolist()
    if status != 0:  # group ids outside [0, 65535]: densify (order of ids is irrelevant per group)
        _, dense = torch.unique(idxs, return_inverse=True)
        keep, info = nms_segments(boxes, scores, dense, [n], iou_threshold, offset_mode=False)
        cnt, status = info.tolist()
        if status != 0:
            raise RuntimeError("batched_nms: more than 65536 distinct groups are not supported")
    return keep[0, :cnt]


# --------------------------------------------------------------------------------- Matcher
def clip_boxes_to_image(boxes: Tensor, size: Tuple[int, int]) -> Tensor:
    """TV ops/boxes.py:149-182 (same signature).  On the training path the clip is fused into
    `rpn_proposals` / `detect_candidates`; this stand-alone form serves FCOS eval post-processing
    (fcos.py:597) and is two clamps on the device."""
    _need_cuda(boxes)
    height, width = size
    x = boxes[..., 0::2].clamp(min=0, max=width)
    y = boxes[..., 1::2].clamp(min=0, max=height)
    return torch.stack((x, y), dim=boxes.dim()).reshape(boxes.shape)


def remove_small_boxes(boxes: Tensor, min_size: float) -> Tensor:
    """TV ops/boxes.py:123-146 (same signature): indices of the boxes with both sides >= min_size."""
    _need_cuda(boxes)
    ws, hs = boxes[:, 2] - boxes[:, 0], boxes[:, 3] - boxes[:, 1]
    return torch.where((ws >= min_size) & (hs >= min_size))[0]


class Matcher:
    """TV models/detection/_utils.py:313-416, same constructor, attributes and errors."""

    BELOW_LOW_THRESHOLD = -1
    BETWEEN_THRESHOLDS = -2

    def __init__(self, high_threshold: float, low_threshold: float, allow_low_quality_matches: bool = False):
        self.BELOW_LOW_THRESHOLD = -1
        self.BETWEEN_THRESHOLDS = -2
        torch._assert(low_threshold <= high_threshold, "low_threshold should be <= high_threshold")
        self.high_threshold = high_threshold
        self.low_threshold = low_threshold
        self.allow_low_quality_matches = allow_low_quality_matches

    def __call__(self, match_quality_matrix: Tensor) -> Tensor:
        if match_quality_matrix.numel() == 0:
            if match_quality_matrix.shape[0] == 0:
                raise ValueError("No ground-truth boxes available for one of the images during training")
            raise ValueError("No proposal boxes available for one of the images during training")
        _need_cuda(match_quality_matrix)
        lib = _lib.load()
        q = _f32c(match_quality_matrix)
        m, n = q.shape
        out = torch.empty(n, dtype=torch.int64, device=q.device)
        wsb = lib.dgod_matcher_workspace_bytes(m)
        ws = _ws(wsb, q.device)
        check(lib.dgod_matcher(_p(q), m, n, float(self.high_threshold), float(self.low_threshold),
                               int(self.allow_low_quality_matches), _p(out), _p(ws), wsb, _stream()),
              ValueError)
        return out


@torch.library.custom_op("dgod_b200::iou_match", mutates_args=())
def _iou_match_op(gt_boxes: Tensor, gt_labels: Optional[Tensor], gt_offsets: Tensor, boxes: Tensor,
                  box_offsets: Optional[Tensor], box_counts: Optional[Tensor], max_boxes_per_img: int, high: float,
                  low: float, allow_low_quality: bool, want: int) -> List[Tensor]:
    """want bitmask: 1 labels_f32, 2 labels_i64, 4 clamped_idx, 8 matched_boxes.
    Returns [matched_idx, labels_f32, labels_i64, clamped_idx, matched_boxes] (empty if not wanted).
    Layouts (include/dgod_b200.h): shared boxes [N,4]; ragged (box_offsets); padded boxes [B,cap,4] + box_counts [B]
    with the ground truths appended, max_boxes_per_img slots per image."""
    _need_cuda(gt_boxes, gt_labels, gt_offsets, boxes, box_offsets, box_counts)
    lib = _lib.load()
    dev = boxes.device
    gt_boxes, boxes = _f32c(gt_boxes), _f32c(boxes)
    n_img = gt_offsets.shape[0] - 1
    total_gt = gt_boxes.shape[0]
    if box_counts is not None:
        box_counts = box_counts.to(torch.int32).contiguous()
        n_boxes = boxes.shape[1]
        shape = (n_img, max_boxes_per_img)
    else:
        n_boxes = boxes.shape[0]
        shape = (n_img, n_boxes) if box_offsets is None else (n_boxes,)
    idx = torch.empty(shape, dtype=torch.int64, device=dev)
    lf = torch.empty(shape if want & 1 else (0,), dtype=torch.float32, device=dev)
    li = torch.empty(shape if want & 2 else (0,), dtype=torch.int64, device=dev)
    ci = torch.empty(shape if want & 4 else (0,), dtype=torch.int64, device=dev)
    mb = torch.empty(shape + (4,) if want & 8 else (0,), dtype=torch.float32, device=dev)
    wsb = lib.dgod_iou_match_workspace_bytes(n_img, total_gt)
    ws = _ws(wsb, dev)
    n_out = idx.numel()
    tok = KernelTimer.start("iou_match", 16 * total_gt + 16 * boxes.numel() // 4 + n_out * (8 + (4 if want & 1 else 0) + (8 if want & 2 else 0)
                                                                                  + (8 if want & 4 else 0) + (16 if want & 8 else 0)))
    check(lib.dgod_iou_match(_p(gt_boxes), _p(gt_labels), _p(gt_offsets), n_img, total_gt, _p(boxes),
                             _p(box_offsets), _p(box_counts), n_boxes, int(max_boxes_per_img), float(high), float(low),
                             int(allow_low_quality), _p(idx), _p(lf) if want & 1 else None,
                             _p(li) if want & 2 else None, _p(ci) if want & 4 else None,
                             _p(mb) if want & 8 else None, _p(ws), wsb, _stream()))
    KernelTimer.stop(tok)
    return [idx, lf, li, ci, mb]


@_iou_match_op.register_fake
def _(gt_boxes, gt_labels, gt_offsets, boxes, box_offsets, box_counts, max_boxes_per_img, high, low, allow_low_quality,
      want):
    n_img = gt_offsets.shape[0] - 1
    if box_counts is not None:
        shape = (n_img, max_boxes_per_img)
    else:
        shape = (n_img, boxes.shape[0]) if box_offsets is None else (boxes.shape[0],)
    e = lambda cond, s, dt: boxes.new_empty(s if cond else (0,), dtype=dt)
    return [boxes.new_empty(shape, dtype=torch.int64), e(want & 1, shape, torch.float32),
            e(want & 2, shape, torch.int64), e(want & 4, shape, torch.int64),
            e(want & 8, shape + (4,), torch.float32)]


def _gt_batch(gt_boxes: Sequence[Tensor], dev) -> Tuple[Tensor, Tensor]:
    """Ground truths of a batch concatenated [sum M_i, 4] fp32 + int32 offsets [B+1] (from the shapes)."""
    gt_cat = torch.cat([g.reshape(-1, 4).float() for g in gt_boxes]) if len(gt_boxes) else torch.zeros((0, 4), device=dev)
    return gt_cat, _offsets([g.shape[0] for g in gt_boxes], dev)


def match_boxes(gt_boxes: Sequence[Tensor], boxes, high_threshold: float, low_threshold: float,
                allow_low_quality_matches: bool, gt_labels: Optional[Sequence[Tensor]] = None,
                want=("labels_f32",)):
    """Fused box_iou + Matcher (+ label / matched-box gather) for a batch of images.

    gt_boxes: list of [M_i,4].  boxes is one of
      * one Tensor [N,4] shared by all images (RPN anchors): results are [B,N];
      * a list of [N_i,4] (proposals): results are concatenated [sum N_i];
      * a pair (padded [B,cap,4], device counts [B]) (RPN output): image i's candidates are its first counts[i] boxes
        followed by its ground truths (add_gt_proposals without the copy) and results are [B, cap + max M_i], -1 labels in
        the slots past count_i + M_i.  Nothing is read back to the host.
    Returns a dict with 'matched_idx' plus the requested 'labels_f32' (TV rpn.py:216-225),
    'labels_i64' / 'clamped_idx' (TV roi_heads.py:597-609), 'matched_boxes'."""
    dev = gt_boxes[0].device if len(gt_boxes) else boxes.device
    gt_cat, gt_off = _gt_batch(gt_boxes, dev)
    gl_cat = None
    if gt_labels is not None:
        gl_cat = torch.cat([l.reshape(-1).to(torch.int64) for l in gt_labels]).contiguous()
    box_off = box_counts = None
    if isinstance(boxes, Tensor):
        bx, max_n = boxes, boxes.shape[0]
    elif isinstance(boxes, tuple):
        bx, box_counts = boxes
        max_n = bx.shape[1] + max([g.shape[0] for g in gt_boxes], default=0)
    else:
        bx = torch.cat(list(boxes))
        box_off = _offsets([b.shape[0] for b in boxes], dev)
        max_n = max([b.shape[0] for b in boxes], default=0)
    bits = {"labels_f32": 1, "labels_i64": 2, "clamped_idx": 4, "matched_boxes": 8}
    mask = 0
    for w in want:
        mask |= bits[w]
    idx, lf, li, ci, mb = _eager(_iou_match_op)(gt_cat, gl_cat, gt_off, bx, box_off, box_counts, max_n,
                                                float(high_threshold), float(low_threshold),
                                                bool(allow_low_quality_matches), mask)
    out = {"matched_idx": idx}
    for name, t in (("labels_f32", lf), ("labels_i64", li), ("clamped_idx", ci), ("matched_boxes", mb)):
        if name in want:
            out[name] = t
    return out


# --------------------------------------------------------------------------------- input side
def resized_shape(h: int, w: int, min_size: int, max_size: int) -> Tuple[int, int]:
    """Output size of TV transform.py:25-83 in eager mode: floor(in * min(min_size/min(h,w), max_size/max(h,w)))
    (double arithmetic, as `interpolate(scale_factor=..., recompute_scale_factor=True)` computes it)."""
    sf = min(float(min_size) / float(min(h, w)), float(max_size) / float(max(h, w)))
    return int(math.floor(float(h) * sf)), int(math.floor(float(w) * sf))


def image_batch(images: Sequence[Tensor], image_mean: Sequence[float], image_std: Sequence[float], min_size: int,
                max_size: int, size_divisible: int = 32):
    """GeneralizedRCNNTransform.forward for the images of a batch (TV transform.py:102-153: normalize,
    resize, batch_images) in one launch.  images: CUDA fp32 [C,H,W] tensors (sizes may differ) — or uint8 tensors with
    values 0..255, in which case the dataset's `image / 255.0` (DrivingDataset.py:53) happens on load inside the kernel
    (bit-identical, a quarter of the host->device bytes).  Returns (batched [B,C,H_pad,W_pad] NCHW tensor,
    [(h_i, w_i)] resized sizes) — what `ImageList` holds."""
    _need_cuda(*images)
    lib = _lib.load()
    n = len(images)
    if n == 0:
        raise RuntimeError("image_batch: empty batch")
    imgs = []
    u8 = images[0].dtype == torch.uint8
    for im in images:
        if im.dim() != 3 or im.dtype != (torch.uint8 if u8 else torch.float32):
            raise RuntimeError("image_batch: images are expected to be [C, H, W] tensors, all float32 or all uint8, got "
                               f"{tuple(im.shape)} {im.dtype}")
        imgs.append(im.contiguous())
    Cn = imgs[0].shape[0]
    if Cn > 4 or Cn != len(image_mean) or Cn != len(image_std):
        raise RuntimeError("image_batch: 1-4 channels with one mean / std each expected")
    in_h, in_w = [int(i.shape[1]) for i in imgs], [int(i.shape[2]) for i in imgs]
    sizes = [resized_shape(h, w, min_size, max_size) for h, w in zip(in_h, in_w)]
    stride = float(size_divisible)
    pad_h = int(math.ceil(max(s[0] for s in sizes) / stride) * stride)      # transform.py:242-247
    pad_w = int(math.ceil(max(s[1] for s in sizes) / stride) * stride)
    out = torch.empty((n, Cn, pad_h, pad_w), dtype=torch.float32, device=imgs[0].device)
    ptrs = (C.c_void_p * n)(*[i.data_ptr() for i in imgs])
    ia = lambda v: (C.c_int * n)(*v)
    fa = lambda v: (C.c_float * Cn)(*[float(x) for x in v])
    tok = KernelTimer.start("image_batch", sum(Cn * h * w * (1 if u8 else 4) for h, w in zip(in_h, in_w)) + out.numel() * 4)
    check((lib.dgod_image_batch_u8 if u8 else lib.dgod_image_batch)(ptrs, ia(in_h), ia(in_w), ia([s[0] for s in sizes]), ia([s[1] for s in sizes]), n, Cn,
                               fa(image_mean), fa(image_std), _p(out), pad_h, pad_w, _stream()))
    KernelTimer.stop(tok)
    return out, sizes


# --------------------------------------------------------------------------------- FCOS
@torch.library.custom_op("dgod_b200::fcos_assign", mutates_args=())
def _fcos_assign_op(anchors: Tensor, n_first: int, n_last: int, radius: float, gt_boxes: Tensor,
                    gt_labels: Optional[Tensor], gt_offsets: Tensor, num_classes: int,
                    want_targets: bool) -> List[Tensor]:
    _need_cuda(anchors, gt_boxes, gt_labels, gt_offsets)
    lib = _lib.load()
    dev = anchors.device
    anchors, gt_boxes = _f32c(anchors), _f32c(gt_boxes)
    n, n_img = anchors.shape[0], gt_offsets.shape[0] - 1
    idx = torch.empty((n_img, n), dtype=torch.int64, device=dev)
    if want_targets:
        cls = torch.empty((n_img, n), dtype=torch.int64, device=dev)
        bt = torch.empty((n_img, n, 4), dtype=torch.float32, device=dev)
        oh = torch.empty((n_img, n, num_classes), dtype=torch.float32, device=dev)
    else:
        cls = torch.empty((0,), dtype=torch.int64, device=dev)
        bt = torch.empty((0,), dtype=torch.float32, device=dev)
        oh = torch.empty((0,), dtype=torch.float32, device=dev)
    tok = KernelTimer.start("fcos_assign", 16 * n + 16 * gt_boxes.shape[0]
                            + n_img * n * (8 + ((8 + 16 + 4 * num_classes) if want_targets else 0)))
    check(lib.dgod_fcos_assign(_p(anchors), n, int(n_first), int(n_last), float(radius), _p(gt_boxes),
                               _p(gt_labels), _p(gt_offsets), n_img, _p(idx),
                               _p(cls) if want_targets else None, _p(bt) if want_targets else None,
                               _p(oh) if want_targets else None, int(num_classes), _stream()))
    KernelTimer.stop(tok)
    return [idx, cls, bt, oh]


@_fcos_assign_op.register_fake
def _(anchors, n_first, n_last, radius, gt_boxes, gt_labels, gt_offsets, num_classes, want_targets):
    n, n_img = anchors.shape[0], gt_offsets.shape[0] - 1
    if want_targets:
        return [anchors.new_empty((n_img, n), dtype=torch.int64), anchors.new_empty((n_img, n), dtype=torch.int64),
                anchors.new_empty((n_img, n, 4), dtype=torch.float32),
                anchors.new_empty((n_img, n, num_classes), dtype=torch.float32)]
    return [anchors.new_empty((n_img, n), dtype=torch.int64), anchors.new_empty((0,), dtype=torch.int64),
            anchors.new_empty((0,), dtype=torch.float32), anchors.new_empty((0,), dtype=torch.float32)]


def fcos_assign(anchors: Tensor, gt_boxes: Sequence[Tensor], num_anchors_per_level: Sequence[int],
                center_sampling_radius: float = 1.5, gt_labels: Optional[Sequence[Tensor]] = None,
                num_classes: int = 0):
    """fcos.py:510-548 for a batch: matched_idx [B,N] int64 (-1 = unmatched).  With gt_labels and
    num_classes also the targets of fcos.py:136-158: (cls_targets [B,N], box_targets [B,N,4],
    gt_classes one-hot [B,N,C])."""
    dev = anchors.device
    gt_cat = torch.cat([g.reshape(-1, 4).float() for g in gt_boxes]) if len(gt_boxes) else torch.zeros((0, 4), device=dev)
    gt_off = _offsets([g.shape[0] for g in gt_boxes], dev)
    want = gt_labels is not None and num_classes > 0
    gl_cat = torch.cat([l.reshape(-1).to(torch.int64) for l in gt_labels]).contiguous() if want else None
    idx, cls, bt, oh = _eager(_fcos_assign_op)(anchors, int(num_anchors_per_level[0]), int(num_anchors_per_level[-1]),
                                       float(center_sampling_radius), gt_cat, gl_cat, gt_off, int(num_classes), want)
    if want:
        return idx, cls, bt, oh
    return idx


@torch.library.custom_op("dgod_b200::fcos_loss", mutates_args=())
def _fcos_loss_op(cls_logits: Tensor, bbox_regression: Tensor, bbox_ctrness: Tensor, anchors: Tensor,
                  cls_targets: Tensor, box_targets: Tensor, alpha: float) -> Tensor:
    _need_cuda(cls_logits, bbox_regression, bbox_ctrness, anchors, cls_targets, box_targets)
    lib = _lib.load()
    B, N, Cn = cls_logits.shape
    out = torch.empty(4, dtype=torch.float32, device=cls_logits.device)
    wsb = lib.dgod_fcos_loss_workspace_bytes(B * N)
    ws = _ws(wsb, cls_logits.device)
    tok = KernelTimer.start("fcos_loss_fwd", B * N * (4 * (Cn + 5) + 8 + 16) + 16 * N)
    check(lib.dgod_fcos_loss_fwd(_p(cls_logits), _p(bbox_regression), _p(bbox_ctrness), _p(anchors), _p(cls_targets),
                                 _p(box_targets), B, N, Cn, float(alpha), _p(out), _p(ws), wsb, _stream()))
    KernelTimer.stop(tok)
    return out


@_fcos_loss_op.register_fake
def _(cls_logits, bbox_regression, bbox_ctrness, anchors, cls_targets, box_targets, alpha):
    return cls_logits.new_empty((4,), dtype=torch.float32)


@torch.library.custom_op("dgod_b200::fcos_loss_backward", mutates_args=())
def _fcos_loss_bwd_op(cls_logits: Tensor, bbox_regression: Tensor, bbox_ctrness: Tensor, anchors: Tensor,
                      cls_targets: Tensor, box_targets: Tensor, alpha: float, losses: Tensor,
                      grad_losses: Tensor) -> List[Tensor]:
    _need_cuda(cls_logits, losses, grad_losses)
    lib = _lib.load()
    B, N, Cn = cls_logits.shape
    g_cls, g_reg, g_ctr = torch.empty_like(cls_logits), torch.empty_like(bbox_regression), torch.empty_like(bbox_ctrness)
    tok = KernelTimer.start("fcos_loss_bwd", 2 * B * N * 4 * (Cn + 5) + B * N * (8 + 16) + 16 * N)
    check(lib.dgod_fcos_loss_bwd(_p(cls_logits), _p(bbox_regression), _p(bbox_ctrness), _p(anchors), _p(cls_targets),
                                 _p(box_targets), B, N, Cn, float(alpha), _p(losses), _p(grad_losses), _p(g_cls),
                                 _p(g_reg), _p(g_ctr), _stream()))
    KernelTimer.stop(tok)
    return [g_cls, g_reg, g_ctr]


@_fcos_loss_bwd_op.register_fake
def _(cls_logits, bbox_regression, bbox_ctrness, anchors, cls_targets, box_targets, alpha, losses, grad_losses):
    return [torch.empty_like(cls_logits), torch.empty_like(bbox_regression), torch.empty_like(bbox_ctrness)]


def _fcos_loss_setup(ctx, inputs, output):
    ctx.save_for_backward(*inputs[:6], output)
    ctx.alpha = inputs[6]


def _fcos_loss_backward(ctx, grad):
    cls_logits, reg, ctr, anchors, ct, bt, losses = ctx.saved_tensors
    g = _fcos_loss_bwd_op(cls_logits, reg, ctr, anchors, ct, bt, ctx.alpha, losses, grad[:3].contiguous().float())
    return g[0], g[1], g[2], None, None, None, None


_fcos_loss_op.register_autograd(_fcos_loss_backward, setup_context=_fcos_loss_setup)


class _FcosLossFn(torch.autograd.Function):
    """Eager path of dgod_b200::fcos_loss (same kernels, no dispatcher round trip)."""

    @staticmethod
    def forward(ctx, cls_logits, reg, ctr, anchors, ct, bt, alpha):
        out = _fcos_loss_op._init_fn(cls_logits, reg, ctr, anchors, ct, bt, alpha)
        ctx.save_for_backward(cls_logits, reg, ctr, anchors, ct, bt, out)
        ctx.alpha = alpha
        ctx.mark_non_differentiable()
        return out

    @staticmethod
    def backward(ctx, grad):
        cls_logits, reg, ctr, anchors, ct, bt, losses = ctx.saved_tensors
        g = _fcos_loss_bwd_op._init_fn(cls_logits, reg, ctr, anchors, ct, bt, ctx.alpha, losses, grad[:3].contiguous().float())
        return g[0], g[1], g[2], None, None, None, None


def fcos_loss(cls_logits: Tensor, bbox_regression: Tensor, bbox_ctrness: Tensor, anchors: Tensor,
              cls_targets: Tensor, box_targets: Tensor, alpha: float = 0.25) -> Tensor:
    """fcos.py:149-202 fused: returns a device tensor [4] = classification, bbox_regression, bbox_ctrness
    (each already divided by max(1, #foreground)) and #foreground — differentiable w.r.t. the three head
    outputs, no host sync.  cls_logits [B,N,C], bbox_regression [B,N,4], bbox_ctrness [B,N,1] fp32;
    anchors [N,4]; cls_targets [B,N] int64 (-1 = background) and box_targets [B,N,4] from `fcos_assign`."""
    for t in (cls_logits, bbox_regression, bbox_ctrness):
        if t.dtype not in (torch.float32, torch.bfloat16):
            raise RuntimeError(f"fcos_loss: float32 or bfloat16 head outputs expected, got {t.dtype}")
    # bf16 head outputs (autocast) go through the fp32 loss kernels, as autocast runs the stock losses in fp32
    cls_logits, bbox_regression, bbox_ctrness = cls_logits.float(), bbox_regression.float(), bbox_ctrness.float()
    B, N, _ = cls_logits.shape
    if bbox_regression.shape != (B, N, 4) or bbox_ctrness.numel() != B * N or cls_targets.shape != (B, N):
        raise RuntimeError("fcos_loss: expected cls_logits [B,N,C], bbox_regression [B,N,4], bbox_ctrness [B,N,1], "
                           "cls_targets [B,N]")
    args = (cls_logits.contiguous(), bbox_regression.contiguous(), bbox_ctrness.contiguous(), _f32c(anchors),
            cls_targets.contiguous(), _f32c(box_targets), float(alpha))
    if torch.compiler.is_compiling():
        return _fcos_loss_op(*args)
    return _FcosLossFn.apply(*args)


def fcos_candidates(cls_logits: Tensor, bbox_regression: Tensor, bbox_ctrness: Tensor, anchors: Tensor,
                    num_anchors_per_level: Sequence[int], image_sizes: Tensor, score_thresh: float = 0.2,
                    topk: int = 1000):
    """fcos.py:576-597 (FCOS.postprocess_detections up to the NMS) for the batch in one launch: cls_logits [B,N,C],
    bbox_regression [B,N,4], bbox_ctrness [B,N,1] over all levels, anchors [N,4], image_sizes float [B,2] = (h, w) on the
    device -> (boxes [B, L*topk, 4], scores [B, L*topk], labels int64 [B, L*topk], valid uint8 [B, L*topk],
    counts int32 [B, L]); level l's survivors start at l*topk, in descending score.  No host synchronisation."""
    _need_cuda(cls_logits, bbox_regression, bbox_ctrness, anchors, image_sizes)
    lib = _lib.load()
    cl, rg, ct, an = _f32c(cls_logits), _f32c(bbox_regression), _f32c(bbox_ctrness), _f32c(anchors)
    B, N, Cn = cl.shape
    if rg.shape != (B, N, 4) or ct.numel() != B * N or an.shape != (N, 4) or sum(num_anchors_per_level) != N:
        raise RuntimeError("fcos_candidates: expected cls_logits [B,N,C], bbox_regression [B,N,4], bbox_ctrness [B,N,1], "
                           "anchors [N,4] and num_anchors_per_level summing to N")
    if not 1 <= int(topk) <= 1024:
        raise RuntimeError("fcos_candidates: topk must be in 1..1024")
    L, dev = len(num_anchors_per_level), cl.device
    off = _offsets(num_anchors_per_level, dev)
    boxes = torch.empty((B, L * topk, 4), dtype=torch.float32, device=dev)
    scores = torch.empty((B, L * topk), dtype=torch.float32, device=dev)
    labels = torch.empty((B, L * topk), dtype=torch.int64, device=dev)
    valid = torch.empty((B, L * topk), dtype=torch.uint8, device=dev)
    counts = torch.empty((B, L), dtype=torch.int32, device=dev)
    tok = KernelTimer.start("fcos_candidates", B * N * (4 * Cn + 4) + B * L * topk * (16 + 16 + 16 + 4 + 8 + 1))
    check(lib.dgod_fcos_candidates(_p(cl), _p(rg), _p(ct), _p(an), N, Cn, _p(off), L, B, _p(_f32c(image_sizes)),
                                   float(score_thresh), int(topk), _p(boxes), _p(scores), _p(labels), _p(valid), _p(counts),
                                   _stream()))
    KernelTimer.stop(tok)
    return boxes, scores, labels, valid, counts


# --------------------------------------------------------------------------------- RoIAlign
def _roi_config(feats: Sequence[Tensor], scales: Sequence[float], ph: int, pw: int, sr: int, aligned: bool,
                k_min: int, k_max: int, s0: float, lvl0: float, eps: float = 1e-6):
    f0 = feats[0]
    if f0.dtype not in (torch.float32, torch.bfloat16):
        raise RuntimeError(f"roi_align: unsupported dtype {f0.dtype} (float32 and bfloat16 only)")
    nhwc = f0.dim() == 4 and not f0.is_contiguous() and f0.is_contiguous(memory_format=torch.channels_last)
    cfg = RoiConfig()
    cfg.n_levels = len(feats)
    cfg.batch, cfg.channels = f0.shape[0], f0.shape[1]
    for l, f in enumerate(feats):
        cfg.height[l], cfg.width[l] = f.shape[2], f.shape[3]
        cfg.spatial_scale[l] = float(scales[l])
    cfg.channels_last = int(nhwc)
    cfg.dtype = _lib.F32 if f0.dtype == torch.float32 else _lib.BF16
    cfg.pooled_h, cfg.pooled_w, cfg.sampling_ratio, cfg.aligned = int(ph), int(pw), int(sr), int(bool(aligned))
    cfg.k_min, cfg.k_max = int(k_min), int(k_max)
    cfg.canonical_scale, cfg.canonical_level, cfg.eps = float(s0), float(lvl0), float(eps)
    return cfg, nhwc


def _level_ptrs(ts: Sequence[Tensor]):
    arr = (C.c_void_p * len(ts))(*[t.data_ptr() for t in ts])
    return C.cast(arr, C.POINTER(C.c_void_p)), arr


def _roi_bytes(feats_numel: Sequence[int], esz: int, n_rois: int, c: int, ph: int, pw: int, sr: int) -> int:
    """Algorithmic bytes of one MSRoIAlign pass (SURVEY.md §8d)."""
    g = sr if sr > 0 else 2
    return n_rois * c * ph * pw * esz + 20 * n_rois + min(sum(feats_numel) * esz, n_rois * c * ph * g * pw * g * 4 * esz)


def _tma_shape(c: int, ph: int, pw: int, sr: int) -> bool:
    """Shapes the TMA RoIAlign kernels are instantiated for (csrc/roi_align_tma.cu)."""
    return ph == 7 and pw == 7 and (c == 256 and sr in (1, 2) or c in (64, 128) and sr == 2)


def to_channels_last(x: Tensor) -> Tensor:
    """NCHW-contiguous [B,C,H,W] -> the same tensor in channels_last memory (dgod_nchw_to_nhwc)."""
    _need_cuda(x)
    if x.dim() != 4 or not x.is_contiguous() or x.dtype not in (torch.float32, torch.bfloat16):
        return x.contiguous(memory_format=torch.channels_last)
    out = torch.empty_like(x, memory_format=torch.channels_last)
    b, c, h, w = x.shape
    tok = KernelTimer.start("nchw_to_nhwc", 2 * x.numel() * x.element_size())
    check(_lib.load().dgod_nchw_to_nhwc(_p(x), _p(out), b, c, h * w, _lib.F32 if x.dtype == torch.float32 else _lib.BF16,
                                        _stream()))
    KernelTimer.stop(tok)
    return out


@torch.library.custom_op("dgod_b200::msroi_align", mutates_args=())
def _msroi_fwd_op(feats: List[Tensor], rois: Tensor, roi_img_offsets: Optional[Tensor], scales: List[float],
                  pooled_h: int, pooled_w: int, sampling_ratio: int, aligned: bool, k_min: int, k_max: int,
                  canonical_scale: float, canonical_level: float) -> Tensor:
    _need_cuda(rois, *feats)
    lib = _lib.load()
    f0 = feats[0]
    if (f0.dim() == 4 and f0.is_contiguous() and f0.shape[2] * f0.shape[3] > 1 and not aligned and rois.shape[0] > 0
            and _tma_shape(f0.shape[1], pooled_h, pooled_w, sampling_ratio)):
        # NCHW maps: one transposing pass, then the channels_last TMA kernel (faster than the generic
        # NCHW kernel even with the extra pass)
        feats = [to_channels_last(f) if f.is_contiguous() else f for f in feats]
        f0 = feats[0]
    cfg, nhwc = _roi_config(feats, scales, pooled_h, pooled_w, sampling_ratio, aligned, k_min, k_max,
                            canonical_scale, canonical_level)
    fs = [f if (f.is_contiguous(memory_format=torch.channels_last) if nhwc else f.is_contiguous())
          else f.contiguous(memory_format=torch.channels_last if nhwc else torch.contiguous_format) for f in feats]
    for f in fs:
        if f.dtype != f0.dtype or f.shape[0] != f0.shape[0] or f.shape[1] != f0.shape[1]:
            raise RuntimeError("multiscale roi_align: all levels must share dtype, batch and channels")
    rois = _f32c(rois)
    n = rois.shape[0]
    out = torch.empty((n, f0.shape[1], pooled_h, pooled_w), dtype=f0.dtype, device=f0.device)
    ptrs, keep_alive = _level_ptrs(fs)
    tok = KernelTimer.start("msroi_align_fwd", _roi_bytes([f.numel() for f in fs], f0.element_size(), n,
                                                          f0.shape[1], pooled_h, pooled_w, sampling_ratio))
    wsb = lib.dgod_msroi_align_fwd_workspace_bytes(n)
    ws = _ws(wsb, f0.device)
    check(lib.dgod_msroi_align_fwd(C.byref(cfg), ptrs, _p(rois), n, _p(out), _p(ws), wsb, _stream()))
    KernelTimer.stop(tok)
    return out


@_msroi_fwd_op.register_fake
def _(feats, rois, roi_img_offsets, scales, pooled_h, pooled_w, sampling_ratio, aligned, k_min, k_max,
      canonical_scale, canonical_level):
    return feats[0].new_empty((rois.shape[0], feats[0].shape[1], pooled_h, pooled_w))


@torch.library.custom_op("dgod_b200::msroi_align_backward", mutates_args=())
def _msroi_bwd_op(grad: Tensor, rois: Tensor, roi_img_offsets: Optional[Tensor], shapes: List[int],
                  channels_last: bool, scales: List[float], pooled_h: int, pooled_w: int, sampling_ratio: int,
                  aligned: bool, k_min: int, k_max: int, canonical_scale: float, canonical_level: float,
                  algo: int) -> List[Tensor]:
    _need_cuda(grad, rois, roi_img_offsets)
    lib = _lib.load()
    n_levels = len(scales)
    b, c = shapes[0], shapes[1]
    if not channels_last and not aligned and algo in (0, 3, 4, 5) and _tma_shape(c, pooled_h, pooled_w, sampling_ratio):
        channels_last = True     # gradients of NCHW maps are returned in channels_last memory (same values)
    mf = torch.channels_last if channels_last else torch.contiguous_format
    grads = [torch.empty((b, c, shapes[2 + 2 * l], shapes[3 + 2 * l]), dtype=grad.dtype, device=grad.device,
                         memory_format=mf) for l in range(n_levels)]
    cfg, _ = _roi_config(grads, scales, pooled_h, pooled_w, sampling_ratio, aligned, k_min, k_max,
                         canonical_scale, canonical_level)
    cfg.channels_last = int(channels_last)
    grad = grad.contiguous()
    rois = _f32c(rois)
    n = rois.shape[0]
    ptrs, keep_alive = _level_ptrs(grads)
    esz = grad.element_size()
    tok = KernelTimer.start("msroi_align_bwd", n * c * pooled_h * pooled_w * esz + 20 * n + sum(g.numel() for g in grads) * esz)
    wsb = lib.dgod_msroi_align_bwd_workspace_bytes_cfg(C.byref(cfg), n)
    ws = _ws(wsb, grad.device)
    check(lib.dgod_msroi_align_bwd(C.byref(cfg), _p(grad), _p(rois), n, _p(roi_img_offsets), ptrs, int(algo),
                                   _p(ws), wsb, _stream()))
    KernelTimer.stop(tok)
    return grads


@_msroi_bwd_op.register_fake
def _(grad, rois, roi_img_offsets, shapes, channels_last, scales, pooled_h, pooled_w, sampling_ratio, aligned,
      k_min, k_max, canonical_scale, canonical_level, algo):
    b, c = shapes[0], shapes[1]
    return [grad.new_empty((b, c, shapes[2 + 2 * l], shapes[3 + 2 * l])) for l in range(len(scales))]


import os as _os

# 0 auto (= 4 where the shape allows), 1 atomic / vector-RED scatter, 2 tile gather, 3 bulk-reduce scatter, 4 owner-computes with
# a static deal of the work items, 5 owner-computes with claimed work items: what ddp.GradSync selects when gradients are
# all-reduced during backward (NCCL kernels then hold SMs when the persistent backward kernel starts)
BACKWARD_ALGO = int(_os.environ.get("DGOD_BWD_ALGO", "0"))


def _msroi_setup(ctx, inputs, output):
    feats, rois, roi_img_offsets, scales, ph, pw, sr, aligned, k_min, k_max, s0, lvl0 = inputs
    f0 = feats[0]
    ctx.save_for_backward(rois)
    ctx.roi_img_offsets = roi_img_offsets
    ctx.meta = ([f0.shape[0], f0.shape[1]] + [d for f in feats for d in (f.shape[2], f.shape[3])],
                (not f0.is_contiguous()) and f0.is_contiguous(memory_format=torch.channels_last),
                list(scales), ph, pw, sr, aligned, k_min, k_max, s0, lvl0)


def _msroi_backward(ctx, grad):
    (rois,) = ctx.saved_tensors
    shapes, nhwc, scales, ph, pw, sr, aligned, k_min, k_max, s0, lvl0 = ctx.meta
    grads = _msroi_bwd_op(grad, rois, ctx.roi_img_offsets, shapes, nhwc, scales, ph, pw, sr, aligned, k_min,
                          k_max, s0, lvl0, BACKWARD_ALGO)
    return (grads,) + (None,) * 11


_msroi_fwd_op.register_autograd(_msroi_backward, setup_context=_msroi_setup)


class _MsroiAlignFn(torch.autograd.Function):
    """Eager path of dgod_b200::msroi_align (same kernels, no dispatcher round trip)."""

    @staticmethod
    def forward(ctx, rois, roi_img_offsets, scales, ph, pw, sr, aligned, k_min, k_max, s0, lvl0, *feats):
        out = _msroi_fwd_op._init_fn(list(feats), rois, roi_img_offsets, scales, ph, pw, sr, aligned, k_min, k_max, s0, lvl0)
        f0 = feats[0]
        ctx.save_for_backward(rois)
        ctx.roi_img_offsets = roi_img_offsets
        ctx.meta = ([f0.shape[0], f0.shape[1]] + [d for f in feats for d in (f.shape[2], f.shape[3])],
                    (not f0.is_contiguous()) and f0.is_contiguous(memory_format=torch.channels_last),
                    list(scales), ph, pw, sr, aligned, k_min, k_max, s0, lvl0)
        return out

    @staticmethod
    def backward(ctx, grad):
        (rois,) = ctx.saved_tensors
        shapes, nhwc, scales, ph, pw, sr, aligned, k_min, k_max, s0, lvl0 = ctx.meta
        grads = _msroi_bwd_op._init_fn(grad, rois, ctx.roi_img_offsets, shapes, nhwc, scales, ph, pw, sr, aligned, k_min,
                                       k_max, s0, lvl0, BACKWARD_ALGO)
        return (None,) * 11 + tuple(grads)


def multiscale_roi_align(feats: Sequence[Tensor], rois: Tensor, scales: Sequence[float], output_size,
                         sampling_ratio: int, k_min: int, k_max: int, canonical_scale: float = 224.0,
                         canonical_level: float = 4.0, aligned: bool = False,
                         roi_img_offsets: Optional[Tensor] = None) -> Tensor:
    """One-launch replacement of TV ops/poolers.py:147-227: `rois` is [K,5] (batch idx, xyxy)."""
    ph, pw = (output_size, output_size) if isinstance(output_size, int) else (int(output_size[0]), int(output_size[1]))
    if torch.compiler.is_compiling():
        return _msroi_fwd_op(list(feats), rois, roi_img_offsets, [float(s) for s in scales], ph, pw, int(sampling_ratio),
                             bool(aligned), int(k_min), int(k_max), float(canonical_scale), float(canonical_level))
    return _MsroiAlignFn.apply(rois, roi_img_offsets, [float(s) for s in scales], ph, pw, int(sampling_ratio), bool(aligned),
                               int(k_min), int(k_max), float(canonical_scale), float(canonical_level), *feats)


def _convert_to_roi_format(boxes: Sequence[Tensor]) -> Tensor:
    """TV ops/poolers.py:87-95."""
    cat = torch.cat(list(boxes), dim=0)
    ids = torch.cat([torch.full_like(b[:, :1], i) for i, b in enumerate(boxes)], dim=0)
    return torch.cat([ids, cat], dim=1)


def roi_align(input: Tensor, boxes, output_size, spatial_scale: float = 1.0, sampling_ratio: int = -1,
              aligned: bool = False) -> Tensor:
    """TV ops/roi_align.py:204-260 (same argument checks and meaning)."""
    if not isinstance(boxes, Tensor):
        if not all(b.dim() == 2 and b.shape[1] == 4 for b in boxes):
            raise AssertionError("The boxes should be a list of Tensor[L, 4]")
        boxes = _convert_to_roi_format(boxes)
    elif boxes.dim() != 2 or boxes.shape[1] != 5:
        raise RuntimeError("rois must have shape as Tensor[K, 5]")
    if boxes.dtype != input.dtype and input.dtype == torch.float32:
        raise RuntimeError("Expected tensor for argument #1 'input' to have the same type as tensor for argument #2 'rois'")
    return multiscale_roi_align([input], boxes, [spatial_scale], output_size, sampling_ratio, 0, 0, aligned=aligned)


# --------------------------------------------------------------------------------- GRL
@torch.library.custom_op("dgod_b200::grl_scale", mutates_args=())
def _grl_scale_op(grad: Tensor, alpha: float) -> Tensor:
    _need_cuda(grad)
    if grad.dtype not in (torch.float32, torch.bfloat16):
        raise RuntimeError(f"grad_reverse: unsupported dtype {grad.dtype}")
    g = grad.contiguous()
    out = torch.empty_like(g)
    tok = KernelTimer.start("grl_scale", 2 * g.numel() * g.element_size())
    check(_lib.load().dgod_grl_scale(_p(g), _p(out), g.numel(), float(alpha),
                                     _lib.F32 if g.dtype == torch.float32 else _lib.BF16, _stream()))
    KernelTimer.stop(tok)
    return out


@_grl_scale_op.register_fake
def _(grad, alpha):
    return torch.empty_like(grad)


class _GRLayer(torch.autograd.Function):
    """DGcommon.py:33-45: identity forward, grad.neg() * 0.1 backward."""

    @staticmethod
    def forward(ctx, x, alpha):
        ctx.alpha = alpha
        return x.view_as(x)

    @staticmethod
    def backward(ctx, grad_output):
        return _eager(_grl_scale_op)(grad_output, ctx.alpha), None


def grad_reverse(x: Tensor, alpha: float = 0.1) -> Tensor:
    return _GRLayer.apply(x, alpha)


class _GRLLinear(torch.autograd.Function):
    """grad_reverse followed by nn.Linear with the reversal scale folded into the input-gradient
    GEMM's alpha (DGcommon.py:40-42 + DGFRCNN.py:19-20): dX = (-alpha) * (dY @ W) in one kernel,
    no separate pass over the [B*512, 1024] gradient."""

    @staticmethod
    def forward(ctx, x, weight, bias, alpha):
        ctx.save_for_backward(x, weight)
        ctx.alpha = alpha
        ctx.has_bias = bias is not None
        return torch.nn.functional.linear(x, weight, bias)

    @staticmethod
    def backward(ctx, gy):
        x, w = ctx.saved_tensors
        # Under autocast the forward ran in gy's dtype: the GEMMs take the operands autocast gave F.linear.
        x, w = x.to(gy.dtype), w.to(gy.dtype)
        gx = gw = gb = None
        gy2 = gy.reshape(-1, gy.shape[-1])
        if ctx.needs_input_grad[0]:
            # beta=0 ignores `input`; alpha is applied to the fp32 accumulator inside the GEMM
            gx = torch.addmm(gy2.new_empty((1, 1)).expand(gy2.shape[0], w.shape[1]), gy2, w,
                             beta=0, alpha=-ctx.alpha).reshape(x.shape)
        if ctx.needs_input_grad[1]:
            gw = gy2.t().mm(x.reshape(-1, x.shape[-1]))
        if ctx.has_bias and ctx.needs_input_grad[2]:
            gb = gy2.sum(0)
        return gx, gw, gb, None


def grl_linear(x: Tensor, weight: Tensor, bias: Optional[Tensor], alpha: float = 0.1) -> Tensor:
    return _GRLLinear.apply(x, weight, bias, alpha)


# --------------------------------------------------------------------------------- box head MLP (fc6 / fc7)
def linear_tc(a: Tensor, b: Tensor, *, a_trans: bool = False, b_trans: bool = False, bias: Optional[Tensor] = None,
              relu: bool = False, mask: Optional[Tensor] = None, name: str = "linear_tc") -> Tensor:
    """fp32 C = A @ B^T on the tensor cores, fp32-accurate (dgod_linear_tc, 3xTF32).  A is `a` [m, k] (or `a`^T when
    a_trans: `a` is [k, m]), B is `b` [n, k] (or `b`^T: [k, n]).  Then + bias, ReLU, * (mask > 0), in that order."""
    _need_cuda(a, b, bias, mask)
    for t in (a, b, bias, mask):
        if t is not None and (t.dtype != torch.float32 or not t.is_contiguous()):
            raise ValueError("linear_tc: operands must be contiguous float32")
    if a.dim() != 2 or b.dim() != 2:
        raise ValueError("linear_tc: a and b must be 2-D")
    m, k = (a.shape[1], a.shape[0]) if a_trans else a.shape
    n, kb = (b.shape[1], b.shape[0]) if b_trans else b.shape
    if k != kb:
        raise ValueError(f"linear_tc: inner dimensions differ ({k} vs {kb})")
    if bias is not None and bias.shape != (n,):
        raise ValueError("linear_tc: bias must be [n]")
    if mask is not None and mask.shape != (m, n):
        raise ValueError("linear_tc: mask must be [m, n]")
    lib = _lib.load()
    c = torch.empty((m, n), dtype=torch.float32, device=a.device)
    wsb = lib.dgod_linear_tc_workspace_bytes(m, n, k)
    ws = _ws(wsb, a.device)
    tok = KernelTimer.start(name, 4 * (m * k + n * k + m * n))
    check(lib.dgod_linear_tc(_p(a), int(a_trans), _p(b), int(b_trans), m, n, k, _p(bias), int(relu), _p(mask), _p(c),
                             _p(ws), ws.numel(), _stream()), ValueError)
    KernelTimer.stop(tok)
    return c


def box_head_mlp_supported(x: Tensor, w6: Tensor, w7: Tensor) -> bool:
    """Whether box_head_mlp takes these operands: CUDA fp32, autocast off, fc widths multiples of 32, x 16-byte aligned."""
    return (x.is_cuda and x.dim() == 2 and x.dtype == torch.float32 and w6.dtype == torch.float32
            and w7.dtype == torch.float32 and not torch.is_autocast_enabled("cuda") and x.shape[0] >= 1
            and x.shape[1] >= 1 and x.data_ptr() % 16 == 0 and w6.shape[1] == x.shape[1] and w6.shape[0] % 32 == 0
            and w7.shape == (w7.shape[0], w6.shape[0]) and w7.shape[0] % 32 == 0)


class _BoxHeadMLP(torch.autograd.Function):
    """relu(fc7(relu(fc6(x)))) on dgod_linear_tc: both ReLUs in the forward products' epilogues, fc6's ReLU mask in
    the epilogue of fc7's input-gradient product.  fc7's ReLU backward and the bias gradients stay ATen."""

    @staticmethod
    def forward(ctx, x, w6, b6, w7, b7):
        h6 = linear_tc(x, w6, bias=b6, relu=True, name="linear_tc_fwd")
        h7 = linear_tc(h6, w7, bias=b7, relu=True, name="linear_tc_fwd")
        ctx.save_for_backward(x, w6, w7, h6, h7)
        return h7

    @staticmethod
    def backward(ctx, g7):
        x, w6, w7, h6, h7 = ctx.saved_tensors
        g7 = torch.ops.aten.threshold_backward(g7.contiguous(), h7, 0)
        gw7 = linear_tc(g7, h6, a_trans=True, b_trans=True, name="linear_tc_wgrad")
        g6 = linear_tc(g7, w7, b_trans=True, mask=h6, name="linear_tc_dgrad")
        gw6 = linear_tc(g6, x, a_trans=True, b_trans=True, name="linear_tc_wgrad")
        gx = linear_tc(g6, w6, b_trans=True, name="linear_tc_dgrad") if ctx.needs_input_grad[0] else None
        return gx, gw6, g6.sum(0), gw7, g7.sum(0)


def box_head_mlp(x: Tensor, w6: Tensor, b6: Tensor, w7: Tensor, b7: Tensor) -> Tensor:
    """relu(linear(relu(linear(x, w6, b6)), w7, b7)) for fp32 x [m, k] with fp32 accuracy on the tensor cores."""
    return _BoxHeadMLP.apply(x.contiguous(), w6.contiguous(), b6.contiguous(), w7.contiguous(), b7.contiguous())


class _GRLConv2d(torch.autograd.Function):
    """grad_reverse followed by nn.Conv2d with the reversal scale folded into the convolution's input-gradient
    (DGcommon.py:73-74 ImageDAFPN.Conv1, DGcommon.py:106-107 ImageDA.Conv1): cuDNN's dgrad runs on the weight
    pre-scaled by -alpha — a pass over the 2-19 MB weight instead of a pass over the feature-map gradient
    (637 MB for [8,256,152,256] fp32).  Weight and bias gradients use the unscaled operands."""

    @staticmethod
    def forward(ctx, x, weight, bias, stride, padding, dilation, groups, alpha):
        ctx.save_for_backward(x, weight)
        ctx.cfg = (stride, padding, dilation, groups, alpha, None if bias is None else list(bias.shape))
        return torch.nn.functional.conv2d(x, weight, bias, stride, padding, dilation, groups)

    @staticmethod
    def backward(ctx, gy):
        x, w = ctx.saved_tensors
        x, w = x.to(gy.dtype), w.to(gy.dtype)         # under autocast: the operands autocast gave F.conv2d
        stride, padding, dilation, groups, alpha, bias_sizes = ctx.cfg
        gx = gw = gb = None
        common = (list(stride), list(padding), list(dilation), False, [0, 0], groups)
        if ctx.needs_input_grad[0]:
            gx = torch.ops.aten.convolution_backward(gy, x, w * (-alpha), bias_sizes, *common, [True, False, False])[0]
        if ctx.needs_input_grad[1] or (bias_sizes is not None and ctx.needs_input_grad[2]):
            _, gw, gb = torch.ops.aten.convolution_backward(gy, x, w, bias_sizes, *common,
                                                            [False, ctx.needs_input_grad[1], bias_sizes is not None])
        return gx, gw, gb, None, None, None, None, None


def grl_conv2d(x: Tensor, conv: "torch.nn.Conv2d", alpha: float = 0.1) -> Tensor:
    """conv(grad_reverse(x)) for an nn.Conv2d with zeros padding, the reversal fused into the conv's dgrad."""
    pad = conv.padding if not isinstance(conv.padding, str) else (0, 0)
    if conv.padding_mode != "zeros" or isinstance(conv.padding, str):
        return conv(grad_reverse(x, alpha))
    return _GRLConv2d.apply(x, conv.weight, conv.bias, tuple(conv.stride), tuple(pad), tuple(conv.dilation), conv.groups, alpha)


# --------------------------------------------------------------------------------- balanced sampler
def balanced_sample(labels: Tensor, keys: Tensor, num_pos: int, batch_size_per_image: int):
    """BalancedPositiveNegativeSampler (TV models/detection/_utils.py:11-71) for a batch in one launch: labels [B,N]
    (float or int64: >= 1 positive, 0 negative, < 0 ignored), keys [B,N] uniform random floats.  Returns
    (pos_idx [B,P'], pos_valid bool, neg_idx [B,S'], neg_valid bool, counts int32 [B,2]) with P' = min(num_pos, N),
    S' = min(batch_size_per_image, N); indices ascending, zero past the counts.  No host synchronisation."""
    _need_cuda(labels, keys)
    if labels.dim() != 2 or keys.shape != labels.shape:
        raise RuntimeError("balanced_sample: labels and keys must be [B, N]")
    if labels.dtype not in (torch.float32, torch.int64):
        labels = labels.to(torch.int64)
    labels, keys = labels.contiguous(), _f32c(keys)
    B, N = labels.shape
    P, S = min(int(num_pos), N), min(int(batch_size_per_image), N)
    dev = labels.device
    pos_idx = torch.empty((B, P), dtype=torch.int64, device=dev)
    neg_idx = torch.empty((B, S), dtype=torch.int64, device=dev)
    pos_valid = torch.empty((B, P), dtype=torch.bool, device=dev)
    neg_valid = torch.empty((B, S), dtype=torch.bool, device=dev)
    counts = torch.empty((B, 2), dtype=torch.int32, device=dev)
    tok = KernelTimer.start("balanced_sample", B * N * (labels.element_size() + 4) + B * (P + S) * 9)
    check(_lib.load().dgod_balanced_sample(_p(labels), int(labels.dtype == torch.int64), _p(keys), B, N, int(num_pos),
                                           int(batch_size_per_image), _p(pos_idx), _p(pos_valid), _p(neg_idx), _p(neg_valid),
                                           _p(counts), _stream()))
    KernelTimer.stop(tok)
    return pos_idx, pos_valid, neg_idx, neg_valid, counts


def sample_rois(pos_idx: Tensor, pos_valid: Tensor, neg_idx: Tensor, neg_valid: Tensor, labels: Tensor,
                clamped_idx: Tensor, boxes: Tensor, counts: Tensor, gt_boxes: Sequence[Tensor],
                batch_size_per_image: int, weights: Sequence[float]):
    """The RoI heads' training samples (TV roi_heads.py:615-678 after the sampler) in one launch, no host
    synchronisation.  `labels` / `clamped_idx` [B,N] are `match_boxes`' results over the padded candidates (boxes
    [B,cap,4], counts [B], ground truths appended) and pos_* / neg_* what `balanced_sample` picked from them.  Returns
    (s_props [B,S,4], s_labels int64 [B,S], reg_targets [B,S,4]) with S = batch_size_per_image: the picked candidates
    in ascending index order, regression targets encoded with `weights`; slots left empty (fewer candidates than S) hold
    a zero box, label -100 and a finite target."""
    _need_cuda(pos_idx, pos_valid, neg_idx, neg_valid, labels, clamped_idx, boxes, counts)
    B, N = labels.shape
    S = int(batch_size_per_image)
    dev = labels.device
    gt_cat, gt_off = _gt_batch(gt_boxes, dev)
    pos_idx, neg_idx = pos_idx.contiguous(), neg_idx.contiguous()
    pos_valid, neg_valid = [(v if v.dtype in (torch.bool, torch.uint8) else v.to(torch.uint8)).contiguous()   # 1 byte each
                            for v in (pos_valid, neg_valid)]
    labels, clamped_idx = labels.contiguous(), clamped_idx.contiguous()
    boxes, counts = _f32c(boxes), counts.to(torch.int32).contiguous()
    s_props = torch.empty((B, S, 4), dtype=torch.float32, device=dev)
    s_labels = torch.empty((B, S), dtype=torch.int64, device=dev)
    reg_targets = torch.empty((B, S, 4), dtype=torch.float32, device=dev)
    tok = KernelTimer.start("sample_rois", B * (pos_idx.shape[1] + neg_idx.shape[1]) * 9 + B * S * (2 * 16 + 16 + 8 + 8 + 16))
    check(_lib.load().dgod_sample_rois(_p(pos_idx), _p(pos_valid), pos_idx.shape[1], _p(neg_idx), _p(neg_valid),
                                       neg_idx.shape[1], _p(labels), _p(clamped_idx), B, N, _p(boxes), _p(counts),
                                       boxes.shape[1], _p(gt_cat), _p(gt_off), S, *[float(w) for w in weights],
                                       _p(s_props), _p(s_labels), _p(reg_targets), _stream()))
    KernelTimer.stop(tok)
    return s_props, s_labels, reg_targets


# --------------------------------------------------------------------------------- RPN
def _rpn_config(n_img: int, grids: Sequence[Tuple[int, int]], strides: Sequence[Tuple[int, int]],
                cell_anchors: Sequence[Sequence[Sequence[float]]], pre_nms_top_n: int, post_nms_top_n: int,
                nms_thresh: float, min_size: float, score_thresh: float) -> RpnConfig:
    cfg = RpnConfig()
    cfg.n_img, cfg.n_levels = int(n_img), len(grids)
    cfg.anchors_per_loc = len(cell_anchors[0])
    for l, ((h, w), (sh, sw)) in enumerate(zip(grids, strides)):
        cfg.height[l], cfg.width[l], cfg.stride_h[l], cfg.stride_w[l] = int(h), int(w), int(sh), int(sw)
        for a, box in enumerate(cell_anchors[l]):
            for c in range(4):
                cfg.cell_anchors[l][a][c] = float(box[c])
    cfg.pre_nms_top_n, cfg.post_nms_top_n = int(pre_nms_top_n), int(post_nms_top_n)
    cfg.nms_thresh = float(nms_thresh)
    cfg.min_size, cfg.score_thresh = float(min_size), float(score_thresh)
    cfg.bbox_xform_clip = math.log(1000.0 / 16)
    return cfg


def rpn_proposals(objectness: Sequence[Tensor], pred_bbox_deltas: Sequence[Tensor], image_sizes: Tensor,
                  strides: Sequence[Tuple[int, int]], cell_anchors: Sequence[Sequence[Sequence[float]]],
                  pre_nms_top_n: int, post_nms_top_n: int, nms_thresh: float, min_size: float = 1e-3,
                  score_thresh: float = 0.0):
    """fasterrcnn.py:166-182 in one fused pipeline: raw RPN head outputs (per level
    [B,A,H,W] / [B,4A,H,W]) -> (boxes [B,post,4], scores [B,post], counts int32 [B]).
    image_sizes: float tensor [B,2] = (h, w) on the device.  No host synchronisation."""
    _need_cuda(image_sizes, *objectness, *pred_bbox_deltas)
    lib = _lib.load()
    dev = objectness[0].device
    n_img = objectness[0].shape[0]
    grids = [(o.shape[2], o.shape[3]) for o in objectness]
    cfg = _rpn_config(n_img, grids, strides, cell_anchors, pre_nms_top_n, post_nms_top_n, nms_thresh,
                      min_size, score_thresh)
    obj = [_f32c(o.detach()) for o in objectness]
    dl = [_f32c(d.detach()) for d in pred_bbox_deltas]
    image_sizes = _f32c(image_sizes)
    boxes = torch.empty((n_img, post_nms_top_n, 4), dtype=torch.float32, device=dev)
    scores = torch.empty((n_img, post_nms_top_n), dtype=torch.float32, device=dev)
    counts = torch.empty((n_img,), dtype=torch.int32, device=dev)
    wsb = lib.dgod_rpn_workspace_bytes(C.byref(cfg))
    ws = _ws(wsb, dev)
    op, _k1 = _level_ptrs(obj)
    dp, _k2 = _level_ptrs(dl)
    n_anchor = sum(o.shape[1] * o.shape[2] * o.shape[3] for o in obj)
    k_tot = sum(min(pre_nms_top_n, o.shape[1] * o.shape[2] * o.shape[3]) for o in obj)
    tok = KernelTimer.start("rpn_proposals", n_img * (4 * n_anchor + 16 * k_tot + 20 * post_nms_top_n))
    check(lib.dgod_rpn_proposals(C.byref(cfg), op, dp, _p(image_sizes), _p(boxes), _p(scores), _p(counts),
                                 _p(ws), wsb, _stream()))
    KernelTimer.stop(tok)
    return boxes, scores, counts


def rpn_filter_proposals(proposals: Tensor, objectness: Tensor, image_sizes: Tensor,
                         num_anchors_per_level: Sequence[int], pre_nms_top_n: int, post_nms_top_n: int,
                         nms_thresh: float, min_size: float = 1e-3, score_thresh: float = 0.0):
    """TV models/detection/rpn.py:242-297 on decoded proposals [B,A,4] and logits [B,A]
    (torchvision's concatenated order) -> (boxes [B,post,4], scores [B,post], counts [B])."""
    _need_cuda(proposals, objectness, image_sizes)
    lib = _lib.load()
    dev = proposals.device
    n_img = proposals.shape[0]
    cfg = RpnConfig()
    cfg.n_img, cfg.n_levels, cfg.anchors_per_loc = n_img, len(num_anchors_per_level), 1
    for l, n in enumerate(num_anchors_per_level):
        cfg.height[l], cfg.width[l], cfg.stride_h[l], cfg.stride_w[l] = 1, int(n), 1, 1
    cfg.pre_nms_top_n, cfg.post_nms_top_n = int(pre_nms_top_n), int(post_nms_top_n)
    cfg.nms_thresh, cfg.min_size, cfg.score_thresh = float(nms_thresh), float(min_size), float(score_thresh)
    cfg.bbox_xform_clip = math.log(1000.0 / 16)
    proposals = _f32c(proposals.detach())
    objectness = _f32c(objectness.detach()).reshape(n_img, -1)
    image_sizes = _f32c(image_sizes)
    boxes = torch.empty((n_img, post_nms_top_n, 4), dtype=torch.float32, device=dev)
    scores = torch.empty((n_img, post_nms_top_n), dtype=torch.float32, device=dev)
    counts = torch.empty((n_img,), dtype=torch.int32, device=dev)
    wsb = lib.dgod_rpn_workspace_bytes(C.byref(cfg))
    ws = _ws(wsb, dev)
    check(lib.dgod_rpn_filter(C.byref(cfg), _p(proposals), _p(objectness), _p(image_sizes), _p(boxes),
                              _p(scores), _p(counts), _p(ws), wsb, _stream()))
    return boxes, scores, counts


# --------------------------------------------------------------------------------- box head post-processing
def box_decode(rel_codes: Tensor, boxes: Tensor, weights=(1.0, 1.0, 1.0, 1.0),
               bbox_xform_clip: float = math.log(1000.0 / 16)) -> Tensor:
    """BoxCoder.decode_single (TV _utils.py:186-224): [n, k*4] codes, [n,4] boxes -> [n, k*4]."""
    _need_cuda(rel_codes, boxes)
    rel, bx = _f32c(rel_codes), _f32c(boxes)
    n = bx.shape[0]
    n_cls = rel.shape[1] // 4 if n else 0
    out = torch.empty_like(rel)
    check(_lib.load().dgod_box_decode(_p(rel), _p(bx), n, n_cls, *[float(w) for w in weights],
                                      float(bbox_xform_clip), _p(out), _stream()))
    return out


def detect_candidates(class_logits: Tensor, box_regression: Tensor, proposals: Tensor,
                      boxes_per_image: Sequence[int], image_sizes: Tensor, weights=(10.0, 10.0, 5.0, 5.0),
                      score_thresh: float = 0.05, min_size: float = 1e-2,
                      bbox_xform_clip: float = math.log(1000.0 / 16)):
    """TV models/detection/roi_heads.py:692-724 for the whole batch in one launch:
    -> (boxes [R, C-1, 4], scores [R, C-1], labels int64 [R, C-1], valid uint8 [R, C-1])."""
    _need_cuda(class_logits, box_regression, proposals, image_sizes)
    dev = class_logits.device
    lg, rg, pr = _f32c(class_logits.detach()), _f32c(box_regression.detach()), _f32c(proposals)
    n_rows, n_cls = lg.shape
    off = _offsets(boxes_per_image, dev)
    cb = torch.empty((n_rows, n_cls - 1, 4), dtype=torch.float32, device=dev)
    cs = torch.empty((n_rows, n_cls - 1), dtype=torch.float32, device=dev)
    cl = torch.empty((n_rows, n_cls - 1), dtype=torch.int64, device=dev)
    cv = torch.empty((n_rows, n_cls - 1), dtype=torch.uint8, device=dev)
    tok = KernelTimer.start("detect_candidates", n_rows * (4 * n_cls + 16 * n_cls + 16) + n_rows * (n_cls - 1) * 29)
    check(_lib.load().dgod_detect_candidates(_p(lg), _p(rg), _p(pr), _p(off), _p(_f32c(image_sizes)),
                                             len(boxes_per_image), n_rows, n_cls, *[float(w) for w in weights],
                                             float(bbox_xform_clip), float(score_thresh), float(min_size),
                                             _p(cb), _p(cs), _p(cl), _p(cv), _stream()))
    KernelTimer.stop(tok)
    return cb, cs, cl, cv


# --------------------------------------------------------------------------------- backbone boundary: FPN merge, stem
def _map_layout(t: Tensor) -> Tuple[Tensor, bool]:
    """(t as NHWC or NCHW dense memory, is NHWC).  A map whose two layouts coincide (1x1 pixels) runs as NCHW."""
    if t.dtype not in (torch.float32, torch.bfloat16) or t.dim() != 4:
        raise RuntimeError(f"backbone kernels take [N, C, H, W] maps (float32 and bfloat16 only), got {t.dtype} "
                           f"{tuple(t.shape)}")
    if t.is_contiguous():
        return t, False
    if t.is_contiguous(memory_format=torch.channels_last):
        return t, True
    return t.contiguous(), False


def _like(t: Tensor, nhwc: bool) -> Tensor:
    return t.contiguous(memory_format=torch.channels_last if nhwc else torch.contiguous_format)


def _map_fn(name: str, t: Tensor):
    """The C entry point `name` for maps of t's dtype: the fp32 one or its `_bf16` sibling."""
    lib = _lib.load()
    return getattr(lib, name) if t.dtype == torch.float32 else getattr(lib, name + "_bf16")


def fpn_merge(lat: Tensor, bias: Tensor, coarse: Tensor) -> Tensor:
    """(lat + bias[c]) + F.interpolate(coarse, size=lat.shape[-2:], mode="nearest") in one pass, bit-exact
    (dgod_fpn_merge_fwd, or dgod_fpn_merge_fwd_bf16 for bf16 maps: then as under autocast, the fp32 bias rounded to bf16
    first); the result has lat's memory layout and dtype."""
    _need_cuda(lat, bias, coarse)
    lat, nhwc = _map_layout(lat)
    coarse, bias = _like(coarse, nhwc), _f32c(bias)
    n, c, h, w = lat.shape
    if coarse.dtype != lat.dtype or coarse.shape[:2] != lat.shape[:2] or bias.shape != (c,):
        raise RuntimeError(f"fpn_merge: lateral {lat.dtype} {tuple(lat.shape)}, bias {tuple(bias.shape)} and coarse "
                           f"{coarse.dtype} {tuple(coarse.shape)}: maps of one dtype, batch and channel count expected")
    out = torch.empty_like(lat)
    tok = KernelTimer.start("fpn_merge_fwd", lat.element_size() * (2 * lat.numel() + coarse.numel()))
    check(_map_fn("dgod_fpn_merge_fwd", lat)(_p(lat), _p(bias), _p(coarse), _p(out), n, h, w, coarse.shape[2],
                                             coarse.shape[3], c, int(nhwc), _stream()))
    KernelTimer.stop(tok)
    return out


def fpn_merge_backward(g_fine: Optional[Tensor], g_lb: Optional[Tensor], coarse_shape) -> Optional[Tensor]:
    """Gradient of a coarse FPN level: g_lb + upsample_nearest2d_backward(g_fine) in one pass, bit-exact with the ATen
    backward followed by autograd's accumulation (dgod_fpn_merge_bwd).  None stands for a zero gradient."""
    if g_fine is None:
        return g_lb
    _need_cuda(g_fine, g_lb)
    g_fine, nhwc = _map_layout(g_fine)
    n, c, h, w = g_fine.shape
    if g_lb is not None:
        g_lb = _like(g_lb, nhwc)
        if g_lb.dtype != g_fine.dtype or tuple(g_lb.shape) != tuple(coarse_shape):
            raise RuntimeError(f"fpn_merge_backward: gradient {g_lb.dtype} {tuple(g_lb.shape)} of the "
                               f"{tuple(coarse_shape)} level, {g_fine.dtype} expected")
        out = torch.empty_like(g_lb)
    else:
        out = torch.empty(tuple(coarse_shape), dtype=g_fine.dtype, device=g_fine.device,
                          memory_format=torch.channels_last if nhwc else torch.contiguous_format)
    hc, wc = out.shape[2], out.shape[3]
    tok = KernelTimer.start("fpn_merge_bwd", g_fine.element_size() * (g_fine.numel() + (2 if g_lb is not None else 1)
                                                                        * out.numel()))
    check(_map_fn("dgod_fpn_merge_bwd", g_fine)(_p(g_fine), _p(g_lb), _p(out), n, h, w, hc, wc, c, int(nhwc),
                                                _stream()))
    KernelTimer.stop(tok)
    return out


class _FpnTopDownFn(torch.autograd.Function):
    """The FPN top-down chain (TV ops/feature_pyramid_network.py, FeaturePyramidNetwork.forward) from the bias-free lateral
    conv outputs: last_inner[i] = (laterals[i] + biases[i]) + upsample(last_inner[i + 1]), last_inner[-1] = top.
    Backward, finest level first: the gradient of level i is its own incoming gradient plus the 2x2 (in general: ATen's
    nearest-backward window) sum of the gradient of level i - 1 — one launch per level, no upsample-backward pass and no
    accumulation add.  A lateral's gradient is its level's gradient, the bias gradient its sum over (N, H, W) as the
    convolution backward computes it."""

    @staticmethod
    def forward(ctx, top, *lats_and_biases):
        k = len(lats_and_biases) // 2
        lats, biases = lats_and_biases[:k], lats_and_biases[k:]
        outs = [top]
        for i in range(k - 1, -1, -1):
            outs.insert(0, fpn_merge(lats[i], biases[i], outs[0]))
        ctx.shapes = [tuple(t.shape) for t in outs]
        ctx.set_materialize_grads(False)
        return tuple(outs)

    @staticmethod
    def backward(ctx, *grads):
        k = len(grads) - 1
        g = grads[0]
        g_lats, g_biases = [], []
        for i in range(k):
            g_lats.append(g)
            g_biases.append(g.sum((0, 2, 3)) if g is not None and ctx.needs_input_grad[1 + k + i] else None)
            g = fpn_merge_backward(g, grads[i + 1], ctx.shapes[i + 1])
        return (g, *g_lats, *g_biases)


def fpn_top_down(laterals: Sequence[Tensor], biases: Sequence[Tensor], top: Tensor) -> List[Tensor]:
    """All K `last_inner` maps of the FPN top-down path, finest first: `laterals` are the K - 1 finer levels' 1x1 conv
    outputs WITHOUT their bias, `biases` those convs' biases, `top` the coarsest level's conv output (bias included).
    Bit-exact with torchvision's interpolate + add chain, forward and backward."""
    if len(laterals) != len(biases):
        raise ValueError("fpn_top_down: one bias per lateral map expected")
    _need_cuda(top, *laterals, *biases)
    return list(_FpnTopDownFn.apply(top, *laterals, *biases))


def stem_pool(conv: Tensor, shift: Tensor) -> Tensor:
    """max_pool2d(relu(conv + shift[c]), kernel 3, stride 2, padding 1) in one pass that reads the conv output once
    (dgod_stem_pool_fwd), bit-exact with the three ATen ops including NaN propagation.  For a frozen stem only: it has
    no backward, so nothing it gets may require grad.  The result has conv's memory layout."""
    _need_cuda(conv, shift)
    if conv.requires_grad or shift.requires_grad:
        raise RuntimeError("stem_pool has no backward: the stem must be frozen and its input must not require grad")
    conv, nhwc = _map_layout(conv)
    shift = _f32c(shift)
    n, c, h, w = conv.shape
    if shift.shape != (c,):
        raise RuntimeError(f"stem_pool: shift of shape ({c},) expected, got {tuple(shift.shape)}")
    ho, wo = (h - 1) // 2 + 1, (w - 1) // 2 + 1
    out = torch.empty((n, c, ho, wo), dtype=conv.dtype, device=conv.device,
                      memory_format=torch.channels_last if nhwc else torch.contiguous_format)
    tok = KernelTimer.start("stem_pool", conv.element_size() * (conv.numel() + out.numel()))
    check(_map_fn("dgod_stem_pool_fwd", conv)(_p(conv), _p(shift), _p(out), n, h, w, c, ho, wo, int(nhwc), _stream()))
    KernelTimer.stop(tok)
    return out


# --------------------------------------------------------------------------------- backbone: folded Bottleneck epilogue
def _shift_relu_fwd(c: Tensor, shift: Tensor, residual: Optional[Tensor], res_shift: Optional[Tensor]) -> Tensor:
    c, nhwc = _map_layout(c)
    shift = _f32c(shift)
    n, ch, h, w = c.shape
    if residual is not None:
        residual = _like(residual, nhwc)
        if residual.dtype != c.dtype or residual.shape != c.shape:
            raise RuntimeError(f"shift_relu: residual {residual.dtype} {tuple(residual.shape)} does not match the "
                               f"{c.dtype} {tuple(c.shape)} conv output")
    if res_shift is not None:
        res_shift = _f32c(res_shift)
    if shift.shape != (ch,) or (res_shift is not None and res_shift.shape != (ch,)):
        raise RuntimeError(f"shift_relu: shifts of shape ({ch},) expected, got {tuple(shift.shape)}"
                           + ("" if res_shift is None else f" and {tuple(res_shift.shape)}"))
    out = torch.empty_like(c)
    tok = KernelTimer.start("shift_relu", c.element_size() * c.numel() * (2 if residual is None else 3))
    check(_map_fn("dgod_shift_relu_fwd", c)(_p(c), _p(shift), _p(residual), _p(res_shift), _p(out), n, h, w, ch,
                                            int(nhwc), _stream()))
    KernelTimer.stop(tok)
    return out


class _ShiftReluFn(torch.autograd.Function):
    """Forward: dgod_shift_relu_fwd.  Backward: the ReLU's threshold_backward — the kernel relu_'s autograd runs — and
    that gradient for both `c` and the residual, as the adds' backward passes it on."""

    @staticmethod
    def forward(ctx, c, shift, residual, res_shift):
        y = _shift_relu_fwd(c, shift, residual, res_shift)
        ctx.save_for_backward(y)
        return y

    @staticmethod
    def backward(ctx, g):
        y, = ctx.saved_tensors
        gc = torch.ops.aten.threshold_backward(g, y, 0)
        return (gc if ctx.needs_input_grad[0] else None), None, (gc if ctx.needs_input_grad[2] else None), None


def shift_relu(c: Tensor, shift: Tensor, residual: Optional[Tensor] = None, res_shift: Optional[Tensor] = None) -> Tensor:
    """The epilogue of a folded ResNet Bottleneck convolution in one pass, bit-exact with torchvision's forward on the
    folded convs (dgod_shift_relu_fwd):  relu(c + shift[c]) for conv1 / conv2; relu((c + shift) + residual) for the
    tail of an identity block; relu((c + shift) + (residual + res_shift)) for the tail of a downsample block, whose
    residual is the downsample conv's output without its shift.  `c` and `residual` may require grad; the shifts are
    frozen-BN buffers and may not.  The result has c's memory layout."""
    _need_cuda(c, shift, residual, res_shift)
    if shift.requires_grad or (res_shift is not None and res_shift.requires_grad):
        raise RuntimeError("shift_relu: the shifts are frozen (no gradient); got a shift that requires grad")
    if res_shift is not None and residual is None:
        raise ValueError("shift_relu: res_shift needs a residual")
    return _ShiftReluFn.apply(c, shift, residual, res_shift)


class _BiasAddFn(torch.autograd.Function):
    """Forward: dgod_bias_add_fwd.  Backward: the gradient itself for the map, and for the bias the
    sum ATen's convolution_backward takes for a cuDNN convolution's bias, so both stay bit-exact with nn.Conv2d."""

    @staticmethod
    def forward(ctx, c, bias):
        c, nhwc = _map_layout(c)
        bias = _f32c(bias)
        n, ch, h, w = c.shape
        if c.dtype != torch.float32 or bias.shape != (ch,):
            raise RuntimeError(f"bias_add: a float32 map and a ({ch},) bias expected, got {c.dtype} and "
                               f"{tuple(bias.shape)}")
        out = torch.empty_like(c)
        tok = KernelTimer.start("bias_add", 8 * c.numel())
        check(_lib.load().dgod_bias_add_fwd(_p(c), _p(bias), _p(out), n, h, w, ch, int(nhwc), _stream()))
        KernelTimer.stop(tok)
        return out

    @staticmethod
    def backward(ctx, g):
        return (g if ctx.needs_input_grad[0] else None), (g.sum((0, 2, 3)) if ctx.needs_input_grad[1] else None)


def bias_add(c: Tensor, bias: Tensor) -> Tensor:
    """c + bias[c] in one pass over an fp32 [N, C, H, W] map (dgod_bias_add_fwd, the shift_relu pass without the ReLU): a biased
    convolution is conv._conv_forward(x, w, None) followed by this, bit-exact with nn.Conv2d forward and backward.  The
    result has c's memory layout."""
    _need_cuda(c, bias)
    return _BiasAddFn.apply(c, bias)


# --------------------------------------------------------------------------------- RPN head after its 3x3 conv
RPN_HEAD_CHANNELS, RPN_HEAD_ANCHORS = 256, 3


def _rpn_head_check(cs: Sequence[Tensor], bias: Tensor, w_cls: Tensor, b_cls: Tensor, w_bbox: Tensor,
                    b_bbox: Tensor) -> None:
    C, A = RPN_HEAD_CHANNELS, RPN_HEAD_ANCHORS
    if not 1 <= len(cs) <= _lib.MAX_LEVELS:
        raise ValueError(f"rpn_head: 1..{_lib.MAX_LEVELS} levels expected, got {len(cs)}")
    for i, c in enumerate(cs):
        if c.dtype != torch.float32 or c.dim() != 4 or c.shape[1] != C or c.shape[0] != cs[0].shape[0]:
            raise ValueError(f"rpn_head: level {i}: float32 [N, {C}, H, W] maps of one batch expected, got {c.dtype} "
                             f"{tuple(c.shape)}")
        if not c.is_contiguous(memory_format=torch.channels_last):
            raise ValueError(f"rpn_head: level {i}: the map must be channels_last (NHWC)")
    for name, t, shape in (("bias", bias, (C,)), ("w_cls", w_cls, (A, C, 1, 1)), ("b_cls", b_cls, (A,)),
                           ("w_bbox", w_bbox, (4 * A, C, 1, 1)), ("b_bbox", b_bbox, (4 * A,))):
        if t.dtype != torch.float32 or tuple(t.shape) != shape:
            raise ValueError(f"rpn_head: {name} must be float32 of shape {shape}, got {t.dtype} {tuple(t.shape)}")


def _rpn_levels(cs: Sequence[Tensor]):
    k = len(cs)
    return (C.c_void_p * k)(*[c.data_ptr() for c in cs]), (C.c_int * k)(*[c.shape[2] for c in cs]), \
        (C.c_int * k)(*[c.shape[3] for c in cs])


def _rpn_head_fwd(cs: Sequence[Tensor], bias: Tensor, w_cls: Tensor, b_cls: Tensor, w_bbox: Tensor, b_bbox: Tensor):
    A, k = RPN_HEAD_ANCHORS, len(cs)
    n = cs[0].shape[0]
    obj = [torch.empty((n, A, c.shape[2], c.shape[3]), dtype=torch.float32, device=c.device) for c in cs]
    dl = [torch.empty((n, 4 * A, c.shape[2], c.shape[3]), dtype=torch.float32, device=c.device) for c in cs]
    cp, hs, ws = _rpn_levels(cs)
    tok = KernelTimer.start("rpn_head_fwd", sum(4 * c.numel() + 4 * 5 * A * c[:, 0].numel() for c in cs))
    check(_lib.load().dgod_rpn_head_fwd(cp, k, hs, ws, n, RPN_HEAD_CHANNELS, A, _p(bias), _p(w_cls), _p(b_cls),
                                        _p(w_bbox), _p(b_bbox), (C.c_void_p * k)(*[o.data_ptr() for o in obj]),
                                        (C.c_void_p * k)(*[d.data_ptr() for d in dl]), _stream()))
    KernelTimer.stop(tok)
    return obj, dl


def _rpn_head_bwd(cs: Sequence[Tensor], bias: Tensor, w_cls: Tensor, w_bbox: Tensor, g_obj: Sequence[Tensor],
                  g_dl: Sequence[Tensor]):
    A, k = RPN_HEAD_ANCHORS, len(cs)
    lib = _lib.load()
    gcs = [torch.empty_like(c, memory_format=torch.channels_last) for c in cs]
    params = torch.empty(RPN_HEAD_CHANNELS * (5 * A + 1) + 5 * A, dtype=torch.float32, device=cs[0].device)
    ws = _ws(lib.dgod_rpn_head_workspace_bytes(), cs[0].device)
    cp, hs, wd = _rpn_levels(cs)
    tok = KernelTimer.start("rpn_head_bwd", sum(8 * c.numel() + 4 * 5 * A * c[:, 0].numel() for c in cs))
    check(lib.dgod_rpn_head_bwd(cp, k, hs, wd, cs[0].shape[0], RPN_HEAD_CHANNELS, A, _p(bias), _p(w_cls), _p(w_bbox),
                                (C.c_void_p * k)(*[g.data_ptr() for g in g_obj]),
                                (C.c_void_p * k)(*[g.data_ptr() for g in g_dl]),
                                (C.c_void_p * k)(*[g.data_ptr() for g in gcs]), _p(params), _p(ws), ws.numel(),
                                _stream()))
    KernelTimer.stop(tok)
    return gcs, params


class _RpnHeadFn(torch.autograd.Function):
    """The RPN head after its 3x3 conv over all levels: forward dgod_rpn_head_fwd, backward dgod_rpn_head_bwd.  Saves
    the bias-free conv outputs (the backward recomputes relu(c + bias) from them) instead of the activations."""

    @staticmethod
    def forward(ctx, bias, w_cls, b_cls, w_bbox, b_bbox, *cs):
        obj, dl = _rpn_head_fwd(cs, bias, w_cls, b_cls, w_bbox, b_bbox)
        ctx.save_for_backward(bias, w_cls, w_bbox, *cs)
        return (*obj, *dl)

    @staticmethod
    def backward(ctx, *grads):
        bias, w_cls, w_bbox, *cs = ctx.saved_tensors
        k, A, Cn = len(cs), RPN_HEAD_ANCHORS, RPN_HEAD_CHANNELS
        gcs, p = _rpn_head_bwd(cs, bias, w_cls, w_bbox, [_f32c(g) for g in grads[:k]], [_f32c(g) for g in grads[k:]])
        o1, o2, o3 = A * Cn, 5 * A * Cn, 5 * A * Cn + Cn
        return (p[o2:o3], p[:o1].view(A, Cn, 1, 1), p[o3:o3 + A], p[o1:o2].view(4 * A, Cn, 1, 1), p[o3 + A:], *gcs)


def rpn_head(cs: Sequence[Tensor], bias: Tensor, w_cls: Tensor, b_cls: Tensor, w_bbox: Tensor, b_bbox: Tensor):
    """torchvision's RPNHead forward after its 3x3 conv, all levels in one launch each way: `cs` are the conv's outputs
    WITHOUT its bias (conv._conv_forward(x, w, None)), fp32 NHWC [N, 256, H, W]; `bias` the conv's bias; w_cls / b_cls
    and w_bbox / b_bbox the cls_logits and bbox_pred 1x1 convs' parameters (3 anchors per location).  Returns
    (objectness, deltas): lists of NCHW-contiguous [N, 3, H, W] / [N, 12, H, W].  The 1x1 products are fp32 fma chains
    (not TF32); relu(c + bias) is bit-identical to the stock conv + relu_."""
    cs = list(cs)
    _rpn_head_check(cs, bias, w_cls, b_cls, w_bbox, b_bbox)
    _need_cuda(*cs, bias, w_cls, b_cls, w_bbox, b_bbox)
    params = tuple(t.contiguous() for t in (bias, w_cls, b_cls, w_bbox, b_bbox))
    k = len(cs)
    if torch.is_grad_enabled() and any(t.requires_grad for t in (*cs, *params)):
        out = _RpnHeadFn.apply(*params, *cs)
        return list(out[:k]), list(out[k:])
    return _rpn_head_fwd(cs, *params)


def rpn_head_supported(feats: Sequence[Tensor], conv: "torch.nn.Conv2d", w_cls: Tensor, w_bbox: Tensor) -> bool:
    """Whether RPNHead's forward can run on rpn_head: CUDA fp32 NHWC maps of 256 channels, autocast off, a 3x3 conv
    with a bias, 3 anchors per location, fp32 parameters 16-byte aligned."""
    params = (conv.weight, conv.bias, w_cls, w_bbox)
    return (len(feats) >= 1 and len(feats) <= _lib.MAX_LEVELS and not torch.is_autocast_enabled("cuda")
            and conv.bias is not None and conv.out_channels == RPN_HEAD_CHANNELS
            and w_cls.shape[0] == RPN_HEAD_ANCHORS
            and all(p.is_cuda and p.dtype == torch.float32 and p.data_ptr() % 16 == 0 for p in params)
            and all(f.is_cuda and f.dtype == torch.float32 and f.dim() == 4 and f.shape[0] == feats[0].shape[0]
                    and f.is_contiguous(memory_format=torch.channels_last) for f in feats))
