"""The oracle against golden vectors produced by the REFERENCE's own modules
(oracle/gen_golden.py, run where /root/reference exists).  CPU only."""
from pathlib import Path

import numpy as np
import torch
from torch import nn

from dgod_b200 import synth
from oracle import cpu as O
from oracle import gen_golden as G

GOLD = Path(__file__).parent / "golden"


def test_fcos_assignment_and_targets_match_reference():
    gold = np.load(GOLD / "fcos_assign.npz")
    anchors, npl, gts, labels = G.fcos_inputs()
    for i, (g, l) in enumerate(zip(gts, labels)):
        idx, cls, _ = O.fcos_assign(anchors, npl[0], npl[-1], g.numpy(), l.numpy(), 1.5)
        assert np.array_equal(idx, gold["matched"][i])
        onehot = np.zeros((len(idx), 9), np.uint8)
        fg = cls >= 0
        onehot[np.nonzero(fg)[0], cls[fg]] = 1
        assert np.array_equal(onehot, gold["gt_classes"][i])
    assert (gold["matched"][2] >= 0).any() and not gold["gt_classes"][2][:, 1:].any()   # the `<= 1` quirk


def test_fcos_loss_tail_matches_reference():
    """oracle o_fcos_loss == fcos.FCOSHead.compute_loss of the reference (fcos.py:149-202) on seeded head outputs."""
    gold = np.load(GOLD / "fcos_loss.npz")
    anchors, npl, gts, labels = G.fcos_inputs()
    ho = G.fcos_loss_inputs()
    cls_t, box_t = [], []
    for g, l in zip(gts, labels):
        _, c, b = O.fcos_assign(anchors, npl[0], npl[-1], g.numpy(), l.numpy(), 1.5)
        cls_t.append(c), box_t.append(b)
    out = O.fcos_loss(ho["cls_logits"].numpy(), ho["bbox_regression"].numpy(), ho["bbox_ctrness"].numpy(), anchors,
                      np.stack(cls_t), np.stack(box_t))
    np.testing.assert_allclose(out[:3], gold["losses"], rtol=1e-5)
    assert out[3] == sum(int((c >= 0).sum()) for c in cls_t) > 0


def test_fcos_eval_candidates_and_nms_match_reference():
    """oracle o_fcos_candidates + batched_nms == fcos.FCOS.postprocess_detections of the reference (fcos.py:552-619) on
    seeded head outputs: labels identical, boxes identical, scores to 1 ulp (expf inside the sigmoid)."""
    gold = np.load(GOLD / "fcos_post.npz")
    anchors, npl, _, _ = G.fcos_inputs()
    ho, shapes = G.fcos_post_inputs()
    for i, (h, w) in enumerate(shapes):
        b, s, l, c = O.fcos_candidates(ho["cls_logits"][i].numpy(), ho["bbox_regression"][i].numpy(),
                                       ho["bbox_ctrness"][i].numpy(), anchors, npl, h, w, 0.2, 300)
        assert c.max() == 300 and c.min() < 300                                   # both the top-k cut and the threshold bite
        v = np.concatenate([np.arange(k) + j * 300 for j, k in enumerate(c)])
        keep = O.batched_nms(b[v], s[v], l[v], 0.6)[:100]
        assert np.array_equal(l[v][keep], gold[f"labels{i}"])
        assert np.array_equal(b[v][keep], gold[f"boxes{i}"])
        np.testing.assert_allclose(s[v][keep], gold[f"scores{i}"], rtol=2e-7)


class _Prefixed(nn.Module):
    """Gives sub-modules the attribute names they have inside the reference's containers so that
    gen_golden.seeded_module_weights draws identical weights."""


def _rpn_and_roi_heads():
    from torchvision.models.detection.faster_rcnn import FastRCNNPredictor
    from torchvision.models.detection.rpn import RPNHead
    from oracle.ref_dgfrcnn import LabelAwareMLPHead
    rpn = _Prefixed()
    rpn.head = RPNHead(256, 3)
    roi = _Prefixed()
    roi.box_head = LabelAwareMLPHead(256 * 49, 1024)
    roi.box_predictor = FastRCNNPredictor(1024, 9)
    G.seeded_module_weights(rpn, 1)
    G.seeded_module_weights(roi, 2)
    return rpn, roi


def test_frcnn_hot_path_chain_matches_reference():
    from torchvision.models.detection._utils import BalancedPositiveNegativeSampler
    gold = np.load(GOLD / "frcnn_hotpath.npz")
    h, w = G.HOT["img"]
    features, targets = G.hotpath_inputs()
    rpn, roi = _rpn_and_roi_heads()
    feats = list(features.values())
    with torch.no_grad():
        objectness, deltas = rpn.head(feats)
    B = feats[0].shape[0]
    grids = [tuple(o.shape[-2:]) for o in objectness]
    strides = [(h // gh, w // gw) for gh, gw in grids]
    from dgod_b200.detector import make_cell_anchors
    cells = make_cell_anchors(((32,), (64,), (128,), (256,), (512,)), ((0.5, 1.0, 2.0),) * 5)
    anchors = np.concatenate([O.grid_anchors(cells[l].numpy(), gh, gw, *strides[l]) for l, (gh, gw) in enumerate(grids)])
    o_flat = torch.cat([x.permute(0, 2, 3, 1).reshape(B, -1) for x in objectness], 1).numpy()
    d_flat = torch.cat([x.view(B, -1, 4, x.shape[2], x.shape[3]).permute(0, 3, 4, 1, 2).reshape(B, -1, 4) for x in deltas], 1).numpy()
    npl = [3 * gh * gw for gh, gw in grids]
    proposals = []
    for i in range(B):
        pb, _ = O.rpn_filter_image(O.box_decode(d_flat[i], anchors), o_flat[i], npl, 600, 600, 0.7, 1e-3, 0.0, h, w)
        g = gold["proposals"][i]
        assert pb.shape == g.shape
        # Same set of boxes (exp within 1 ulp); the ORDER is only defined up to scores that are
        # equal or 1 ulp apart: torch's final sort is unstable (TV ops/boxes.py:120) and its
        # sigmoid may round the last bit differently.
        key = lambda a: a[np.lexsort(np.round(a, 2).T[::-1])]
        np.testing.assert_allclose(key(pb), key(g), rtol=0, atol=2e-4)
        moved = np.abs(pb - g).max(1) > 2e-4
        assert moved.mean() < 0.02
        proposals.append(pb)
    # anchor labels: bit-exact (no transcendental involved)
    lab = [O.rpn_assign(t["boxes"].numpy(), anchors)[1] for t in targets]
    assert np.array_equal(np.stack(lab).astype(np.int8), gold["anchor_labels"])
    # replay the reference's RNG consumption: RPN sampler (per image) then RoI sampler (batched call)
    torch.manual_seed(1234)
    s256 = BalancedPositiveNegativeSampler(256, 0.5)
    for l in lab:
        s256([torch.from_numpy(l)])
    roi_lab, props_gt = [], []
    for i, t in enumerate(targets):
        p = np.concatenate([gold["proposals"][i], t["boxes"].numpy()])
        _, lb = O.roi_assign(t["boxes"].numpy(), t["labels"].numpy(), p, 0.5, 0.5)
        roi_lab.append(torch.from_numpy(lb))
        props_gt.append(p)
    pos, neg = BalancedPositiveNegativeSampler(512, 0.25)(roi_lab)
    sampled = [torch.where(p | n)[0].numpy() for p, n in zip(pos, neg)]
    got_labels = np.stack([roi_lab[i].numpy()[s] for i, s in enumerate(sampled)])
    assert np.array_equal(got_labels, gold["roi_labels"])
    rois = synth.rois_from_boxes([torch.from_numpy(props_gt[i][s]) for i, s in enumerate(sampled)]).numpy()
    pooled = O.msroi_align_fwd([f.numpy() for f in feats[:4]], rois, [1 / 4, 1 / 8, 1 / 16, 1 / 32], 7, 7, 2, 2, 5)
    np.testing.assert_allclose(pooled.astype(np.float64).sum(axis=(1, 2, 3)), gold["pooled_sum"], rtol=1e-6, atol=1e-6)


def test_restated_training_step_reproduces_reference_losses():
    from oracle.ref_dgfrcnn import build_like_reference_factory
    gold = np.load(GOLD / "frcnn_step.npz")
    s = G.STEP
    torch.manual_seed(0)
    model = build_like_reference_factory(9, s["min_size"], s["max_size"]).train()
    imgs = synth.random_images(s["batch"], *s["img"], s["seed"])
    targets, _ = synth.random_targets(s["batch"], s["n_gt"], *s["img"], s["seed"])
    torch.manual_seed(4321)
    det = model(imgs, targets)
    for k in gold.files:
        got = torch.stack([d["losses"][k] for d in det]).detach().numpy()
        np.testing.assert_allclose(got, gold[k], rtol=1e-5, atol=1e-6)
