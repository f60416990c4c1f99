"""The DG training step without device->host synchronisation, and the RoI heads' sampled RoIs it produces.

The RoI heads take the RPN's proposals padded [B, cap, 4] with their counts on the device: the matcher appends each
image's ground truths virtually and one kernel turns the sampler's picks into the sampled boxes, labels and
regression targets.  The eager composition that did this before (per-image cat + matcher over ragged lists, padding,
sort of the picked indices, gathers, torch `encode_boxes`) is restated here as the reference, and the new path has to
reproduce it bit for bit."""
import pytest
import torch

from dgod_b200 import synth

H, W = 608, 1024


def _reference_samples(roi, proposals, targets, keys):
    """RoIHeads.select_training_samples as the eager torch composition over a list of per-image proposals."""
    from dgod_b200 import ops
    from dgod_b200.detector import encode_boxes
    gt_boxes = [t["boxes"].to(proposals[0].dtype) for t in targets]
    gt_labels = [t["labels"] for t in targets]
    proposals = [torch.cat((p, g)) for p, g in zip(proposals, gt_boxes)]
    sizes = [p.shape[0] for p in proposals]
    m = ops.match_boxes(gt_boxes, proposals, roi.fg_iou_thresh, roi.bg_iou_thresh, False,
                        gt_labels=gt_labels, want=("labels_i64", "clamped_idx"))
    B, N, S = len(proposals), max(sizes), roi.batch_size_per_image
    dev = proposals[0].device
    labels = torch.full((B, N), -1, dtype=torch.int64, device=dev)
    idxs = torch.zeros((B, N), dtype=torch.int64, device=dev)
    props = torch.zeros((B, N, 4), dtype=proposals[0].dtype, device=dev)
    for i, (l, c, p) in enumerate(zip(m["labels_i64"].split(sizes), m["clamped_idx"].split(sizes), proposals)):
        labels[i, :sizes[i]], idxs[i, :sizes[i]], props[i, :sizes[i]] = l, c, p
    pos_idx, pos_valid, neg_idx, neg_valid = roi.sampler(labels, keys)
    chosen = torch.cat([torch.where(pos_valid, pos_idx, torch.full_like(pos_idx, N)),
                        torch.where(neg_valid, neg_idx, torch.full_like(neg_idx, N))], dim=1)
    if chosen.shape[1] < S:
        chosen = torch.cat([chosen, torch.full((B, S - chosen.shape[1]), N, dtype=chosen.dtype, device=dev)], dim=1)
    sel = torch.sort(chosen, dim=1).values[:, :S]
    slot_valid = sel < N
    sel = sel.clamp(max=N - 1)
    s_props = torch.gather(props, 1, sel[..., None].expand(-1, -1, 4)) * slot_valid[..., None]
    s_labels = torch.where(slot_valid, torch.gather(labels, 1, sel), torch.full_like(sel, -100))
    s_idxs = torch.gather(idxs, 1, sel) * slot_valid
    max_gt = max([g.shape[0] for g in gt_boxes] + [1])
    gt_pad = torch.zeros((B, max_gt, 4), dtype=props.dtype, device=dev)
    for i, g in enumerate(gt_boxes):
        gt_pad[i, :g.shape[0]] = g
    matched_gt = torch.gather(gt_pad, 1, s_idxs[..., None].expand(-1, -1, 4))
    safe = s_props.clone()
    safe[..., 2:] += (~slot_valid)[..., None]
    return s_props, s_labels, encode_boxes(matched_gt, safe, roi.weights), N


def _same_bits(a, b):
    return a.shape == b.shape and a.dtype == b.dtype and torch.equal(a.view(torch.int32) if a.is_floating_point() else a,
                                                                      b.view(torch.int32) if b.is_floating_point() else b)


def _inputs(n_props, n_gts, seed):
    from dgod_b200.detector import RoIHeads
    props, targets = [], []
    for i, (n, m) in enumerate(zip(n_props, n_gts)):
        g = synth.gen(seed + i)
        gt = synth.random_boxes(m, H, W, g)
        p = synth.random_boxes(n, H, W, g)
        if m > 0:                          # a share of the proposals near the ground truths: positives at 0.5 IoU
            near = gt[torch.randint(0, m, (n // 4,), generator=g)] + torch.randn(n // 4, 4, generator=g) * 8
            p[: n // 4] = torch.minimum(near.clamp(min=0), torch.tensor([W, H, W, H], dtype=torch.float32))
            p[: n // 4, 2:] = torch.maximum(p[: n // 4, 2:], p[: n // 4, :2] + 1)
        props.append(p.cuda())
        targets.append({"boxes": gt.cuda(), "labels": torch.randint(1, 9, (m,), generator=g).cuda()})
    return RoIHeads(256, 9).cuda().train(), props, targets


@pytest.mark.gpu
@pytest.mark.parametrize("n_props,n_gts", [
    ((2000, 2000), (20, 20)),              # bench.py's case: every image full, N = cap + max_gt = max(sizes)
    ((700, 650, 90), (3, 5, 4)),           # unequal counts (padding), image 2 has fewer candidates than 512 slots
    ((600, 400), (6, 0)),                  # an image without ground truth: every candidate is background
])
def test_sampled_rois_bit_exact_with_eager_composition(n_props, n_gts):
    roi, props, targets = _inputs(n_props, n_gts, 17)
    g = torch.Generator(device="cuda")
    g.manual_seed(5)
    n_ref = max(n + m for n, m in zip(n_props, n_gts))
    keys = torch.rand((len(props), n_ref), device="cuda", generator=g)
    want = _reference_samples(roi, props, targets, keys)[:3]
    # the list form, and the RPN's padded form with garbage past each image's count
    cap = max(n_props) + 37
    padded = synth.random_boxes(len(props) * cap, H, W, synth.gen(3)).view(len(props), cap, 4).cuda()
    for i, p in enumerate(props):
        padded[i, :p.shape[0]] = p
    counts = torch.tensor(n_props, dtype=torch.int32, device="cuda")
    for proposals in (props, (padded, counts)):
        got = roi.select_training_samples(proposals, targets, keys)
        for name, a, b in zip(("s_props", "s_labels", "reg_targets"), got, want):
            assert _same_bits(a, b), name
    s_labels = want[1]
    for i, (n, m) in enumerate(zip(n_props, n_gts)):
        assert int((s_labels[i] >= 0).sum()) == min(512, n + m)
        if m == 0:
            assert int((s_labels[i] > 0).sum()) == 0


@pytest.mark.gpu
def test_dg_cycle_has_no_host_sync():
    """A full 8-step dg cycle of dg.DGFRCNN (forward, backward, SGD) enqueues without a single synchronising call."""
    from dgod_b200 import dg
    torch.manual_seed(0)
    B, D = 2, 2
    m = dg.DGFRCNN(9, B, "dg", [0.5, 0.5, 0.5, 0.05, 0.0001], num_domains=D).cuda().train()
    opt = m.configure_optimizer(lr=1e-5)
    imgs = [i.cuda() for i in synth.random_images(B, H, W, 3)]
    targets, dom = synth.random_targets(B, 6, H, W, 3, n_domains=D)
    batch = (imgs, [t["boxes"].cuda() for t in targets], [t["labels"].cuda() for t in targets], dom)  # ids on the host

    def cycle():
        losses = []
        for _ in range(8):
            loss = m.training_step(batch)
            opt.zero_grad(set_to_none=True)
            loss.backward()
            opt.step()
            losses.append(loss.detach())
        return losses

    cycle()                                # warm-up: allocator, cached device constants, cuDNN / cuBLAS handles
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        losses = cycle()
    finally:
        torch.cuda.set_sync_debug_mode(0)
    assert bool(torch.isfinite(torch.stack(losses)).all())
    assert m.mode == 0 and m.sub_mode == 0
