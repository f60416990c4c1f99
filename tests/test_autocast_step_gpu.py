"""Training and validation under torch.autocast("cuda", dtype=torch.bfloat16): the fused gradient-reversal layers against
grad_reverse + the stock layer under the same autocast, a FasterRCNN step, full DGFRCNN / DGFCOS mode cycles (batched and
per-image modes) with backward and the optimizer step outside the context, and the validation hooks."""
import pytest
import torch

from dgod_b200 import synth

pytestmark = pytest.mark.gpu

DEV = "cuda"
BF = torch.bfloat16
IMG_H, IMG_W = 800, 1333                  # bench.py's synthetic images (the detector resizes them to 608x1024)
REG_WEIGHTS = [0.5, 0.5, 0.5, 0.05, 0.0001]
CYCLE = [0, 1, 0, 2, 0, 3, 0, 4]
# Input-gradient bound of the fused GRL layers: they fold -alpha into the bf16 product (the GEMM's alpha / the
# pre-scaled bf16 weight), where the stock chain rounds the product to bf16 and then scales it.  Each side is within a
# few bf16 roundings (2^-8 relative) of the exact product, and the pre-scaled weight adds one rounding per term, so the
# two agree to 2^-6 relative plus 2^-8 of the largest magnitude (for sums that cancel).
GRL_RTOL, GRL_ATOL_OF_MAX = 2.0 ** -6, 2.0 ** -8


@pytest.fixture
def deterministic_convs():
    old = (torch.backends.cudnn.deterministic, torch.backends.cudnn.benchmark)
    torch.backends.cudnn.deterministic, torch.backends.cudnn.benchmark = True, False
    yield
    torch.backends.cudnn.deterministic, torch.backends.cudnn.benchmark = old


def _same_bits(a, b):
    return a.dtype == b.dtype and a.shape == b.shape and torch.equal(a.contiguous().view(torch.int16 if a.dtype == BF
                                                                                          else torch.int32),
                                                                     b.contiguous().view(torch.int16 if b.dtype == BF
                                                                                          else torch.int32))


def _grl_bound(got, want):
    torch.testing.assert_close(got, want, rtol=GRL_RTOL, atol=GRL_ATOL_OF_MAX * float(want.abs().max()))


@pytest.mark.parametrize("x_dtype", [torch.float32, BF], ids=["x_fp32", "x_bf16"])
@pytest.mark.parametrize("shape", [(1024, 1024), (2, 600, 256)], ids=["2d", "3d"])
def test_grl_linear_under_autocast(x_dtype, shape):
    from dgod_b200 import ops
    g = synth.gen(12)
    lin = torch.nn.Linear(shape[-1], 512).to(DEV)
    x0 = torch.randn(*shape, generator=g).to(DEV, x_dtype)
    go = torch.randn(*shape[:-1], 512, generator=g).to(DEV, BF)

    def run(fn):
        x = x0.clone().requires_grad_(True)
        lin.weight.grad = lin.bias.grad = None
        with torch.autocast("cuda", dtype=BF):
            y = fn(x)
        y.backward(go)
        return y.detach(), x.grad, lin.weight.grad, lin.bias.grad

    y1, gx1, gw1, gb1 = run(lambda x: ops.grl_linear(x, lin.weight, lin.bias))
    y0, gx0, gw0, gb0 = run(lambda x: lin(ops.grad_reverse(x)))
    assert y1.dtype == BF and gx1.dtype == x_dtype and gw1.dtype == gb1.dtype == torch.float32
    assert _same_bits(y1, y0) and _same_bits(gw1, gw0) and _same_bits(gb1, gb0)
    _grl_bound(gx1.float(), gx0.float())


@pytest.mark.parametrize("x_dtype", [torch.float32, BF], ids=["x_fp32", "x_bf16"])
def test_grl_conv2d_under_autocast(deterministic_convs, x_dtype):
    from dgod_b200 import ops
    g = synth.gen(13)
    for cin, cout, stride, shape in [(256, 256, (2, 4), (2, 256, 38, 64)), (64, 32, 2, (1, 64, 19, 32))]:
        conv = torch.nn.Conv2d(cin, cout, 3, stride=stride).to(DEV)
        x0 = torch.randn(*shape, generator=g).to(DEV, x_dtype)

        def run(fn, go=None):
            x = x0.clone().requires_grad_(True)
            conv.weight.grad = conv.bias.grad = None
            with torch.autocast("cuda", dtype=BF):
                y = fn(x)
            if go is None:
                go = torch.randn(y.shape, generator=g).to(DEV, BF)
            y.backward(go)
            return go, y.detach(), x.grad, conv.weight.grad, conv.bias.grad

        go, y1, gx1, gw1, gb1 = run(lambda x: ops.grl_conv2d(x, conv))
        _, y0, gx0, gw0, gb0 = run(lambda x: conv(ops.grad_reverse(x)), go)
        assert y1.dtype == BF and gx1.dtype == x_dtype and gw1.dtype == gb1.dtype == torch.float32
        assert _same_bits(y1, y0) and _same_bits(gw1, gw0) and _same_bits(gb1, gb0)
        _grl_bound(gx1.float(), gx0.float())


def test_faster_rcnn_training_step_under_autocast():
    from dgod_b200.detector import FasterRCNN
    from dgod_b200.utils import calibrate_frozen_bn, fold_frozen_bn
    torch.manual_seed(0)
    det = FasterRCNN(num_classes=10, min_size=600, max_size=1200, trainable_backbone_layers=3).to(DEV).train()
    det = det.to(memory_format=torch.channels_last)
    imgs = [i.to(DEV) for i in synth.random_images(2, IMG_H, IMG_W, 3)]
    with torch.no_grad():
        calibrate_frozen_bn(det.backbone, det.transform(imgs, None)[0].tensors)
    fold_frozen_bn(det.backbone)
    targets, _ = synth.random_targets(2, 6, IMG_H, IMG_W, 3)
    targets = [{k: v.to(DEV) for k, v in t.items()} for t in targets]
    with torch.autocast("cuda", dtype=BF):
        out = det(imgs, targets)
    feats = det.last["features"]
    assert all(v.dtype == BF for v in feats.values())
    losses = [v for d in out for v in d["losses"].values()]
    assert losses and all(bool(torch.isfinite(v).all()) for v in losses)
    sum(losses).backward()
    assert all(p.grad is None or p.grad.dtype == torch.float32 for p in det.parameters())
    assert det.backbone.fpn.inner_blocks[0][0].bias.grad is not None


def _dg_model(arch, batched, B=2, D=2):
    from dgod_b200 import dg, dg_fcos
    from dgod_b200.utils import calibrate_frozen_bn, fold_frozen_bn
    torch.manual_seed(0)
    cls = dg.DGFRCNN if arch == "frcnn" else dg_fcos.DGFCOS
    m = cls(9, B, "dg", REG_WEIGHTS, num_domains=D).to(DEV).train().to(memory_format=torch.channels_last)
    if hasattr(m, "batched_modes"):
        m.batched_modes = batched
    imgs = [i.to(DEV) for i in synth.random_images(B, IMG_H, IMG_W, 3)]
    with torch.no_grad():
        calibrate_frozen_bn(m.detector.backbone, m.detector.transform(imgs, None)[0].tensors)
    fold_frozen_bn(m.detector.backbone)
    targets, dom = synth.random_targets(B, 6, IMG_H, IMG_W, 3, n_domains=D)
    batch = (imgs, [t["boxes"].to(DEV) for t in targets], [t["labels"].to(DEV) for t in targets], dom)
    return m, batch


def _cycle(m, batch, opt, amp):
    """One 8-step mode cycle; the forward under autocast when `amp`, backward and the optimizer step outside it.
    Returns the losses and, per step, the names of the parameters that received a gradient."""
    losses, touched = [], []
    for _ in CYCLE:
        with torch.autocast("cuda", dtype=BF, enabled=amp):
            loss = m.training_step(batch)
        opt.zero_grad(set_to_none=True)
        loss.backward()
        touched.append({n for n, p in m.named_parameters() if p.grad is not None})
        for n, p in m.named_parameters():
            assert p.grad is None or (p.dtype == p.grad.dtype == torch.float32), n
        opt.step()
        losses.append(loss.detach())
    return losses, touched


@pytest.mark.parametrize("batched", [True, False], ids=["batched", "per_image"])
def test_dgfrcnn_cycle_under_autocast(batched):
    m, batch = _dg_model("frcnn", batched)
    opt = m.configure_optimizer(lr=1e-5)
    _, touched32 = _cycle(m, batch, opt, amp=False)
    losses, touched16 = _cycle(m, batch, opt, amp=True)
    assert all(bool(torch.isfinite(v)) for v in losses)
    assert touched16 == touched32
    assert m.mode == 0 and m.sub_mode == 0


def test_dgfrcnn_autocast_cycle_has_no_host_sync():
    """With the domain ids on the host, as the reference's collate_fn leaves them: nothing in the autocast cycle reads
    from the device (the same check as the fp32 cycle's)."""
    m, batch = _dg_model("frcnn", True)
    opt = m.configure_optimizer(lr=1e-5)
    _cycle(m, batch, opt, amp=True)                 # warm-up: allocator, cached constants, cuDNN / cuBLAS handles
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        losses = []
        for _ in CYCLE:
            with torch.autocast("cuda", dtype=BF):
                loss = m.training_step(batch)
            opt.zero_grad(set_to_none=True)
            loss.backward()
            opt.step()
            losses.append(loss.detach())
    finally:
        torch.cuda.set_sync_debug_mode(0)
    assert bool(torch.isfinite(torch.stack(losses)).all())


def test_dgfcos_cycle_under_autocast():
    m, batch = _dg_model("fcos", True)
    opt = m.configure_optimizer()
    _, touched32 = _cycle(m, batch, opt, amp=False)
    losses, touched16 = _cycle(m, batch, opt, amp=True)
    assert all(bool(torch.isfinite(v)) for v in losses)
    assert touched16 == touched32


@pytest.mark.parametrize("arch", ["frcnn", "fcos"])
def test_validation_under_autocast(arch):
    m, _ = _dg_model(arch, True)
    if arch == "fcos":
        m.detector.score_thresh = 0.0
    with torch.autocast("cuda", dtype=BF):
        for b in range(2):
            imgs = [i.to(DEV) for i in synth.random_images(2, 320, 416, 11 + b)]
            tg, dom = synth.random_targets(2, 6, 320, 416, 11 + b)
            preds = m.validation_step((imgs, [t["boxes"].to(DEV) for t in tg], [t["labels"].to(DEV) for t in tg], dom))
            assert all(bool(torch.isfinite(p["scores"]).all()) for p in preds)
        out = m.on_validation_epoch_end()
    assert bool(torch.isfinite(torch.as_tensor(out["val_acc"])).all())
    assert m.detector.training
