"""The native FPN top-down merge (ops.fpn_top_down, detector.FusedFPN) and the fused frozen stem (ops.stem_pool,
utils.fold_frozen_bn) against the stock torchvision / ATen ops they replace, bit for bit: at the benchmarked shapes
(batch 8, 608x1024 padded input, channels_last), at sizes that are not a factor 2 apart, and in NCHW memory."""
import copy
from collections import OrderedDict

import pytest
import torch
import torch.nn.functional as F
from torch import nn

pytestmark = pytest.mark.gpu

DEV = "cuda"
B, IMG_H, IMG_W = 8, 608, 1024
BENCH_LEVELS = [(IMG_H // s, IMG_W // s) for s in (4, 8, 16, 32)]      # C2..C5 of ResNet-50: 152x256 .. 19x32
IN_CHANNELS = [256, 512, 1024, 2048]


@pytest.fixture
def deterministic_convs():
    """cuDNN algorithms without atomics, so that two evaluations of the same convolution agree bit for bit."""
    old = (torch.backends.cudnn.deterministic, torch.backends.cudnn.benchmark)
    torch.backends.cudnn.deterministic, torch.backends.cudnn.benchmark = True, False
    yield
    torch.backends.cudnn.deterministic, torch.backends.cudnn.benchmark = old


def _assert_bits(got, want, what):
    assert got.shape == want.shape, f"{what}: shape {tuple(got.shape)} != {tuple(want.shape)}"
    diff = (got.contiguous().view(torch.int32) != want.contiguous().view(torch.int32))
    assert not bool(diff.any()), (f"{what}: {int(diff.sum())} of {diff.numel()} values differ, "
                                  f"max |diff| {float((got - want).abs().nan_to_num().max())}")


def _fpn_pair(in_channels, out_channels=256, memory_format=torch.channels_last):
    from torchvision.ops.feature_pyramid_network import FeaturePyramidNetwork, LastLevelMaxPool
    from dgod_b200.detector import fuse_fpn
    torch.manual_seed(0)
    stock = FeaturePyramidNetwork(in_channels, out_channels, extra_blocks=LastLevelMaxPool())
    for m in stock.modules():
        if isinstance(m, nn.Conv2d):
            nn.init.uniform_(m.bias, -0.5, 0.5)          # nonzero biases: the bias add is part of what is compared
    stock = stock.to(DEV).to(memory_format=memory_format)
    fused = copy.deepcopy(stock)
    fuse_fpn(fused)
    return stock, fused


def _output_grads(outs, seed):
    """Fixed random gradients for `outs`, each in its output's memory layout (the layout of a gradient decides the
    summation order of the convolution's bias gradient)."""
    g = torch.Generator(device=DEV).manual_seed(seed)
    return [torch.randn(v.shape, generator=g, device=DEV).contiguous(
        memory_format=torch.channels_last if v.is_contiguous(memory_format=torch.channels_last) else torch.contiguous_format)
        for v in outs]


def _run(fpn, xs, seed=1):
    """Forward, then backward of a fixed random linear functional of every output -> (outputs, input grads, param grads)."""
    xs = OrderedDict((k, v.detach().clone().requires_grad_(True)) for k, v in xs.items())
    out = fpn(xs)
    torch.autograd.backward(list(out.values()), _output_grads(out.values(), seed))
    return ([v.detach() for v in out.values()], [x.grad for x in xs.values()],
            {n: p.grad for n, p in fpn.named_parameters()})


def _compare_fpn(sizes, in_channels, memory_format, batch=B):
    stock, fused = _fpn_pair(in_channels, memory_format=memory_format)
    g = torch.Generator(device=DEV).manual_seed(0)
    xs = OrderedDict((str(i), torch.randn(batch, c, h, w, generator=g, device=DEV).contiguous(memory_format=memory_format))
                     for i, (c, (h, w)) in enumerate(zip(in_channels, sizes)))
    o0, gx0, gp0 = _run(stock, xs)
    o1, gx1, gp1 = _run(fused, xs)
    assert len(o0) == len(o1) == len(sizes) + 1
    for i, (a, b) in enumerate(zip(o1, o0)):
        _assert_bits(a, b, f"output {i}")
    for i, (a, b) in enumerate(zip(gx1, gx0)):
        _assert_bits(a, b, f"input gradient {i}")
    assert gp1.keys() == gp0.keys()
    for n in gp0:
        _assert_bits(gp1[n], gp0[n], f"gradient of {n}")


def test_fpn_top_down_bit_exact_at_bench_shapes(deterministic_convs):
    _compare_fpn(BENCH_LEVELS, IN_CHANNELS, torch.channels_last)


@pytest.mark.parametrize("sizes", [
    [(100, 168), (50, 84), (25, 42), (13, 21)],           # 2x steps, then 13 -> 25 and 21 -> 42: not a factor 2
    [(37, 53), (19, 27), (10, 14), (5, 7)],               # odd sizes throughout
    [(30, 40), (11, 17), (7, 5), (3, 6)],                 # arbitrary ratios; the coarsest map is wider than the next
])
@pytest.mark.parametrize("memory_format", [torch.channels_last, torch.contiguous_format], ids=["nhwc", "nchw"])
def test_fpn_top_down_bit_exact_at_other_sizes(deterministic_convs, sizes, memory_format):
    _compare_fpn(sizes, [32, 64, 96, 128], memory_format, batch=2)


def test_fpn_ops_reject_cpu_tensors():
    from dgod_b200 import ops
    x = torch.rand(1, 4, 4, 4)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        ops.fpn_top_down([x], [torch.rand(4)], torch.rand(1, 4, 2, 2))
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        ops.stem_pool(x, torch.rand(4))


# ------------------------------------------------------------------------------------------ stem
def _stem_reference(conv, shift):
    return F.max_pool2d(torch.relu_(conv + shift.view(1, -1, 1, 1)), 3, 2, 1)


@pytest.mark.parametrize("shape,memory_format", [
    ((B, 64, IMG_H // 2, IMG_W // 2), torch.channels_last),      # the bench's stem: 8 x 64 x 304 x 512
    ((2, 64, 37, 50), torch.channels_last),
    ((2, 8, 37, 51), torch.contiguous_format),
], ids=["bench_nhwc", "odd_nhwc", "odd_nchw"])
def test_stem_pool_bit_exact_with_nan(shape, memory_format):
    from dgod_b200 import ops
    g = torch.Generator(device=DEV).manual_seed(3)
    conv = torch.randn(shape, generator=g, device=DEV)
    idx = torch.randint(0, conv.numel() - 1, (max(conv.numel() // 5000, 4),), generator=g, device=DEV)
    conv.view(-1)[idx] = float("nan")                            # NaN in some windows
    conv.view(-1)[idx[: len(idx) // 2] + 1] = -float("inf")
    conv[:, :, :3, :3] = -5.0                                    # a window where everything is below zero
    conv = conv.contiguous(memory_format=memory_format)
    shift = torch.randn(shape[1], generator=g, device=DEV)
    got = ops.stem_pool(conv, shift)
    want = _stem_reference(conv.clone(), shift)
    assert bool(torch.isnan(want).any())
    assert got.is_contiguous(memory_format=memory_format)
    _assert_bits(got, want, "stem_pool")


def test_stem_pool_refuses_inputs_that_require_grad():
    from dgod_b200 import ops
    conv = torch.randn(1, 4, 8, 8, device=DEV, requires_grad=True)
    with pytest.raises(RuntimeError, match="no backward"):
        ops.stem_pool(conv, torch.zeros(4, device=DEV))


def _backbone(trainable_layers=3):
    from torchvision.models.detection.backbone_utils import resnet_fpn_backbone
    from dgod_b200.utils import calibrate_frozen_bn
    torch.manual_seed(0)
    bb = resnet_fpn_backbone(backbone_name="resnet50", weights=None, trainable_layers=trainable_layers).to(DEV)
    bb = bb.to(memory_format=torch.channels_last).train()
    calibrate_frozen_bn(bb, torch.rand(2, 3, 64, 96, device=DEV))
    return bb


def _backbone_step(bb, x, seed=2):
    for p in bb.parameters():
        p.grad = None
    out = bb(x)
    torch.autograd.backward(list(out.values()), _output_grads(out.values(), seed))
    return [v.detach().clone() for v in out.values()], {n: p.grad.clone() for n, p in bb.named_parameters()
                                                         if p.grad is not None}


def test_folded_backbone_with_fused_stem_and_fpn_equals_stock(deterministic_convs):
    """The whole rebound backbone (fused stem + FusedFPN) against the same folded backbone with the stock stem ops and
    the stock FPN, at the bench's input size; unfold_frozen_bn restores the stock modules."""
    from dgod_b200.detector import fuse_fpn
    from dgod_b200 import utils
    bb = _backbone()
    assert utils.fold_frozen_bn(bb) == 53
    assert type(bb.body.conv1) is utils._FoldedStem
    stock = copy.deepcopy(bb)
    stock.body.conv1.__class__, stock.body.relu.__class__ = utils._FoldedConv2d, nn.ReLU
    stock.body.maxpool.__class__ = nn.MaxPool2d
    keys = list(bb.state_dict().keys())
    fuse_fpn(bb.fpn)
    assert list(bb.state_dict().keys()) == keys
    x = torch.rand(B, 3, IMG_H, IMG_W, device=DEV)
    o0, g0 = _backbone_step(stock, x)
    o1, g1 = _backbone_step(bb, x)
    for i, (a, b) in enumerate(zip(o1, o0)):
        _assert_bits(a, b, f"backbone output {i}")
    assert g1.keys() == g0.keys() and "body.conv1.weight" not in g0
    for n in g0:
        _assert_bits(g1[n], g0[n], f"gradient of {n}")
    utils.unfold_frozen_bn(bb)
    assert type(bb.body.conv1) is nn.Conv2d and type(bb.body.relu) is nn.ReLU and type(bb.body.maxpool) is nn.MaxPool2d


def test_trainable_stem_is_not_fused():
    from dgod_b200 import utils
    bb = _backbone(trainable_layers=5)
    assert utils.fold_frozen_bn(bb) == 53
    assert type(bb.body.conv1) is utils._FoldedConv2d and type(bb.body.maxpool) is nn.MaxPool2d


def test_graph_captured_backbone_equals_eager(deterministic_convs):
    """bench.py captures the backbone's forward and backward with make_graphed_callables: the fused stem and FPN launch on
    the capturing stream and allocate from the torch allocator, so the replay computes what eager mode computes."""
    from dgod_b200.detector import fuse_fpn
    from dgod_b200.utils import fold_frozen_bn
    bb = _backbone()
    fold_frozen_bn(bb)
    fuse_fpn(bb.fpn)
    x = torch.rand(B, 3, IMG_H, IMG_W, device=DEV)
    o0, g0 = _backbone_step(bb, x)
    graphed = torch.cuda.make_graphed_callables(bb, (torch.rand_like(x),), num_warmup_iters=3)
    for p in bb.parameters():
        p.grad = None
    out = list(graphed(x.clone()).values())
    torch.autograd.backward(out, _output_grads(out, 2))
    for i, (a, b) in enumerate(zip(out, o0)):
        _assert_bits(a.detach(), b, f"graphed output {i}")
    for n, p in bb.named_parameters():
        if n in g0:
            _assert_bits(p.grad, g0[n], f"graphed gradient of {n}")
