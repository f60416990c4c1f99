"""The bf16 backbone epilogues (dgod_*_bf16 behind ops.shift_relu, ops.stem_pool, ops.fpn_merge / fpn_top_down) against
the ATen bf16 compositions they replace, bit for bit: each op against the stock ops written out below, and the fused
modules (_FusedBottleneck, _FoldedStem, FusedFPN) under torch.autocast(dtype=bfloat16) against their stock forms under
the same autocast — outputs, input gradients and parameter gradients."""
import copy
from collections import OrderedDict

import pytest
import torch
import torch.nn.functional as F
from torch import nn
from torchvision.models.resnet import Bottleneck

pytestmark = pytest.mark.gpu

DEV = "cuda"
BF = torch.bfloat16
B, IMG_H, IMG_W = 8, 608, 1024
FORMS = ["plain", "residual", "shifted_residual"]
NHWC, NCHW = torch.channels_last, torch.contiguous_format


@pytest.fixture
def deterministic_convs():
    """cuDNN algorithms without atomics, so that two evaluations of the same convolution agree bit for bit."""
    old = (torch.backends.cudnn.deterministic, torch.backends.cudnn.benchmark)
    torch.backends.cudnn.deterministic, torch.backends.cudnn.benchmark = True, False
    yield
    torch.backends.cudnn.deterministic, torch.backends.cudnn.benchmark = old


def _bits(t):
    return t.contiguous().view(torch.int16 if t.dtype == BF else torch.int32)


def _assert_bits(got, want, what):
    assert got.dtype == want.dtype, f"{what}: dtype {got.dtype} != {want.dtype}"
    assert got.shape == want.shape, f"{what}: shape {tuple(got.shape)} != {tuple(want.shape)}"
    diff = _bits(got) != _bits(want)
    assert not bool(diff.any()), (f"{what}: {int(diff.sum())} of {diff.numel()} values differ, "
                                  f"max |diff| {float((got.float() - want.float()).abs().nan_to_num().max())}")


def _randn(shape, g, memory_format=NCHW, special=False):
    """A bf16 map; with `special`, NaN, +-inf and -0.0 at random places and all of channel 0 -0.0."""
    x = torch.randn(shape, generator=g, device=DEV)
    if special:
        idx = torch.randint(0, x.numel(), (max(x.numel() // 5000, 8),), generator=g, device=DEV)
        k = len(idx) // 4
        x.view(-1)[idx[:k]] = float("nan")
        x.view(-1)[idx[k:2 * k]] = float("inf")
        x.view(-1)[idx[2 * k:3 * k]] = -float("inf")
        x.view(-1)[idx[3 * k:]] = -0.0
        x[:, 0] = -0.0
    return x.to(BF).contiguous(memory_format=memory_format)


def _channel(v):
    return v.to(BF).view(1, -1, 1, 1)


# ------------------------------------------------------------------------------------------ shift_relu
def _shift_relu_reference(c, shift, residual, res_shift):
    """torchvision's Bottleneck on folded convs under autocast: the conv's bias (the shift) cast to bf16 and added by
    ATen's add_, the identity (the downsample conv plus its bf16 bias) added in place, relu_ — all bf16 ops."""
    out = c + _channel(shift)
    if residual is not None:
        out += residual if res_shift is None else residual + _channel(res_shift)
    return torch.relu_(out)


def _compare_shift_relu(shape, memory_format, form, special):
    from dgod_b200 import ops
    g = torch.Generator(device=DEV).manual_seed(0)
    c = _randn(shape, g, memory_format, special)
    r = _randn(shape, g, memory_format, special) if form != "plain" else None
    shift = torch.randn(shape[1], generator=g, device=DEV)
    t = torch.randn(shape[1], generator=g, device=DEV) if form == "shifted_residual" else None
    if special:
        shift[0] = -0.0
        c[:, 1] = -shift[1].to(BF)                # channel 1: the (bf16) shift cancels exactly
    gy = _randn(shape, g, memory_format)

    def run(fn):
        cc = c.detach().clone().requires_grad_(True)
        rr = None if r is None else r.detach().clone().requires_grad_(True)
        y = fn(cc, shift, rr, t)
        y.backward(gy)
        return y.detach(), cc.grad, None if rr is None else rr.grad

    y1, gc1, gr1 = run(ops.shift_relu)
    y0, gc0, gr0 = run(_shift_relu_reference)
    assert y1.is_contiguous(memory_format=memory_format)
    if special:
        assert bool(torch.isnan(y0).any()) and bool(torch.isinf(y0).any())
    _assert_bits(y1, y0, f"{form} output")
    _assert_bits(gc1, gc0, f"{form} gradient of c")
    if r is not None:
        _assert_bits(gr1, gr0, f"{form} gradient of the residual")


@pytest.mark.parametrize("form", FORMS)
def test_shift_relu_bf16_bit_exact_at_bench_shape(form):
    _compare_shift_relu((B, 256, IMG_H // 4, IMG_W // 4), NHWC, form, special=False)   # layer1's 8x256x152x256


@pytest.mark.parametrize("form", FORMS)
@pytest.mark.parametrize("shape,memory_format", [
    ((2, 64, 37, 53), NHWC),
    ((3, 24, 19, 7), NHWC),
    ((2, 12, 37, 53), NCHW),
    ((3, 7, 5, 9), NCHW),
], ids=["odd_nhwc", "odd_nhwc_c24", "odd_nchw", "odd_nchw_c7"])
@pytest.mark.parametrize("special", [False, True], ids=["finite", "nan_inf_zero"])
def test_shift_relu_bf16_bit_exact_at_odd_sizes(form, shape, memory_format, special):
    _compare_shift_relu(shape, memory_format, form, special)


# ------------------------------------------------------------------------------------------ stem
@pytest.mark.parametrize("shape,memory_format", [
    ((B, 64, IMG_H // 2, IMG_W // 2), NHWC),      # the bench's stem: 8 x 64 x 304 x 512
    ((2, 64, 37, 50), NHWC),
    ((2, 8, 37, 51), NCHW),
    ((2, 5, 6, 7), NCHW),
], ids=["bench_nhwc", "odd_nhwc", "odd_nchw", "tiny_nchw"])
def test_stem_pool_bf16_bit_exact_with_specials(shape, memory_format):
    from dgod_b200 import ops
    g = torch.Generator(device=DEV).manual_seed(3)
    conv = _randn(shape, g, memory_format, special=True)
    conv[:, :, :3, :3] = -5.0                                  # a window where everything is below zero
    shift = torch.randn(shape[1], generator=g, device=DEV)
    got = ops.stem_pool(conv, shift)
    want = F.max_pool2d(torch.relu_(conv + _channel(shift)), 3, 2, 1)
    assert bool(torch.isnan(want).any()) and bool(torch.isinf(want).any())
    assert got.is_contiguous(memory_format=memory_format)
    _assert_bits(got, want, "stem_pool")


# ------------------------------------------------------------------------------------------ FPN merge
MERGE_CASES = [
    ((B, 256, 152, 256), (76, 128), NHWC),        # the bench's P2 <- P3 merge
    ((2, 32, 13, 21), (7, 11), NHWC),             # not a factor 2 apart
    ((2, 16, 30, 40), (11, 17), NHWC),            # arbitrary ratio
    ((2, 12, 37, 53), (19, 27), NCHW),
    ((2, 5, 7, 5), (3, 6), NCHW),                 # the coarse map is wider than the fine one
]
MERGE_IDS = ["bench_nhwc", "non2x_nhwc", "ratio_nhwc", "odd_nchw", "wide_nchw"]


@pytest.mark.parametrize("fine,coarse_hw,memory_format", MERGE_CASES, ids=MERGE_IDS)
@pytest.mark.parametrize("special", [False, True], ids=["finite", "nan_inf_zero"])
def test_fpn_merge_bf16_forward_and_backward_bit_exact(fine, coarse_hw, memory_format, special):
    from dgod_b200 import ops
    g = torch.Generator(device=DEV).manual_seed(5)
    n, c = fine[:2]
    lat = _randn(fine, g, memory_format, special)
    coarse = _randn((n, c) + coarse_hw, g, memory_format, special)
    bias = torch.randn(c, generator=g, device=DEV)
    got = ops.fpn_merge(lat, bias, coarse)
    want = (lat + _channel(bias)) + F.interpolate(coarse, size=fine[-2:], mode="nearest")
    assert got.is_contiguous(memory_format=memory_format)
    _assert_bits(got, want, "merge forward")

    g_fine = _randn(fine, g, memory_format, special)
    g_lb = _randn(coarse.shape, g, memory_format, special)
    leaf = coarse.detach().clone().requires_grad_(True)
    F.interpolate(leaf, size=fine[-2:], mode="nearest").backward(g_fine)
    _assert_bits(ops.fpn_merge_backward(g_fine, None, coarse.shape), leaf.grad, "merge backward without g_lb")
    _assert_bits(ops.fpn_merge_backward(g_fine, g_lb, coarse.shape), g_lb + leaf.grad, "merge backward")


def test_mismatched_dtypes_raise():
    from dgod_b200 import ops
    x16 = torch.randn(1, 8, 4, 4, device=DEV, dtype=BF)
    x32 = x16.float()
    b = torch.zeros(8, device=DEV)
    with pytest.raises(RuntimeError, match="one dtype"):
        ops.fpn_merge(x16, b, x32[:, :, :2, :2])
    with pytest.raises(RuntimeError, match="one dtype"):
        ops.fpn_merge(x32, b, x16[:, :, :2, :2])
    with pytest.raises(RuntimeError, match="bfloat16 expected"):
        ops.fpn_merge_backward(x16, x32[:, :, :2, :2], (1, 8, 2, 2))
    with pytest.raises(RuntimeError, match="does not match"):
        ops.shift_relu(x16, b, x32)
    with pytest.raises(RuntimeError, match="does not match"):
        ops.shift_relu(x32, b, x16)
    for fn in (lambda t: ops.shift_relu(t, b), lambda t: ops.stem_pool(t, b), lambda t: ops.fpn_merge(t, b, t)):
        with pytest.raises(RuntimeError, match="float32 and bfloat16 only"):
            fn(x32.half())


# ------------------------------------------------------------------------------------------ fused modules under autocast
def _output_grads(outs, seed):
    g = torch.Generator(device=DEV).manual_seed(seed)
    return [torch.randn(v.shape, generator=g, device=DEV).to(v.dtype).contiguous(
        memory_format=NHWC if v.is_contiguous(memory_format=NHWC) else NCHW) for v in outs]


def _autocast_step(model, x, seed=2):
    """Forward under bf16 autocast, backward outside it: (outputs, input gradient, parameter gradients)."""
    for p in model.parameters():
        p.grad = None
    x = x.detach().clone().requires_grad_(x.is_floating_point() and x.requires_grad)
    with torch.autocast("cuda", dtype=BF):
        out = model(x)
    outs = list(out.values())
    torch.autograd.backward(outs, _output_grads(outs, seed))
    return ([v.detach() for v in outs], x.grad,
            {n: p.grad for n, p in model.named_parameters() if p.grad is not None})


def _compare_models(fused, stock, x):
    o0, gx0, gp0 = _autocast_step(stock, x)
    o1, gx1, gp1 = _autocast_step(fused, x)
    assert len(o0) == len(o1)
    for i, (a, b) in enumerate(zip(o1, o0)):
        assert a.dtype == BF
        _assert_bits(a, b, f"output {i}")
    if gx0 is not None:
        _assert_bits(gx1, gx0, "input gradient")
    assert gp1.keys() == gp0.keys() and len(gp0) > 0
    for n in gp0:
        assert gp1[n].dtype == torch.float32, n
        _assert_bits(gp1[n], gp0[n], f"gradient of {n}")
    return gp0


def _fpn_pair(in_channels, memory_format):
    from torchvision.ops.feature_pyramid_network import FeaturePyramidNetwork, LastLevelMaxPool
    from dgod_b200.detector import fuse_fpn
    torch.manual_seed(0)
    stock = FeaturePyramidNetwork(in_channels, 256, extra_blocks=LastLevelMaxPool())
    for m in stock.modules():
        if isinstance(m, nn.Conv2d):
            nn.init.uniform_(m.bias, -0.5, 0.5)
    stock = stock.to(DEV).to(memory_format=memory_format)
    fused = copy.deepcopy(stock)
    fuse_fpn(fused)
    return fused, stock


class _Features(nn.Module):
    """An FPN fed from one tensor: the four levels are slices of a packed bf16 input, so that one input gradient
    covers every level."""

    def __init__(self, fpn, in_channels, sizes):
        super().__init__()
        self.fpn, self.in_channels, self.sizes = fpn, in_channels, sizes

    def forward(self, flat):
        xs, off = OrderedDict(), 0
        mf = NHWC if self.fpn.inner_blocks[0][0].weight.is_contiguous(memory_format=NHWC) else NCHW
        for i, (c, (h, w)) in enumerate(zip(self.in_channels, self.sizes)):
            n = flat.shape[0]
            xs[str(i)] = flat[:, off:off + c * h * w].view(n, c, h, w).contiguous(memory_format=mf)
            off += c * h * w
        return self.fpn(xs)


@pytest.mark.parametrize("sizes,in_channels,memory_format,batch", [
    ([(IMG_H // s, IMG_W // s) for s in (4, 8, 16, 32)], [256, 512, 1024, 2048], NHWC, B),
    ([(37, 53), (19, 27), (10, 14), (5, 7)], [32, 64, 96, 128], NHWC, 2),
    ([(30, 40), (11, 17), (7, 5), (3, 6)], [32, 64, 96, 128], NCHW, 2),
], ids=["bench_nhwc", "odd_nhwc", "ratio_nchw"])
def test_fused_fpn_under_autocast_equals_stock(deterministic_convs, sizes, in_channels, memory_format, batch):
    """FusedFPN against torchvision's FeaturePyramidNetwork, both under the same autocast.  Under autocast the stock
    merge is fp32 (F.interpolate is on autocast's fp32 list, so a bf16 lateral is added to an fp32 map), and FusedFPN
    runs the fp32 merge kernels on the upcast laterals: outputs, input gradients and every parameter gradient (the
    lateral biases' included, from the same convolution_backward) bitwise equal."""
    fused, stock = _fpn_pair(in_channels, memory_format)
    g = torch.Generator(device=DEV).manual_seed(0)
    numel = sum(c * h * w for c, (h, w) in zip(in_channels, sizes))
    flat = torch.randn(batch, numel, generator=g, device=DEV).to(BF).requires_grad_(True)
    grads = _compare_models(_Features(fused, in_channels, sizes), _Features(stock, in_channels, sizes), flat)
    assert any(n.endswith("inner_blocks.0.0.bias") for n in grads)


def _backbone(trainable_layers, memory_format):
    from torchvision.models.detection.backbone_utils import resnet_fpn_backbone
    from dgod_b200 import utils
    from dgod_b200.detector import fuse_fpn
    torch.manual_seed(0)
    bb = resnet_fpn_backbone(backbone_name="resnet50", weights=None, trainable_layers=trainable_layers).to(DEV)
    bb = bb.to(memory_format=memory_format).train()
    utils.calibrate_frozen_bn(bb, torch.rand(2, 3, 64, 96, device=DEV))
    assert utils.fold_frozen_bn(bb) == 53
    stock = copy.deepcopy(bb)
    fuse_fpn(bb.fpn)
    for m in stock.modules():                          # the unfused forms: folded convs + stock relu, add, max-pool
        if type(m) is utils._FusedBottleneck:
            m.__class__ = Bottleneck
        elif type(m) is utils._FoldedStem:
            m.__class__ = utils._FoldedConv2d
        elif type(m) is utils._StemReLU:
            m.__class__ = nn.ReLU
        elif type(m) is utils._StemMaxPool:
            m.__class__ = nn.MaxPool2d
    return bb, stock


@pytest.mark.parametrize("trainable_layers,memory_format,shape", [
    (3, NHWC, (B, 3, IMG_H, IMG_W)),                   # the bench's backbone: fused stem, layer1 forward-only
    (3, NCHW, (2, 3, 200, 328)),
    (5, NHWC, (2, 3, 200, 328)),                       # every block through the op's backward (stock stem: trainable)
], ids=["bench_tl3_nhwc", "tl3_nchw", "tl5_nhwc"])
def test_fused_backbone_under_autocast_equals_stock(deterministic_convs, trainable_layers, memory_format, shape):
    """The folded ResNet-50-FPN with _FoldedStem, _FusedBottleneck (identity and downsample blocks) and FusedFPN under
    autocast against the same folded backbone with the stock stem ops, Bottleneck and FeaturePyramidNetwork under the
    same autocast: outputs and every parameter gradient bit for bit."""
    from dgod_b200 import utils
    bb, stock = _backbone(trainable_layers, memory_format)
    assert (type(bb.body.conv1) is utils._FoldedStem) == (trainable_layers < 5)
    x = torch.rand(shape, device=DEV).contiguous(memory_format=memory_format)
    grads = _compare_models(bb, stock, x)
    assert any(".downsample.0.weight" in n for n in grads) and any(".conv3.weight" in n for n in grads)


def test_fused_bottleneck_input_gradient_under_autocast(deterministic_convs):
    """A single downsample block and an identity block with a bf16 input that requires grad: the input gradient (the
    residual's threshold_backward plus the convolutions' dgrad) is bitwise the stock one."""
    from torchvision.ops.misc import FrozenBatchNorm2d
    from dgod_b200 import utils
    torch.manual_seed(1)
    ds = nn.Sequential(nn.Conv2d(64, 256, 1, bias=False), FrozenBatchNorm2d(256))
    model = nn.Sequential(Bottleneck(64, 64, downsample=ds, norm_layer=FrozenBatchNorm2d),
                          Bottleneck(256, 64, norm_layer=FrozenBatchNorm2d)).to(DEV).to(memory_format=NHWC)
    for m in model.modules():
        if isinstance(m, FrozenBatchNorm2d):
            m.running_var.uniform_(0.5, 2.0)
            m.bias.uniform_(-0.5, 0.5)
    assert utils.fold_frozen_bn(model) == 7
    stock = copy.deepcopy(model)
    for m in stock.modules():
        if type(m) is utils._FusedBottleneck:
            m.__class__ = Bottleneck

    class _Dict(nn.Module):
        def __init__(self, m):
            super().__init__()
            self.m = m

        def forward(self, x):
            return {"out": self.m(x)}

    x = torch.randn(2, 64, 38, 52, device=DEV).to(BF).contiguous(memory_format=NHWC).requires_grad_(True)
    _compare_models(_Dict(model), _Dict(stock), x)
