"""The folded ResNet Bottleneck epilogue (ops.shift_relu, utils._FusedBottleneck) against the stock ATen composition and
torchvision's Bottleneck, bit for bit, forward and every gradient: at the benchmarked shapes (batch 8, 608x1024 padded
input, channels_last), at odd sizes, in NCHW memory, and with NaN, infinities and signed zeros in the inputs."""
import copy

import pytest
import torch
from torchvision.models.resnet import Bottleneck

pytestmark = pytest.mark.gpu

DEV = "cuda"
B, IMG_H, IMG_W = 8, 608, 1024
FORMS = ["plain", "residual", "shifted_residual"]


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


def _reference(c, shift, residual, res_shift):
    """What torchvision's Bottleneck.forward runs on folded convs: ATen's bias add after the convolution, the identity
    (itself the downsample conv plus its bias add) added in place, relu_."""
    out = c + shift.view(1, -1, 1, 1)
    if residual is not None:
        out += residual if res_shift is None else residual + res_shift.view(1, -1, 1, 1)
    return torch.relu_(out)


def _inputs(shape, memory_format, form, special, seed=0):
    g = torch.Generator(device=DEV).manual_seed(seed)
    n, ch = shape[0], shape[1]
    c = torch.randn(shape, generator=g, device=DEV)
    r = torch.randn(shape, generator=g, device=DEV) if form != "plain" else None
    shift = torch.randn(ch, generator=g, device=DEV)
    t = torch.randn(ch, generator=g, device=DEV) if form == "shifted_residual" else None
    if special:
        for x in [c] + ([r] if r is not None else []):
            idx = torch.randint(0, x.numel(), (max(x.numel() // 5000, 8),), generator=g, device=DEV)
            k = len(idx) // 4
            x.view(-1)[idx[:k]] = float("nan")
            x.view(-1)[idx[k:2 * k]] = float("inf")
            x.view(-1)[idx[2 * k:3 * k]] = -float("inf")
            x[:, 0] = -0.0                        # channel 0: every term -0.0, so the sum entering the ReLU is -0.0
        shift[0] = -0.0
        if t is not None:
            t[0] = -0.0
        c[:, 1] = -shift[1]                       # channel 1: the shift cancels exactly (+0.0)
    cvt = lambda x: None if x is None else x.contiguous(memory_format=memory_format)
    return cvt(c), shift, cvt(r), t


def _compare_op(shape, memory_format, form, special):
    from dgod_b200 import ops
    c, shift, r, t = _inputs(shape, memory_format, form, special)
    g = torch.randn(shape, generator=torch.Generator(device=DEV).manual_seed(7), device=DEV)
    g = g.contiguous(memory_format=memory_format)

    def run(fn):
        cc = c.detach().clone().requires_grad_(True)
        rr = None if r is None else r.detach().clone().requires_grad_(True)
        y = fn(cc, shift, rr, t)
        y.backward(g)
        return y.detach(), cc.grad, None if rr is None else rr.grad

    y1, gc1, gr1 = run(ops.shift_relu)
    y0, gc0, gr0 = run(_reference)
    assert y1.is_contiguous(memory_format=memory_format)
    if special:
        assert bool(torch.isnan(y0).any()) and bool(torch.isinf(y0).any())
        assert bool(torch.signbit(c[:, 0] + shift[0]).all()), "the -0.0 case does not reach the ReLU"
    _assert_bits(y1, y0, f"{form} output")
    _assert_bits(gc1, gc0, f"{form} gradient of c")
    if r is not None:
        _assert_bits(gr1, gr0, f"{form} gradient of the residual")


@pytest.mark.parametrize("form", FORMS)
def test_shift_relu_bit_exact_at_bench_shape(form):
    _compare_op((B, 256, IMG_H // 4, IMG_W // 4), torch.channels_last, form, special=False)   # layer1's 8x256x152x256


@pytest.mark.parametrize("form", FORMS)
@pytest.mark.parametrize("shape,memory_format", [
    ((2, 64, 37, 53), torch.channels_last),
    ((3, 20, 19, 7), torch.channels_last),
    ((2, 12, 37, 53), torch.contiguous_format),
    ((3, 7, 5, 9), torch.contiguous_format),
], ids=["odd_nhwc", "odd_nhwc_c20", "odd_nchw", "odd_nchw_c7"])
@pytest.mark.parametrize("special", [False, True], ids=["finite", "nan_inf_zero"])
def test_shift_relu_bit_exact_at_odd_sizes(form, shape, memory_format, special):
    _compare_op(shape, memory_format, form, special)


def test_shift_relu_refuses_shifts_that_require_grad():
    from dgod_b200 import ops
    c = torch.randn(1, 4, 8, 8, device=DEV, requires_grad=True)
    with pytest.raises(RuntimeError, match="frozen"):
        ops.shift_relu(c, torch.zeros(4, device=DEV, requires_grad=True))
    with pytest.raises(RuntimeError, match="frozen"):
        ops.shift_relu(c, torch.zeros(4, device=DEV), torch.randn_like(c), torch.zeros(4, device=DEV, requires_grad=True))


# ------------------------------------------------------------------------------------------ whole backbone
def _backbone(trainable_layers, memory_format):
    from torchvision.models.detection.backbone_utils import resnet_fpn_backbone
    from dgod_b200 import utils
    torch.manual_seed(0)
    bb = resnet_fpn_backbone(backbone_name="resnet50", weights=None, trainable_layers=trainable_layers).to(DEV)
    bb = bb.to(memory_format=memory_format).train()
    utils.calibrate_frozen_bn(bb, torch.rand(2, 3, 64, 96, device=DEV))
    keys = list(bb.state_dict().keys())
    assert utils.fold_frozen_bn(bb) == 53
    assert list(bb.state_dict().keys()) == keys
    blocks = [m for m in bb.modules() if isinstance(m, Bottleneck)]
    assert len(blocks) == 16 and all(type(m) is utils._FusedBottleneck for m in blocks)
    stock = copy.deepcopy(bb)
    for m in stock.modules():
        if type(m) is utils._FusedBottleneck:
            m.__class__ = Bottleneck
    return bb, stock


def _grads(outs, seed=2):
    g = torch.Generator(device=DEV).manual_seed(seed)
    return [torch.randn(v.shape, generator=g, device=DEV).contiguous(
        memory_format=torch.channels_last if v.is_contiguous(memory_format=torch.channels_last) else torch.contiguous_format)
        for v in outs]


def _step(bb, x):
    out = bb(x)
    torch.autograd.backward(list(out.values()), _grads(out.values()))
    return [v.detach() for v in out.values()], {n: p.grad for n, p in bb.named_parameters() if p.grad is not None}


def _compare_backbones(trainable_layers, memory_format, shape):
    bb, stock = _backbone(trainable_layers, memory_format)
    x = torch.rand(shape, device=DEV).contiguous(memory_format=memory_format)
    o0, g0 = _step(stock, x)
    o1, g1 = _step(bb, x)
    for i, (a, b) in enumerate(zip(o1, o0)):
        _assert_bits(a, b, f"backbone output {i}")
    assert g1.keys() == g0.keys()
    assert any(n.startswith("body.layer2.") for n in g0)
    for n in g0:
        _assert_bits(g1[n], g0[n], f"gradient of {n}")
    return bb


def test_fused_backbone_equals_stock_at_bench_shape(deterministic_convs):
    """trainable_layers=3 as in the bench: layer1 runs forward-only, layers 2-4 through the op's backward."""
    from dgod_b200 import utils
    bb = _compare_backbones(3, torch.channels_last, (B, 3, IMG_H, IMG_W))
    keys = list(bb.state_dict().keys())
    utils.unfold_frozen_bn(bb)
    assert list(bb.state_dict().keys()) == keys
    assert all(type(m) is Bottleneck for m in bb.modules() if isinstance(m, Bottleneck))
    assert not any(isinstance(m, utils._FoldedConv2d) for m in bb.modules())


@pytest.mark.parametrize("trainable_layers,memory_format", [
    (3, torch.contiguous_format),
    (5, torch.channels_last),
    (5, torch.contiguous_format),
], ids=["tl3_nchw", "tl5_nhwc", "tl5_nchw"])
def test_fused_backbone_equals_stock_at_other_settings(deterministic_convs, trainable_layers, memory_format):
    _compare_backbones(trainable_layers, memory_format, (2, 3, 200, 328))
