"""utils.fold_frozen_bn's Bottleneck rebinding on the host: which blocks become _FusedBottleneck, that on CPU such a block
computes exactly what torchvision's Bottleneck computes on the same folded convolutions, and that unfold_frozen_bn
restores the stock classes."""
import copy

import pytest
import torch
from torchvision.models.resnet import Bottleneck


def _folded_backbone(trainable_layers):
    from torchvision.models.detection.backbone_utils import resnet_fpn_backbone
    from dgod_b200.utils import calibrate_frozen_bn, fold_frozen_bn
    torch.manual_seed(0)
    bb = resnet_fpn_backbone(backbone_name="resnet50", weights=None, trainable_layers=trainable_layers)
    calibrate_frozen_bn(bb, torch.rand(1, 3, 64, 96))
    keys = list(bb.state_dict().keys())
    assert fold_frozen_bn(bb) == 53
    assert list(bb.state_dict().keys()) == keys
    return bb


@pytest.mark.parametrize("trainable_layers", [3, 5])
def test_fused_bottleneck_on_cpu_equals_stock(trainable_layers):
    from dgod_b200 import utils
    bb = _folded_backbone(trainable_layers)
    blocks = [m for m in bb.modules() if isinstance(m, Bottleneck)]
    assert len(blocks) == 16 and all(type(m) is utils._FusedBottleneck for m in blocks)
    assert sum(m.downsample is not None for m in blocks) == 4
    stock = copy.deepcopy(bb)
    for m in stock.modules():
        if type(m) is utils._FusedBottleneck:
            m.__class__ = Bottleneck
    x = torch.rand(1, 3, 64, 96)

    def run(model):
        out = model(x)
        sum(v.square().mean() for v in out.values()).backward()
        return out, {n: p.grad for n, p in model.named_parameters() if p.grad is not None}

    (o1, g1), (o0, g0) = run(bb), run(stock)
    for k in o0:
        assert torch.equal(o1[k], o0[k]), k
    assert g1.keys() == g0.keys() and len(g0) > 0
    for n in g0:
        assert torch.equal(g1[n], g0[n]), n

    keys = list(bb.state_dict().keys())
    utils.unfold_frozen_bn(bb)
    assert list(bb.state_dict().keys()) == keys
    assert all(type(m) is Bottleneck for m in bb.modules() if isinstance(m, Bottleneck))


def test_bottleneck_with_unfolded_conv_is_not_fused():
    """A block is rebound only when all its convolutions (and its downsample conv) carry a folded frozen BN."""
    from torchvision.ops.misc import FrozenBatchNorm2d
    from dgod_b200 import utils
    plain = Bottleneck(64, 16, norm_layer=FrozenBatchNorm2d)               # identity block, every conv folded
    mixed = Bottleneck(64, 16, norm_layer=FrozenBatchNorm2d)
    mixed.bn2 = torch.nn.BatchNorm2d(16)                                     # conv2 + a trainable BN: not folded
    model = torch.nn.Sequential(plain, mixed)
    assert utils.fold_frozen_bn(model) == 5
    assert type(plain) is utils._FusedBottleneck and type(mixed) is Bottleneck


def test_shift_relu_rejects_cpu_tensors():
    from dgod_b200 import ops
    x = torch.rand(1, 4, 4, 4)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        ops.shift_relu(x, torch.rand(4), torch.rand(1, 4, 4, 4))
