"""Host-side utilities shared by bench.py's two arms and the tests (no kernels here)."""
from __future__ import annotations

import torch
from torch import nn
from torchvision.models.resnet import Bottleneck


@torch.no_grad()
def calibrate_frozen_bn(backbone: nn.Module, images: torch.Tensor) -> int:
    """Data-dependent initialisation of the FrozenBatchNorm2d statistics of a randomly initialised
    backbone: one forward pass in which every frozen BN layer first sets running_mean / running_var
    to the statistics of its own input.

    The reference trains from COCO-pretrained weights (DGFRCNN.py:81), which cannot be downloaded
    here.  A random-init ResNet-50 whose frozen BN layers are the identity (mean 0, var 1) has
    activations that grow by orders of magnitude with depth and diverges to NaN on the first
    SGD step at the reference's learning rate, after which the RPN proposes nothing and the timed
    work collapses.  Calibrated statistics give the activations the unit scale they have in a trained
    network without changing the architecture or the amount of work.  Returns the number of layers."""
    from torchvision.ops.misc import FrozenBatchNorm2d
    hooks, count = [], 0

    def pre(mod, inputs):
        x = inputs[0]
        mod.running_mean.copy_(x.mean(dim=(0, 2, 3)))
        mod.running_var.copy_(x.var(dim=(0, 2, 3), unbiased=False).clamp_min(1e-6))

    for m in backbone.modules():
        if isinstance(m, FrozenBatchNorm2d):
            hooks.append(m.register_forward_pre_hook(pre))
            count += 1
    was_training = backbone.training
    backbone.eval()
    backbone(images)
    backbone.train(was_training)
    for h in hooks:
        h.remove()
    return count


# ------------------------------------------------------------------ frozen-BN folding (host side, PyTorch/cuDNN only)
class _FoldedConv2d(nn.Conv2d):
    """conv followed by a FrozenBatchNorm2d, evaluated as ONE cuDNN convolution:
    bn(conv(x, w)) = conv(x, w * s) + (b - m * s) with s = gamma / sqrt(var + eps), per output channel.
    The parameter stays `weight` (same state_dict key, same weight decay, gradients flow through the
    product), the BN buffers stay in the BN module; only the two elementwise passes over the
    activation (x*s, +shift) and their backward disappear."""

    def _scale_shift(self):
        bn = self._folded_bn[0]
        scale = bn.weight * (bn.running_var + bn.eps).rsqrt()
        return scale, bn.bias - bn.running_mean * scale

    def forward(self, x):
        scale, shift = self._scale_shift()
        return self._conv_forward(x, self.weight * scale.view(-1, 1, 1, 1), shift)

    def _bias_free(self, x):
        """(conv(x, w * s) without the shift, shift): the same cuDNN call as forward() makes, for a native epilogue
        that adds the shift itself."""
        scale, shift = self._scale_shift()
        return self._conv_forward(x, self.weight * scale.view(-1, 1, 1, 1), None), shift


class _FoldedStem(_FoldedConv2d):
    """The folded conv1 of a frozen ResNet stem together with the ReLU and 3x3 / stride-2 max-pool behind it.  On CUDA:
    the cuDNN convolution with w * s and no bias, then ONE native pass (ops.stem_pool) that adds the shift, applies the
    ReLU and pools — it reads the conv output once and writes only the pooled map, where the stock ops make three
    full-resolution passes (bias add, ReLU, pool).  The stem's `relu` and `maxpool` modules then pass through.  On CPU
    it is the folded conv and the stock modules do the rest.  Only for a stem whose weights and input need no
    gradient (trainable_layers <= 4): the fused pass has no backward."""

    def forward(self, x):
        if not x.is_cuda:
            return super().forward(x)
        from . import ops
        return ops.stem_pool(*self._bias_free(x))


class _StemReLU(nn.ReLU):
    """A fused stem's ReLU: already applied by _FoldedStem on CUDA."""

    def forward(self, x):
        return x if x.is_cuda else super().forward(x)


class _StemMaxPool(nn.MaxPool2d):
    """A fused stem's max-pool: already applied by _FoldedStem on CUDA."""

    def forward(self, x):
        return x if x.is_cuda else super().forward(x)


class _FusedBottleneck(Bottleneck):
    """A torchvision Bottleneck whose convolutions (and downsample conv) are folded.  On CUDA: each cuDNN convolution
    without its shift, then ONE native pass per convolution (ops.shift_relu) that adds the shift, the block's identity or
    shifted downsample output, and applies the ReLU — where the stock forward makes a bias add, a ReLU and, at the
    tail, a residual add (plus the downsample's bias add) as separate full-size passes.  The convolutions are the calls
    ATen makes in the stock forward, so outputs and gradients are bit-identical.  On CPU it is the stock forward."""

    def forward(self, x):
        if not x.is_cuda:
            return super().forward(x)
        from . import ops
        out = ops.shift_relu(*self.conv1._bias_free(x))
        out = ops.shift_relu(*self.conv2._bias_free(out))
        c, shift = self.conv3._bias_free(out)
        if self.downsample is None:
            return ops.shift_relu(c, shift, x)
        return ops.shift_relu(c, shift, *self.downsample[0]._bias_free(x))


def _fuse_bottleneck(block: nn.Module) -> None:
    """Rebinds a torchvision Bottleneck whose conv1-3 (and downsample conv, if any) are folded to _FusedBottleneck."""
    pairs = [(block.conv1, block.bn1), (block.conv2, block.bn2), (block.conv3, block.bn3)]
    ds = block.downsample
    if ds is not None:
        if not (type(ds) is nn.Sequential and len(ds) == 2):
            return
        pairs.append((ds[0], ds[1]))
    if type(block.relu) is nn.ReLU and all(type(c) is _FoldedConv2d and c._folded_bn[0] is bn for c, bn in pairs):
        block.__class__ = _FusedBottleneck


def _pair(v):
    return tuple(v) if isinstance(v, (tuple, list)) else (v, v)


def _fuse_frozen_stem(parent: nn.Module) -> None:
    """Rebinds a ResNet stem (children conv1, bn1, relu, maxpool in that order, conv1 folded and frozen, the torchvision
    pooling 3x3 / 2 / pad 1) to _FoldedStem + pass-through relu and maxpool."""
    names = [k for k, _ in parent.named_children()][:4]
    if names != ["conv1", "bn1", "relu", "maxpool"]:
        return
    conv, relu, pool = parent.conv1, parent.relu, parent.maxpool
    if (type(conv) is _FoldedConv2d and not conv.weight.requires_grad and type(relu) is nn.ReLU
            and type(pool) is nn.MaxPool2d and _pair(pool.kernel_size) == (3, 3) and _pair(pool.stride) == (2, 2)
            and _pair(pool.padding) == (1, 1) and _pair(pool.dilation) == (1, 1) and not pool.ceil_mode):
        conv.__class__ = _FoldedStem
        relu.__class__ = _StemReLU
        pool.__class__ = _StemMaxPool


def fold_frozen_bn(module: nn.Module) -> int:
    """Rebinds every (Conv2d without bias, FrozenBatchNorm2d) sibling pair that torchvision's ResNet applies
    back to back (stem, Bottleneck conv1-3, downsample) so that the BN becomes the conv's epilogue.
    A frozen stem additionally runs its shift, ReLU and max-pool as one native pass on CUDA (_FoldedStem), and every
    folded Bottleneck its shifts, residual add and ReLUs as one native pass per convolution (_FusedBottleneck).
    Call after `calibrate_frozen_bn`.  State-dict keys and parameters are unchanged.  Returns the
    number of folded pairs; `unfold_frozen_bn` restores the stock modules."""
    from torchvision.ops.misc import FrozenBatchNorm2d

    class _Identity(FrozenBatchNorm2d):
        def forward(self, x):
            return x

    n = 0
    for parent in module.modules():
        prev = None
        for child in parent.children():
            if (type(child) is FrozenBatchNorm2d and type(prev) is nn.Conv2d and prev.bias is None
                    and prev.out_channels == child.weight.numel()):
                prev.__class__ = _FoldedConv2d
                prev._folded_bn = [child]          # a list: not registered as a sub-module
                child.__class__ = _Identity
                n += 1
            prev = child
        _fuse_frozen_stem(parent)
    for m in module.modules():                     # after the loop above: a block's downsample is folded after the block
        if type(m) is Bottleneck:
            _fuse_bottleneck(m)
    return n


def unfold_frozen_bn(module: nn.Module) -> None:
    from torchvision.ops.misc import FrozenBatchNorm2d
    for m in module.modules():
        if type(m) is _FusedBottleneck:
            m.__class__ = Bottleneck
        elif type(m) is _StemReLU:
            m.__class__ = nn.ReLU
        elif type(m) is _StemMaxPool:
            m.__class__ = nn.MaxPool2d
        elif isinstance(m, _FoldedConv2d):
            m._folded_bn[0].__class__ = FrozenBatchNorm2d
            del m._folded_bn
            m.__class__ = nn.Conv2d
