"""The box head's fc6 / fc7 products on the tensor cores (dgod_linear_tc, 3xTF32) against a float64 matmul, and
TwoMLPHead's native path against the stock fp32 chain.  Error metric of a product C = A B^T: |C - C64| / (|A| |B|^T),
the denominator in float64; its max and RMS are compared with cuBLAS's fp32 SGEMM (TF32 off) and single-pass TF32 on
the same inputs."""
import pytest
import torch
import torch.nn.functional as F

from dgod_b200 import ops
from dgod_b200.detector import TwoMLPHead

pytestmark = pytest.mark.gpu
DEV = "cuda"
SHAPES = {"fc6": (1024, 256 * 7 * 7), "fc7": (1024, 1024)}


def _err(c, a, b):
    a64, b64 = a.double(), b.double()
    e = (c.double() - a64 @ b64.t()).abs() / (a64.abs() @ b64.abs().t()).clamp_min(1e-300)
    return float(e.max()), float(e.square().mean().sqrt())


def _sgemm(a, b):
    prev = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        return a @ b.t()
    finally:
        torch.backends.cuda.matmul.allow_tf32 = prev


def _tf32(t):
    """fp32 -> tf32 (round to nearest, ties away), kept in fp32 storage."""
    i = t.contiguous().view(torch.int32)
    return ((i + 0x1000) & ~0x1FFF).view(torch.float32)


def _single_tf32(a, b):
    """A plain single-pass TF32 product: operands rounded to tf32, then summed exactly (float64).  Explicit, as cuBLAS
    runs single rows on fp32 kernels whatever allow_tf32 says."""
    return (_tf32(a).double() @ _tf32(b).double().t()).float()


@pytest.mark.parametrize("layer", ["fc6", "fc7"])
@pytest.mark.parametrize("m", [4096, 8000, 1, 37, 1000])
@pytest.mark.parametrize("product", ["forward", "dgrad", "wgrad"])
def test_product_accuracy(layer, m, product):
    n_out, k_in = SHAPES[layer]
    g = torch.Generator(device=DEV).manual_seed(m + n_out + k_in)
    x = torch.randn(m, k_in, device=DEV, generator=g)
    w = torch.randn(n_out, k_in, device=DEV, generator=g) * k_in ** -0.5
    dy = torch.randn(m, n_out, device=DEV, generator=g)
    if product == "forward":
        c, a, b = ops.linear_tc(x, w), x, w
    elif product == "dgrad":
        c, a, b = ops.linear_tc(dy, w, b_trans=True), dy, w.t()
    else:
        c, a, b = ops.linear_tc(dy, x, a_trans=True, b_trans=True), dy.t(), x.t()
    assert c.shape == (a.shape[0], b.shape[0])
    tc, sgemm, tf32 = _err(c, a, b), _err(_sgemm(a, b), a, b), _err(_single_tf32(a, b), a, b)
    # Each MMA's addition into the tensor-core accumulator truncates and the split drops the lo*lo term (<= 2^-22 of a
    # product): for short sums (wgrad at a few RoIs, k = m) and for a single row (torch's fp32 matmul then sums more
    # accurately than its tiled SGEMM) that exceeds twice torch's error; the bound there is 4x (RMS) and 12x (max).
    short = min(a.shape) < 37 or a.shape[1] < 1000
    factor = (12.0, 4.0) if short else (2.0, 2.0)
    assert tc[0] <= factor[0] * sgemm[0] and tc[1] <= factor[1] * sgemm[1], (tc, sgemm)
    assert tc[0] <= tf32[0] / 16 and tc[1] <= tf32[1] / 16, (tc, tf32)


def test_epilogues():
    g = torch.Generator(device=DEV).manual_seed(1)
    x = torch.randn(300, 96, device=DEV, generator=g)
    w = torch.randn(64, 96, device=DEV, generator=g)
    bias = torch.randn(64, device=DEV, generator=g)
    mask = torch.relu(torch.randn(300, 64, device=DEV, generator=g))
    ref = x.double() @ w.double().t()
    torch.testing.assert_close(ops.linear_tc(x, w, bias=bias, relu=True).double(), torch.relu(ref + bias.double()),
                               rtol=1e-5, atol=1e-5)
    torch.testing.assert_close(ops.linear_tc(x, w, mask=mask).double(), ref * (mask > 0), rtol=1e-5, atol=1e-5)


@pytest.mark.parametrize("where", ["x", "w"])
def test_non_finite_positions_match_sgemm(where):
    g = torch.Generator(device=DEV).manual_seed(2)
    x = torch.randn(200, 128, device=DEV, generator=g)
    w = torch.randn(96, 128, device=DEV, generator=g)
    t = x if where == "x" else w
    t[3, 5], t[7, 9], t[11, 13] = float("inf"), float("-inf"), float("nan")
    ref = _sgemm(x, w)
    out = ops.linear_tc(x, w)
    assert torch.equal(torch.isfinite(out), torch.isfinite(ref))
    assert torch.equal(torch.isnan(ref) & ~torch.isnan(out), torch.zeros_like(ref, dtype=torch.bool))


def _head_grads(head, x):
    x = x.detach().clone().requires_grad_(True)
    out = head(x)
    (out * torch.linspace(-1, 1, out.shape[1], device=DEV)).sum().backward()
    return [out.detach(), x.grad] + [p.grad for p in head.parameters()]


@pytest.mark.parametrize("m", [1000, 37])
def test_two_mlp_head_matches_stock(m):
    torch.manual_seed(0)
    head = TwoMLPHead(256 * 7 * 7, 1024).to(DEV)
    with torch.no_grad():   # pre-activations far from 0, so that no ReLU flips between the two paths' roundings
        head.fc6.bias.copy_(4 * torch.randn(1024, device=DEV).sign())
        head.fc7.bias.copy_(12 * torch.randn(1024, device=DEV).sign())
    x = torch.randn(m, 256, 7, 7, device=DEV)
    assert ops.box_head_mlp_supported(x.flatten(1), head.fc6.weight, head.fc7.weight)
    native = _head_grads(head, x)
    head.zero_grad(set_to_none=True)
    stock = TwoMLPHead(256 * 7 * 7, 1024).to(DEV)
    stock.load_state_dict(head.state_dict())
    orig = ops.box_head_mlp_supported
    ops.box_head_mlp_supported = lambda *a: False
    try:
        ref = _head_grads(stock, x)
    finally:
        ops.box_head_mlp_supported = orig
    for name, a, b in zip(["out", "x", "w6", "b6", "w7", "b7"], native, ref):
        assert a.shape == b.shape, name
        assert float((a - b).norm() / b.norm()) <= 1e-5, name


def test_autocast_and_unsupported_shapes_use_the_stock_chain():
    torch.manual_seed(0)
    head = TwoMLPHead(256, 1024).to(DEV)
    x = torch.randn(64, 256, device=DEV)
    with torch.autocast("cuda", dtype=torch.bfloat16):
        assert not ops.box_head_mlp_supported(x, head.fc6.weight, head.fc7.weight)
        out = head(x)
        ref = F.relu(head.fc7(F.relu(head.fc6(x))))
    assert out.dtype == torch.bfloat16 and torch.equal(out, ref)
    odd = TwoMLPHead(256, 1000).to(DEV)
    assert not ops.box_head_mlp_supported(x, odd.fc6.weight, odd.fc7.weight)
    assert torch.equal(odd(x), F.relu(odd.fc7(F.relu(odd.fc6(x)))))
