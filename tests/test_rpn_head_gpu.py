"""The native RPN head (ops.rpn_head, detector.RPNHead) against torchvision's RPNHead run by ATen / cuDNN with TF32
off, both measured against a float64 evaluation of the same head.  Error of a tensor: max |x - x64| / max |x64|.  The
native 1x1 products are fp32 fma chains, so they are held to fp32 accuracy and to stock's own distance from float64
(with a little slack: the two sum in different orders).  relu(c + bias) is bit-identical to stock's, so the ReLU mask
of the gradient must match exactly."""
import pytest
import torch
import torch.nn.functional as F
from torchvision.models.detection.rpn import RPNHead as TVRPNHead

from dgod_b200 import ops
from dgod_b200.detector import RPNHead

pytestmark = pytest.mark.gpu
DEV = "cuda"
BENCH_LEVELS = ((152, 256), (76, 128), (38, 64), (19, 32), (10, 16))   # bench.py's P2-P6 at batch 8
ODD_LEVELS = ((37, 23), (9, 13), (1, 1), (5, 3), (16, 16))


@pytest.fixture(autouse=True)
def _no_tf32():
    prev = torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
    yield
    torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = prev


def _params(seed, dtype=torch.float32):
    g = torch.Generator(device=DEV).manual_seed(seed)
    r = lambda *s, std=1.0: (torch.randn(*s, device=DEV, generator=g) * std).to(dtype)
    return [r(256, std=0.5), r(3, 256, 1, 1, std=0.06), r(3, std=0.1), r(12, 256, 1, 1, std=0.06), r(12, std=0.1)]


def _maps(levels, n, seed):
    g = torch.Generator(device=DEV).manual_seed(seed)
    return [torch.randn(n, 256, h, w, device=DEV, generator=g).to(memory_format=torch.channels_last)
            for h, w in levels]


def _stock(cs, bias, w_cls, b_cls, w_bbox, b_bbox):
    """What torchvision's RPNHead does after its 3x3 conv: ATen's bias add_, relu_, the two biased 1x1 convs."""
    obj, dl = [], []
    for c in cs:
        t = torch.relu_(c + bias.view(1, -1, 1, 1))
        obj.append(F.conv2d(t, w_cls, b_cls))
        dl.append(F.conv2d(t, w_bbox, b_bbox))
    return obj, dl


def _run(fn, cs, params, g_obj, g_dl):
    cs = [c.detach().clone().requires_grad_(True) for c in cs]
    params = [p.detach().clone().requires_grad_(True) for p in params]
    obj, dl = fn(cs, *params)
    torch.autograd.backward([*obj, *dl], [*g_obj, *g_dl])
    return [o.detach() for o in obj], [d.detach() for d in dl], [c.grad for c in cs], [p.grad for p in params]


def _err(x, ref):
    return float((x.double() - ref).abs().max() / ref.abs().max().clamp_min(1e-300))


def _case(levels, n, seed):
    cs, params = _maps(levels, n, seed), _params(seed + 1)
    g = torch.Generator(device=DEV).manual_seed(seed + 2)
    g_obj = [torch.randn(n, 3, h, w, device=DEV, generator=g) for h, w in levels]
    g_dl = [torch.randn(n, 12, h, w, device=DEV, generator=g) for h, w in levels]
    return cs, params, g_obj, g_dl


@pytest.mark.parametrize("levels,n", [(BENCH_LEVELS, 8), (ODD_LEVELS, 3), (((7, 5),), 1)])
def test_matches_stock_and_float64(levels, n):
    cs, params, g_obj, g_dl = _case(levels, n, 7)
    nat = _run(ops.rpn_head, cs, params, g_obj, g_dl)
    stk = _run(_stock, cs, params, g_obj, g_dl)
    ref = _run(_stock, [c.double() for c in cs], [p.double() for p in params], [g.double() for g in g_obj],
               [g.double() for g in g_dl])
    for kind, a, b, r in zip(("objectness", "deltas", "grad c", "grad params"), nat, stk, ref):
        for i, (x, y, z) in enumerate(zip(a, b, r)):
            e_nat, e_stk = _err(x, z), _err(y, z)
            assert x.shape == y.shape and x.dtype == torch.float32, (kind, i)
            assert e_nat < 1e-5, (kind, i, e_nat, e_stk)
            assert e_nat <= 2 * e_stk + 2e-7, (kind, i, e_nat, e_stk)
    for x, y in zip(nat[2], stk[2]):     # the ReLU mask: the same t, so zero exactly where stock's gradient is
        assert torch.equal(x == 0, y == 0)
    # the layout rpn_proposals reads: no copy there
    assert all(o.is_contiguous() for o in nat[0] + nat[1])


def test_nonfinite_inputs_give_nonfinite_results_where_stock_does():
    levels, n = ODD_LEVELS, 2
    cs, params, g_obj, g_dl = _case(levels, n, 11)
    cs[0][0, 5, 3, 4] = float("nan")
    cs[0][1, 17, 30, 2] = float("inf")
    cs[0][1, 18, 30, 2] = float("-inf")
    cs[1][0, 200, 8, 12] = float("inf")
    cs[4][1, 0, 0, 0] = float("nan")
    g_obj[1][0, :, 8, 12] = 0.0                   # a zero gradient still turns inf * 0 into a NaN weight gradient
    nat = _run(ops.rpn_head, cs, params, g_obj, g_dl)
    stk = _run(_stock, cs, params, g_obj, g_dl)
    saw_nonfinite = False
    for a, b in zip(nat, stk):
        for x, y in zip(a, b):
            assert torch.equal(torch.isfinite(x), torch.isfinite(y))
            saw_nonfinite |= not bool(torch.isfinite(y).all())
    assert saw_nonfinite


def test_backward_is_deterministic():
    cs, params, g_obj, g_dl = _case(BENCH_LEVELS, 8, 3)
    a = _run(ops.rpn_head, cs, params, g_obj, g_dl)
    b = _run(ops.rpn_head, cs, params, g_obj, g_dl)
    for u, v in zip(a, b):
        for x, y in zip(u, v):
            assert torch.equal(x, y)


def test_no_grad_forward_matches_and_records_nothing():
    cs, params, _, _ = _case(ODD_LEVELS, 2, 5)
    cs = [c.requires_grad_(True) for c in cs]
    obj, dl = ops.rpn_head(cs, *params)
    with torch.no_grad():
        obj0, dl0 = ops.rpn_head(cs, *params)
    for x, y in zip(obj + dl, obj0 + dl0):
        assert y.grad_fn is None and not y.requires_grad
        assert torch.equal(x, y)


def _heads(seed):
    torch.manual_seed(seed)
    ref = TVRPNHead(256, 3).to(DEV)
    with torch.no_grad():
        for p in ref.parameters():
            p.normal_(0, 0.05)
    head = RPNHead(256, 3).to(DEV)
    head.load_state_dict(ref.state_dict())
    return head, ref


def test_module_matches_stock_and_float64():
    head, ref = _heads(0)
    ref64 = TVRPNHead(256, 3).to(DEV).double()
    ref64.load_state_dict(ref.state_dict())
    x = _maps(ODD_LEVELS, 2, 1)
    outs = []
    ops.KernelTimer.reset()
    ops.KernelTimer.enabled = True
    for m, dt in ((head, torch.float32), (ref, torch.float32), (ref64, torch.float64)):
        xs = [f.detach().to(dt).requires_grad_(True) for f in x]
        obj, dl = m(xs)
        loss = sum((o * (k + 1)).sum() + (d.square() * 0.5).sum() for k, (o, d) in enumerate(zip(obj, dl)))
        m.zero_grad()
        loss.backward()
        outs.append([*obj, *dl, *[f.grad for f in xs], *[p.grad for p in m.parameters()]])
    ops.KernelTimer.enabled = False
    assert {"rpn_head_fwd", "rpn_head_bwd"} <= set(ops.KernelTimer.records)     # the native path ran
    ops.KernelTimer.reset()
    for y_nat, y_stk, y64 in zip(*outs):
        e_nat, e_stk = _err(y_nat.detach(), y64.detach()), _err(y_stk.detach(), y64.detach())
        assert e_nat < 1e-5 and e_nat <= 2 * e_stk + 2e-7, (e_nat, e_stk)


@pytest.mark.parametrize("case", ["autocast", "nchw"])
def test_fallback_is_torchvisions_forward(case):
    head, ref = _heads(1)
    x = _maps(ODD_LEVELS, 2, 2)
    if case == "nchw":
        x = [f.contiguous() for f in x]
    with torch.autocast("cuda", dtype=torch.bfloat16, enabled=case == "autocast"):
        a, b = head(x), ref(x)
    for u, v in zip(a, b):
        for s, t in zip(u, v):
            assert s.dtype == t.dtype and torch.equal(s, t)


def test_bias_add_is_bit_exact_with_conv_bias():
    g = torch.Generator(device=DEV).manual_seed(0)
    conv = torch.nn.Conv2d(256, 256, 3, padding=1).to(DEV).to(memory_format=torch.channels_last)
    x = torch.randn(2, 256, 19, 33, device=DEV, generator=g).to(memory_format=torch.channels_last)
    gy = torch.randn(2, 256, 19, 33, device=DEV, generator=g).to(memory_format=torch.channels_last)
    y_ref = conv(x)
    gb_ref, = torch.autograd.grad(y_ref, conv.bias, gy)
    y = ops.bias_add(conv._conv_forward(x, conv.weight, None), conv.bias)
    gb, = torch.autograd.grad(y, conv.bias, gy)
    assert y.is_contiguous(memory_format=torch.channels_last)
    assert torch.equal(y, y_ref) and torch.equal(gb, gb_ref)
