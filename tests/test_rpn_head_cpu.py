"""Host-side checks of the native RPN head (dgod_rpn_head_fwd / _bwd): the C entry points reject invalid arguments
before they touch the device, ops.rpn_head validates shapes, dtypes and layouts and refuses CPU tensors, and
detector.RPNHead keeps torchvision's forward and state-dict keys on CPU."""
import ctypes as C

import pytest
import torch
from torchvision.models.detection.rpn import RPNHead as TVRPNHead

from dgod_b200 import _lib, ops
from dgod_b200.detector import RPNHead

DGOD_ERR_ARG = -1


def _fwd(n_levels=2, channels=256, anchors=3, ptr=1024, n_img=2, h=4, w=4, null_out=False):
    lib = _lib.load()
    k = max(n_levels, 1)
    ptrs = (C.c_void_p * k)(*[ptr] * k)
    hs, ws = (C.c_int * k)(*[h] * k), (C.c_int * k)(*[w] * k)
    p = C.c_void_p(1024)
    outs = (C.c_void_p * k)(*[None if null_out else 1024] * k)
    return lib.dgod_rpn_head_fwd(ptrs, n_levels, hs, ws, n_img, channels, anchors, p, p, p, p, p, outs, outs, None)


def _bwd(ws_bytes=None, ptr=1024):
    lib = _lib.load()
    ptrs = (C.c_void_p * 1)(ptr)
    hs, ws = (C.c_int * 1)(4), (C.c_int * 1)(4)
    p = C.c_void_p(1024)
    return lib.dgod_rpn_head_bwd(ptrs, 1, hs, ws, 2, 256, 3, p, p, p, ptrs, ptrs, ptrs, p, p,
                                 0 if ws_bytes is None else ws_bytes, None)


@pytest.mark.parametrize("kw,msg", [
    (dict(channels=128), "only 256 channels and 3 anchors"),
    (dict(anchors=9), "only 256 channels and 3 anchors"),
    (dict(n_levels=0), "levels expected"),
    (dict(n_levels=9), "levels expected"),
    (dict(ptr=1028), "16-byte aligned"),
    (dict(h=-1), "negative size"),
    (dict(null_out=True), "null output"),
])
def test_fwd_entry_point_rejects_invalid_arguments(kw, msg):
    assert _fwd(**kw) == DGOD_ERR_ARG
    assert msg in _lib.load().dgod_last_error().decode()


def test_bwd_entry_point_rejects_misaligned_map_and_small_workspace():
    lib = _lib.load()
    assert _bwd(ptr=1028) == DGOD_ERR_ARG
    assert "16-byte aligned" in lib.dgod_last_error().decode()
    # an empty workspace is refused before anything is launched (without a device the size query already fails)
    assert _bwd(ws_bytes=0) == DGOD_ERR_ARG


def _args(levels=((8, 8), (4, 4)), n=2, layout=torch.channels_last, dtype=torch.float32):
    cs = [torch.zeros(n, 256, h, w, dtype=dtype).to(memory_format=layout) for h, w in levels]
    return [cs, torch.zeros(256), torch.zeros(3, 256, 1, 1), torch.zeros(3), torch.zeros(12, 256, 1, 1), torch.zeros(12)]


@pytest.mark.parametrize("mutate,msg", [
    (lambda a: a.__setitem__(0, []), "levels expected"),
    (lambda a: a.__setitem__(0, a[0] * 5), "levels expected"),
    (lambda a: a[0].__setitem__(1, torch.zeros(3, 256, 4, 4).to(memory_format=torch.channels_last)), "one batch"),
    (lambda a: a[0].__setitem__(0, torch.zeros(2, 128, 8, 8).to(memory_format=torch.channels_last)), "[N, 256, H, W]"),
    (lambda a: a[0].__setitem__(0, torch.zeros(2, 256, 8, 8, dtype=torch.float64)), "float32"),
    (lambda a: a[0].__setitem__(0, torch.zeros(2, 256, 8, 8)), "channels_last"),
    (lambda a: a.__setitem__(1, torch.zeros(255)), "bias must be"),
    (lambda a: a.__setitem__(2, torch.zeros(9, 256, 1, 1)), "w_cls must be"),
    (lambda a: a.__setitem__(4, torch.zeros(12, 256)), "w_bbox must be"),
    (lambda a: a.__setitem__(5, torch.zeros(12, dtype=torch.float64)), "b_bbox must be"),
])
def test_rpn_head_validates_arguments(mutate, msg):
    a = _args()
    mutate(a)
    with pytest.raises(ValueError, match=msg.replace("[", r"\[").replace("]", r"\]")):
        ops.rpn_head(*a)


def test_rpn_head_refuses_cpu_tensors():
    with pytest.raises(RuntimeError, match="need CUDA tensors"):
        ops.rpn_head(*_args())


def test_bias_add_refuses_cpu_tensors():
    with pytest.raises(RuntimeError, match="need CUDA tensors"):
        ops.bias_add(torch.zeros(1, 4, 2, 2), torch.zeros(4))


def test_rpn_head_module_is_torchvisions_on_cpu():
    torch.manual_seed(0)
    ref = TVRPNHead(256, 3)
    head = RPNHead(256, 3)
    assert list(head.state_dict().keys()) == list(ref.state_dict().keys())
    head.load_state_dict(ref.state_dict())
    x = [torch.randn(2, 256, 6, 5), torch.randn(2, 256, 3, 3)]
    for a, b in zip(head(x), ref(x)):
        for u, v in zip(a, b):
            assert torch.equal(u, v)
