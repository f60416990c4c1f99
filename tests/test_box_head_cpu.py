"""Host-side checks of the box-head matrix product (dgod_linear_tc): the C entry point rejects invalid arguments before
it touches the device, the Python wrapper validates shapes and dtypes, and TwoMLPHead keeps the stock path on CPU."""
import ctypes as C

import pytest
import torch
import torch.nn.functional as F

from dgod_b200 import _lib, ops
from dgod_b200.detector import TwoMLPHead

DGOD_ERR_ARG = -1


def _call(a=1, b=1, m=128, n=256, k=64, c=1, ws=1, ws_bytes=None):
    lib = _lib.load()
    if ws_bytes is None:
        ws_bytes = lib.dgod_linear_tc_workspace_bytes(m, n, k)
    p = lambda v: None if v is None else C.c_void_p(v * 1024)
    return lib.dgod_linear_tc(p(a), 0, p(b), 0, m, n, k, None, 0, None, p(c), p(ws), ws_bytes, None)


def test_workspace_bytes():
    lib = _lib.load()
    assert lib.dgod_linear_tc_workspace_bytes(0, 32, 8) == 0
    assert lib.dgod_linear_tc_workspace_bytes(4, 32, -1) == 0
    # hi and lo of A [m, kp] and B [n, kp], kp = k rounded up to 32, plus alignment slack
    assert lib.dgod_linear_tc_workspace_bytes(4096, 1024, 12544) == 2 * (4096 + 1024) * 12544 * 4 + 1024
    assert lib.dgod_linear_tc_workspace_bytes(37, 1024, 40) == 2 * (37 + 1024) * 64 * 4 + 1024


@pytest.mark.parametrize("kw,msg", [
    (dict(a=None), "must not be NULL"),
    (dict(ws=None), "must not be NULL"),
    (dict(m=0), "must be >= 1"),
    (dict(k=0), "must be >= 1"),
    (dict(n=100), "multiple of 32"),
    (dict(ws_bytes=1024), "workspace"),
])
def test_entry_point_rejects_invalid_arguments(kw, msg):
    assert _call(**kw) == DGOD_ERR_ARG
    assert msg in _lib.load().dgod_last_error().decode()


def test_entry_point_rejects_misaligned_pointers():
    lib = _lib.load()
    ws = lib.dgod_linear_tc_workspace_bytes(128, 256, 64)
    rc = lib.dgod_linear_tc(C.c_void_p(1028), 0, C.c_void_p(2048), 0, 128, 256, 64, None, 0, None, C.c_void_p(4096),
                            C.c_void_p(8192), ws, None)
    assert rc == DGOD_ERR_ARG and "16-byte aligned" in lib.dgod_last_error().decode()


def test_wrapper_validation():
    with pytest.raises(RuntimeError, match="CUDA"):
        ops.linear_tc(torch.zeros(4, 8), torch.zeros(32, 8))
    x = torch.zeros(4, 8)
    assert not ops.box_head_mlp_supported(x, torch.zeros(32, 8), torch.zeros(32, 32))


def test_two_mlp_head_on_cpu_is_stock():
    torch.manual_seed(0)
    head = TwoMLPHead(64, 32)
    x = torch.randn(5, 4, 4, 4)
    ref = F.relu(head.fc7(F.relu(head.fc6(x.flatten(1)))))
    assert torch.equal(head(x), ref)
    assert list(head.state_dict()) == ["fc6.weight", "fc6.bias", "fc7.weight", "fc7.bias"]
