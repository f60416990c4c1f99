"""Host-side argument validation of the bf16 backbone entry points (dgod_*_bf16): every check runs before a launch, so
no GPU is needed.  Pointers are fake device addresses that are never dereferenced."""
import ctypes

import pytest

A = 1 << 20          # a 16-byte aligned stand-in for a device pointer
U = A + 8            # 8-byte aligned only


@pytest.fixture(scope="module")
def lib():
    from dgod_b200 import _lib
    return _lib.load()


def _err(lib):
    return lib.dgod_last_error().decode()


def _calls(lib, p):
    """name -> call of the entry point on an NHWC 2x16x8x8 map (coarse / pooled / fine sizes to match), every pointer
    p(i) for argument i."""
    return {
        "dgod_fpn_merge_fwd_bf16": lambda c=16, nhwc=1: lib.dgod_fpn_merge_fwd_bf16(p(0), p(1), p(2), p(3), 2, 8, 8, 4,
                                                                                    4, c, nhwc, None),
        "dgod_fpn_merge_bwd_bf16": lambda c=16, nhwc=1: lib.dgod_fpn_merge_bwd_bf16(p(0), p(1), p(2), 2, 8, 8, 4, 4, c,
                                                                                    nhwc, None),
        "dgod_stem_pool_fwd_bf16": lambda c=16, nhwc=1: lib.dgod_stem_pool_fwd_bf16(p(0), p(1), p(2), 2, 8, 8, c, 4, 4,
                                                                                    nhwc, None),
        "dgod_shift_relu_fwd_bf16": lambda c=16, nhwc=1: lib.dgod_shift_relu_fwd_bf16(p(0), p(1), p(2), p(3), p(4), 2,
                                                                                      8, 8, c, nhwc, None),
    }


NAMES = ["dgod_fpn_merge_fwd_bf16", "dgod_fpn_merge_bwd_bf16", "dgod_stem_pool_fwd_bf16", "dgod_shift_relu_fwd_bf16"]
# the pointer argument whose absence is an error (merge backward's g_lb and shift_relu's res / res_shift are optional)
REQUIRED = {"dgod_fpn_merge_fwd_bf16": 0, "dgod_fpn_merge_bwd_bf16": 0, "dgod_stem_pool_fwd_bf16": 1,
            "dgod_shift_relu_fwd_bf16": 4}


@pytest.mark.parametrize("name", NAMES)
def test_null_pointer_is_rejected(lib, name):
    miss = REQUIRED[name]
    rc = _calls(lib, lambda i: None if i == miss else ctypes.c_void_p(A))[name]()
    assert rc == -1 and _err(lib) == f"{name}: null pointer"


@pytest.mark.parametrize("name", NAMES)
def test_channels_last_needs_eight_channels(lib, name):
    calls = _calls(lib, lambda i: ctypes.c_void_p(A))
    assert calls[name](c=12) == -1
    assert _err(lib) == f"{name}: channels_last needs channels % 8 == 0, got 12"


@pytest.mark.parametrize("name", NAMES)
@pytest.mark.parametrize("arg", [0, 1, 2])
def test_channels_last_needs_16_byte_alignment(lib, name, arg):
    calls = _calls(lib, lambda i: ctypes.c_void_p(U if i == arg else A))
    assert calls[name]() == -1
    assert _err(lib) == f"{name}: channels_last needs 16-byte aligned pointers"


@pytest.mark.parametrize("name", NAMES)
def test_empty_maps_are_a_no_op(lib, name):
    """Zero channels: nothing to do, no pointer is looked at (the same rule as the fp32 entry points)."""
    assert _calls(lib, lambda i: None)[name](c=0) == 0


def test_stem_pool_output_size_is_checked(lib):
    p = ctypes.c_void_p(A)
    assert lib.dgod_stem_pool_fwd_bf16(p, p, p, 2, 8, 8, 16, 5, 4, 1, None) == -1
    assert "is not the 3x3 / stride 2 / pad 1 pooling of 8x8" in _err(lib)


def test_shift_relu_res_shift_needs_res(lib):
    p = ctypes.c_void_p(A)
    assert lib.dgod_shift_relu_fwd_bf16(p, p, None, p, p, 2, 8, 8, 16, 1, None) == -1
    assert _err(lib) == "dgod_shift_relu_fwd_bf16: res_shift given without res"


def test_nchw_takes_any_channel_count_and_alignment(lib):
    """NCHW runs one element per thread: C % 8 and 16-byte alignment are NHWC-only rules.  A null pointer is still
    caught first, which keeps the call from launching."""
    u = ctypes.c_void_p(U)
    assert lib.dgod_fpn_merge_fwd_bf16(None, u, u, u, 2, 8, 8, 4, 4, 12, 0, None) == -1
    assert _err(lib) == "dgod_fpn_merge_fwd_bf16: null pointer"
