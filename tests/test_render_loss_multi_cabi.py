"""CPU (-m "not gpu"): the multi-scale rendered-target loss entries (lhn_render_loss_multi,
lhn_render_loss_backward_multi) reject bad calls with LHN_E* codes before touching the device, and their
workspace size follows the documented formula."""
import ctypes as C

import pytest

from litehandnet_b200 import _lib as L

EINVAL, EDTYPE, EWORKSPACE = -1, -2, -4
FAKE = C.c_void_p(0x1000)          # never dereferenced: every call below is rejected on the host
SIZES = (16, 16, 32, 64)


def _rp(mode=L.LOSS_DISTANCE_BALANCE, unbiased=0, image=256.0):
    rp = L.RenderParams()
    rp.loss_mode, rp.unbiased, rp.num_stacks = mode, unbiased, 1
    rp.image_w = rp.image_h = image
    rp.pos_value = 0.5
    return rp


def _scales(n=4, K=21, **override):
    arr = (L.LossScale * max(n, 1))()
    for i in range(n):
        s = arr[i]
        hw = SIZES[i % len(SIZES)]
        s.output, s.grad, s.out_weight = 0x1000, 0x2000, None
        s.H, s.W, s.stride_c, s.stride_b = hw, hw, hw * hw, K * hw * hw
        s.sigma, s.loss_weight = 2.0, 1.0
    for k, v in override.items():
        setattr(arr[n - 1], k, v)
    return arr


def _fwd(lib, n=4, scales=None, dtype=L.F32, B=2, K=21, rp=None, joints=FAKE, vis=FAKE, ws=FAKE, ws_bytes=1 << 20):
    scales = scales if scales is not None else _scales(n, K)
    rp = rp if rp is not None else _rp()
    return lib.lhn_render_loss_multi(n, scales, dtype, B, K, C.byref(rp), joints, 3, vis, 1, 0, 1.0, ws, ws_bytes,
                                     None, None, None, None)


def _bwd(lib, n=4, scales=None, dtype=L.F32, B=2, K=21, rp=None, joints=FAKE, vis=FAKE, sums=FAKE):
    scales = scales if scales is not None else _scales(n, K)
    rp = rp if rp is not None else _rp()
    return lib.lhn_render_loss_backward_multi(n, scales, dtype, B, K, C.byref(rp), joints, 3, vis, 1, sums, 0, None,
                                              None)


def test_workspace_formula():
    lib = L.lib()
    f = lib.lhn_render_loss_multi_workspace_bytes()
    # the explicit-target multi-tensor loss's workspace: 256 header bytes + one 32-byte row per CTA of a grid of at
    # most 8 CTAs per SM, plus one per tensor
    assert f == lib.lhn_loss_mse_workspace_bytes()
    rows = (f - 256) // 32
    assert (f - 256) % 32 == 0 and rows > L.LOSS_MAX_TENSORS and (rows - L.LOSS_MAX_TENSORS) % 8 == 0


@pytest.mark.parametrize("call", [_fwd, _bwd])
@pytest.mark.parametrize("n", [0, L.LOSS_MAX_TENSORS + 1, -1])
def test_rejects_scale_count(call, n):
    assert call(L.lib(), n=n, scales=_scales(max(n, 1))) == EINVAL


@pytest.mark.parametrize("field", ["joints", "vis", "ws"])
def test_forward_rejects_null_pointers(field):
    assert _fwd(L.lib(), **{field: None}) == EINVAL


@pytest.mark.parametrize("field", ["joints", "vis", "sums"])
def test_backward_rejects_null_pointers(field):
    assert _bwd(L.lib(), **{field: None}) == EINVAL


@pytest.mark.parametrize("call", [_fwd, _bwd])
def test_rejects_null_descriptor_array_and_output(call):
    lib = L.lib()
    rp = _rp()
    if call is _fwd:
        assert lib.lhn_render_loss_multi(4, None, L.F32, 2, 21, C.byref(rp), FAKE, 3, FAKE, 1, 0, 1.0, FAKE, 1 << 20,
                                         None, None, None, None) == EINVAL
    else:
        assert lib.lhn_render_loss_backward_multi(4, None, L.F32, 2, 21, C.byref(rp), FAKE, 3, FAKE, 1, FAKE, 0, None,
                                                  None) == EINVAL
    assert call(lib, scales=_scales(output=None)) == EINVAL


@pytest.mark.parametrize("call", [_fwd, _bwd])
@pytest.mark.parametrize("bad", [dict(B=0), dict(B=-3), dict(K=0), dict(K=-1)])
def test_rejects_bad_batch_and_joints(call, bad):
    assert call(L.lib(), **bad) == EINVAL


@pytest.mark.parametrize("call", [_fwd, _bwd])
@pytest.mark.parametrize("bad", [dict(H=0), dict(W=0), dict(H=-16), dict(W=-1), dict(sigma=0.0), dict(sigma=-2.0),
                                 dict(sigma=float("nan"))])
def test_rejects_bad_scale(call, bad):
    assert call(L.lib(), scales=_scales(**bad)) == EINVAL


@pytest.mark.parametrize("call", [_fwd, _bwd])
def test_rejects_bad_render_params(call):
    lib = L.lib()
    assert call(lib, rp=_rp(unbiased=3)) == EINVAL
    assert call(lib, rp=_rp(unbiased=-1)) == EINVAL
    assert call(lib, rp=_rp(mode=L.LOSS_NONE)) == EINVAL
    assert call(lib, rp=_rp(mode=4)) == EINVAL
    assert call(lib, rp=_rp(image=0.0)) == EINVAL
    # UDP divides by W - 1 and H - 1
    assert call(lib, rp=_rp(unbiased=2), scales=_scales(W=1)) == EINVAL


@pytest.mark.parametrize("call", [_fwd, _bwd])
@pytest.mark.parametrize("dtype", [L.F64, 7, -1])
def test_rejects_bad_dtype(call, dtype):
    assert call(L.lib(), dtype=dtype) == EDTYPE


def test_forward_rejects_small_workspace():
    lib = L.lib()
    need = lib.lhn_render_loss_multi_workspace_bytes()
    assert _fwd(lib, ws_bytes=need - 1) == EWORKSPACE
    assert _fwd(lib, ws_bytes=0) == EWORKSPACE


def test_descriptor_layout_matches_header():
    # lhn_loss_scale: three pointers, two int64 strides, H, W, sigma, loss_weight
    assert C.sizeof(L.LossScale) == 3 * 8 + 2 * 8 + 4 * 4
    assert L.LossScale.stride_b.offset == 24 and L.LossScale.H.offset == 40 and L.LossScale.loss_weight.offset == 52
