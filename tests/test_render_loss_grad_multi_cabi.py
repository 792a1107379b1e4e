"""CPU (-m "not gpu"): the one-pass multi-scale loss + gradient entries (lhn_render_loss_grad_multi,
lhn_render_loss_backward_multi_cond) reject bad calls with LHN_E* codes before touching the device, and the one-pass
workspace size follows the documented formula."""
import ctypes as C

import pytest

from litehandnet_b200 import _lib as L

EINVAL, EDTYPE, EALIGN, EWORKSPACE = -1, -2, -3, -4
FAKE = C.c_void_p(0x1000)          # never dereferenced: every call below is rejected on the host
SIZES = (16, 16, 32, 64)
WS_BYTES = 1 << 24


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


def _one_pass(lib, n=4, scales=None, dtype=L.F32, B=2, K=21, rp=None, joints=FAKE, vis=FAKE, ws=FAKE,
              ws_bytes=WS_BYTES, sums=None):
    scales = scales if scales is not None else _scales(n, K)
    rp = rp if rp is not None else _rp()
    return lib.lhn_render_loss_grad_multi(n, scales, dtype, B, K, C.byref(rp), joints, 3, vis, 1, 0, 1.0, ws,
                                          ws_bytes, sums, None, None, None, None, None)


def _cond(lib, n=4, scales=None, dtype=L.F32, B=2, K=21, rp=None, joints=FAKE, vis=FAKE, sums=FAKE, used=FAKE):
    scales = scales if scales is not None else _scales(n, K)
    rp = rp if rp is not None else _rp()
    return lib.lhn_render_loss_backward_multi_cond(n, scales, dtype, B, K, C.byref(rp), joints, 3, vis, 1, sums, 0,
                                                   None, used, None, None)


@pytest.mark.parametrize("n,B,K", [(1, 1, 1), (4, 2, 21), (4, 1024, 21), (8, 3, 5), (2, 7, 1)])
def test_workspace_formula(n, B, K):
    # 256 header bytes (one u64 N_pos counter per scale, the ticket) + one 16-byte row per CTA of 8 warps, a warp per
    # plane, every scale starting on a fresh CTA
    f = L.lib().lhn_render_loss_grad_multi_workspace_bytes(n, B, K)
    assert f == 256 + 16 * n * ((B * K + 7) // 8)


@pytest.mark.parametrize("n,B,K", [(0, 2, 21), (L.LOSS_MAX_TENSORS + 1, 2, 21), (-1, 2, 21), (4, 0, 21), (4, -2, 21),
                                   (4, 2, 0), (4, 2, -1)])
def test_workspace_formula_of_invalid_arguments_is_zero(n, B, K):
    assert L.lib().lhn_render_loss_grad_multi_workspace_bytes(n, B, K) == 0


@pytest.mark.parametrize("call", [_one_pass, _cond])
@pytest.mark.parametrize("n", [0, L.LOSS_MAX_TENSORS + 1, -1])
def test_rejects_scale_count(call, n):
    assert call(L.lib(), n=n, scales=_scales(max(n, 1))) == EINVAL


@pytest.mark.parametrize("field", ["joints", "vis", "ws"])
def test_one_pass_rejects_null_pointers(field):
    assert _one_pass(L.lib(), **{field: None}) == EINVAL


@pytest.mark.parametrize("field", ["joints", "vis", "sums", "used"])
def test_cond_rejects_null_pointers(field):
    assert _cond(L.lib(), **{field: None}) == EINVAL


@pytest.mark.parametrize("call", [_one_pass, _cond])
def test_rejects_null_descriptor_array_and_output(call):
    lib = L.lib()
    rp = _rp()
    if call is _one_pass:
        assert lib.lhn_render_loss_grad_multi(4, None, L.F32, 2, 21, C.byref(rp), FAKE, 3, FAKE, 1, 0, 1.0, FAKE,
                                              WS_BYTES, None, None, None, None, None, None) == EINVAL
    else:
        assert lib.lhn_render_loss_backward_multi_cond(4, None, L.F32, 2, 21, C.byref(rp), FAKE, 3, FAKE, 1, FAKE, 0,
                                                       None, FAKE, None, None) == EINVAL
    assert call(lib, scales=_scales(output=None)) == EINVAL


@pytest.mark.parametrize("call", [_one_pass, _cond])
@pytest.mark.parametrize("bad", [dict(B=0), dict(B=-3), dict(K=0), dict(K=-1)])
def test_rejects_bad_batch_and_joints(call, bad):
    assert call(L.lib(), **bad) == EINVAL


@pytest.mark.parametrize("call", [_one_pass, _cond])
def test_rejects_bad_joint_strides(call):
    lib = L.lib()
    rp = _rp()
    if call is _one_pass:
        args = lambda js, vs: (4, _scales(), L.F32, 2, 21, C.byref(rp), FAKE, js, FAKE, vs, 0, 1.0, FAKE, WS_BYTES,
                               None, None, None, None, None, None)
        fn = lib.lhn_render_loss_grad_multi
    else:
        args = lambda js, vs: (4, _scales(), L.F32, 2, 21, C.byref(rp), FAKE, js, FAKE, vs, FAKE, 0, None, FAKE, None,
                               None)
        fn = lib.lhn_render_loss_backward_multi_cond
    assert fn(*args(1, 1)) == EINVAL
    assert fn(*args(3, 0)) == EINVAL


@pytest.mark.parametrize("call", [_one_pass, _cond])
@pytest.mark.parametrize("bad", [dict(H=0), dict(W=0), dict(H=-16), dict(W=-1), dict(sigma=0.0), dict(sigma=-2.0),
                                 dict(sigma=float("nan"))])
def test_rejects_bad_scale(call, bad):
    assert call(L.lib(), scales=_scales(**bad)) == EINVAL


@pytest.mark.parametrize("call", [_one_pass, _cond])
def test_rejects_bad_render_params(call):
    lib = L.lib()
    assert call(lib, rp=_rp(unbiased=3)) == EINVAL
    assert call(lib, rp=_rp(unbiased=-1)) == EINVAL
    assert call(lib, rp=_rp(mode=L.LOSS_NONE)) == EINVAL
    assert call(lib, rp=_rp(mode=4)) == EINVAL
    assert call(lib, rp=_rp(image=0.0)) == EINVAL
    # UDP divides by W - 1 and H - 1
    assert call(lib, rp=_rp(unbiased=2), scales=_scales(W=1)) == EINVAL


@pytest.mark.parametrize("call", [_one_pass, _cond])
@pytest.mark.parametrize("dtype", [L.F64, 7, -1])
def test_rejects_bad_dtype(call, dtype):
    assert call(L.lib(), dtype=dtype) == EDTYPE


def test_one_pass_rejects_small_workspace():
    lib = L.lib()
    need = lib.lhn_render_loss_grad_multi_workspace_bytes(4, 2, 21)
    assert _one_pass(lib, ws_bytes=need - 1) == EWORKSPACE
    assert _one_pass(lib, ws_bytes=0) == EWORKSPACE
    # the size depends on the batch: enough for B = 2 is too little for B = 1024
    assert _one_pass(lib, B=1024, ws_bytes=need) == EWORKSPACE


def test_one_pass_rejects_misaligned_workspace_and_sums():
    lib = L.lib()
    assert _one_pass(lib, ws=C.c_void_p(0x1008)) == EALIGN
    assert _one_pass(lib, ws=C.c_void_p(0x1001)) == EALIGN
    assert _one_pass(lib, sums=C.c_void_p(0x2004)) == EALIGN
