"""CPU (-m "not gpu"): the one-pass loss + gradient entries (lhn_render_loss_grad,
lhn_render_loss_backward_cond) reject bad calls with LHN_E* codes before touching the device, and their
workspace size follows the documented formula."""
import ctypes as C

import pytest

from litehandnet_b200 import _lib as L

EINVAL, EDTYPE, EWORKSPACE = -1, -2, -4
FAKE = C.c_void_p(0x1000)          # never dereferenced: every call below is rejected on the host


def _rp(**kw):
    rp = L.RenderParams()
    rp.loss_mode, rp.unbiased, rp.num_stacks = kw.get("mode", L.LOSS_DISTANCE_BALANCE), kw.get("unbiased", 1), kw.get("S", 1)
    rp.image_w = rp.image_h = 256.0
    rp.pos_value = 0.5
    for i in range(min(rp.num_stacks, L.MAX_STACKS)):
        rp.sigma[i] = 2.0
    return rp


def _grad(lib, hm=FAKE, dtype=L.F32, B=2, K=21, H=64, W=64, rp=None, joints=FAKE, vis=FAKE, ws=FAKE, ws_bytes=1 << 20,
          grad=FAKE):
    rp = rp if rp is not None else _rp()
    return lib.lhn_render_loss_grad(hm, dtype, B, K, H, W, K * H * W, H * W, C.byref(rp), joints, 3, vis, 1, None,
                                    ws, ws_bytes, None, 0, 1.0, None, None, None, grad, None)


def _cond(lib, hm=FAKE, dtype=L.F32, B=2, K=21, H=64, W=64, rp=None, sums=FAKE, used=FAKE, grad=FAKE):
    rp = rp if rp is not None else _rp()
    return lib.lhn_render_loss_backward_cond(hm, dtype, B, K, H, W, K * H * W, H * W, C.byref(rp), FAKE, 3, FAKE, 1,
                                             sums, 0, 1.0, None, used, None, grad, None)


def test_workspace_formula():
    lib = L.lib()
    f = lib.lhn_render_loss_grad_workspace_bytes
    # 256 header bytes + one 32-byte row per CTA of the persistent grid (at most one per plane, at most 4096)
    assert f(1, 21, 1) == 256 + 32 * 21
    assert f(3, 21, 2) == 256 + 32 * 126
    assert f(1024, 21, 1) == 256 + 32 * 4096
    assert f(0, 21, 1) == 256
    assert f(-1, 21, 1) == 0 and f(4, 0, 1) == 0
    assert f(4, 21, 0) == f(4, 21, 1)


@pytest.mark.parametrize("field", ["hm", "joints", "vis", "ws", "grad"])
def test_loss_grad_rejects_null_pointers(field):
    assert _grad(L.lib(), **{field: None}) == EINVAL


@pytest.mark.parametrize("shape", [dict(B=-1), dict(K=0), dict(H=0), dict(W=-4)])
def test_loss_grad_rejects_bad_shapes(shape):
    assert _grad(L.lib(), **shape) == EINVAL


def test_loss_grad_rejects_bad_params_dtype_and_small_workspace():
    lib = L.lib()
    assert _grad(lib, rp=_rp(mode=L.LOSS_NONE)) == EINVAL
    assert _grad(lib, rp=_rp(unbiased=3)) == EINVAL
    assert _grad(lib, rp=_rp(S=L.MAX_STACKS + 1)) == EINVAL
    assert _grad(lib, rp=_rp(unbiased=2), W=1) == EINVAL
    assert _grad(lib, dtype=L.F64) == EDTYPE
    need = lib.lhn_render_loss_grad_workspace_bytes(2, 21, 1)
    assert _grad(lib, ws_bytes=need - 1) == EWORKSPACE
    need2 = lib.lhn_render_loss_grad_workspace_bytes(2, 21, 2)
    assert _grad(lib, rp=_rp(S=2), ws_bytes=need2 - 1) == EWORKSPACE


@pytest.mark.parametrize("field", ["hm", "sums", "used", "grad"])
def test_backward_cond_rejects_null_pointers(field):
    assert _cond(L.lib(), **{field: None}) == EINVAL


@pytest.mark.parametrize("shape", [dict(B=-1), dict(K=0), dict(H=0), dict(W=0)])
def test_backward_cond_rejects_bad_shapes(shape):
    assert _cond(L.lib(), **shape) == EINVAL


def test_backward_cond_rejects_bad_params_and_dtype():
    lib = L.lib()
    assert _cond(lib, rp=_rp(mode=4)) == EINVAL
    assert _cond(lib, dtype=7) == EDTYPE
